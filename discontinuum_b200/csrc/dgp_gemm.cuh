// FP64 tensor-pipe tile engine: C(128x64 tile) = init -/+ sum_k A[rows, k] * B[rows', k]^T  ("NT" form,
// both operands K-contiguous), DMMA.8x8x4 (mma.sync.m8n8k4.f64) fed from a TMA + mbarrier ring.
//
// One CTA = one 128x64 output tile, 256 threads in two warpgroups: warps 0-3 are DMMA consumers (2x2, 64x32 per warp, 128
// accumulator registers), warp 4 is the TMA producer, warps 5-7 only hand their registers over (setmaxnreg: producer
// warpgroup 40 registers per thread, consumers 216).  Two CTAs are co-resident per SM so that one CTA's tile
// prologue/epilogue overlaps the other's main loop.  Operand tiles are 64-row x 16-col (128 B) TMA boxes with the
// 128-byte swizzle; the k-index permutation kperm() makes every fragment load conflict free.
//
// The same kernel runs every O(n^3) phase of the marginal-likelihood evaluation; `mode` selects how a
// tile index maps to operand panels (decode_job) and the template flags select what the tile starts from
// (nothing / its old value / a generated covariance tile -- added in the epilogue, the accumulators always start at
// zero) and the epilogue (store / row sum of squares).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "dgp_cov.cuh"

namespace dgp {

constexpr int BM = 128, BN = 64, BK = 16;
constexpr int STAGES = 4;
constexpr int A_BYTES = BM * BK * 8;   // 16 KB
constexpr int B_BYTES = BN * BK * 8;   //  8 KB
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int GEMM_THREADS = 256;      // 2 warpgroups: 4 consumer warps | 1 producer warp + 3 warps that only give up their registers
constexpr int WS = BN + 1;             // padded row stride of the W tile in the first-touch epilogue
#ifndef DGP_COV_V
#define DGP_COV_V 8
#endif
constexpr int COV_V = DGP_COV_V;       // covariance entries a thread evaluates side by side when it generates a tile

enum { M_TRSM = 0, M_TRAIL_COL = 2, M_INV_M = 3, M_LAUUM = 4, M_PREDVAR = 5, M_GENERIC = 6, M_INV_U = 7, M_ZL = 8 };
enum { INIT_ZERO = 0, INIT_LOAD = 1, INIT_COV = 2 };
enum { EPI_STORE = 0, EPI_SUMSQ = 2 };

struct GemmArgs {
  int mode, step, nb, n;        // nb = npad / 128, n = valid points
  int ntiles, aux0, aux1, aux2; // mode dependent (M_PREDVAR: aux0 = row blocks of the chunk; M_GENERIC: see decode)
  double* C; long long ldc;     // in/out matrix of the tile
  double sign;                  // EPI_STORE: C = sign * acc  (INIT_LOAD loads sign * C)
  const double* Xw;             // feature table [npad][DGP_XS]          (INIT_COV)
  const double* noise;          // fixed noise [npad]                    (INIT_COV)
  const double* theta;          // natural parameters on device          (INIT_COV)
  const void* reserved0_;       // unused (see reserved3_)
  double* part;                 // EPI_SUMSQ: [2 nb][rows] (batched: [site][2 nbmax][rows])
  const void* reserved1_;       // unused (see reserved3_)
  double jitter;
  int latent;                   // INIT_COV: add only `jitter` on the diagonal (latent posterior covariance)
  int reserved2_;               // unused (see reserved3_)
  int reserved3_[3];            // unused: k_gemm spills more with a shorter GemmArgs (ptxas -v), so the layout stays fixed
};

// Batched launches (dgp_batch_*: several independent sites per launch).  A launch covers the tiles of up to
// DGP_BATCH_MAX sites: entry e owns tile indices [e.tile0, next.tile0) and carries the per-site values of the mode
// dependent GemmArgs fields.  Every per-site array lives in a slab indexed by the site: matrices [site][ld][ld] behind 3-D
// tensor maps (the site is the third TMA coordinate), per-point vectors [site][ld], theta [site][DGP_MAX_THETA].
// count == 0: a plain single-site launch (GemmArgs as given, 2-D tensor maps).
struct BatchEnt { int tile0, site, step, nb, n, aux0, aux1, aux2; };
struct BatchTab {
  int count, pad_;
  long long ld;                 // leading dimension of every slab matrix = rows of a per-point vector slab
  const double* jitv;           // [sites] diagonal jitter of each site
  BatchEnt e[DGP_BATCH_MAX];
};

// tile slots of an M_LAUUM launch over nb block rows (8-row bands of 8 x 16 cells, see decode_job)
__host__ __device__ inline int lauum_slots(int nb) {
  const int B = (nb + 7) / 8;
  return 64 * B * (B + 1);
}

// the fields of GemmArgs that decode_job reads (per site in a batched launch)
struct JobCtx { int mode, step, nb, aux0, aux1, aux2; };

struct Job {
  int rowA, kA, rowB, kB, nk;   // operand panel origins (elements) and number of 16-wide k steps
  int crow, ccol;               // output tile origin
  int init;                     // INIT_* actually used by this tile
  int valid;                    // 0: tile index falls outside the (ragged) problem, the CTA exits
};

__device__ __forceinline__ int isqrt_floor(int x) {
  int r = (int)sqrt((double)x);
  while (r * r > x) --r;
  while ((r + 1) * (r + 1) <= x) ++r;
  return r;
}

__device__ __forceinline__ Job decode_job(const JobCtx& g, int tile, int init_default) {
  Job j;
  j.init = init_default;
  j.valid = 1;
  const int s = g.step;
  switch (g.mode) {
    case M_TRSM: {  // L[i, s] = A[i, s] * Linv_s^T            A: work panel, B: diagonal-inverse table, or (aux1 = 1)
                    // the diagonal block of the work matrix itself, where the diagonal-block kernel left T_ss
      const int i = s + 1 + (tile >> 1), h = tile & 1;
      j.rowA = i * 128; j.kA = s * 128;
      j.rowB = s * 128 + h * 64; j.kB = g.aux1 ? s * 128 : 0;
      j.nk = h ? 8 : 4;
      j.crow = i * 128; j.ccol = (g.aux0 ? 0 : s * 128) + h * 64;  // aux0 = 1: into a [rows][128] panel buffer
    } break;
    case M_TRAIL_COL: {  // A[i, c] -= L[i, K] L[c, K]^T, K = block columns [step, step + aux1), on the block columns
                         // [o, o + w) (aux0 = o | (w << 16)): rows i >= o, tiles above the diagonal exit.  aux2 = 0: first
                         // touch of these tiles, generate the covariance
      const int o = g.aux0 & 0xffff, w2 = 2 * (g.aux0 >> 16);
      const int i = o + tile / w2, c = 2 * o + tile % w2;
      j.valid = c <= 2 * i + 1;
      j.rowA = i * 128; j.kA = s * 128;
      j.rowB = c * 64; j.kB = s * 128;
      j.nk = 8 * g.aux1;
      j.crow = i * 128; j.ccol = c * 64;
      j.init = g.aux2 ? INIT_LOAD : INIT_COV;
    } break;
    case M_INV_M:    // recursive triangular inverse, merge of block ranges [o, o+h) and [o+h, o+2h):
    case M_INV_U: {  //   M' = U11 L21'  (M_INV_M, scratch in the upper triangle of the work matrix)
                     //   U12 = -M' T22' (M_INV_U), T = L^-1 lower, U = T' upper.  aux0 = h, aux1 = pairs of this launch,
                     //   step = first pair of this launch (the pairs of a level are launched as their columns of L become final)
      const int hb = g.aux0, np_ = g.aux1;
      const int pr = tile % np_, w = tile / np_;
      const int o = (s + pr) * 2 * hb;
      // L2-aware order: the hb x 2hb tiles of a pair in cells of R x 2R tiles (R = min(8, hb)), so that the CTAs resident
      // together share R row panels and 2R column panels instead of one row panel and ~150 column panels
      const int R = hb < 8 ? hb : 8, C2 = 2 * R, per = R * C2, cpr = hb / R;
      const int cell = w / per, within = w % per;
      int jb, ic;
      if (g.mode == M_INV_M) { jb = (cell / cpr) * R + within / C2; ic = (cell % cpr) * C2 + within % C2; }
      else { jb = (cell % cpr) * R + within % R; ic = 2 * hb - 1 - ((cell / cpr) * C2 + within / R); }
      const int cb64 = 2 * (o + hb) + ic;
      j.valid = cb64 < 2 * g.nb;
      j.rowA = (o + jb) * 128;
      j.rowB = cb64 * 64;
      if (g.mode == M_INV_M) { j.kA = (o + jb) * 128; j.nk = (hb - jb) * 8; }
      else { j.kA = (o + hb) * 128; j.nk = (ic + 1) * 4; }
      j.kB = j.kA;
      j.crow = j.rowA; j.ccol = j.rowB;
    } break;
    case M_LAUUM: {  // Kinv[i, c] = sum_{k >= i} U[i, k] U[c, k]^T  (lower tiles, longest K first)
      // L2-aware order: bands of 8 block rows, inside a band cells of 8 x 16 tiles (band b has b + 1 cells, 64 b (b + 1)
      // tile slots before it); slots beyond the triangle exit.  Grid = lauum_slots(nb).
      const int ip = (isqrt_floor(4 * (tile >> 6) + 1) - 1) >> 1;
      const int rem = tile - 64 * ip * (ip + 1);
      const int i = ip * 8 + ((rem & 127) >> 4);
      const int c = (rem >> 7) * 16 + (rem & 15);
      j.valid = i < g.nb && c <= 2 * i + 1;
      j.rowA = i * 128; j.kA = i * 128;
      j.rowB = c * 64; j.kB = i * 128;
      j.nk = (g.nb - i) * 8;
      j.crow = i * 128; j.ccol = c * 64;
    } break;
    case M_PREDVAR: {  // V^T[i*, c] = sum_{k < (c+1)64} Kx[i*, k] T[c, k]   (T = L^-1), longest K first
      const int rb = g.aux0;
      const int c = 2 * g.nb - 1 - tile / rb, i = tile % rb;
      j.rowA = i * 128; j.kA = 0;
      j.rowB = c * 64; j.kB = 0;
      j.nk = (c + 1) * 4;
      j.crow = i * 128; j.ccol = c * 64;
    } break;
    case M_ZL: {  // draws[:, c] += Z[:, K] L[c, K]^T for the block columns K = [step, step + aux1) of L (one panel of a
                  // column-distributed factor), rows c of L from block `step` on; k limited to the row's own 64-block
      const int ncb = 2 * (g.nb - s);
      const int sb = tile / ncb, cbi = tile % ncb;
      j.rowA = sb * 128; j.kA = s * 128;
      j.rowB = (2 * s + cbi) * 64; j.kB = s * 128;
      j.nk = min(8 * g.aux1, (cbi + 1) * 4);
      j.crow = sb * 128; j.ccol = j.rowB;
    } break;
    default: {  // M_GENERIC: C[i, c] (+)= A[i, :] B[c, :]^T, aux0 = col blocks(64), aux1 = k steps,
                // aux2 = 1: lower-triangular B (k <= row), 2: lower tiles only (SYRK), 0: dense
      const int ncb = g.aux0;
      int i = tile / ncb, c = tile % ncb;
      if (g.aux2 == 2) {
        i = (isqrt_floor(4 * tile + 1) - 1) >> 1;
        c = tile - i * (i + 1);
      }
      j.rowA = i * 128; j.kA = 0;
      j.rowB = c * 64; j.kB = 0;
      j.nk = g.aux1;
      if (g.aux2 == 1) j.nk = min(g.aux1, (c + 1) * 4);
      j.crow = i * 128; j.ccol = c * 64;
    } break;
  }
  return j;
}

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {}
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void consumer_bar() { asm volatile("bar.sync 1, 128;" ::: "memory"); }
__device__ __forceinline__ void dmma(double (&c)[2], double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
      : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}

// dynamic shared memory map (bytes from a 1024-aligned base)
constexpr int SM_STAGES = 0;
constexpr int SM_XS = STAGES * STAGE_BYTES;                 // 192 feature rows (INIT_COV)
constexpr int SM_COVC = SM_XS + (BM + BN) * DGP_XS * 8;     // CovC
constexpr int SM_BAR = SM_COVC + ((sizeof(CovC) + 15) / 16) * 16;
constexpr int SM_TOTAL = SM_BAR + 2 * STAGES * 8 + 1024;    // + alignment slack

// MT = 8-row fragments per consumer warp along M: 8 -> the 128x64 tile; 4 -> 64x64 half tiles (blockIdx = 2 tile + half)
// for the short launches of the panel chain, whose few tiles leave most SMs idle: twice the CTAs, half the DMMA time.
template <int INIT, int EPI, int MT = 8>
__global__ void __launch_bounds__(GEMM_THREADS, 2)
k_gemm(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
       const __grid_constant__ dgp_spec spec, const GemmArgs g, const __grid_constant__ BatchTab bt) {
  static_assert(MT == 8 || (MT == 4 && INIT != INIT_COV && EPI == EPI_STORE), "half tiles: plain load/store tiles only");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full = (uint64_t*)(smem + SM_BAR);
  uint64_t* empty = full + STAGES;
  CovC* cc = (CovC*)(smem + SM_COVC);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int tile = MT == 8 ? blockIdx.x : (blockIdx.x >> 1);
  JobCtx jc{g.mode, g.step, g.nb, g.aux0, g.aux1, g.aux2};
  int site = -1;   // site >= 0: batched launch
  if (bt.count > 0) {
    int k = 0;
#pragma unroll 1
    for (int i = 1; i < bt.count; i++) if (tile >= bt.e[i].tile0) k = i;
    const BatchEnt& e = bt.e[k];
    tile -= e.tile0; site = e.site;
    jc.step = e.step; jc.nb = e.nb; jc.aux0 = e.aux0; jc.aux1 = e.aux1; jc.aux2 = e.aux2;
  }
  // slab offsets of this site (0 for a single-site launch)
  const size_t soff_m = site >= 0 ? (size_t)site * (size_t)bt.ld * (size_t)bt.ld : 0;  // matrices
  Job job = decode_job(jc, tile, INIT);
  if (!job.valid) return;
  if (MT == 4) { job.rowA += 64 * (blockIdx.x & 1); job.crow += 64 * (blockIdx.x & 1); }

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 4); }
    fence_mbar_init();
  }
  __syncthreads();
  // dependent launch (panel chain): everything above overlapped the predecessor's tail; no global access before this
  asm volatile("griddepcontrol.wait;" ::: "memory");

  // Register reallocation between the warpgroups (setmaxnreg): the kernel is compiled for 128 registers per thread
  // (2 CTAs x 256 threads = the whole register file); the producer warpgroup shrinks to 40 and the consumer warpgroup
  // grows to 216, which is what lets the accumulators (128), rolling fragments and addresses live without spills.
  if (warp >= 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 40;");
    if (warp > 4) return;
    // ------------------------------------------------------------ TMA producer
    if (lane == 0) {
      for (int it = 0; it < job.nk; it++) {
        const int s = it % STAGES;
        if (it >= STAGES) mbar_wait(&empty[s], ((it / STAGES) - 1) & 1);
        uint8_t* st = smem + SM_STAGES + s * STAGE_BYTES;
        mbar_expect_tx(&full[s], MT == 8 ? STAGE_BYTES : STAGE_BYTES - 64 * BK * 8);
        if (site < 0) {
          tma_load_2d(st, &tmA, &full[s], job.kA + it * BK, job.rowA);
          if (MT == 8) tma_load_2d(st + 64 * BK * 8, &tmA, &full[s], job.kA + it * BK, job.rowA + 64);
          tma_load_2d(st + A_BYTES, &tmB, &full[s], job.kB + it * BK, job.rowB);
        } else {
          tma_load_3d(st, &tmA, &full[s], job.kA + it * BK, job.rowA, site);
          if (MT == 8) tma_load_3d(st + 64 * BK * 8, &tmA, &full[s], job.kA + it * BK, job.rowA + 64, site);
          tma_load_3d(st + A_BYTES, &tmB, &full[s], job.kB + it * BK, job.rowB, site);
        }
      }
    }
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    return;
  }

  // -------------------------------------------------------------- DMMA consumers
  asm volatile("setmaxnreg.inc.sync.aligned.u32 216;");
  const int g8 = lane >> 2, q = lane & 3;
  const int wm = warp >> 1, wn = warp & 1;
  double acc[MT][4][2];
  constexpr int WROWS = 8 * MT;  // rows per consumer warp

  // ---- accumulators start at zero in every variant: what the tile starts from (its old value, INIT_LOAD, or the
  // covariance entries, INIT_COV) is added in the epilogue, out = start + sign * sum.  The main loop is then the same code
  // for all variants, nothing waits for the start values before the first DMMA, and an INIT_LOAD tile is prefetched to L2
  // here so that the epilogue's loads do not pay the DRAM latency.
#pragma unroll
  for (int mi = 0; mi < MT; mi++)
#pragma unroll
    for (int ni = 0; ni < 4; ni++) { acc[mi][ni][0] = 0.0; acc[mi][ni][1] = 0.0; }
  if constexpr (INIT == INIT_LOAD || INIT == INIT_COV) if (job.init == INIT_LOAD) {
    const int t = threadIdx.x;   // 0..127: 8 * MT rows x 4 lines of 128 B
    const int pr = MT == 8 ? t : (t & 63);
    const char* rowp = reinterpret_cast<const char*>(g.C + soff_m + (size_t)(job.crow + pr) * g.ldc + job.ccol);
    if (MT == 8) {
#pragma unroll
      for (int l = 0; l < 4; l++) asm volatile("prefetch.global.L2 [%0];" ::"l"(rowp + 128 * l));
    } else {
      asm volatile("prefetch.global.L2 [%0];" ::"l"(rowp + 256 * (t >> 6)));
      asm volatile("prefetch.global.L2 [%0];" ::"l"(rowp + 256 * (t >> 6) + 128));
    }
  }

  // ---- main loop.  Fragment addressing: row r of a 64-row box sits at r*128 B; logical 16-byte chunk
  // ch of that row is stored at chunk (ch ^ (r & 7)) (TMA 128B swizzle).  Lane (g8, q) takes, for the
  // s-th k4 step of a stage, k = (q>>1)*8 + 2s + (q&1), i.e. chunk (q>>1)*4 + s, word q&1: the 16
  // lanes of each half warp then hit 16 distinct 8-byte bank pairs.
  const uint32_t a_off = (uint32_t)((WROWS * wm + g8) * 128 + (q & 1) * 8);
  const uint32_t b_off = (uint32_t)(A_BYTES + (32 * wn + g8) * 128 + (q & 1) * 8);
  const uint32_t chq = (uint32_t)((q >> 1) * 4);
  uint32_t sbase = smem_u32(smem + SM_STAGES);
  asm volatile("" : "+r"(sbase));   // one register, not a re-derivation of the shared window base at every use
  // Fragment loads roll across k4 steps AND across stages, in the 24 registers one step needs: a step issues its DMMAs as
  // columns {0,1} of every row block, then columns {2,3}; fb[0..1] are reloaded for the next step after the first half,
  // fa[mi] after row block mi of the second half, fb[2..3] at the end -- each at least 14 DMMAs (> 200 cycles) before its
  // first use.  The first fragments of stage it + 1 are loaded under the last DMMAs of stage it (its full barrier is
  // polled one step earlier), so a warp's DMMA issue does not stop at a stage boundary for the barrier round trip plus
  // a shared-memory load latency, and one CTA alone keeps the tensor pipe busy while its co-resident CTA is in its tile
  // prologue / epilogue.
  double fa[MT], fb[4];
  auto lds = [&](double& dst, uint32_t addr) { asm volatile("ld.shared.f64 %0, [%1];" : "=d"(dst) : "r"(addr)); };
  // chunk of k4 step ks: ((chq + ks) ^ g8) << 4 = sw0 ^ (ks << 4)  (chq is 0 or 4, ks < 4); bits 4..6 of a row base are zero
  const uint32_t pa = a_off + (((chq) ^ (uint32_t)g8) << 4), pb = b_off + (((chq) ^ (uint32_t)g8) << 4);
  if (job.nk > 0) {
    mbar_wait(&full[0], 0);
#pragma unroll
    for (int mi = 0; mi < MT; mi++) lds(fa[mi], sbase + pa + mi * 1024);
#pragma unroll
    for (int ni = 0; ni < 4; ni++) lds(fb[ni], sbase + pb + ni * 1024);
  }
  const int nk = job.nk;
  uint32_t st = sbase;
  int s = 0;
  uint32_t ph = 0;   // parity of the full barrier of stage s in this round of the ring
  for (int it = 0; it < nk; it++) {
    // Release the PREVIOUS stage only now.  Its fragment loads are known to have returned: every DMMA of
    // that stage was issued (in order, operands scoreboarded) before the loop back-edge.  Releasing at
    // the end of the stage itself is not safe: the arrive can overtake shared-memory loads still queued
    // behind the co-resident CTA's global-load burst, and the TMA refill then lands under them.
    if (it > 0) {
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[(s + STAGES - 1) % STAGES]);
    }
    const int s2 = (s + 1 == STAGES) ? 0 : s + 1;
    const uint32_t ph2 = (s + 1 == STAGES) ? (ph ^ 1u) : ph;
    const uint32_t st2 = sbase + s2 * STAGE_BYTES;
    const bool more = it + 1 < nk;
    bool ready = true;
    // next step's fragments: this stage, or k4 step 0 of the next one (after the last stage: this stage again, unused)
    const uint32_t stn = more ? st2 : st;
#pragma unroll
    for (int ks = 0; ks < 4; ks++) {
      if (ks == 2 && more) ready = mbar_try_wait(&full[s2], ph2);
      if (ks == 3 && more && !ready) mbar_wait(&full[s2], ph2);
      const uint32_t na = (((ks < 3) ? st : stn) + pa) ^ (uint32_t)(((ks + 1) & 3) << 4);
      const uint32_t nb_ = (((ks < 3) ? st : stn) + pb) ^ (uint32_t)(((ks + 1) & 3) << 4);
#pragma unroll
      for (int mi = 0; mi < MT; mi++) {
        dmma(acc[mi][0], fa[mi], fb[0]);
        dmma(acc[mi][1], fa[mi], fb[1]);
      }
      lds(fb[0], nb_);
      lds(fb[1], nb_ + 1024);
#pragma unroll
      for (int mi = 0; mi < MT; mi++) {
        dmma(acc[mi][2], fa[mi], fb[2]);
        dmma(acc[mi][3], fa[mi], fb[3]);
        lds(fa[mi], na + mi * 1024);
      }
      lds(fb[2], nb_ + 2 * 1024);
      lds(fb[3], nb_ + 3 * 1024);
    }
    st = st2; s = s2; ph = ph2;
  }

  // ---- epilogue
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if constexpr (EPI == EPI_STORE) {
    // The output address is recomputed from the block index (through an opaque copy, so that the compiler cannot keep
    // the values of the prologue alive instead): the main loop needs every register for accumulators and fragments.
    int bx = blockIdx.x, tx = threadIdx.x;
    asm volatile("" : "+r"(bx), "+r"(tx));
    int tile_e = MT == 8 ? bx : (bx >> 1);
    JobCtx je{g.mode, g.step, g.nb, g.aux0, g.aux1, g.aux2};
    size_t soff_e = 0;
    int site_e = -1, npts_e = g.n;
    if (bt.count > 0) {
      int k = 0;
#pragma unroll 1
      for (int i = 1; i < bt.count; i++) if (tile_e >= bt.e[i].tile0) k = i;
      const BatchEnt& e = bt.e[k];
      tile_e -= e.tile0; site_e = e.site; npts_e = e.n;
      je.step = e.step; je.nb = e.nb; je.aux0 = e.aux0; je.aux1 = e.aux1; je.aux2 = e.aux2;
      soff_e = (size_t)e.site * (size_t)bt.ld * (size_t)bt.ld;
    }
    const Job jo = decode_job(je, tile_e, INIT);
    const int crow_e = jo.crow + (MT == 4 ? 64 * (bx & 1) : 0);
    const int lane_e = tx & 31, warp_e = tx >> 5;
    const int g8e = lane_e >> 2, qe = lane_e & 3, wme = warp_e >> 1, wne = warp_e & 1;
    bool gen = false;
    if constexpr (INIT == INIT_COV) gen = jo.init == INIT_COV;
    if (gen) {
      if constexpr (INIT == INIT_COV) {
        // First touch of the tile: out = K + sign * sum.  The accumulators are parked in the (now idle) operand ring as a
        // padded tile, thread t then generates row t of the covariance tile, 8 columns at a time (cov_vals<8>, with every
        // register free for it), combines it with the parked sums in place, and the tile leaves in 512-byte rows.
        const double jit_e = site_e >= 0 ? bt.jitv[site_e] : g.jitter;
        const size_t soff_ve = site_e >= 0 ? (size_t)site_e * (size_t)bt.ld : 0;
        double* xaT = (double*)(smem + SM_XS);          // [DGP_XS][128] row-point features, column-major
        double* xb = xaT + DGP_XS * BM;                 // [64][DGP_XS]  column-point features
        double* W = (double*)(smem + SM_STAGES);        // [128][WS]
        const double* Xw_s = g.Xw + soff_ve * DGP_XS;
        const double* noise_s = g.noise + soff_ve;
        consumer_bar();                                  // every warp is done reading the ring
#pragma unroll
        for (int mi = 0; mi < 8; mi++)
#pragma unroll
          for (int ni = 0; ni < 4; ni++) {
            double* wp = W + (64 * wme + 8 * mi + g8e) * WS + 32 * wne + 8 * ni + 2 * qe;
            wp[0] = g.sign * acc[mi < MT ? mi : 0][ni][0];
            wp[1] = g.sign * acc[mi < MT ? mi : 0][ni][1];
          }
        cov_compile(cc, spec, g.theta + (site_e >= 0 ? site_e * DGP_MAX_THETA : 0), jit_e, tx, 128);
        for (int e = tx; e < BM * DGP_XS; e += 128) xaT[(e % DGP_XS) * BM + e / DGP_XS] = Xw_s[(size_t)jo.crow * DGP_XS + e];
        for (int e = tx; e < BN * DGP_XS; e += 128) xb[e] = Xw_s[(size_t)jo.ccol * DGP_XS + e];
        consumer_bar();
        {
          const int gr = jo.crow + tx;
          const double dn = (gr < npts_e) ? (g.latent ? jit_e : noise_s[gr] + cc->extra_noise) : 0.0;
#pragma unroll 1
          for (int c0 = 0; c0 < BN; c0 += COV_V) {
            double val[COV_V];
            cov_vals<COV_V>(cc, xaT, BM, tx, xb + c0 * DGP_XS, val);
#pragma unroll
            for (int v = 0; v < COV_V; v++) {
              const int gc = jo.ccol + c0 + v;
              double x = val[v];
              if (gr < npts_e && gc < npts_e) { if (gr == gc) x += dn; }
              else x = (gr == gc) ? 1.0 : 0.0;
              W[tx * WS + c0 + v] += x;
            }
          }
        }
        consumer_bar();
        {  // warp w stores rows 32 w .. 32 w + 31, one 512-byte row per instruction
          double* cbase = g.C + soff_e + (size_t)jo.crow * g.ldc + jo.ccol + 2 * lane_e;
#pragma unroll 4
          for (int r = 32 * warp_e; r < 32 * warp_e + 32; r++) {
            double2 o;
            o.x = W[r * WS + 2 * lane_e];
            o.y = W[r * WS + 2 * lane_e + 1];
            *reinterpret_cast<double2*>(cbase + (size_t)r * g.ldc) = o;
          }
        }
      }
    } else {
      const bool ldc = (INIT == INIT_LOAD || INIT == INIT_COV) && jo.init == INIT_LOAD;
#pragma unroll
      for (int mi = 0; mi < MT; mi++) {
        double* crow = g.C + soff_e + (size_t)(crow_e + WROWS * wme + 8 * mi + g8e) * g.ldc + jo.ccol + 32 * wne + 2 * qe;
        double2 old[4];
        if (ldc) {
#pragma unroll
          for (int ni = 0; ni < 4; ni++) old[ni] = *reinterpret_cast<const double2*>(crow + 8 * ni);
        }
#pragma unroll
        for (int ni = 0; ni < 4; ni++) {
          double2 v;
          if (ldc) {
            v.x = fma(g.sign, acc[mi][ni][0], old[ni].x);
            v.y = fma(g.sign, acc[mi][ni][1], old[ni].y);
          } else {
            v.x = g.sign * acc[mi][ni][0];
            v.y = g.sign * acc[mi][ni][1];
          }
          *reinterpret_cast<double2*>(crow + 8 * ni) = v;
        }
      }
    }
  } else if constexpr (EPI == EPI_SUMSQ) {
    // row sums of squares of the tile -> part[cblock][row]; a batched launch writes site s's partials at part[s][2 nbmax]
    // [rows] (nbmax = bt.ld / 128), the site found again from the block index like the store epilogue does
    size_t cb = job.ccol / 64;
    if (bt.count > 0) {
      int bx = blockIdx.x;
      asm volatile("" : "+r"(bx));
      int k = 0;
#pragma unroll 1
      for (int i = 1; i < bt.count; i++) if (bx >= bt.e[i].tile0) k = i;
      cb += (size_t)bt.e[k].site * (size_t)(bt.ld / 64);
    }
    double rs[8];
#pragma unroll
    for (int mi = 0; mi < 8; mi++) {
      double s = 0.0;
#pragma unroll
      for (int ni = 0; ni < 4; ni++) s += acc[mi][ni][0] * acc[mi][ni][0] + acc[mi][ni][1] * acc[mi][ni][1];
      s += __shfl_xor_sync(0xffffffffu, s, 1);
      s += __shfl_xor_sync(0xffffffffu, s, 2);
      rs[mi] = s;
    }
    // two warps (wn = 0, 1) share a row: combine through the (now idle) stage ring
    double* red = (double*)(smem + SM_STAGES);
    consumer_bar();
    if (q == 0 && wn == 1) {
#pragma unroll
      for (int mi = 0; mi < 8; mi++) red[64 * wm + 8 * mi + g8] = rs[mi];
    }
    consumer_bar();
    if (q == 0 && wn == 0) {
#pragma unroll
      for (int mi = 0; mi < 8; mi++) {
        const int lr = 64 * wm + 8 * mi + g8;
        g.part[cb * g.aux1 + job.crow + lr] = rs[mi] + red[lr];
      }
    }
  }
}

}  // namespace dgp
