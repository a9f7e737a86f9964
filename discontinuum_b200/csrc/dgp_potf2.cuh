// Diagonal block of the blocked Cholesky, second generation: L_ss, T_ss = L_ss^-1 and U_ss = L_ss^-T of one 128x128
// block in one CTA that is small enough (95 KB of shared memory, <= 144 registers) to share an SM with one CTA of the
// DMMA tile engine.  Written around one measured fact: a dependent FP64 operation costs ~40 cycles on B200 (DMMA ~64),
// so the kernel is a latency chain, not a throughput problem, and everything that can leave the chain does.
//
// The block is held as the 10 lower 32x32 sub-blocks B[i][j] (i >= j), row stride 36 doubles: with that stride the
// A (row g8, k = q), B^T (row g8, k = q), B (k = q, column g8) and C fragments of DMMA.8x8x4 are all conflict free.
// The factorisation runs in L D L^T form (unit-lower Lu, pivots d, w = 1/d): no square root, no logarithm and no
// division is on the chain; L = Lu sqrt(D), T = D^-1/2 Lu^-1 are scaled on the way out.  Step k = 0..3:
//   A  warp 0 factors the diagonal sub-block, lane = row, rows in registers.  Every lane evaluates the next pivot
//      redundantly from the two exchanged columns, d' = a' - l^2 w, so that the recurrence is one FMA plus a reciprocal
//      (MUFU.RCP64H and two Newton steps arranged as three dependent operations); the shared-memory exchange of the
//      column and the updates of the row run beside it.  Warps 1-7 meanwhile finish row k-1 of the inverse,
//      Tu[k-1][j] = -Tu_kk sum_l Lu[k-1][l] Tu[l][j] (in place over the dead row of L), and stream finished rows out.
//   B  unit-lower forward substitution by columns, one row per lane: warp 0 on the identity (-> Tu_kk), warps 1.. on
//      the rows below (-> u[i][k] = Lu[i][k] D_k); warp 7 takes 1/sqrt(d), log d and writes L_kk.
//   C  results back into shared memory (Tu_kk over Lu_kk).
//   D  B[i][j] -= (u[i][k] W_k) u[j][k]^T by DMMA in 16x32 jobs (8 independent accumulator chains per warp).
#pragma once
#include <cuda_runtime.h>
#include "dgp_gemm.cuh"

namespace dgp {

constexpr int P2_THREADS = 256;
constexpr int P2_LD = 36;
constexpr int P2_BLK = 32 * P2_LD;
constexpr int P2_OFF_EX = 10 * P2_BLK;          // [2][2][32] exchange buffers of the diagonal factorisation
constexpr int P2_OFF_W = P2_OFF_EX + 128;       // [128] w = 1 / d
constexpr int P2_OFF_D = P2_OFF_W + 128;        // [128] pivots d
constexpr int P2_OFF_RS = P2_OFF_D + 128;       // [128] 1 / sqrt(d) = 1 / L_ii
constexpr int P2_OFF_SQ = P2_OFF_RS + 128;      // [128] sqrt(d)
constexpr int P2_OFF_PROG = P2_OFF_SQ + 128;   // int: pivots published so far
#ifdef P2_TIMING
constexpr int P2_SMEM = (P2_OFF_PROG + 2 + 128) * 8;
#else
constexpr int P2_SMEM = (P2_OFF_PROG + 2) * 8;  // 97 296 B
#endif

#ifdef P2_TIMING
__device__ long long p2_ts[64];
#define P2_STAMP(i) do { if (threadIdx.x == 0) reinterpret_cast<long long*>(p2_smem + P2_OFF_PROG + 2)[i] = clock64(); } while (0)
#define P2_WSTAMP(b, k) do { if ((threadIdx.x & 31) == 0) reinterpret_cast<long long*>(p2_smem + P2_OFF_PROG + 2)[64 + (b) * 32 + (k) * 8 + (threadIdx.x >> 5)] = clock64(); } while (0)
__device__ long long p2_wts[64];
#else
#define P2_WSTAMP(b, k) do { } while (0)
#define P2_STAMP(i) do { } while (0)
#endif

// 1 / d: MUFU.RCP64H seed (20 bits) and two Newton steps, the second one on e^2 so that only three operations depend
// on each other (e ; x1 and e^2 ; x2).  d > 0 normal; the result is within an ulp or two of 1 / d.
__device__ __forceinline__ double rcp_newton(double d) {
  double x;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(d));
  const double e = fma(-d, x, 1.0);
  const double x1 = fma(x, e, x);
  const double e2 = e * e;
  return fma(x1, e2, x1);
}

__device__ __forceinline__ double* p2_blk(double* sm, int i, int j) { return sm + ((i * (i + 1)) / 2 + j) * P2_BLK; }

// acc (16 x 32: rows g8 and 8 + g8, columns 8 ni + 2q, +1) += sum over nks k4-steps of A[row][4 ks + q] * Bop
//   NN = false: Bop = Bm[8 ni + g8][4 ks + q]   (A Bm^T);   NN = true: Bop = Bm[4 ks + q][8 ni + g8]   (A Bm)
//   SCALE: A[row][k] is multiplied by wk[k] on the way in;  NEG: the product is subtracted
//   LOWB: Bm (NN) is lower triangular, B[k][c] = 0 for k < c: column group ni only sees k >= 8 ni
//   nmax: column groups ni >= nmax are not needed (upper half of a diagonal tile)
template <bool NN, bool NEG, bool SCALE, int NKS, bool LOWB = false>
__device__ __forceinline__ void p2_strip2(double (&acc)[2][4][2], const double* A, const double* Bm,
                                          const double* wk, int g8, int q, int nmax = 4) {
  const double* ap = A + g8 * P2_LD + q;
  const double* bp = NN ? Bm + q * P2_LD + g8 : Bm + g8 * P2_LD + q;
#pragma unroll
  for (int ks = 0; ks < NKS; ks++) {
    double a0 = ap[4 * ks], a1 = ap[8 * P2_LD + 4 * ks];
    if (SCALE) { const double w = wk[4 * ks + q]; a0 *= w; a1 *= w; }
    if (NEG) { a0 = -a0; a1 = -a1; }
#pragma unroll
    for (int ni = 0; ni < 4; ni++) {
      if (LOWB && ks < 2 * ni) continue;
      if (ni < nmax) {
        const double b = NN ? bp[4 * ks * P2_LD + 8 * ni] : bp[8 * ni * P2_LD + 4 * ks];
        dmma(acc[0][ni], a0, b);
        dmma(acc[1][ni], a1, b);
      }
    }
  }
}

__device__ __forceinline__ void p2_zero(double (&acc)[2][4][2]) {
#pragma unroll
  for (int h = 0; h < 2; h++)
#pragma unroll
    for (int ni = 0; ni < 4; ni++) { acc[h][ni][0] = 0.0; acc[h][ni][1] = 0.0; }
}

__device__ __forceinline__ void p2_store2(double* C, const double (&acc)[2][4][2], int g8, int q) {
#pragma unroll
  for (int h = 0; h < 2; h++)
#pragma unroll
    for (int ni = 0; ni < 4; ni++) {
      double2 v; v.x = acc[h][ni][0]; v.y = acc[h][ni][1];
      *reinterpret_cast<double2*>(C + (8 * h + g8) * P2_LD + 8 * ni + 2 * q) = v;
    }
}

// The unit inverse Tu = Lu^-1 is built right-looking, in place over the dead blocks of u, one row per step:
//   M[i][j] = sum_{l = j}^{i-1} Lu[i][l] Tu[l][j]   accumulates as the rows l of Tu become final (Lu[i][l] = u[i][l] W_l),
//   Tu[R][j] = -Tu_RR M[R][j]                        closes row R once Tu_RR is known (Tu_RR unit lower: k <= row).
// Jobs are 16 x 32 halves (mh) of a 32x32 block.
__device__ __forceinline__ void p2_load2(double (&acc)[2][4][2], const double* C, int g8, int q) {
#pragma unroll
  for (int h = 0; h < 2; h++)
#pragma unroll
    for (int ni = 0; ni < 4; ni++) {
      const double2 v = *reinterpret_cast<const double2*>(C + (8 * h + g8) * P2_LD + 8 * ni + 2 * q);
      acc[h][ni][0] = v.x; acc[h][ni][1] = v.y;
    }
}
// job (j, mh), j < R: acc = -Tu_RR[rows of mh] M[R][j]
__device__ __forceinline__ void p2_inv_t(double (&acc)[2][4][2], double* sm, int R, int job, int g8, int q) {
  p2_zero(acc);
  if (job < 2 * R) {
    const int j = job >> 1, mh = job & 1;
    if (mh == 0) p2_strip2<true, true, false, 4>(acc, p2_blk(sm, R, R), p2_blk(sm, R, j), nullptr, g8, q);
    else p2_strip2<true, true, false, 8>(acc, p2_blk(sm, R, R) + 16 * P2_LD, p2_blk(sm, R, j), nullptr, g8, q);
  }
}
__device__ __forceinline__ void p2_inv_t_store(const double (&acc)[2][4][2], double* sm, int R, int job, int g8, int q) {
  if (job < 2 * R) p2_store2(p2_blk(sm, R, job >> 1) + 16 * (job & 1) * P2_LD, acc, g8, q);
}
// M[i][j] += Lu[i][R] Tu[R][j] for i > R, j < R  (each job reads and writes its own 16 rows of block (i, j))
__device__ __forceinline__ void p2_inv_update(double* sm, int R, int hx, int nh, int g8, int q) {
  const int njobs = (3 - R) * R * 2;
  for (int job = hx; job < njobs; job += nh) {
    const int mh = job & 1, t = job >> 1, j = t % R, i = R + 1 + t / R;
    double acc[2][4][2];
    double* C = p2_blk(sm, i, j) + 16 * mh * P2_LD;
    p2_load2(acc, C, g8, q);
    p2_strip2<true, false, true, 8>(acc, p2_blk(sm, i, R) + 16 * mh * P2_LD, p2_blk(sm, R, j), sm + P2_OFF_W + 32 * R, g8, q);
    p2_store2(C, acc, g8, q);
  }
}
// M[i][R] = Lu[i][R] Tu_RR for i > R, in place over u[i][R] (a job reads only its own 16 rows of it)
__device__ __forceinline__ void p2_inv_first(double* sm, int R, int hx, int nh, int g8, int q) {
  const int njobs = (3 - R) * 2;
  for (int job = hx; job < njobs; job += nh) {
    const int mh = job & 1, i = R + 1 + (job >> 1);
    double acc[2][4][2];
    double* C = p2_blk(sm, i, R) + 16 * mh * P2_LD;
    p2_zero(acc);
    p2_strip2<true, false, true, 8, true>(acc, C, p2_blk(sm, R, R), sm + P2_OFF_W + 32 * R, g8, q);
    __syncwarp();
    p2_store2(C, acc, g8, q);
  }
}

// Row R of T = D^-1/2 Tu -> DIblk, Tblk (rows 32 R .., row-major) and U = T^T (columns 32 R ..), by nt threads.
__device__ __forceinline__ void p2_out_row(double* sm, int R, int t, int nt, double* DIblk, double* Tblk, double* Ublk, long long ld) {
  const double* rs = sm + P2_OFF_RS + 32 * R;
  for (int e = t; e < (R + 1) * 512; e += nt) {
    const int j = e >> 9, r = (e >> 4) & 31, c2 = (e & 15) * 2;
    double2 v = *reinterpret_cast<const double2*>(p2_blk(sm, R, j) + r * P2_LD + c2);
    const double s = rs[r];
    v.x *= s; v.y *= s;
    if (DIblk != nullptr) *reinterpret_cast<double2*>(DIblk + (32 * R + r) * 128 + 32 * j + c2) = v;
    if (Tblk != nullptr) *reinterpret_cast<double2*>(Tblk + (size_t)(32 * R + r) * ld + 32 * j + c2) = v;
  }
  if (Ublk != nullptr)
    for (int e = t; e < (R + 1) * 512; e += nt) {
      const int j = e >> 9, c = (e >> 4) & 31, r2 = (e & 15) * 2;
      const double* tb = p2_blk(sm, R, j) + r2 * P2_LD + c;
      double2 v; v.x = tb[0] * rs[r2]; v.y = tb[P2_LD] * rs[r2 + 1];
      *reinterpret_cast<double2*>(Ublk + (size_t)(32 * j + c) * ld + 32 * R + r2) = v;
    }
}

// Zero sub-blocks: above the diagonal in L^-1 (both copies, when present) and, with zero_lu, in L, below it in U.
__device__ __forceinline__ void p2_out_zeros(int t, int nt, double* Lblk, double* DIblk, double* Tblk, double* Ublk, long long ld,
                                             int zero_lu) {
  double2 z; z.x = 0.0; z.y = 0.0;
  for (int e = t; e < 6 * 512; e += nt) {
    const int b = e >> 9, r = (e >> 4) & 31, c2 = (e & 15) * 2;
    const int j = (b >= 3) ? 3 : (b >= 1) ? 2 : 1, i = b - (j * (j - 1)) / 2;  // i < j
    if (zero_lu) *reinterpret_cast<double2*>(Lblk + (size_t)(32 * i + r) * ld + 32 * j + c2) = z;
    if (DIblk != nullptr) *reinterpret_cast<double2*>(DIblk + (32 * i + r) * 128 + 32 * j + c2) = z;
    if (Tblk != nullptr) *reinterpret_cast<double2*>(Tblk + (size_t)(32 * i + r) * ld + 32 * j + c2) = z;
    if (zero_lu && Ublk != nullptr) *reinterpret_cast<double2*>(Ublk + (size_t)(32 * j + r) * ld + 32 * i + c2) = z;
  }
}

__device__ __forceinline__ int p2_ld_prog(const int* prog) {
  int v;
  asm volatile("ld.volatile.shared.s32 %0, [%1];" : "=r"(v) : "r"(smem_u32(prog)) : "memory");
  return v;
}
__device__ __forceinline__ void p2_st_prog(int* prog, int v) {
  asm volatile("st.volatile.shared.s32 [%0], %1;" ::"r"(smem_u32(prog)), "r"(v) : "memory");
}

#define P2_BARH(nh) asm volatile("bar.sync 1, %0;" ::"r"((nh) * 32) : "memory")

// Factors the 128x128 diagonal block A_ss = L L^T (lower triangle of Ablk, leading dimension ld) and produces its inverses
// in the same CTA: Lblk <- L (zeros above the diagonal), Ublk <- L^-T (upper, optional), DIblk <- L^-1 ([128][128]
// contiguous, optional), Tblk <- L^-1 as a full block with zeros above the diagonal (optional, leading dimension ld: the
// diagonal block of T for the recursive inverse; may alias Ablk: the block is staged in shared memory before anything is
// written), scal[SC_LOGDET] += sum log L_ii, first bad pivot -> scal[SC_INFO].
// zero_lu = 0: the 32x32 sub-blocks above the diagonal of Lblk / below the diagonal of Ublk are known to be zero already.
//
// Warp roles in phase A of step k: warp 0 pivots; warps 1..3-k follow with the rows of the sub-blocks below and warp 5
// with the rows of the identity (one pivot behind, through the published columns of Lu); warp 4 waits for the last pivot
// and takes the scalings; the helpers (warps 6, 7; at k = 3 warps 1, 2, 3, 6, 7) finish the previous row of the inverse.
//
// Batched launch (pb.count > 0, one CTA per site): Ablk / Lblk / Ublk / Tblk are then the bases of the [site][ld][ld]
// slabs and scal the base of [site][SC_SIZE]; CTA b factors the diagonal block pb.step[b] of site pb.site[b].
struct P2Batch {
  int count, pad_;
  long long slab;               // elements between the matrices of consecutive sites
  short site[DGP_BATCH_MAX], step[DGP_BATCH_MAX];
};

__global__ void __maxnreg__(144)
k_potf2_v2(const double* Ablk, double* Lblk, double* Ublk, long long ld, double* DIblk, double* __restrict__ scal, int base,
           double* Tblk, int zero_lu, const __grid_constant__ P2Batch pb) {
  extern __shared__ __align__(16) double p2_smem[];
  if (pb.count > 0) {
    const int st = pb.site[blockIdx.x], s = pb.step[blockIdx.x];
    const size_t off = (size_t)st * (size_t)pb.slab + (size_t)s * 128 * (size_t)ld + (size_t)s * 128;
    Ablk += off; Lblk += off;
    if (Ublk != nullptr) Ublk += off;
    if (Tblk != nullptr) Tblk += off;
    scal += (size_t)st * SC_SIZE;
    base = s * 128;
  }
  double* sm = p2_smem;
  double* ex = sm + P2_OFF_EX;
  double* wv = sm + P2_OFF_W;
  double* dvs = sm + P2_OFF_D;
  double* rsv = sm + P2_OFF_RS;
  double* sqv = sm + P2_OFF_SQ;
  int* prog = reinterpret_cast<int*>(sm + P2_OFF_PROG);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g8 = lane >> 2, q = lane & 3;
  P2_STAMP(0);
  asm volatile("griddepcontrol.wait;" ::: "memory");

  // ---- stage the lower sub-blocks (upper triangles of the diagonal sub-blocks zeroed): 20 independent 16-byte loads
  {
    double2 v[20];
#pragma unroll
    for (int u = 0; u < 20; u++) {
      const int e = u * P2_THREADS + tid;          // 0 .. 5119 = 10 blocks x 32 rows x 16 pairs
      const int b = e >> 9, r = (e >> 4) & 31, c2 = (e & 15) * 2;
      const int i = (b >= 6) ? 3 : (b >= 3) ? 2 : (b >= 1) ? 1 : 0, j = b - (i * (i + 1)) / 2;
      v[u] = *reinterpret_cast<const double2*>(Ablk + (size_t)(32 * i + r) * ld + 32 * j + c2);
    }
    if (tid == 0) p2_st_prog(prog, 0);
#pragma unroll
    for (int u = 0; u < 20; u++) {
      const int e = u * P2_THREADS + tid;
      const int b = e >> 9, r = (e >> 4) & 31, c2 = (e & 15) * 2;
      const int i = (b >= 6) ? 3 : (b >= 3) ? 2 : (b >= 1) ? 1 : 0, j = b - (i * (i + 1)) / 2;
      double2 w = v[u];
      if (i == j) { if (c2 > r) w.x = 0.0; if (c2 + 1 > r) w.y = 0.0; }
      *reinterpret_cast<double2*>(sm + b * P2_BLK + r * P2_LD + c2) = w;
    }
  }
  __syncthreads();
  P2_STAMP(1);

  int bad = 0;

#pragma unroll 1
  for (int k = 0; k < 4; k++) {
    double* Bkk = p2_blk(sm, k, k);
    const bool row_follower = warp >= 1 && warp <= 3 - k;
    const bool follower = row_follower || warp == 5;
    double x[32];
    // ---------------------------------------------------------------- phase A
    if (warp == 0) {
      double a[32];
#pragma unroll
      for (int p = 0; p < 16; p++) {
        const double2 v = *reinterpret_cast<const double2*>(Bkk + lane * P2_LD + 2 * p);
        a[2 * p] = v.x; a[2 * p + 1] = v.y;
      }
      ex[lane] = a[0];
      ex[32 + lane] = a[1];
      __syncwarp();
      double d = ex[0];
#pragma unroll
      for (int c = 0; c < 32; c++) {
        const double* cA = ex + (c & 1) * 64;
        const double* cB = cA + 32;
        double lc1sq = 0.0, cb1 = 0.0;
        if (c + 1 < 32) { const double lc1 = cA[c + 1]; lc1sq = lc1 * lc1; cb1 = cB[c + 1]; }
        if (!(d > 0.0) && bad == 0) bad = 32 * k + c + 1;
        const double w = rcp_newton(d);
        const double dnext = fma(-lc1sq, w, cb1);
        if (lane == 0) { wv[32 * k + c] = w; dvs[32 * k + c] = d; }
        const double tfac = a[c] * w;
        if (c < lane) Bkk[lane * P2_LD + c] = tfac;  // Lu[lane][c]
        if (c + 1 < 32) {
#pragma unroll
          for (int p = (c + 1) / 2; p < 16; p++) {
            const double2 v = *reinterpret_cast<const double2*>(cA + 2 * p);
            if (2 * p >= c + 1) a[2 * p] = fma(-tfac, v.x, a[2 * p]);
            a[2 * p + 1] = fma(-tfac, v.y, a[2 * p + 1]);
          }
          double* nA = ex + ((c + 1) & 1) * 64;
          nA[lane] = a[c + 1];
          if (c + 2 < 32) nA[32 + lane] = a[c + 2];
        }
        __syncwarp();
        if (lane == 0) p2_st_prog(prog, 32 * k + c + 1);  // column c of Lu, w_c, d_c are out
        d = dnext;
      }
      P2_STAMP(2 + 6 * k);
    } else if (follower) {
      // x <- Lu_kk^-1 x by columns, column c as soon as the pivot warp has published it
      if (row_follower) {
        const double* row = p2_blk(sm, k + warp, k) + lane * P2_LD;
#pragma unroll
        for (int p = 0; p < 16; p++) {
          const double2 v = *reinterpret_cast<const double2*>(row + 2 * p);
          x[2 * p] = v.x; x[2 * p + 1] = v.y;
        }
      } else {
#pragma unroll
        for (int c = 0; c < 32; c++) x[c] = (c == lane) ? 1.0 : 0.0;
      }
#pragma unroll
      for (int c = 0; c < 31; c++) {
        while (p2_ld_prog(prog) < 32 * k + c + 1) { }
#pragma unroll
        for (int c2 = c + 1; c2 < 32; c2++) x[c2] = fma(-x[c], Bkk[c2 * P2_LD + c], x[c2]);
      }
    } else if (warp == 4) {
      // scalings of this sub-block, log-determinant, and L_kk = Lu_kk sqrt(D_k) -> global, once the last pivot is out
      while (p2_ld_prog(prog) < 32 * k + 32) __nanosleep(200);  // (shares a scheduler with the pivot warp: poll rarely)
      const double d = dvs[32 * k + lane];
      const double rs = rsqrt(d), sq = d * rs;
      rsv[32 * k + lane] = rs;
      sqv[32 * k + lane] = sq;
      __syncwarp();
      double* Lrow = Lblk + (size_t)(32 * k + lane) * ld + 32 * k;
#pragma unroll
      for (int p = 0; p < 16; p++) {
        const double2 l2 = *reinterpret_cast<const double2*>(Bkk + lane * P2_LD + 2 * p);
        const double2 s2 = *reinterpret_cast<const double2*>(sqv + 32 * k + 2 * p);
        double2 v;
        v.x = (2 * p < lane) ? l2.x * s2.x : (2 * p == lane ? sq : 0.0);
        v.y = (2 * p + 1 < lane) ? l2.y * s2.y : (2 * p + 1 == lane ? sq : 0.0);
        *reinterpret_cast<double2*>(Lrow + 2 * p) = v;
      }
    } else if (warp >= 6 || warp >= 4 - k) {
      // helpers (warps 6, 7 and the follower warps already out of work: 2 + k of them): global stores that nothing on
      // the chain waits for, and the inverse: close row R = k-1, push its contributions into the rows below
      const int nh = 2 + k;
      const int hx = (warp >= 6) ? k + warp - 6 : warp - (4 - k);
      const int ht = hx * 32 + lane, nht = nh * 32;
      if (k == 0) { p2_out_zeros(ht, nht, Lblk, DIblk, Tblk, Ublk, ld, zero_lu); goto phase_a_done; }
      const int R = k - 1;
      // L[i][R] = u[i][R] D_R^-1/2, i > R
      for (int e = ht; e < (3 - R) * 256; e += nht) {
        const int i = R + 1 + (e >> 8), r = (e >> 3) & 31, c4 = (e & 7) * 4;
        const double* src = p2_blk(sm, i, R) + r * P2_LD + c4;
        const double* rk = rsv + 32 * R + c4;
        double* dst = Lblk + (size_t)(32 * i + r) * ld + 32 * R + c4;
        double2 v0 = *reinterpret_cast<const double2*>(src), v1 = *reinterpret_cast<const double2*>(src + 2);
        v0.x *= rk[0]; v0.y *= rk[1]; v1.x *= rk[2]; v1.y *= rk[3];
        *reinterpret_cast<double2*>(dst) = v0;
        *reinterpret_cast<double2*>(dst + 2) = v1;
      }
      if (R >= 1) {
        double acc[2][4][2];
        p2_inv_t(acc, sm, R, hx, g8, q);
        P2_BARH(nh);
        p2_inv_t_store(acc, sm, R, hx, g8, q);
        P2_BARH(nh);
        p2_inv_update(sm, R, hx, nh, g8, q);
      }
      P2_BARH(nh);  // every read of u[i][R] above is done
      p2_inv_first(sm, R, hx, nh, g8, q);
      p2_out_row(sm, R, ht, nht, DIblk, Tblk, Ublk, ld);
    }
  phase_a_done:
    P2_STAMP(3 + 6 * k);
    P2_WSTAMP(0, k);
    __syncthreads();
    P2_STAMP(4 + 6 * k);
    P2_STAMP(5 + 6 * k);
    // ---------------------------------------------------------------- phase C: followers' results back
    if (follower) {
      if (!row_follower) {
#pragma unroll
        for (int c = 0; c < 32; c++) Bkk[c * P2_LD + lane] = (c >= lane) ? x[c] : 0.0;  // Tu_kk[c][lane]
      } else {
        double* row = p2_blk(sm, k + warp, k) + lane * P2_LD;
#pragma unroll
        for (int p = 0; p < 16; p++) {
          double2 v; v.x = x[2 * p]; v.y = x[2 * p + 1];
          *reinterpret_cast<double2*>(row + 2 * p) = v;
        }
      }
    }
    P2_WSTAMP(1, k);
    __syncthreads();
    P2_STAMP(6 + 6 * k);
    // ---------------------------------------------------------------- phase D
    if (k < 3) {
      // B[i][j] -= (u[i][k] W_k) u[j][k]^T, k < j <= i: jobs (tile, half)
      const int rem = 3 - k, njobs = rem * (rem + 1);
      for (int job = warp; job < njobs; job += 8) {
        const int t = job >> 1, mh = job & 1;
        int ii = 0;
        while ((ii + 1) * (ii + 2) / 2 <= t) ii++;
        const int jj = t - ii * (ii + 1) / 2;
        const int i = k + 1 + ii, j = k + 1 + jj;
        double* Cst = p2_blk(sm, i, j) + 16 * mh * P2_LD;
        double acc[2][4][2];
#pragma unroll
        for (int h = 0; h < 2; h++)
#pragma unroll
          for (int ni = 0; ni < 4; ni++) {
            const double2 v = *reinterpret_cast<const double2*>(Cst + (8 * h + g8) * P2_LD + 8 * ni + 2 * q);
            acc[h][ni][0] = v.x; acc[h][ni][1] = v.y;
          }
        p2_strip2<false, true, true, 8>(acc, p2_blk(sm, i, k) + 16 * mh * P2_LD, p2_blk(sm, j, k), wv + 32 * k, g8, q,
                                        (i == j && mh == 0) ? 2 : 4);  // a diagonal tile is only used below its diagonal
        p2_store2(Cst, acc, g8, q);
      }
      __syncthreads();
    }
    P2_STAMP(7 + 6 * k);
  }
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // the panel solve may start its prologue
  // ---- row 3 of the inverse: Tu[3][j] = -Tu_33 M[3][j], 6 jobs on warps 0..5
  {
    double acc[2][4][2];
    p2_inv_t(acc, sm, 3, warp, g8, q);
    __syncthreads();
    p2_inv_t_store(acc, sm, 3, warp, g8, q);
    if (tid < 128) {  // log-determinant: one logarithm per thread, summed in a fixed order
      double lg = 0.5 * log(dvs[tid]);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) lg += __shfl_xor_sync(0xffffffffu, lg, o);
      if (lane == 0) ex[warp] = lg;
    }
    __syncthreads();
  }
  P2_STAMP(26);
  p2_out_row(sm, 3, tid, P2_THREADS, DIblk, Tblk, Ublk, ld);
  if (tid == 0) {
    scal[SC_LOGDET] += (ex[0] + ex[1]) + (ex[2] + ex[3]);
    if (bad != 0 && scal[SC_INFO] == 0.0) scal[SC_INFO] = (double)(base + bad);
  }
  P2_STAMP(27);
#ifdef P2_TIMING
  __syncthreads();
  if (tid < 64) p2_ts[tid] = reinterpret_cast<long long*>(p2_smem + P2_OFF_PROG + 2)[tid];
  if (tid < 64) p2_wts[tid] = reinterpret_cast<long long*>(p2_smem + P2_OFF_PROG + 2)[64 + tid];
#endif
}

}  // namespace dgp
