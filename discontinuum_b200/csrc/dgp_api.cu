// libdgp.so -- C ABI (include/dgp.h) and host-side schedule of the B200 exact-GP engine.
//
// Per evaluation (DESIGN.md 4.5), on four streams (P: panel chain, highest priority; T and T2: trailing updates;
// W: everything after the factorisation, lowest priority):
//   features/residual -> [block-column 0 covariance panel] ->
//   two-level right-looking Cholesky, panels of 4 block columns:
//     P: for s in panel: k_potf2_v2(s) -> panel solve(s) (GEMM against T_ss) -> rank-128 update of the panel's columns
//        (programmatic dependent launches; 64-row half tiles while a launch is smaller than the GPU)
//     T / T2: rank-512 update right of the panel in fixed column strips, strip j on stream j mod 2; the next panel's
//        columns are the head of their strip: first column | its other columns | the rest of the strip       (n^3/3, DMMA)
//     from SYRK_MIN_NB block columns split at hs: left of hs the updates stop at column hs, and the lower-right quadrant
//        takes them all at once as A22 -= L21 L21' on the INT8 tensor cores (syrk_i8)               (44 % of the n^3/3)
//   W: U = L^-T by recursive doubling (two long-K products and a transpose per level; up to 96 block columns and in batches
//      the merges are launched as the factorisation passes them)                                            (n^3/3, DMMA)
//      z = U'r, alpha = U z, LAUUM -> Ky^-1 (lower tiles), gradient contraction W (.) dK/dtheta              (n^3/3, DMMA)
//   deterministic reductions -> {nlml, info, grad} -> pinned host buffer.
// Three padded n x n panels: bufA (work matrix, then T = L^-1 and scratch, then Ky^-1), bufL (L, lower), bufU (U = L^-T,
// upper).  Covariance tiles come from one of two generators with the same per-entry arithmetic (dgp_cov.cuh): up to
// DGP_PREGEN_MIN_NB block columns and for the prediction / sampling matrices a tile is generated in shared
// memory in the epilogue of its first trailing update (out = K - sum) and K itself is never stored; for larger training
// matrices a standalone generator writes the lower tiles of K into the work matrix strip by strip on the low-priority stream
// while the first panel is factored (measured faster: the generator's FP64 arithmetic shares the datapath with DMMA and is
// latency-bound inside a GEMM epilogue; the extra 2 x 8 n^2 bytes are 3 % of the evaluation's DRAM traffic, DESIGN 4.6).
#include <cuda.h>
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <tuple>
#include <utility>
#include <vector>

#include "../../include/dgp.h"
#include "dgp_cov.cuh"
#include "dgp_gemm.cuh"
#include "dgp_lauum8.cuh"
#include "dgp_panel.cuh"
#include "dgp_potf2.cuh"

using namespace dgp;

namespace {

thread_local std::string g_create_error;

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (PFN_encodeTiled)p;
  }
  return fn;
}

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

// the factorisation schedule of both engines (DESIGN.md 4.5): panels of PANEL_BLOCKS block columns; trailing updates in
// column strips of STRIP_BLOCKS block columns, strip j on stream j mod 2
constexpr int PANEL_BLOCKS = 4;
constexpr int STRIP_BLOCKS = 8;
static_assert(STRIP_BLOCKS % PANEL_BLOCKS == 0, "a strip holds whole panels");
// the merges of the inverse are launched as the factorisation passes them up to this many block columns (single-site engine)
constexpr int EAGER_INV_MAX_NB = 96;
// sites of at least this many padded points form Ky^-1 for the gradient on the INT8 tensor cores (dgp_lauum8.cuh), in both
// engines alike; below it the FP64 DMMA LAUUM is faster (tools/lauum_emul_probe.py)
constexpr int L8_MIN_NPAD = 8192;
inline bool lauum_emulated(int npad) { return npad >= L8_MIN_NPAD && npad <= L8_MAX_NPAD; }
// a merge of the inverse (block ranges of hb and w2 <= hb blocks) forms its two products on the INT8 tensor cores
// (inv_merge_i8) when hb >= INV8_MIN_HB and w2 >= INV8_MIN_W2, in both engines alike; smaller merges stay on the FP64 DMMA
// tile engine.  Measured per merge (tools/inv_emul_probe.py, DESIGN.md 4.1b): 16 | 16 loses, 32 | 32, 64 | 16 and above
// win; hb = 32 stays on DMMA so that the batched sites up to 64 blocks keep their shared launches.  Monotone in w2: at one
// level only the ragged last pair can fall below it.
constexpr int INV8_MIN_HB = 64;
constexpr int INV8_MIN_W2 = 16;
inline bool inv_emulated(int hb, int w2) { return hb >= INV8_MIN_HB && w2 >= INV8_MIN_W2 && 128 * hb <= L8_MAX_NPAD; }
// a training matrix of SYRK_MIN_NB block columns or more is factorised split at hs = syrk_split(nb) block columns
// (potrf_core): the panels left of hs update only the block columns left of it, and the lower-right quadrant receives all
// their updates as one product A22 -= L21 L21' on the INT8 tensor cores (syrk_i8), K = 128 hs.  In both engines alike, a
// function of nb only.  hs = 3 nb / 8 rounded to a whole strip (DESIGN.md 4.5, tools/syrk_emul_probe.py).
constexpr int SYRK_MIN_NB = 96;
constexpr int SYRK_NUM = 3, SYRK_DEN = 8;
static_assert(SYRK_MIN_NB > DGP_PREGEN_MIN_NB, "the quadrant is always a pre-generated matrix");
static_assert(EAGER_INV_MAX_NB < 2 * INV8_MIN_HB, "no INT8 merge of the eager inverse shares the residue buffers with syrk_i8");
inline int syrk_split(int nb) {
  if (nb < SYRK_MIN_NB || 128 * nb > L8_MAX_NPAD) return 0;
  return (SYRK_NUM * nb + SYRK_DEN * STRIP_BLOCKS / 2) / (SYRK_DEN * STRIP_BLOCKS) * STRIP_BLOCKS;
}
// blocks of the second range of merge pair pr at level hb of an nb-block inverse
inline int pair_w2(int nb, int hb, int pr) { return std::min(hb, nb - (2 * pr + 1) * hb); }

// residue buffers of the emulated LAUUM and inverse merges, allocated by the first evaluation that needs them and kept until
// destroy: R [16][npad][npad] int8 (LAUUM: operand residues in the upper block triangle, product residues in the strictly
// lower one; a merge: the planes of its two operands and of its product, 16 (hb^2 + 2 hb w2) 128^2 <= 16 npad^2 bytes),
// D [16][npad][128] int8 (LAUUM: product residues of the diagonal blocks), the row scale exponents [npad]
struct L8Work {
  int8_t *R = nullptr, *D = nullptr;
  int* sexp = nullptr;
  void release() {
    if (R) cudaFree(R);
    if (D) cudaFree(D);
    if (sexp) cudaFree(sexp);
    R = D = nullptr; sexp = nullptr;
  }
};

}  // namespace

struct dgp_handle_s {
  int device = 0;
  cudaStream_t stream = nullptr;     // trailing updates and everything outside the factorisation
  cudaStream_t stream_hi = nullptr;  // look-ahead: diagonal block + panel solve of the next block column (high priority)
  cudaStream_t stream_lo = nullptr;  // inverse, LAUUM and gradient contraction (lowest priority, own streams only): grids are
                                     // served in priority, then launch order, so that the trailing updates of one site's
                                     // factorisation do not wait for the dispatch of another site's multi-millisecond grids
  cudaEvent_t ev_lo[2] = {nullptr, nullptr};
  bool own_stream = false;
  std::vector<cudaEvent_t> evs;      // look-ahead dependencies (no timing)
  cudaStream_t stream_t2 = nullptr;  // second trailing-update stream (same priority as `stream`): column strips alternate
  int max_n = 0, max_pad = 0, max_m = 0;
  int n = 0, npad = 0, nb = 0, sms = 148;
  bool have_train = false, factorized = false, have_T = false, debug_kinv = false, timing = false;
  bool lu_zeroed = false;  // bufL / bufU cleared for the current leading dimension (see k_potf2_v2, zero_lu)
  int zeroed_npad = 0;     // ... which is this one
  dgp_spec spec;       // internal copy: the caller's spec + derived sin/cos feature columns of periodic factors
  // device buffers
  double *bufA = nullptr, *bufL = nullptr, *bufU = nullptr, *DI = nullptr;
  double *X = nullptr, *y = nullptr, *noise = nullptr, *Xw = nullptr, *r = nullptr, *z = nullptr, *alpha = nullptr;
  double *theta = nullptr, *scal = nullptr, *gpart = nullptr, *zpart = nullptr;
  // adjoint of the posterior mean (dgp_mean_functional_grad)
  double *cvec = nullptr, *vvec = nullptr, *gam = nullptr, *tmpz = nullptr, *mfg_out = nullptr, *wpart = nullptr;
  double* h_mfg = nullptr;
  size_t wpart_count = 0;
  // m-sized workspace of dgp_sample_ex / dgp_dist_begin: one grow-only arena (dgp_reserve sizes it ahead of time, so that the
  // calls themselves allocate nothing; a call that needs more than was reserved grows it once and keeps it)
  double* arena = nullptr;
  size_t arena_count = 0;
  // prediction chunk
  double *Kx = nullptr, *Xs = nullptr, *Xws = nullptr, *means = nullptr, *dot = nullptr, *vpart = nullptr;
  double *mu = nullptr, *var = nullptr;
  // pinned host staging
  double *h_theta = nullptr, *h_scal = nullptr;
  L8Work l8;
  CUtensorMap tmA, tmL, tmU, tmDI, tmKx;
  cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  double last_ms[4] = {0, 0, 0, 0};
  bool pending = false;
  int pending_grad = 0;
  long long launches = 0;
  // DGP_TRACE=<file>: one timing event before/after every launch of the factorisation, dumped per evaluation
  struct TraceMark { cudaEvent_t ev; const char* tag; int lane; int arg; };
  std::vector<TraceMark> trace;
  const char* trace_path = nullptr;
  std::string err;
};

#define DGP_FAIL(h, code, ...)                                   \
  do {                                                           \
    char buf_[512];                                              \
    snprintf(buf_, sizeof(buf_), __VA_ARGS__);                   \
    if (h) (h)->err = buf_; else g_create_error = buf_;          \
    return (code);                                               \
  } while (0)

#define CK(h, call)                                                                                   \
  do {                                                                                                \
    cudaError_t e_ = (call);                                                                          \
    if (e_ != cudaSuccess) DGP_FAIL(h, -2, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

static inline void trace_mark(dgp_handle h, cudaStream_t st, const char* tag, int arg) {
  if (!h->trace_path) return;
  cudaEvent_t e;
  if (cudaEventCreate(&e) != cudaSuccess) return;
  cudaEventRecord(e, st);
  h->trace.push_back({e, tag, st == h->stream ? 0 : 1, arg});
}

static void trace_dump(dgp_handle h) {
  if (!h->trace_path || h->trace.empty()) return;
  FILE* f = fopen(h->trace_path, "a");
  if (f) {
    fprintf(f, "# evaluation n=%d\n", h->n);
    for (auto& m : h->trace) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, h->trace[0].ev, m.ev);
      fprintf(f, "%d,%s,%d,%.3f\n", m.lane, m.tag, m.arg, ms * 1e3);
    }
    fclose(f);
  }
  for (auto& m : h->trace) cudaEventDestroy(m.ev);
  h->trace.clear();
}

static int make_map(dgp_handle h, CUtensorMap* m, double* base, int rows, int cols, long long ld) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) DGP_FAIL(h, -3, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 8};
  cuuint32_t box[2] = {BK, 64};
  cuuint32_t es[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) DGP_FAIL(h, -3, "cuTensorMapEncodeTiled failed (%d) rows=%d cols=%d ld=%lld", (int)r, rows, cols, ld);
  return 0;
}

// Programmatic dependent launch: the kernel may be scheduled while its predecessor in the stream is still in its
// tail (after the predecessor's griddepcontrol.launch_dependents); it blocks in griddepcontrol.wait, before its
// first global access, until the predecessor has completed and flushed.  Hides the launch latency between the short,
// strictly dependent kernels of the panel chain.
template <typename... KArgs, typename... Args>
static cudaError_t launch_ex(void (*kern)(KArgs...), int grid, int block, size_t smem, cudaStream_t st, bool pdl, Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(block); cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

// the residue buffers, allocated on first use for sites of up to cap padded points
template <typename HT>
static int l8_ensure(HT h, L8Work& w, long long cap) {
  if (w.R) return 0;
  const size_t c = (size_t)cap;
  cudaError_t e = cudaMalloc((void**)&w.R, L8_NMOD * c * c);
  if (e == cudaSuccess) e = cudaMalloc((void**)&w.D, L8_NMOD * c * 128);
  if (e == cudaSuccess) e = cudaMalloc((void**)&w.sexp, c * sizeof(int));
  if (e != cudaSuccess) {
    cudaGetLastError();
    w.release();
    DGP_FAIL(h, -2, "INT8 emulation workspace (%zu B for %lld padded points) not allocated: %s",
             (size_t)L8_NMOD * c * (c + 128) + c * sizeof(int), cap, cudaGetErrorString(e));
  }
  static bool attr_set[64] = {false};
  const int dev = (h->device >= 0 && h->device < 64) ? h->device : 0;
  if (!attr_set[dev]) {
    CK(h, cudaFuncSetAttribute(k_l8_gemm, cudaFuncAttributeMaxDynamicSharedMemorySize, L8_SMEM));
    CK(h, cudaFuncSetAttribute(k_l8_gemm_ab, cudaFuncAttributeMaxDynamicSharedMemorySize, L8_SMEM));
    attr_set[dev] = true;
  }
  return 0;
}

// 3-D map of 16 int8 residue planes [16][rows][kw] (128 x 128 boxes, the operand layout of l8_tile)
template <typename HT>
static int l8_map(HT h, CUtensorMap* tm, int8_t* base, long long rows, long long kw) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) DGP_FAIL(h, -3, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[3] = {(cuuint64_t)kw, (cuuint64_t)rows, (cuuint64_t)L8_NMOD};
  cuuint64_t strides[2] = {(cuuint64_t)kw, (cuuint64_t)kw * (cuuint64_t)rows};
  cuuint32_t box[3] = {128, 128, 1};
  cuuint32_t es[3] = {1, 1, 1};
  CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) DGP_FAIL(h, -3, "cuTensorMapEncodeTiled (int8 residues) failed (%d) rows=%lld kw=%lld", (int)r, rows, kw);
  return 0;
}

// Ky^-1 = U U' (lower block triangle of K, leading dimension ld) of one site of npad points on the INT8 tensor cores
template <typename HT>
static int lauum_i8(HT h, L8Work& w, long long cap, const double* U, double* K, long long ld, int npad, cudaStream_t st) {
  const int nb = npad / 128;
  int rc;
  if ((rc = l8_ensure(h, w, cap))) return rc;
  CUtensorMap tm;
  if ((rc = l8_map(h, &tm, w.R, npad, npad))) return rc;
  k_l8_convert<<<npad, 256, 0, st>>>(U, ld, npad, l8_bits(npad), true, false, w.R, npad, (long long)npad * npad, w.sexp);
  k_l8_gemm<<<L8_NMOD * l8_slots(nb), 128, L8_SMEM, st>>>(tm, nb, w.R, w.D, npad);
  k_l8_recon<<<nb * (nb + 1) / 2, 256, 0, st>>>(w.R, w.D, npad, w.sexp, K, ld);
  h->launches += 3;
  CK(h, cudaGetLastError());
  return 0;
}

// C = sign A B' (ra x rb tiles, leading dimension ldc) on the INT8 tensor cores, A = rows [0, 128 ra) and B = rows
// [0, 128 rb) of their k ranges [0, 128 kb) (leading dimension ld): A upper block triangular and the k blocks [i, kb) of
// tile row i when kupper, else B lower triangular at 64-row granularity and the k blocks [0, c + 1) of tile column c.
// The operand width b depends on the k extent 128 kb alone.
template <typename HT>
static int gemm_ab_i8(HT h, L8Work& w, const double* A, const double* B, long long ld, int ra, int rb, int kb, bool kupper,
                      double sign, double* C, long long ldc, cudaStream_t st) {
  const long long kw = 128LL * kb, rowsA = 128LL * ra, rowsB = 128LL * rb;
  int8_t* PA = w.R;
  int8_t* PB = PA + L8_NMOD * rowsA * kw;
  int8_t* PC = PB + L8_NMOD * rowsB * kw;
  int* sa = w.sexp;
  int* sb = w.sexp + rowsA;
  const int b = l8_bits(kw);
  int rc;
  CUtensorMap tmA, tmB;
  if ((rc = l8_map(h, &tmA, PA, rowsA, kw)) || (rc = l8_map(h, &tmB, PB, rowsB, kw))) return rc;
  k_l8_convert<<<(unsigned)rowsA, 256, 0, st>>>(A, ld, (int)kw, b, kupper, false, PA, kw, rowsA * kw, sa);
  k_l8_convert<<<(unsigned)rowsB, 256, 0, st>>>(B, ld, (int)kw, b, false, !kupper, PB, kw, rowsB * kw, sb);
  k_l8_gemm_ab<<<L8_NMOD * 64 * ((ra + 7) / 8) * ((rb + 7) / 8), 128, L8_SMEM, st>>>(tmA, tmB, ra, rb, kb,
                                                                                      kupper ? L8_KUPPER_A : L8_KLOWER_B, PC);
  k_l8_recon_ab<<<ra * rb, 256, 0, st>>>(PC, ra, rb, sa, sb, sign, C, ldc, false);
  h->launches += 4;
  CK(h, cudaGetLastError());
  return 0;
}

// the lower-right quadrant update of a split factorisation (potrf_core) on the INT8 tensor cores: A22 -= L21 L21', L21 = rows
// [128 hs, 128 nb) x columns [0, 128 hs) of L, over the lower tiles of A22 with its diagonal blocks in full (the region the
// DMMA trailing updates write).  Operand planes [16][128 r][128 hs], product planes [16][128 r][128 r] (r = nb - hs): together
// 16 128^2 r nb bytes, inside the LAUUM's 16 npad^2.  Every entry is the exact product rounded once, then one subtraction.
template <typename HT>
static int syrk_i8(HT h, L8Work& w, long long cap, const double* L, double* A, long long ld, int nb, int hs, cudaStream_t st) {
  int rc;
  if ((rc = l8_ensure(h, w, cap))) return rc;
  const int r = nb - hs;
  const long long kw = 128LL * hs, rows = 128LL * r;
  int8_t* PA = w.R;
  int8_t* PC = PA + L8_NMOD * rows * kw;
  CUtensorMap tm;
  if ((rc = l8_map(h, &tm, PA, rows, kw))) return rc;
  const size_t o = (size_t)hs * 128;
  k_l8_convert<<<(unsigned)rows, 256, 0, st>>>(L + o * ld, ld, (int)kw, l8_bits(kw), false, false, PA, kw, rows * kw, w.sexp);
  k_l8_gemm_ab<<<L8_NMOD * l8_slots(r), 128, L8_SMEM, st>>>(tm, tm, r, r, hs, L8_KFULL_SYRK, PC);
  k_l8_recon_ab<<<r * (r + 1) / 2, 256, 0, st>>>(PC, r, r, w.sexp, w.sexp, -1.0, A + o * ld + o, ld, true);
  h->launches += 3;
  CK(h, cudaGetLastError());
  return 0;
}

// one merge of the inverse (block ranges [o, o + hb) | [o + hb, o + hb + w2)) on the INT8 tensor cores, the products of
// M_INV_M and M_INV_U (dgp_gemm.cuh) over the same operand entries:
//   M'  = U11 L21'  -> upper triangle of A (work matrix), k over the blocks [row block, hb) of range 1
//   U12 = -M' T22'  -> U, k over range 2 up to the 64-row half of T22's row (T22 in the lower triangle of A)
template <typename HT>
static int inv_merge_i8(HT h, L8Work& w, long long cap, double* A, const double* L, double* U, long long ld, int o, int hb,
                        int w2, cudaStream_t st) {
  int rc;
  if ((rc = l8_ensure(h, w, cap))) return rc;
  const size_t r1 = (size_t)o * 128, r2 = (size_t)(o + hb) * 128;
  double* Mp = A + r1 * ld + r2;
  if ((rc = gemm_ab_i8(h, w, U + r1 * ld + r1, L + r2 * ld + r1, ld, hb, w2, hb, true, 1.0, Mp, ld, st))) return rc;
  return gemm_ab_i8(h, w, Mp, A + r2 * ld + r2, ld, hb, w2, w2, false, -1.0, U + r1 * ld + r2, ld, st);
}

static const BatchTab g_no_batch = {};   // count == 0: single-site launch
static const P2Batch g_no_p2batch = {};

template <int INIT, int EPI, int MT = 8, typename HT>
static int launch_gemm(HT h, const CUtensorMap& a, const CUtensorMap& b, const GemmArgs& g,
                       cudaStream_t st = nullptr, bool pdl = false, const BatchTab* bt = nullptr) {
  if (g.ntiles <= 0) return 0;
  if (st == nullptr) st = h->stream;
  if (bt == nullptr) bt = &g_no_batch;
  static bool attr_set[64] = {false};  // per device: function attributes belong to the device's context
  const int dev = (h->device >= 0 && h->device < 64) ? h->device : 0;
  if (!attr_set[dev]) {
    CK(h, cudaFuncSetAttribute(k_gemm<INIT, EPI, MT>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_TOTAL));
    attr_set[dev] = true;
  }
  CK(h, launch_ex(k_gemm<INIT, EPI, MT>, g.ntiles * (MT == 8 ? 1 : 2), GEMM_THREADS, (size_t)SM_TOTAL, st, pdl, a, b, h->spec, g, *bt));
  h->launches++;
  return 0;
}

extern "C" {

int dgp_abi_version(void) { return DGP_ABI_VERSION; }

size_t dgp_workspace_bytes(int max_n, int max_m) {
  const size_t np = round_up(max_n > 0 ? max_n : 128, 128);
  const size_t mc = round_up(max_m > 0 ? max_m : 2048, 128);
  const size_t nb = np / 128;
  size_t b = 3 * np * np * 8 + np * 128 * 8;
  b += nb * (nb + 1) * DGP_MAX_THETA * 8 + nb * np * 8;
  b += mc * np * 8 + (nb + 2 * nb) * mc * 8;
  return b;
}

const char* dgp_last_error(dgp_handle h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int dgp_create(dgp_handle* out, int device, int max_n, int max_m, void* stream) {
  if (!out || max_n <= 0) DGP_FAIL((dgp_handle) nullptr, -1, "dgp_create: bad arguments");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    DGP_FAIL((dgp_handle) nullptr, -2, "dgp_create: no CUDA device (this engine has no CPU fallback)");
  dgp_handle h = new dgp_handle_s();
  h->device = device;
  cudaError_t e = cudaSetDevice(device);
  if (e != cudaSuccess) { g_create_error = cudaGetErrorString(e); delete h; return -2; }
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, device);
  if (prop.major != 10) {
    g_create_error = "dgp_create: libdgp is built for sm_100a (B200) only";
    delete h; return -2;
  }
  h->sms = prop.multiProcessorCount;
  h->max_n = max_n;
  h->max_pad = round_up(max_n, 128);
  h->max_m = round_up(max_m > 0 ? max_m : 2048, 128);
  {
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);
    if (stream) { h->stream = (cudaStream_t)stream; }
    else {
      cudaStreamCreateWithPriority(&h->stream, cudaStreamNonBlocking, (lo + hi) / 2);
      h->own_stream = true;
    }
    // the phases after the factorisation get a lowest-priority stream of the handle's own, also behind a caller's stream
    cudaStreamCreateWithPriority(&h->stream_lo, cudaStreamNonBlocking, lo);
    cudaEventCreateWithFlags(&h->ev_lo[0], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&h->ev_lo[1], cudaEventDisableTiming);
    cudaStreamCreateWithPriority(&h->stream_hi, cudaStreamNonBlocking, hi);
    {  // second trailing-update stream at the priority of `stream` (whoever created that)
      int pr = (lo + hi) / 2;
      if (cudaStreamGetPriority(h->stream, &pr) != cudaSuccess) { cudaGetLastError(); pr = (lo + hi) / 2; }
      cudaStreamCreateWithPriority(&h->stream_t2, cudaStreamNonBlocking, pr);
    }
    h->trace_path = getenv("DGP_TRACE");
  }
  const size_t np = h->max_pad, mc = h->max_m, nbm = np / 128;
  auto A = [&](double** p, size_t count) { return cudaMalloc((void**)p, count * sizeof(double)); };
  cudaError_t r = cudaSuccess;
  auto acc = [&](cudaError_t x) { if (r == cudaSuccess) r = x; };
  acc(A(&h->bufA, np * np)); acc(A(&h->bufL, np * np)); acc(A(&h->bufU, np * np)); acc(A(&h->DI, np * 128));
  acc(A(&h->X, np * DGP_MAX_COLS)); acc(A(&h->y, np)); acc(A(&h->noise, np)); acc(A(&h->Xw, np * DGP_XS));
  acc(A(&h->r, np)); acc(A(&h->z, np)); acc(A(&h->alpha, np));
  acc(A(&h->theta, DGP_MAX_THETA)); acc(A(&h->scal, SC_SIZE)); acc(A(&h->gpart, nbm * (nbm + 1) * DGP_MAX_THETA));
  acc(A(&h->zpart, nbm * np));
  acc(A(&h->cvec, mc)); acc(A(&h->vvec, np)); acc(A(&h->gam, np)); acc(A(&h->tmpz, np)); acc(A(&h->mfg_out, 1 + DGP_MAX_THETA));
  h->wpart_count = (mc / 128 + nbm) * (np / 64) * DGP_MAX_THETA;  // dgp_mean_functional_grad partials at the largest m, n
  acc(A(&h->wpart, h->wpart_count));
  acc(cudaMallocHost((void**)&h->h_mfg, (1 + DGP_MAX_THETA) * sizeof(double)));
  acc(A(&h->Kx, mc * np)); acc(A(&h->Xs, mc * DGP_MAX_COLS)); acc(A(&h->Xws, mc * DGP_XS)); acc(A(&h->means, mc));
  acc(A(&h->dot, nbm * mc)); acc(A(&h->vpart, 2 * nbm * mc)); acc(A(&h->mu, mc)); acc(A(&h->var, mc));
  acc(cudaMallocHost((void**)&h->h_theta, DGP_MAX_THETA * sizeof(double)));
  acc(cudaMallocHost((void**)&h->h_scal, SC_SIZE * sizeof(double)));
  for (int i = 0; i < 5; i++) acc(cudaEventCreate(&h->ev[i]));
  if (r != cudaSuccess) {
    g_create_error = std::string("dgp_create: allocation failed: ") + cudaGetErrorString(r);
    dgp_destroy(h);
    return -2;
  }
  cudaFuncSetAttribute(k_potf2_v2, cudaFuncAttributeMaxDynamicSharedMemorySize, P2_SMEM);
  *out = h;
  return 0;
}

int dgp_destroy(dgp_handle h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->stream_hi) { cudaStreamSynchronize(h->stream_hi); cudaStreamDestroy(h->stream_hi); }
  if (h->stream_lo) { cudaStreamSynchronize(h->stream_lo); cudaStreamDestroy(h->stream_lo); }
  if (h->stream_t2) { cudaStreamSynchronize(h->stream_t2); cudaStreamDestroy(h->stream_t2); }
  for (int i = 0; i < 2; i++) if (h->ev_lo[i]) cudaEventDestroy(h->ev_lo[i]);
  for (cudaEvent_t e : h->evs) cudaEventDestroy(e);
  double* bufs[] = {h->bufA, h->bufL, h->bufU, h->DI, h->X, h->y, h->noise, h->Xw, h->r, h->z, h->alpha, h->theta,
                    h->scal, h->gpart, h->zpart, h->cvec, h->vvec, h->gam, h->tmpz, h->mfg_out, h->wpart, h->Kx, h->Xs, h->Xws, h->means, h->dot, h->vpart, h->mu, h->var};
  for (double* p : bufs) if (p) cudaFree(p);
  if (h->arena) cudaFree(h->arena);
  h->l8.release();
  if (h->h_theta) cudaFreeHost(h->h_theta);
  if (h->h_scal) cudaFreeHost(h->h_scal);
  if (h->h_mfg) cudaFreeHost(h->h_mfg);
  for (int i = 0; i < 5; i++) if (h->ev[i]) cudaEventDestroy(h->ev[i]);
  if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return 0;
}

extern "C++" {
template <typename HT>
static int check_spec(HT h, const dgp_spec* sp) {
  if (sp->abi != DGP_ABI_VERSION) DGP_FAIL(h, -1, "spec abi %d != %d", sp->abi, DGP_ABI_VERSION);
  if (sp->ndim < 1 || sp->ndim > DGP_MAX_COLS || sp->ncols < 1 || sp->ncols > DGP_MAX_COLS)
    DGP_FAIL(h, -1, "spec: ndim/ncols out of range");
  if (sp->nterms < 1 || sp->nterms > DGP_MAX_TERMS) DGP_FAIL(h, -1, "spec: nterms out of range");
  if (sp->ntheta < 1 || sp->ntheta > DGP_MAX_THETA) DGP_FAIL(h, -1, "spec: ntheta out of range");
  auto bad = [&](int idx) { return idx < -1 || idx >= sp->ntheta; };
  if (bad(sp->noise_theta)) DGP_FAIL(h, -1, "spec: noise_theta out of range");
  if (sp->mean_kind < DGP_MEAN_ZERO || sp->mean_kind > DGP_MEAN_POWERLAW) DGP_FAIL(h, -1, "spec: mean kind %d", sp->mean_kind);
  for (int c = 0; c < sp->ncols; c++) {
    const dgp_col& k = sp->col[c];
    // the internal DGP_COL_SINP / DGP_COL_COSP kinds are appended by augment_spec, never accepted from a caller
    if (k.kind < DGP_COL_COPY || k.kind > DGP_COL_GATE) DGP_FAIL(h, -1, "spec: col %d kind %d", c, k.kind);
    if (k.src < 0 || k.src >= sp->ndim) DGP_FAIL(h, -1, "spec: col %d src out of range", c);
    if (k.kind == DGP_COL_GATE && (k.theta < 0 || k.theta >= sp->ntheta)) DGP_FAIL(h, -1, "spec: gate col %d theta", c);
  }
  for (int t = 0; t < sp->nterms; t++) {
    const dgp_term& tm = sp->term[t];
    if (bad(tm.scale) || tm.nfactors < 0 || tm.nfactors > DGP_MAX_FACTORS) DGP_FAIL(h, -1, "spec: term %d", t);
    if (tm.gate < DGP_GATE_NONE || tm.gate > DGP_GATE_INV_SIGMOID) DGP_FAIL(h, -1, "spec: term %d gate kind %d", t, tm.gate);
    if (tm.gate != DGP_GATE_NONE && (tm.gate_col < 0 || tm.gate_col >= sp->ncols || sp->col[tm.gate_col].kind != DGP_COL_GATE))
      DGP_FAIL(h, -1, "spec: term %d gate column", t);
    for (int f = 0; f < tm.nfactors; f++) {
      const dgp_factor& fa = tm.factor[f];
      if (fa.kind < DGP_RBF || fa.kind > DGP_PERIODIC || fa.ndims < 1 || fa.ndims > DGP_MAX_FDIMS)
        DGP_FAIL(h, -1, "spec: term %d factor %d kind/ndims", t, f);
      for (int d = 0; d < fa.ndims; d++) {
        if (fa.col[d] < 0 || fa.col[d] >= sp->ncols || fa.ls[d] < 0 || fa.ls[d] >= sp->ntheta)
          DGP_FAIL(h, -1, "spec: term %d factor %d dim %d", t, f, d);
        // a gate column depends on theta[col.theta]; the gradient slots of a factor have no place for that dependence
        if (sp->col[fa.col[d]].kind == DGP_COL_GATE)
          DGP_FAIL(h, -1, "spec: term %d factor %d dim %d reads gate column %d", t, f, d, fa.col[d]);
      }
      if (fa.kind == DGP_PERIODIC && (fa.ndims != 1 || fa.period < 0 || fa.period >= sp->ntheta))
        DGP_FAIL(h, -1, "spec: term %d factor %d periodic", t, f);
    }
  }
  if (sp->mean_kind == DGP_MEAN_CONST && (sp->mean_theta[0] < 0 || sp->mean_theta[0] >= sp->ntheta))
    DGP_FAIL(h, -1, "spec: mean theta");
  if (sp->mean_kind == DGP_MEAN_POWERLAW)
    for (int k = 0; k < 3; k++)
      if (sp->mean_theta[k] < 0 || sp->mean_theta[k] >= sp->ntheta || sp->mean_col < 0 || sp->mean_col >= sp->ndim)
        DGP_FAIL(h, -1, "spec: power-law mean");
  return 0;
}
}  // extern "C++"

// Append sinpi / cospi feature columns for periodic factors while the feature table has room (see dgp_cov.cuh).
static void augment_spec(dgp_spec* sp) {
  for (int t = 0; t < sp->nterms; t++)
    for (int f = 0; f < sp->term[t].nfactors; f++) {
      dgp_factor& fa = sp->term[t].factor[f];
      fa.pad_ = 0;
      if (fa.kind != DGP_PERIODIC) continue;
      // reuse the pair of an earlier factor on the same column and period
      for (int c = 0; c + 1 < sp->ncols && fa.pad_ == 0; c++)
        if (sp->col[c].kind == DGP_COL_SINP && sp->col[c].src == fa.col[0] && sp->col[c].theta == fa.period) fa.pad_ = c + 1;
      if (fa.pad_ == 0 && sp->ncols + 2 <= DGP_XS) {
        const int c = sp->ncols;
        sp->col[c].kind = DGP_COL_SINP; sp->col[c].src = fa.col[0]; sp->col[c].theta = fa.period; sp->col[c].pad_ = 0; sp->col[c].aux = 0.0;
        sp->col[c + 1] = sp->col[c];
        sp->col[c + 1].kind = DGP_COL_COSP;
        sp->ncols += 2;
        fa.pad_ = c + 1;
      }
    }
}

int dgp_set_train(dgp_handle h, const dgp_spec* spec, const double* X, const double* y, const double* noise, int n,
                  int on_device) {
  if (!h) return -1;
  if (!spec || !X || !y || !noise || n < 1 || n > h->max_n) DGP_FAIL(h, -1, "dgp_set_train: bad arguments (n=%d, max_n=%d)", n, h->max_n);
  int rc = check_spec(h, spec);
  if (rc) return rc;
  CK(h, cudaSetDevice(h->device));
  h->spec = *spec;
  augment_spec(&h->spec);
  h->n = n;
  h->npad = round_up(n, 128);
  h->nb = h->npad / 128;
  h->factorized = false;
  h->have_T = false;
  const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  // The zero sub-blocks of bufL / bufU (above / below the diagonal) are only ever written by the diagonal-block kernel, and
  // only with zeros: with an unchanged leading dimension they are still clear from the previous training set.
  if (!h->lu_zeroed || h->zeroed_npad != h->npad) {
    CK(h, cudaMemsetAsync(h->bufL, 0, (size_t)h->npad * h->npad * 8, h->stream));
    CK(h, cudaMemsetAsync(h->bufU, 0, (size_t)h->npad * h->npad * 8, h->stream));
    h->lu_zeroed = true;
    h->zeroed_npad = h->npad;
  }
  CK(h, cudaMemsetAsync(h->noise, 0, (size_t)h->npad * 8, h->stream));
  CK(h, cudaMemcpyAsync(h->X, X, (size_t)n * spec->ndim * 8, kind, h->stream));
  CK(h, cudaMemcpyAsync(h->y, y, (size_t)n * 8, kind, h->stream));
  CK(h, cudaMemcpyAsync(h->noise, noise, (size_t)n * 8, kind, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  const long long ld = h->npad;
  if ((rc = make_map(h, &h->tmA, h->bufA, h->npad, h->npad, ld))) return rc;
  if ((rc = make_map(h, &h->tmL, h->bufL, h->npad, h->npad, ld))) return rc;
  if ((rc = make_map(h, &h->tmU, h->bufU, h->npad, h->npad, ld))) return rc;
  if ((rc = make_map(h, &h->tmDI, h->DI, h->npad, 128, 128))) return rc;
  if ((rc = make_map(h, &h->tmKx, h->Kx, h->max_m, h->npad, ld))) return rc;
  h->have_train = true;
  return 0;
}

// ------------------------------------------------------------------ schedule pieces
static int upload_theta(dgp_handle h, const double* theta) {
  memcpy(h->h_theta, theta, sizeof(double) * h->spec.ntheta);
  CK(h, cudaMemcpyAsync(h->theta, h->h_theta, sizeof(double) * h->spec.ntheta, cudaMemcpyHostToDevice, h->stream));
  return 0;
}

static GemmArgs base_args(dgp_handle h, int mode, int step) {
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.mode = mode; g.step = step; g.nb = h->nb; g.n = h->n;
  g.ldc = h->npad; g.sign = 1.0;
  g.Xw = h->Xw; g.noise = h->noise; g.theta = h->theta; g.part = h->gpart;
  return g;
}

static int run_features(dgp_handle h) {
  k_features<<<(h->npad + 255) / 256, 256, 0, h->stream>>>(h->spec, h->theta, h->X, h->y, h->Xw, h->r, nullptr, h->n,
                                                        h->npad, h->scal);
  h->launches++;
  CK(h, cudaGetLastError());
  return 0;
}

// Right-looking blocked Cholesky of the padded matrix in `A` (lower tiles), L -> `Lm`.  generate: block
// column 0 and every tile at its first trailing update come from the covariance generator instead of memory.
struct CholBufs {
  double *A, *L, *U, *DI, *scal;
  const CUtensorMap *tA, *tL, *tDI;
  int nb;
  long long ld;
  double* P = nullptr;  // in-place factorisation (L == A): [rows][128] staging buffer of the panel solve
};

static int ensure_events(dgp_handle h, size_t count) {
  while (h->evs.size() < count) {
    cudaEvent_t e;
    CK(h, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    h->evs.push_back(e);
  }
  return 0;
}

// Two-level right-looking Cholesky with look-ahead.  Block columns are grouped in panels of PANEL_BLOCKS blocks.
// Stream P (high priority) runs the latency-bound work of one panel, block column by block column:
//   potf2(s) -> TRSM(s) (all rows below) [-> forward substitution(s)] -> rank-128 update of the panel's own
//   remaining columns.
// Streams T and T2 run the throughput-bound rank-(128 pw) update of everything right of the panel in column strips: the
// next panel's columns first (all panel p+1 reads), then the rest, which overlaps panel p+1 on P.
// The wide update reads/writes each trailing tile once per panel instead of once per block column.
// one rank-(128 kb) update launch of block columns [o, o + w)
static int launch_trail(dgp_handle h, const CholBufs& b, int k0, int kb, int o, int w, int ntiles, bool first_touch,
                        double jitter, cudaStream_t st, bool half_tiles = false, bool pdl = false) {
  GemmArgs g = base_args(h, M_TRAIL_COL, k0);
  g.nb = b.nb; g.ldc = b.ld;
  g.aux0 = o | (w << 16);
  g.aux1 = kb;
  g.aux2 = first_touch ? 0 : 1;
  g.C = b.A; g.ntiles = ntiles; g.sign = -1.0; g.jitter = jitter;
  if (first_touch) return launch_gemm<INIT_COV, EPI_STORE>(h, *b.tL, *b.tL, g, st, pdl);
  if (half_tiles) return launch_gemm<INIT_LOAD, EPI_STORE, 4>(h, *b.tL, *b.tL, g, st, pdl);
  return launch_gemm<INIT_LOAD, EPI_STORE>(h, *b.tL, *b.tL, g, st, pdl);
}

// the latency-bound chain of one panel [pb, pe) on stream P:
//   for s: potf2(s) -> TRSM(s) on every row below [-> forward substitution(s)] -> rank-128 update of columns (s, pe)
// mid_wait: event the in-panel update of the first block column has to wait for (the trailing update of the panel's
// other columns, which stream T applies while the first column is already being factored)
// piv0: index of b's row 0 in the whole matrix, so that a failing pivot is reported as a global 1-based index when b is a
// trailing submatrix (the panel slabs of dgp_dist_*)
static int factor_panel(dgp_handle h, const CholBufs& b, int pb, int pe, bool generate, double jitter, bool fwd, cudaStream_t P,
                        cudaEvent_t mid_wait = nullptr, int piv0 = 0) {
  const int nb = b.nb;
  const long long ld = b.ld;
  int rc;
  const bool pdl = !h->trace_path;  // the trace's events would sit between the kernels
  // timing experiments only (results are garbage), compiled in with -DDGP_EXPERIMENTS and never in the shipped library:
  // DGP_SKIP bit 0: no diagonal-block kernel, 1: no panel solve, 2: no in-panel update
#ifdef DGP_EXPERIMENTS
  static const int skip = getenv("DGP_SKIP") ? atoi(getenv("DGP_SKIP")) : 0;
#else
  constexpr int skip = 0;
#endif
  for (int s = pb; s < pe; s++) {
    const size_t off = (size_t)s * 128 * ld + (size_t)s * 128;
    const bool inplace = (b.L == b.A);
    trace_mark(h, P, "potf2<", s);
    // T_ss is read by the panel solve from the diagonal block of the work matrix: the contiguous copy in DI is only
    // written for the in-place factorisation and for the forward-substitution kernel of the NLML-only path
    const bool t_in_a = !inplace && !fwd;
    // the zero sub-blocks of bufL / bufU were cleared by dgp_set_train and only this kernel ever writes them
    const bool lu_clean = !inplace && h->lu_zeroed && b.L == h->bufL && (b.U == nullptr || b.U == h->bufU);
    if (!(skip & 1))  // dependent launch behind the in-panel update of the previous block column (same stream, nothing in between)
      CK(h, launch_ex(k_potf2_v2, 1, P2_THREADS, (size_t)P2_SMEM, P, pdl && s > pb && !inplace && !fwd, (const double*)(b.A + off), b.L + off,
                      b.U ? b.U + off : (double*)nullptr, ld, t_in_a ? (double*)nullptr : b.DI + (size_t)s * 128 * 128, b.scal, piv0 + s * 128,
                      inplace ? (double*)nullptr : b.A + off, lu_clean ? 0 : 1, g_no_p2batch));
    h->launches++;
    CK(h, cudaGetLastError());
    trace_mark(h, P, "potf2>", s);
    const int m = nb - s - 1;
    if (m > 0 && !(skip & 2)) {
      GemmArgs g = base_args(h, M_TRSM, s);
      g.nb = nb; g.ldc = ld;
      g.C = b.L; g.ntiles = 2 * m;
      if (inplace) { g.C = b.P; g.ldc = 128; g.aux0 = 1; }  // both half-tiles read the whole block: stage, then copy
      g.aux1 = t_in_a ? 1 : 0;
      const CUtensorMap& tB = t_in_a ? *b.tA : *b.tDI;
      // half tiles while the launch is smaller than the GPU (2 m 64x64-row CTAs fit the 2 x SMs slots)
      if (4 * m <= 2 * h->sms) { if ((rc = launch_gemm<INIT_ZERO, EPI_STORE, 4>(h, *b.tA, tB, g, P, pdl))) return rc; }
      else if ((rc = launch_gemm<INIT_ZERO, EPI_STORE>(h, *b.tA, tB, g, P, pdl))) return rc;
      if (inplace) {
        k_copy_panel<<<m, 256, 0, P>>>(b.P, b.A, ld, s);
        h->launches++;
        CK(h, cudaGetLastError());
      }
      trace_mark(h, P, "trsm>", s);
    }
    if (fwd) {
      k_fwd_step<<<nb - s, 256, 0, P>>>(b.L, ld, b.DI, h->r, h->z, s);
      h->launches++;
      CK(h, cudaGetLastError());
    }
    if (s + 1 < pe && !(skip & 4)) {  // in-panel update: rank-128 update of the panel's own block columns (s, pe), rows >= s + 1
      const bool waited = (s == pb && mid_wait != nullptr);
      if (waited) CK(h, cudaStreamWaitEvent(P, mid_wait, 0));
      const int w = pe - s - 1;
      if ((rc = launch_trail(h, b, s, 1, s + 1, w, m * 2 * w, generate && s == 0, jitter, P, 4 * m * w <= 2 * h->sms,
                             pdl && !inplace && !fwd && !waited))) return rc;
      trace_mark(h, P, "inpanel>", s);
    }
  }
  return 0;
}

// after_panel(p, pe): called once the chain of panel p is enqueued and ev_panel(p) = h->evs[3 p] is recorded (the first pe
// block columns of L, and the diagonal blocks of T and U up to there, are final behind that event)
struct PanelHook { int (*fn)(dgp_handle, void*, cudaEvent_t, int) = nullptr; void* ctx = nullptr; };

// the standalone generator covers every matrix it is used for with at least two column strips
static_assert(DGP_PREGEN_MIN_NB >= STRIP_BLOCKS, "pre-generated matrices span more than one strip");

// hs > 0 (training matrices, syrk_split): the panels ending at or before block column hs update the block columns [pe, hs)
// only, all rows below included, so L21 comes out exactly as without the split; after the panel ending at hs, syrk_i8
// applies all their updates to the lower-right quadrant at once and the panels from hs on run as without the split.
static int potrf_core(dgp_handle h, const CholBufs& b, bool generate, double jitter, bool fwd, PanelHook hook = PanelHook(),
                      int hs = 0) {
  const int nb = b.nb;
  const long long ld = b.ld;
  int rc;
  cudaStream_t T = h->stream, P = h->stream_hi, T2 = h->stream_t2;
  constexpr int pw = PANEL_BLOCKS, sw = STRIP_BLOCKS;
  const int npanels = (nb + pw - 1) / pw;
  bool any2 = false;
  const int nstrips = (nb + sw - 1) / sw;
  // above DGP_PREGEN_MIN_NB block columns the covariance matrix is written by a standalone generator, strip by strip on the
  // low-priority stream while the first panel is factored, and the first trailing update reads it like any later one
  const bool pregen = generate && nb > DGP_PREGEN_MIN_NB;
  if ((rc = ensure_events(h, 3 * (size_t)npanels + 3 + (size_t)nstrips))) return rc;
  auto ev_gen = [&](int j) { return h->evs[3 * (size_t)npanels + 2 + j]; };
  auto ev_panel = [&](int p) { return h->evs[3 * p]; };
  auto ev_cols = [&](int p) { return h->evs[3 * p + 1]; };   // all columns of panel p have the updates of panels < p
  auto ev_col0 = [&](int p) { return h->evs[3 * p + 2]; };   // ... its first block column has them
  if (pregen) {
    k_cov_lower<<<dim3(nb * 4, sw), 256, 0, T>>>(h->spec, h->theta, h->Xw, h->noise, jitter, b.A, ld, h->n, 0);
    h->launches++;
    CK(h, cudaGetLastError());
    CK(h, cudaEventRecord(h->evs[3 * (size_t)npanels + 1], T));
    cudaStream_t G = h->stream_lo;
    CK(h, cudaStreamWaitEvent(G, h->evs[3 * (size_t)npanels + 1], 0));
    for (int j = 1; j < nstrips; j++) {
      const int o = j * sw, wj = (o + sw < nb) ? sw : nb - o;
      k_cov_lower<<<dim3((nb - o) * 4, wj), 256, 0, G>>>(h->spec, h->theta, h->Xw, h->noise, jitter, b.A, ld, h->n, o);
      h->launches++;
      CK(h, cudaGetLastError());
      CK(h, cudaEventRecord(ev_gen(j), G));
    }
  } else if (generate) {
    k_cov_rect<<<dim3(nb * 4, 1), 256, 0, T>>>(h->spec, h->theta, h->Xw, h->Xw, h->noise, jitter, b.A, ld, h->n,
                                               h->n, 1, 1, nullptr, nullptr, 0);
    h->launches++;
    CK(h, cudaGetLastError());
  }
  CK(h, cudaEventRecord(ev_cols(0), T));
  CK(h, cudaStreamWaitEvent(P, ev_cols(0), 0));
  for (int p = 0; p < npanels; p++) {
    const int pb = p * pw, pe = (pb + pw < nb) ? pb + pw : nb;
    if (p > 0) CK(h, cudaStreamWaitEvent(P, ev_col0(p), 0));
    if ((rc = factor_panel(h, b, pb, pe, generate && !pregen, jitter, fwd, P, p > 0 ? ev_cols(p) : nullptr))) return rc;
    CK(h, cudaEventRecord(ev_panel(p), P));
    CK(h, cudaStreamWaitEvent(T, ev_panel(p), 0));
    if (hook.fn && pe < nb && (rc = hook.fn(h, hook.ctx, ev_panel(p), pe))) return rc;
    if (pe == hs) {   // the quadrant update; the generator's strips right of hs have not been waited for yet
      CK(h, cudaStreamWaitEvent(T, ev_gen(nstrips - 1), 0));
      trace_mark(h, T, "syrk<", p);
      if ((rc = syrk_i8(h, h->l8, h->max_pad, b.L, b.A, ld, nb, hs, T))) return rc;
      trace_mark(h, T, "syrk>", p);
      CK(h, cudaEventRecord(ev_col0(p + 1), T));
      CK(h, cudaEventRecord(ev_cols(p + 1), T));
    } else if (pe < nb) {
      // Column strips on two streams.  The trailing matrix is cut into fixed strips of `sw` block columns; strip j is
      // always updated on stream j mod 2, so the strips of one stream form their own dependency chain (panel after
      // panel) and the two streams never wait for each other: while one launch drains its last partial wave, the other
      // stream's CTAs take the free slots (a single stream loses about half a wave per launch, 3 launches per panel).
      // The next panel's columns are the head of their strip: first column | its other columns | the rest of the strip.
      // Launches with fewer tiles than the GPU has CTA slots run on 64-row half tiles (a K = 512 tile is 34 us on its own).
      const int ce = pe < hs ? hs : nb;   // end of the block columns this panel updates
      const int ne = (pe + pw < nb) ? pe + pw : nb, w = ne - pe, m = nb - pe;
      const int slots = 2 * h->sms;
      const bool first = generate && p == 0 && !pregen;
      const int j0 = pe / sw;
      bool used2 = false;
      auto strip_stream = [&](int j) -> cudaStream_t {
        cudaStream_t S = T;
        if (j & 1) {
          if (!used2) { used2 = true; cudaStreamWaitEvent(T2, ev_panel(p), 0); }
          S = T2;
        }
        if (pregen && p == 0 && j > 0) cudaStreamWaitEvent(S, ev_gen(j), 0);
        return S;
      };
      cudaStream_t S0 = strip_stream(j0);
      trace_mark(h, S0, "cols<", p);
      if ((rc = launch_trail(h, b, pb, pe - pb, pe, 1, m * 2, first, jitter, S0, m * 2 <= slots))) return rc;
      CK(h, cudaEventRecord(ev_col0(p + 1), S0));
      if (w > 1 && (rc = launch_trail(h, b, pb, pe - pb, pe + 1, w - 1, (m - 1) * 2 * (w - 1), first, jitter, S0,
                                      (m - 1) * 2 * (w - 1) <= slots))) return rc;
      trace_mark(h, S0, "cols>", p);
      CK(h, cudaEventRecord(ev_cols(p + 1), S0));
      const int e0 = ((j0 + 1) * sw < ce) ? (j0 + 1) * sw : ce;
      if (ne < e0) {
        const int tiles = (nb - ne) * 2 * (e0 - ne);
        if ((rc = launch_trail(h, b, pb, pe - pb, ne, e0 - ne, tiles, first, jitter, S0, tiles <= slots))) return rc;
      }
      for (int j = j0 + 1; j * sw < ce; j++) {
        const int o = j * sw, wj = (o + sw < ce) ? sw : ce - o, tiles = (nb - o) * 2 * wj;
        if ((rc = launch_trail(h, b, pb, pe - pb, o, wj, tiles, first, jitter, strip_stream(j), tiles <= slots))) return rc;
      }
      trace_mark(h, T, "rest>", p);
      if (used2) any2 = true;
    }
  }
  if (any2) {  // the caller continues on T
    CK(h, cudaEventRecord(h->evs[3 * (size_t)npanels], T2));
    CK(h, cudaStreamWaitEvent(T, h->evs[3 * (size_t)npanels], 0));
  }
  return 0;
}

static int run_potrf(dgp_handle h, double jitter, bool fwd, PanelHook hook = PanelHook()) {
  CholBufs b{h->bufA, h->bufL, h->bufU, h->DI, h->scal, &h->tmA, &h->tmL, &h->tmDI, h->nb, h->npad};
  return potrf_core(h, b, true, jitter, fwd, hook, syrk_split(h->nb));
}

// U = L^-T (upper) by recursive doubling: the diagonal 128-blocks come from k_potf2_v2 (U_ss in bufU, T_ss = L_ss^-1 in
// the diagonal blocks of bufA); level h merges neighbouring block ranges [o, o+h) | [o+h, o+2h):
//   M'  = U11 L21'          -> scratch, upper triangle of bufA          (long-K tiles, no read-modify-write)
//   U12 = -M' T22'          -> bufU
//   T21 = U12'              -> lower triangle of bufA (operand of the next level / of the prediction kernels)
// log2(nb) levels x 3 launches instead of 2 nb launches of rank-128 updates.  want_T: also transpose the last level.
// The merges of a level are launched pair by pair as the factorisation passes them (trtri_advance(F): every merge whose
// block range lies inside the first F block columns and has not been launched yet), on the lowest-priority stream: the
// inverse of the leading ranges fills the SM slots the factorisation leaves idle (partial last waves, the latency-bound
// chain of its last panels).  Same products in the same order as one launch per level: bit-identical.
struct InvProgress {
  int done[16];       // per level (hb = 1 << l): leading pairs already launched
  bool want_T;
  cudaStream_t W;
};

static int trtri_advance(dgp_handle h, InvProgress& ip, int F) {
  const int nb = h->nb;
  int rc, lv = 0;
  for (int hb = 1; hb < nb; hb *= 2, lv++) {
    const int npairs = (nb - hb + 2 * hb - 1) / (2 * hb);  // pairs whose second range is non-empty
    const int avail = F >= nb ? npairs : F / (2 * hb);
    const int pr0 = ip.done[lv], cnt = avail - pr0;
    if (cnt <= 0) continue;
    int pe = pr0;   // pairs [pr0, pe) on the INT8 tensor cores, [pe, avail) on the DMMA tile engine
    for (; pe < avail && inv_emulated(hb, pair_w2(nb, hb, pe)); pe++)
      if ((rc = inv_merge_i8(h, h->l8, h->max_pad, h->bufA, h->bufL, h->bufU, h->npad, pe * 2 * hb, hb, pair_w2(nb, hb, pe),
                             ip.W))) return rc;
    if (pe < avail) {
      {
        GemmArgs g = base_args(h, M_INV_M, pe);
        g.aux0 = hb; g.aux1 = avail - pe; g.C = h->bufA; g.ntiles = (avail - pe) * hb * 2 * hb;
        if ((rc = launch_gemm<INIT_ZERO, EPI_STORE>(h, h->tmU, h->tmL, g, ip.W))) return rc;
      }
      {
        GemmArgs g = base_args(h, M_INV_U, pe);
        g.aux0 = hb; g.aux1 = avail - pe; g.C = h->bufU; g.ntiles = (avail - pe) * hb * 2 * hb; g.sign = -1.0;
        if ((rc = launch_gemm<INIT_ZERO, EPI_STORE>(h, h->tmA, h->tmA, g, ip.W))) return rc;
      }
    }
    if (ip.want_T || 2 * hb < nb) {
      k_transpose_pairs<<<cnt * 16 * hb * hb, 256, 0, ip.W>>>(h->bufU, h->bufA, h->npad, hb, h->npad, pr0);
      h->launches++;
      CK(h, cudaGetLastError());
    }
    ip.done[lv] = avail;
  }
  return 0;
}

static int eager_hook(dgp_handle h, void* ctx, cudaEvent_t ev_panel, int pe) {
  InvProgress& ip = *(InvProgress*)ctx;
  if ((pe & 7) != 0) return 0;   // every 8 block columns: 4 / 2 / 1 new pairs at the three lowest levels
  CK(h, cudaStreamWaitEvent(ip.W, ev_panel, 0));
  return trtri_advance(h, ip, pe);
}

static int run_trtri(dgp_handle h, InvProgress& ip) {
  const int nb = h->nb;
  int rc;
  if ((rc = trtri_advance(h, ip, nb))) return rc;
  // z = U' r (= L^-1 r), alpha = U z
  k_upperT_gemv_part<<<dim3(nb, nb), 256, 0, ip.W>>>(h->bufU, h->npad, h->r, h->zpart, h->npad);
  k_upperT_gemv_sum<<<(h->npad + 255) / 256, 256, 0, ip.W>>>(h->zpart, h->npad, h->z, h->npad);
  k_upper_gemv<<<h->npad / 8, 256, 0, ip.W>>>(h->bufU, h->npad, h->z, h->alpha, h->npad);
  h->launches += 3;
  CK(h, cudaGetLastError());
  return 0;
}

// LAUUM stores the lower tiles of Ky^-1 (8 n^2 / 2 B, over T, which is dead by now) and a separate high-occupancy pass
// contracts W = alpha alpha' - Ky^-1 with the regenerated dK/dtheta tiles (measured 3-4 ms faster at n = 16384 than the
// contraction fused into the LAUUM epilogue, whose dependent FP64 chains wait behind the co-resident CTA's DMMA issue).
static int run_lauum_grad(dgp_handle h) {
  int rc;
  if (lauum_emulated(h->npad)) {
    rc = lauum_i8(h, h->l8, h->max_pad, h->bufU, h->bufA, h->npad, h->npad, h->stream);
  } else {
    GemmArgs g = base_args(h, M_LAUUM, 0);
    g.C = h->bufA; g.ntiles = lauum_slots(h->nb);
    rc = launch_gemm<INIT_ZERO, EPI_STORE>(h, h->tmU, h->tmU, g);
  }
  if (rc) return rc;
  k_grad_contract<<<h->nb * (h->nb + 1), 128, 0, h->stream>>>(h->spec, h->theta, h->Xw, h->alpha, h->bufA, h->npad, h->n, h->gpart);
  h->launches++;
  CK(h, cudaGetLastError());
  return 0;
}

static int run_finish(dgp_handle h, int want_grad) {
  k_finish<<<h->spec.ntheta + 1, 256, 0, h->stream>>>(h->spec, h->theta, h->gpart, h->nb * (h->nb + 1), h->z, h->alpha,
                                                     h->X, h->n, h->npad, h->scal, want_grad);
  h->launches++;
  CK(h, cudaGetLastError());
  CK(h, cudaMemcpyAsync(h->h_scal, h->scal, SC_SIZE * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  return 0;
}

static int evaluate_enqueue(dgp_handle h, double jitter, int level) {
  int rc;
  CK(h, cudaMemcpyAsync(h->theta, h->h_theta, sizeof(double) * h->spec.ntheta, cudaMemcpyHostToDevice, h->stream));
  if ((rc = run_features(h))) return rc;
  // the O(n^3) phases after the factorisation go to the low-priority stream
  cudaStream_t main_stream = h->stream;
  InvProgress ip;
  memset(&ip, 0, sizeof(ip));
  ip.want_T = (level == 2); ip.W = h->stream_lo;
  // (measured: releasing the merges as the factorisation passes them is a gain at every level up to n = 8192 and for
  // batches; at n = 16384 the long low-priority tiles cost the chain of the last panels as much as they fill, and no level
  // gained there -- above EAGER_INV_MAX_NB block columns the inverse starts after the factorisation)
  PanelHook hook;
  if (level >= 1 && h->nb <= EAGER_INV_MAX_NB) { hook.fn = eager_hook; hook.ctx = &ip; }
  if ((rc = run_potrf(h, jitter, level == 0, hook))) return rc;  // level >= 1: z = U'r after the inverse instead
  if (h->timing) CK(h, cudaEventRecord(h->ev[1], h->stream));
  if (level >= 1) {
    CK(h, cudaEventRecord(h->ev_lo[0], main_stream));
    CK(h, cudaStreamWaitEvent(h->stream_lo, h->ev_lo[0], 0));
    h->stream = h->stream_lo;
    rc = run_trtri(h, ip);
    if (!rc && h->timing) { cudaEventRecord(h->ev[2], h->stream); }
    if (!rc && level == 1) rc = run_lauum_grad(h);
    if (!rc && h->timing) { cudaEventRecord(h->ev[3], h->stream); }
    cudaEventRecord(h->ev_lo[1], h->stream_lo);
    h->stream = main_stream;
    CK(h, cudaStreamWaitEvent(main_stream, h->ev_lo[1], 0));
    if (rc) return rc;
  }
  if ((rc = run_finish(h, level == 1))) return rc;
  return 0;
}

static int evaluate_launch(dgp_handle h, const double* theta, double jitter, int level) {
  // level 0: nlml ; 1: nlml + grad ; 2: factorize for prediction (L, U, alpha, T)
  if (!h) return -1;
  if (!h->have_train) DGP_FAIL(h, -1, "no training data: call dgp_set_train first");
  if (!theta) DGP_FAIL(h, -1, "theta is NULL");
  CK(h, cudaSetDevice(h->device));
  int rc;
  h->factorized = false; h->have_T = false;
  memcpy(h->h_theta, theta, sizeof(double) * h->spec.ntheta);
  if (h->timing) CK(h, cudaEventRecord(h->ev[0], h->stream));
  if ((rc = evaluate_enqueue(h, jitter, level))) return rc;
  if (h->timing) CK(h, cudaEventRecord(h->ev[4], h->stream));
  h->pending = true;
  h->pending_grad = level;
  return 0;
}

static int evaluate_wait(dgp_handle h, double* nlml_out, double* grad_out) {
  if (!h) return -1;
  if (!h->pending) DGP_FAIL(h, -1, "no evaluation in flight");
  CK(h, cudaSetDevice(h->device));
  CK(h, cudaStreamSynchronize(h->stream));
  h->pending = false;
  trace_dump(h);
  const int level = h->pending_grad;
  if (h->timing) {
    float ms;
    for (int i = 0; i < 4; i++) h->last_ms[i] = 0.0;
    cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]); h->last_ms[0] = ms;
    if (level >= 1) {
      cudaEventElapsedTime(&ms, h->ev[1], h->ev[2]); h->last_ms[1] = ms;
      cudaEventElapsedTime(&ms, h->ev[2], h->ev[3]); h->last_ms[2] = ms;
      cudaEventElapsedTime(&ms, h->ev[3], h->ev[4]); h->last_ms[3] = ms;
    } else {
      cudaEventElapsedTime(&ms, h->ev[1], h->ev[4]); h->last_ms[3] = ms;
    }
  }
  if (nlml_out) *nlml_out = h->h_scal[SC_NLML];
  if (grad_out && level == 1) memcpy(grad_out, h->h_scal + SC_GRAD, sizeof(double) * h->spec.ntheta);
  const int info = (int)h->h_scal[SC_INFO];
  h->factorized = (info == 0);
  h->have_T = (info == 0 && level == 2);
  return info;
}

int dgp_nlml(dgp_handle h, const double* theta, double jitter, double* nlml_out) {
  int rc = evaluate_launch(h, theta, jitter, 0);
  if (rc) return rc;
  return evaluate_wait(h, nlml_out, nullptr);
}

int dgp_nlml_grad(dgp_handle h, const double* theta, double jitter, double* nlml_out, double* grad_out) {
  int rc = evaluate_launch(h, theta, jitter, 1);
  if (rc) return rc;
  return evaluate_wait(h, nlml_out, grad_out);
}

int dgp_nlml_grad_launch(dgp_handle h, const double* theta, double jitter) { return evaluate_launch(h, theta, jitter, 1); }
int dgp_nlml_grad_wait(dgp_handle h, double* nlml_out, double* grad_out) { return evaluate_wait(h, nlml_out, grad_out); }
int dgp_nlml_grad_ready(dgp_handle h) {
  if (!h) return -1;
  if (!h->pending) DGP_FAIL(h, -1, "no evaluation in flight");
  CK(h, cudaSetDevice(h->device));
  const cudaError_t e = cudaStreamQuery(h->stream);
  if (e == cudaSuccess) return 1;
  if (e == cudaErrorNotReady) return 0;
  DGP_FAIL(h, -2, "cudaStreamQuery failed: %s", cudaGetErrorString(e));
}

int dgp_factorize(dgp_handle h, const double* theta, double jitter, double* nlml_out) {
  int rc = evaluate_launch(h, theta, jitter, 2);
  if (rc) return rc;
  return evaluate_wait(h, nlml_out, nullptr);
}

// ------------------------------------------------------------------ dense covariance (parity entries)
static int copy_out(dgp_handle h, double* dst, const double* src_dev, size_t rows, size_t cols, size_t ld, int on_device) {
  CK(h, cudaMemcpy2DAsync(dst, cols * 8, src_dev, ld * 8, cols * 8, rows,
                          on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return 0;
}

int dgp_covmat(dgp_handle h, const double* theta, double* K_out, int out_on_device) {
  if (!h) return -1;
  if (!h->have_train || !theta || !K_out) DGP_FAIL(h, -1, "dgp_covmat: bad arguments");
  CK(h, cudaSetDevice(h->device));
  int rc;
  h->factorized = false; h->have_T = false;
  if ((rc = upload_theta(h, theta))) return rc;
  if ((rc = run_features(h))) return rc;
  k_cov_rect<<<dim3(h->npad / 32, h->nb), 256, 0, h->stream>>>(h->spec, h->theta, h->Xw, h->Xw, h->noise, 0.0, h->bufA,
                                                               h->npad, h->n, h->n, 0, 0, nullptr, nullptr, 0);
  h->launches++;
  CK(h, cudaGetLastError());
  return copy_out(h, K_out, h->bufA, h->n, h->n, h->npad, out_on_device);
}

static int stage_xs(dgp_handle h, const double* Xs, int m0, int mc, int on_device) {
  CK(h, cudaMemcpyAsync(h->Xs, Xs + (size_t)m0 * h->spec.ndim, (size_t)mc * h->spec.ndim * 8,
                        on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, h->stream));
  const int mpad = round_up(mc, 128);
  k_features<<<(mpad + 255) / 256, 256, 0, h->stream>>>(h->spec, h->theta, h->Xs, nullptr, h->Xws, nullptr, h->means, mc,
                                                     mpad, nullptr);
  h->launches++;
  CK(h, cudaGetLastError());
  return 0;
}

int dgp_cross_covmat(dgp_handle h, const double* theta, const double* Xs, int m, int xs_on_device, double* K_out,
                     int out_on_device) {
  if (!h) return -1;
  if (!h->have_train || !theta || !Xs || !K_out || m < 1) DGP_FAIL(h, -1, "dgp_cross_covmat: bad arguments");
  CK(h, cudaSetDevice(h->device));
  int rc;
  h->factorized = false; h->have_T = false;
  if ((rc = upload_theta(h, theta))) return rc;
  if ((rc = run_features(h))) return rc;
  for (int m0 = 0; m0 < m; m0 += h->max_m) {
    const int mc = (m - m0 < h->max_m) ? m - m0 : h->max_m;
    if ((rc = stage_xs(h, Xs, m0, mc, xs_on_device))) return rc;
    const int mpad = round_up(mc, 128);
    k_cov_rect<<<dim3(mpad / 32, h->nb), 256, 0, h->stream>>>(h->spec, h->theta, h->Xws, h->Xw, h->noise, 0.0, h->Kx,
                                                             h->npad, mc, h->n, 0, 0, nullptr, nullptr, 0);
    h->launches++;
    CK(h, cudaGetLastError());
    if ((rc = copy_out(h, K_out + (size_t)m0 * h->n, h->Kx, mc, h->n, h->npad, out_on_device))) return rc;
  }
  return 0;
}

// ------------------------------------------------------------------ prediction
int dgp_predict(dgp_handle h, const double* Xs, int m, int on_device, double* mu_out, double* var_out) {
  if (!h) return -1;
  if (!Xs || !mu_out || m < 1) DGP_FAIL(h, -1, "dgp_predict: bad arguments");
  if (!h->factorized || (var_out && !h->have_T))
    DGP_FAIL(h, -1, "dgp_predict: call dgp_factorize first (the mean alone is also available after dgp_nlml_grad)");
  CK(h, cudaSetDevice(h->device));
  int rc;
  const cudaMemcpyKind okind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
  for (int m0 = 0; m0 < m; m0 += h->max_m) {
    const int mc = (m - m0 < h->max_m) ? m - m0 : h->max_m;
    const int mpad = round_up(mc, 128);
    if ((rc = stage_xs(h, Xs, m0, mc, on_device))) return rc;
    // cross covariance chunk (kept for the variance GEMM) fused with the mean partial dot products
    k_cov_rect<<<dim3(mpad / 32, h->nb), 256, 0, h->stream>>>(h->spec, h->theta, h->Xws, h->Xw, h->noise, 0.0, h->Kx,
                                                             h->npad, mc, h->n, 0, 0, h->alpha, h->dot, h->max_m);
    h->launches++;
    CK(h, cudaGetLastError());
    if (var_out) {
      GemmArgs g = base_args(h, M_PREDVAR, 0);
      g.aux0 = mpad / 128; g.aux1 = h->max_m; g.part = h->vpart;
      g.ntiles = (mpad / 128) * 2 * h->nb;
      if ((rc = launch_gemm<INIT_ZERO, EPI_SUMSQ>(h, h->tmKx, h->tmA, g))) return rc;
    }
    k_pred_finish<<<(mc + 255) / 256, 256, 0, h->stream>>>(h->spec, h->theta, h->Xws, h->means, h->dot, h->nb, h->vpart,
                                                          2 * h->nb, h->max_m, mc, h->mu, var_out ? h->var : nullptr);
    h->launches++;
    CK(h, cudaGetLastError());
    CK(h, cudaMemcpyAsync(mu_out + m0, h->mu, (size_t)mc * 8, okind, h->stream));
    if (var_out) CK(h, cudaMemcpyAsync(var_out + m0, h->var, (size_t)mc * 8, okind, h->stream));
    CK(h, cudaStreamSynchronize(h->stream));
  }
  return 0;
}

// ------------------------------------------------------------------ adjoint of the posterior mean
// F = sum_p c_p mu(x*_p) and dF/dtheta at the theta of the last dgp_nlml_grad / dgp_factorize (U = L^-T and alpha
// resident).  Used by the rating-curve monotonicity penalty (src/rating_gp/models/gpytorch.py:126-187), whose value
// is such a functional once the active set is fixed.  m <= the handle's prediction chunk.
int dgp_mean_functional_grad(dgp_handle h, const double* Xs, int m, const double* c, double* val_out, double* grad_out) {
  if (!h) return -1;
  if (!Xs || !c || !grad_out || m < 1) DGP_FAIL(h, -1, "dgp_mean_functional_grad: bad arguments");
  if (m > h->max_m) DGP_FAIL(h, -1, "dgp_mean_functional_grad: m=%d exceeds the prediction chunk %d", m, h->max_m);
  if (!h->factorized || h->pending_grad < 1) DGP_FAIL(h, -1, "dgp_mean_functional_grad: call dgp_nlml_grad or dgp_factorize first");
  CK(h, cudaSetDevice(h->device));
  int rc;
  const int mpad = round_up(m, 128), npad = h->npad, nb = h->nb;
  const size_t nparts = (size_t)(mpad / 128 + nb) * (npad / 64);
  if (h->wpart_count < nparts * DGP_MAX_THETA) DGP_FAIL(h, -1, "dgp_mean_functional_grad: partials workspace too small (internal)");
  cudaStream_t st = h->stream;
  if ((rc = stage_xs(h, Xs, 0, m, 0))) return rc;
  CK(h, cudaMemsetAsync(h->cvec, 0, (size_t)mpad * 8, st));
  CK(h, cudaMemcpyAsync(h->cvec, c, (size_t)m * 8, cudaMemcpyHostToDevice, st));
  k_cov_rect<<<dim3(mpad / 32, nb), 256, 0, st>>>(h->spec, h->theta, h->Xws, h->Xw, h->noise, 0.0, h->Kx, npad, m, h->n,
                                                  0, 0, h->alpha, h->dot, h->max_m);
  k_pred_finish<<<(m + 255) / 256, 256, 0, st>>>(h->spec, h->theta, h->Xws, h->means, h->dot, nb, nullptr, 0, h->max_m, m,
                                                 h->mu, nullptr);
  // gamma = Ky^-1 (Kx*' c) = U (U' v)
  k_colsum_weighted<<<npad / 256 + (npad % 256 ? 1 : 0), 256, 0, st>>>(h->Kx, npad, h->cvec, mpad, h->vvec);
  k_upperT_gemv_part<<<dim3(nb, nb), 256, 0, st>>>(h->bufU, npad, h->vvec, h->zpart, npad);
  k_upperT_gemv_sum<<<(npad + 255) / 256, 256, 0, st>>>(h->zpart, npad, h->tmpz, npad);
  k_upper_gemv<<<npad / 8, 256, 0, st>>>(h->bufU, npad, h->tmpz, h->gam, npad);
  // the two weighted contractions of dK/dtheta
  k_wgrad<<<dim3(npad / 64, mpad / 128), 128, 0, st>>>(h->spec, h->theta, h->Xws, h->Xw, h->cvec, h->alpha, 1.0, h->wpart);
  k_wgrad<<<dim3(npad / 64, nb), 128, 0, st>>>(h->spec, h->theta, h->Xw, h->Xw, h->gam, h->alpha, -1.0,
                                               h->wpart + (size_t)(mpad / 128) * (npad / 64) * DGP_MAX_THETA);
  k_mfg_finish<<<h->spec.ntheta + 1, 256, 0, st>>>(h->spec, h->theta, h->wpart, (int)nparts, h->cvec, h->mu, h->Xs, m, h->gam,
                                                   h->alpha, h->X, h->n, h->mfg_out);
  h->launches += 9;
  CK(h, cudaGetLastError());
  CK(h, cudaMemcpyAsync(h->h_mfg, h->mfg_out, (1 + DGP_MAX_THETA) * sizeof(double), cudaMemcpyDeviceToHost, st));
  CK(h, cudaStreamSynchronize(st));
  if (val_out) *val_out = h->h_mfg[0];
  memcpy(grad_out, h->h_mfg + 1, sizeof(double) * h->spec.ntheta);
  return 0;
}

// ------------------------------------------------------------------ joint posterior samples
// Sigma* = K** - V'V with V = L^-1 Kx* (n x m), Lpost = chol(Sigma* + jitter I), out = mu* + Z Lpost'.
// Work buffers (m-sized) are allocated per call; everything runs on the tile engine:
//   V'  [m, n] = Kx [m, n] T'          (T = L^-1 lower: triangular k range)
//   Sigma* lower tiles = cov tile(x*_i, x*_j) - V'[i, :] V'[j, :]'   (covariance tile generated as accumulator init)
//   Lpost by the same blocked Cholesky as the training factorisation
//   out [S, m] = Z [S, m] Lpost'     (triangular k range) + mu
// bump allocation out of the handle's arena (256-byte granules)
struct ArenaCarver {
  double* base; size_t used = 0;
  explicit ArenaCarver(double* b) : base(b) {}
  double* take(size_t count) { double* p = base ? base + used : nullptr; used += (count + 31) / 32 * 32; return p; }
};
// doubles dgp_sample_ex(m, S, ngroups) carves for a training set padded to npad (nb blocks)
static size_t sample_arena_count(size_t mpad, size_t Spad, size_t npad, size_t nb, size_t S, size_t ngroups) {
  ArenaCarver c(nullptr);
  c.take(mpad * DGP_MAX_COLS); c.take(mpad * DGP_XS); c.take(mpad); c.take(nb * mpad);
  c.take(mpad); c.take(mpad * npad);
  c.take(mpad * mpad); c.take(mpad * 128); c.take(mpad * 128); c.take(Spad * mpad);
  c.take(Spad * mpad);
  c.take(mpad); c.take(SC_SIZE);
  if (ngroups) { c.take(mpad); c.take(S * ngroups); c.take((ngroups + 2) / 2 + 1); }
  return c.used;
}
static size_t dist_arena_count(int m, int S, int world, int rank, size_t nb);  // dgp_dist_begin's (below)
static int ensure_arena(dgp_handle h, size_t count) {
  if (h->arena_count >= count) return 0;
  CK(h, cudaStreamSynchronize(h->stream));
  if (h->arena) cudaFree(h->arena);
  h->arena = nullptr; h->arena_count = 0;
  cudaError_t e = cudaMalloc((void**)&h->arena, count * sizeof(double));
  if (e != cudaSuccess) {
    cudaGetLastError();
    DGP_FAIL(h, -2, "workspace allocation of %.1f GB failed: %s", (double)count * 8e-9, cudaGetErrorString(e));
  }
  h->arena_count = count;
  return 0;
}

int dgp_reserve(dgp_handle h, int max_m_sample, int max_S, int max_groups) {
  if (!h) return -1;
  if (max_m_sample < 0 || max_S < 0 || max_groups < 0) DGP_FAIL(h, -1, "dgp_reserve: bad arguments");
  CK(h, cudaSetDevice(h->device));
  if (max_m_sample == 0) {  // release
    CK(h, cudaStreamSynchronize(h->stream));
    if (h->arena) cudaFree(h->arena);
    h->arena = nullptr; h->arena_count = 0;
    return 0;
  }
  const size_t mpad = round_up(max_m_sample, 128), Spad = round_up(max_S > 0 ? max_S : 1, 128), npad = h->max_pad, nb = npad / 128;
  const size_t a = sample_arena_count(mpad, Spad, npad, nb, (size_t)(max_S > 0 ? max_S : 1), (size_t)max_groups);
  const size_t b = dist_arena_count(max_m_sample, max_S > 0 ? max_S : 1, 1, 0, nb);  // world 1: the slabs of every panel
  return ensure_arena(h, a > b ? a : b);
}

int dgp_sample(dgp_handle h, const double* Xs, int m, const double* Z, int S, double jitter, double* out, int on_device) {
  if (!h) return -1;
  if (!Z) DGP_FAIL(h, -1, "dgp_sample: Z is NULL (use dgp_sample_ex for device-generated normals)");
  return dgp_sample_ex(h, Xs, m, Z, 0ull, S, jitter, nullptr, out, on_device);
}

// the checks dgp_sample_ex and dgp_dist_finish_ex apply to a reduction over an m-point grid
static int check_flux_reduce(dgp_handle h, const dgp_flux_reduce* red, int m, const char* who) {
  if (red->ngroups < 1 || !red->weight || !red->group_start) DGP_FAIL(h, -1, "%s: bad reduction spec", who);
  if (red->group_start[0] < 0 || red->group_start[red->ngroups] > m) DGP_FAIL(h, -1, "%s: group range outside the grid", who);
  for (int g = 0; g < red->ngroups; g++)
    if (red->group_start[g] > red->group_start[g + 1]) DGP_FAIL(h, -1, "%s: group_start must be non-decreasing", who);
  return 0;
}

int dgp_sample_ex(dgp_handle h, const double* Xs, int m, const double* Z, unsigned long long seed, int S, double jitter,
                  const dgp_flux_reduce* red, double* out, int on_device) {
  if (!h) return -1;
  if (!Xs || !out || m < 1 || S < 1) DGP_FAIL(h, -1, "dgp_sample: bad arguments");
  if (red) {
    int rc = check_flux_reduce(h, red, m, "dgp_sample_ex");
    if (rc) return rc;
  }
  if (!h->factorized || !h->have_T) DGP_FAIL(h, -1, "dgp_sample: call dgp_factorize first");
  CK(h, cudaSetDevice(h->device));
  const int mpad = round_up(m, 128), Spad = round_up(S, 128), npad = h->npad, mb = mpad / 128;
  const cudaMemcpyKind ikind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  const cudaMemcpyKind okind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
  // m-sized work buffers, carved out of the handle's arena (dgp_reserve sizes it ahead of time; otherwise it grows here,
  // once, and stays): V' (m x n), Sigma* (m x m, factorised in place), the panel staging buffer and block inverses of that
  // factorisation, Z and the draws.  The cross covariance goes through the handle's prediction chunk, so the footprint is
  // 8 (m n + m^2) B + O(m): 106 GB at m = 100k, n = 32k.
  {
    int rca = ensure_arena(h, sample_arena_count(mpad, Spad, npad, h->nb, S, red ? red->ngroups : 0));
    if (rca) return rca;
  }
  ArenaCarver ar(h->arena);
  double* Xsd = ar.take((size_t)mpad * DGP_MAX_COLS); double* Xws = ar.take((size_t)mpad * DGP_XS); double* means = ar.take(mpad);
  double* dot = ar.take((size_t)h->nb * mpad); double* mu = ar.take(mpad); double* VT = ar.take((size_t)mpad * npad);
  double* Sig = ar.take((size_t)mpad * mpad); double* Pb = ar.take((size_t)mpad * 128); double* DI2 = ar.take((size_t)mpad * 128);
  double* Zd = ar.take((size_t)Spad * mpad); double* Od = ar.take((size_t)Spad * mpad); double* zero = ar.take(mpad);
  double* scal2 = ar.take(SC_SIZE);
  double *wd = nullptr, *gout = nullptr, *gstart = nullptr;
  if (red) { wd = ar.take(mpad); gout = ar.take((size_t)S * red->ngroups); gstart = ar.take((size_t)(red->ngroups + 2) / 2 + 1); }
  int rc;
  CK(h, cudaMemsetAsync(zero, 0, (size_t)mpad * 8, h->stream));
  CK(h, cudaMemsetAsync(scal2, 0, SC_SIZE * 8, h->stream));
  CK(h, cudaMemsetAsync(Zd, 0, (size_t)Spad * mpad * 8, h->stream));
  CK(h, cudaMemsetAsync(Xsd, 0, (size_t)mpad * DGP_MAX_COLS * 8, h->stream));
  CK(h, cudaMemcpyAsync(Xsd, Xs, (size_t)m * h->spec.ndim * 8, ikind, h->stream));
  if (Z != nullptr) {
    CK(h, cudaMemcpy2DAsync(Zd, (size_t)mpad * 8, Z, (size_t)m * 8, (size_t)m * 8, S, ikind, h->stream));
  } else {
    k_fill_normals<<<dim3((m + 255) / 256, S), 256, 0, h->stream>>>(Zd, mpad, m, seed);
    h->launches++;
  }
  k_features<<<(mpad + 255) / 256, 256, 0, h->stream>>>(h->spec, h->theta, Xsd, nullptr, Xws, nullptr, means, m, mpad, nullptr);
  h->launches++;
  CK(h, cudaGetLastError());
  CUtensorMap tVT, tSig, tDI2, tZ;
  if ((rc = make_map(h, &tVT, VT, mpad, npad, npad))) return rc;
  if ((rc = make_map(h, &tSig, Sig, mpad, mpad, mpad))) return rc;
  if ((rc = make_map(h, &tDI2, DI2, mpad, 128, 128))) return rc;
  if ((rc = make_map(h, &tZ, Zd, Spad, mpad, mpad))) return rc;
  // cross covariance (+ posterior-mean partials) and V' = Kx T', one prediction chunk of rows at a time
  for (int m0 = 0; m0 < mpad; m0 += h->max_m) {
    const int mc = (mpad - m0 < h->max_m) ? mpad - m0 : h->max_m;  // multiple of 128
    const int mv = (m - m0 < mc) ? m - m0 : mc;                     // valid rows of the chunk
    k_cov_rect<<<dim3(mc / 32, h->nb), 256, 0, h->stream>>>(h->spec, h->theta, Xws + (size_t)m0 * DGP_XS, h->Xw, h->noise,
                                                           0.0, h->Kx, npad, mv, h->n, 0, 0, h->alpha, dot + m0, mpad);
    h->launches++;
    CK(h, cudaGetLastError());
    GemmArgs g = base_args(h, M_GENERIC, 0);
    g.nb = mc / 128; g.n = mv; g.aux0 = 2 * h->nb; g.aux1 = npad / 16; g.aux2 = 1;
    g.ntiles = (mc / 128) * 2 * h->nb; g.C = VT + (size_t)m0 * npad; g.ldc = npad;
    if ((rc = launch_gemm<INIT_ZERO, EPI_STORE>(h, h->tmKx, h->tmA, g))) return rc;
  }
  k_pred_finish<<<(m + 255) / 256, 256, 0, h->stream>>>(h->spec, h->theta, Xws, means, dot, h->nb, nullptr, 0, mpad, m, mu, nullptr);
  h->launches++;
  CK(h, cudaGetLastError());
  {  // Sigma* = K** + jitter I - V'V  (lower tiles)
    GemmArgs g = base_args(h, M_GENERIC, 0);
    g.nb = mb; g.n = m; g.aux0 = 2 * mb; g.aux1 = npad / 16; g.aux2 = 2;
    g.ntiles = mb * (mb + 1); g.C = Sig; g.ldc = mpad; g.sign = -1.0;
    g.Xw = Xws; g.noise = zero; g.jitter = jitter; g.latent = 1;
    if ((rc = launch_gemm<INIT_COV, EPI_STORE>(h, tVT, tVT, g))) return rc;
  }
  {  // Lpost, in place
    CholBufs b{Sig, Sig, nullptr, DI2, scal2, &tSig, &tSig, &tDI2, mb, mpad, Pb};
    if ((rc = potrf_core(h, b, false, 0.0, false))) return rc;
  }
  {  // out = Z Lpost'
    GemmArgs g = base_args(h, M_GENERIC, 0);
    g.nb = Spad / 128; g.n = S; g.aux0 = 2 * mb; g.aux1 = mpad / 16; g.aux2 = 1;
    g.ntiles = (Spad / 128) * 2 * mb; g.C = Od; g.ldc = mpad;
    if ((rc = launch_gemm<INIT_ZERO, EPI_STORE>(h, tZ, tSig, g))) return rc;
  }
  k_add_rowvec<<<dim3((m + 255) / 256, S), 256, 0, h->stream>>>(Od, mpad, mu, m);
  h->launches++;
  CK(h, cudaGetLastError());
  if (red == nullptr) {
    CK(h, cudaMemcpy2DAsync(out, (size_t)m * 8, Od, (size_t)mpad * 8, (size_t)m * 8, S, okind, h->stream));
  } else {  // annual (grouped) flux of every draw, reduced where the draws are
    CK(h, cudaMemcpyAsync(wd, red->weight, (size_t)m * 8, cudaMemcpyHostToDevice, h->stream));
    CK(h, cudaMemcpyAsync(gstart, red->group_start, (size_t)(red->ngroups + 1) * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    k_flux_reduce<<<dim3(red->ngroups, (S + 7) / 8), 256, 0, h->stream>>>(Od, mpad, wd, (const int*)gstart, red->ngroups, S,
                                                                      red->y_mean, red->y_scale, red->log_transform, gout);
    h->launches++;
    CK(h, cudaGetLastError());
    CK(h, cudaMemcpyAsync(out, gout, (size_t)S * red->ngroups * 8, okind, h->stream));
  }
  CK(h, cudaMemcpyAsync(h->h_scal, scal2, SC_SIZE * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return (int)h->h_scal[SC_INFO];
}

// ------------------------------------------------------------------ distributed joint posterior sampling
// SURVEY 8e: exact joint draws need the Cholesky factor of the m x m posterior covariance.  Across G ranks the block
// columns are dealt out panel-cyclically (panel p -> rank p mod G); every rank holds the training factorisation and
// stores, generates, updates and factors only ITS panels' columns:
//   V'   rows sharded over ranks              -> caller all-gathers V'        (m n^2 / G flop per rank)
//   Sigma* columns of my panels               (m^2 n / G flop per rank)
//   for p: owner factors panel p, packs its sub-diagonal rows -> caller broadcasts -> others unpack
//          every rank applies the rank-(128 pw) update to its own panels right of p        (m^3 / 3G flop per rank)
//   draws: partial Z[:, my columns] L[:, my columns]' -> caller all-reduces, adds the mean
// Storage: one slab per owned panel j of block columns [jb, je): the trailing submatrix Sigma*[jb 128 :, jb 128 : je 128],
// (mb - jb) 128 rows, leading dimension (je - jb) 128, the slabs one after another in the handle's arena -- the lower
// trapezoids of the rank's panels, about 4 mpad^2 / G bytes.  A slab has the same offset on rows and columns, so the
// tile modes of the single-GPU factorisation run on it unchanged in slab coordinates (block indices minus jb); every
// operand that lives in a larger buffer (V', Z, another panel) gets a tensor map based at the matching offset into it.  A
// received panel p goes to receive slot p mod 2, indexed by global row, so that the maps of a slot serve all its panels.
// The caller (multisite.sample_sharded: torch.distributed over NCCL) owns the exchanged buffers and the collectives;
// this side is the per-rank kernels, all on the handle's stream.
struct dgp_dist_s {
  dgp_handle h = nullptr;
  int m = 0, mpad = 0, mb = 0, S = 0, Spad = 0, pw = 0, npanels = 0, rank = 0, world = 1;
  double jitter = 0.0;
  double *VT = nullptr, *Od = nullptr, *mu = nullptr;  // caller-owned device buffers
  int vt_rows = 0;                                      // rows of VT (world rows_per_rank)
  double *Xsd = nullptr, *Xws = nullptr, *means = nullptr, *dot = nullptr, *zero = nullptr, *scal2 = nullptr;
  double *Pb = nullptr, *DI2 = nullptr, *Zd = nullptr;  // from Pb on, nothing is read after the partial draws
  double* slot[2] = {nullptr, nullptr};                 // received panels: row = global row, leading dimension pw 128
  std::vector<double*> slab;                            // slab of owned panel p: slab[p / world]
  CUtensorMap tDI2;
  std::map<std::tuple<const double*, int, int, long long>, CUtensorMap> maps;  // (base, rows, cols, ld) -> map
  bool mine(int p) const { return p % world == rank; }
  int pbeg(int p) const { return p * pw; }
  int pend(int p) const { return (p * pw + pw < mb) ? p * pw + pw : mb; }
  // tensor map of the rows x cols matrix at `base`: encoded on first use, then reused (a world-1 run at m = 100 000 makes
  // about 19 000 trailing launches)
  int map(const double* base, int rows, int cols, long long ld, const CUtensorMap** out) {
    const auto key = std::make_tuple(base, rows, cols, ld);
    auto it = maps.find(key);
    if (it == maps.end()) {
      CUtensorMap tm;
      int rc = make_map(h, &tm, const_cast<double*>(base), rows, cols, ld);
      if (rc) return rc;
      it = maps.emplace(key, tm).first;
    }
    *out = &it->second;
    return 0;
  }
};

static void dist_geometry(dgp_dist_s* d, int m, int S, int world, int rank) {
  d->m = m; d->mpad = round_up(m, 128); d->mb = d->mpad / 128; d->S = S; d->Spad = round_up(S, 128);
  d->pw = PANEL_BLOCKS; d->npanels = (d->mb + d->pw - 1) / d->pw; d->rank = rank; d->world = world;
}

// carve d's buffers out of `base` (nullptr: count only) -> doubles used.  The slabs come last: everything before them is
// the same on every rank.
static size_t dist_carve(dgp_dist_s* d, double* base, size_t nb) {
  ArenaCarver ar(base);
  const size_t mpad = d->mpad, pcols = (size_t)d->pw * 128;
  d->Xsd = ar.take(mpad * DGP_MAX_COLS); d->Xws = ar.take(mpad * DGP_XS); d->means = ar.take(mpad); d->dot = ar.take(nb * mpad);
  d->zero = ar.take(mpad); d->scal2 = ar.take(SC_SIZE);
  d->Pb = ar.take(mpad * 128); d->DI2 = ar.take(pcols * 128); d->Zd = ar.take((size_t)d->Spad * mpad);
  for (int k = 0; k < 2; k++) d->slot[k] = ar.take(mpad * pcols);
  d->slab.clear();
  for (int p = d->rank; p < d->npanels; p += d->world)
    d->slab.push_back(ar.take((size_t)(d->mb - d->pbeg(p)) * 128 * (size_t)(d->pend(p) - d->pbeg(p)) * 128));
  return ar.used;
}

static size_t dist_arena_count(int m, int S, int world, int rank, size_t nb) {
  dgp_dist_s d;
  dist_geometry(&d, m, S, world, rank);
  return dist_carve(&d, nullptr, nb);
}

size_t dgp_dist_arena_bytes(dgp_handle h, int m, int S, int world, int rank) {
  if (!h || m < 1 || S < 1 || world < 1 || rank < 0 || rank >= world || !h->have_train) return 0;
  return dist_arena_count(m, S, world, rank, h->nb) * sizeof(double);
}

int dgp_dist_dims(dgp_handle h, int m, int S, int world, long long* dims) {
  if (!h || !dims || m < 1 || S < 1 || world < 1) return -1;
  if (!h->have_train) DGP_FAIL(h, -1, "dgp_dist_dims: no training data");
  const long long mpad = round_up(m, 128), mb = mpad / 128;
  const long long rows_per_rank = ((mb + world - 1) / world) * 128;
  dims[0] = mpad; dims[1] = h->npad; dims[2] = round_up(S, 128); dims[3] = (long long)PANEL_BLOCKS * 128;
  dims[4] = (mb + PANEL_BLOCKS - 1) / PANEL_BLOCKS; dims[5] = rows_per_rank;
  return 0;
}

int dgp_dist_begin(dgp_handle h, const double* Xs, int m, int S, const double* Z, unsigned long long seed, double jitter,
                   int rank, int world, double* VT, double* Od, double* mu, dgp_dist* out) {
  if (!h) return -1;
  if (!Xs || !VT || !Od || !mu || !out || m < 1 || S < 1 || world < 1 || rank < 0 || rank >= world)
    DGP_FAIL(h, -1, "dgp_dist_begin: bad arguments");
  if (!h->factorized || !h->have_T) DGP_FAIL(h, -1, "dgp_dist_begin: call dgp_factorize first");
  CK(h, cudaSetDevice(h->device));
  dgp_dist d = new dgp_dist_s();
  d->h = h; d->jitter = jitter;
  dist_geometry(d, m, S, world, rank);
  d->VT = VT; d->Od = Od; d->mu = mu;
  const size_t mpad = d->mpad;
  {
    int rca = ensure_arena(h, dist_carve(d, nullptr, h->nb));
    if (rca) { delete d; return rca; }
  }
  dist_carve(d, h->arena, h->nb);
  cudaStream_t st = h->stream;
  int rc;
  CK(h, cudaMemsetAsync(d->zero, 0, mpad * 8, st));
  CK(h, cudaMemsetAsync(d->scal2, 0, SC_SIZE * 8, st));
  CK(h, cudaMemsetAsync(d->Zd, 0, (size_t)d->Spad * mpad * 8, st));
  CK(h, cudaMemsetAsync(d->Od, 0, (size_t)d->Spad * mpad * 8, st));
  CK(h, cudaMemsetAsync(d->mu, 0, mpad * 8, st));
  CK(h, cudaMemsetAsync(d->Xsd, 0, mpad * DGP_MAX_COLS * 8, st));
  CK(h, cudaMemcpyAsync(d->Xsd, Xs, (size_t)m * h->spec.ndim * 8, cudaMemcpyHostToDevice, st));
  if (Z != nullptr) CK(h, cudaMemcpy2DAsync(d->Zd, mpad * 8, Z, (size_t)m * 8, (size_t)m * 8, S, cudaMemcpyHostToDevice, st));
  else k_fill_normals<<<dim3((m + 255) / 256, S), 256, 0, st>>>(d->Zd, mpad, m, seed);
  k_features<<<(d->mpad + 255) / 256, 256, 0, st>>>(h->spec, h->theta, d->Xsd, nullptr, d->Xws, nullptr, d->means, m, d->mpad, nullptr);
  h->launches += 2;
  CK(h, cudaGetLastError());
  long long dims[6];
  dgp_dist_dims(h, m, S, world, dims);
  d->vt_rows = (int)(dims[5] * world);
  if ((rc = make_map(h, &d->tDI2, d->DI2, d->pw * 128, 128, 128))) { dgp_dist_end(d); return rc; }
  *out = d;
  return 0;
}

int dgp_dist_end(dgp_dist d) {
  if (!d) return 0;
  if (d->h) { cudaSetDevice(d->h->device); cudaStreamSynchronize(d->h->stream); }
  delete d;  // its buffers live in the handle's arena
  return 0;
}

// rows [row0, row1) (multiples of 128) of V' = Kx T' and of the posterior mean.  Both ends are clamped to mpad first: a
// shard of rows_per_rank rows lies wholly past mpad when world is large for mb (world 3, mb 1: rank 2 gets [256, 384)),
// and such a range is an empty shard, not an error.
int dgp_dist_vt_rows(dgp_dist d, int row0, int row1) {
  if (!d) return -1;
  dgp_handle h = d->h;
  if (row0 < 0 || row0 % 128 || row1 % 128) DGP_FAIL(h, -1, "dgp_dist_vt_rows: bad row range");
  if (row0 > d->mpad) row0 = d->mpad;
  if (row1 > d->mpad) row1 = d->mpad;
  if (row1 < row0) DGP_FAIL(h, -1, "dgp_dist_vt_rows: bad row range");
  CK(h, cudaSetDevice(h->device));
  int rc;
  const int npad = h->npad;
  for (int m0 = row0; m0 < row1; m0 += h->max_m) {
    const int mc = (row1 - m0 < h->max_m) ? row1 - m0 : h->max_m;
    const int mv = (d->m - m0 < mc) ? (d->m - m0 > 0 ? d->m - m0 : 0) : mc;
    k_cov_rect<<<dim3(mc / 32, h->nb), 256, 0, h->stream>>>(h->spec, h->theta, d->Xws + (size_t)m0 * DGP_XS, h->Xw, h->noise,
                                                           0.0, h->Kx, npad, mv, h->n, 0, 0, h->alpha, d->dot + m0, d->mpad);
    h->launches++;
    CK(h, cudaGetLastError());
    GemmArgs g = base_args(h, M_GENERIC, 0);
    g.nb = mc / 128; g.n = mv; g.aux0 = 2 * h->nb; g.aux1 = npad / 16; g.aux2 = 1;
    g.ntiles = (mc / 128) * 2 * h->nb; g.C = d->VT + (size_t)m0 * npad; g.ldc = npad;
    if ((rc = launch_gemm<INIT_ZERO, EPI_STORE>(h, h->tmKx, h->tmA, g))) return rc;
  }
  if (row1 > row0) {
    const int cnt = ((d->m < row1) ? d->m : row1) - row0;
    if (cnt > 0) {
      k_pred_finish<<<(cnt + 255) / 256, 256, 0, h->stream>>>(h->spec, h->theta, d->Xws + (size_t)row0 * DGP_XS, d->means + row0,
                                                             d->dot + row0, h->nb, nullptr, 0, d->mpad, cnt, d->mu + row0, nullptr);
      h->launches++;
      CK(h, cudaGetLastError());
    }
  }
  return 0;
}

// Sigma* = K** + jitter I - V'V on the slabs of this rank's panels (needs the complete V').  In slab coordinates: V' from
// row jb 128 on, the features from point jb 128 on and n = m - jb 128, so the diagonal, the jitter and the identity
// padding land where they are in the full matrix.
int dgp_dist_sigma(dgp_dist d) {
  if (!d) return -1;
  dgp_handle h = d->h;
  CK(h, cudaSetDevice(h->device));
  int rc;
  for (size_t k = 0; k < d->slab.size(); k++) {
    const int p = d->rank + (int)k * d->world, jb = d->pbeg(p), w = d->pend(p) - jb, r0 = jb * 128;
    const CUtensorMap* tv;
    if ((rc = d->map(d->VT + (size_t)r0 * h->npad, d->vt_rows - r0, h->npad, h->npad, &tv))) return rc;
    GemmArgs g = base_args(h, M_TRAIL_COL, 0);
    g.nb = d->mb - jb; g.n = d->m - r0; g.ldc = (long long)w * 128;
    g.aux0 = 0 | (w << 16); g.aux1 = h->npad / 128; g.aux2 = 0;
    g.C = d->slab[k]; g.ntiles = (d->mb - jb) * 2 * w; g.sign = -1.0;
    g.Xw = d->Xws + (size_t)r0 * DGP_XS; g.noise = d->zero; g.jitter = d->jitter; g.latent = 1;
    if ((rc = launch_gemm<INIT_COV, EPI_STORE>(h, *tv, *tv, g))) return rc;
  }
  return 0;
}

// owner of panel p: factor it in place and pack the rows below its diagonal blocks into `pack` for the broadcast.
// stream: where to run (NULL: the handle's stream) -- a high-priority side stream lets the factorisation of the next
// panel overlap this rank's trailing updates (look-ahead); the caller orders the streams with events.
int dgp_dist_panel_factor(dgp_dist d, int p, double* pack, void* stream) {
  if (!d) return -1;
  dgp_handle h = d->h;
  if (!pack || p < 0 || p >= d->npanels || !d->mine(p)) DGP_FAIL(h, -1, "dgp_dist_panel_factor: panel %d is not owned by rank %d", p, d->rank);
  CK(h, cudaSetDevice(h->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
  const int pb = d->pbeg(p), w = d->pend(p) - pb, nbl = d->mb - pb;
  const long long ld = (long long)w * 128;
  double* sl = d->slab[p / d->world];
  const CUtensorMap* ts;
  int rc = d->map(sl, nbl * 128, w * 128, ld, &ts);
  if (rc) return rc;
  CholBufs b{sl, sl, nullptr, d->DI2, d->scal2, ts, ts, &d->tDI2, nbl, ld, d->Pb};
  if ((rc = factor_panel(h, b, 0, w, false, 0.0, false, st, nullptr, pb * 128))) return rc;
  const long long rows = (long long)(nbl - w) * 128;
  if (rows > 0) {
    k_pack_panel<<<(unsigned)(rows / 8), 256, 0, st>>>(sl, ld, ld, 0, w * 128, pack, 0);
    h->launches++;
    CK(h, cudaGetLastError());
  }
  return 0;
}

// other ranks: copy the received panel (rows below its diagonal blocks) into receive slot p mod 2.  The handle's stream
// orders the slot's reuse (by panel p + 2) behind the trailing updates with panel p.
int dgp_dist_panel_unpack(dgp_dist d, int p, double* pack) {
  if (!d) return -1;
  dgp_handle h = d->h;
  if (!pack || p < 0 || p >= d->npanels) DGP_FAIL(h, -1, "dgp_dist_panel_unpack: bad panel");
  CK(h, cudaSetDevice(h->device));
  const int pb = d->pbeg(p), pe = d->pend(p);
  const long long rows = (long long)(d->mb - pe) * 128;
  if (rows > 0) {
    k_pack_panel<<<(unsigned)(rows / 8), 256, 0, h->stream>>>(d->slot[p & 1], (long long)d->pw * 128, (long long)pe * 128, 0,
                                                              (pe - pb) * 128, pack, 1);
    h->launches++;
    CK(h, cudaGetLastError());
  }
  return 0;
}

// rank-(128 pw) update, with panel p, of this rank's panels j in [j_first, j_last].  Panel p's rows from jb 128 on (its
// own slab on the owner, the receive slot elsewhere) are the operand, behind a map based at that row; the update is the
// single-GPU factorisation's, on slab j at o = 0 with step 0.
int dgp_dist_trail(dgp_dist d, int p, int j_first, int j_last) {
  if (!d) return -1;
  dgp_handle h = d->h;
  if (p < 0 || p >= d->npanels) DGP_FAIL(h, -1, "dgp_dist_trail: bad panel");
  CK(h, cudaSetDevice(h->device));
  const int pb = d->pbeg(p), wp = d->pend(p) - pb;
  int rc;
  if (j_first < p + 1) j_first = p + 1;
  if (j_last > d->npanels - 1) j_last = d->npanels - 1;
  for (int j = j_first; j <= j_last; j++) {
    if (!d->mine(j)) continue;
    const int jb = d->pbeg(j), wj = d->pend(j) - jb, nbl = d->mb - jb;
    const double* src;
    long long ld;
    if (d->mine(p)) { ld = (long long)wp * 128; src = d->slab[p / d->world] + (size_t)(jb - pb) * 128 * ld; }
    else { ld = (long long)d->pw * 128; src = d->slot[p & 1] + (size_t)jb * 128 * ld; }
    const CUtensorMap* tp;
    if ((rc = d->map(src, nbl * 128, wp * 128, ld, &tp))) return rc;
    CholBufs b{d->slab[j / d->world], nullptr, nullptr, nullptr, nullptr, nullptr, tp, nullptr, nbl, (long long)wj * 128};
    if ((rc = launch_trail(h, b, 0, wp, 0, wj, nbl * 2 * wj, false, 0.0, h->stream))) return rc;
  }
  return 0;
}

// Od += Z[:, my columns] L[:, my columns]'   (partial sums of the draws; the caller all-reduces Od).  Panel p in slab
// coordinates: Z from column pb 128 on, the draws' columns from pb 128 on.
int dgp_dist_draws_partial(dgp_dist d) {
  if (!d) return -1;
  dgp_handle h = d->h;
  CK(h, cudaSetDevice(h->device));
  int rc;
  for (size_t k = 0; k < d->slab.size(); k++) {
    const int p = d->rank + (int)k * d->world, pb = d->pbeg(p), w = d->pend(p) - pb, nbl = d->mb - pb;
    const CUtensorMap *tz, *ts;
    if ((rc = d->map(d->Zd + (size_t)pb * 128, d->Spad, d->mpad - pb * 128, d->mpad, &tz))) return rc;
    if ((rc = d->map(d->slab[k], nbl * 128, w * 128, (long long)w * 128, &ts))) return rc;
    GemmArgs g = base_args(h, M_ZL, 0);
    g.nb = nbl; g.n = d->S; g.aux1 = w;
    g.ntiles = (d->Spad / 128) * 2 * nbl; g.C = d->Od + (size_t)pb * 128; g.ldc = d->mpad;
    if ((rc = launch_gemm<INIT_LOAD, EPI_STORE>(h, *tz, *ts, g))) return rc;
  }
  return 0;
}

// after the all-reduce of Od and of mu: Od + mu, then out[S, m] = the draws, or (red) out[S, ngroups] = their grouped
// flux sums (k_flux_reduce, as dgp_sample_ex); returns the LAPACK-style info of THIS rank's panels
int dgp_dist_finish_ex(dgp_dist d, const dgp_flux_reduce* red, double* out) {
  if (!d) return -1;
  dgp_handle h = d->h;
  if (!out) DGP_FAIL(h, -1, "dgp_dist_finish: out is NULL");
  if (red) {
    int rc = check_flux_reduce(h, red, d->m, "dgp_dist_finish_ex");
    if (rc) return rc;
  }
  CK(h, cudaSetDevice(h->device));
  k_add_rowvec<<<dim3((d->m + 255) / 256, d->S), 256, 0, h->stream>>>(d->Od, d->mpad, d->mu, d->m);
  h->launches++;
  CK(h, cudaGetLastError());
  if (red == nullptr) {
    CK(h, cudaMemcpy2DAsync(out, (size_t)d->m * 8, d->Od, (size_t)d->mpad * 8, (size_t)d->m * 8, d->S, cudaMemcpyDeviceToHost, h->stream));
  } else {
    // the reduction's buffers take the place of the panel staging, Z, the receive slots and the slabs, which nothing
    // reads any more
    ArenaCarver ar(d->Pb);
    double* wd = ar.take(d->mpad);
    double* gstart = ar.take((size_t)(red->ngroups + 2) / 2 + 1);
    double* gout = ar.take((size_t)d->S * red->ngroups);
    if ((size_t)(d->Pb - h->arena) + ar.used > h->arena_count)
      DGP_FAIL(h, -1, "dgp_dist_finish_ex: %d groups of %d draws do not fit the workspace", red->ngroups, d->S);
    CK(h, cudaMemcpyAsync(wd, red->weight, (size_t)d->m * 8, cudaMemcpyHostToDevice, h->stream));
    CK(h, cudaMemcpyAsync(gstart, red->group_start, (size_t)(red->ngroups + 1) * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    k_flux_reduce<<<dim3(red->ngroups, (d->S + 7) / 8), 256, 0, h->stream>>>(d->Od, d->mpad, wd, (const int*)gstart, red->ngroups,
                                                                            d->S, red->y_mean, red->y_scale, red->log_transform, gout);
    h->launches++;
    CK(h, cudaGetLastError());
    CK(h, cudaMemcpyAsync(out, gout, (size_t)d->S * red->ngroups * 8, cudaMemcpyDeviceToHost, h->stream));
  }
  CK(h, cudaMemcpyAsync(h->h_scal, d->scal2, SC_SIZE * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return (int)h->h_scal[SC_INFO];
}

int dgp_dist_finish(dgp_dist d, double* out) { return dgp_dist_finish_ex(d, nullptr, out); }

// ------------------------------------------------------------------ generic NT product on the tile engine
int dgp_gemm_nt(dgp_handle h, const double* A, long long lda, const double* B, long long ldb, double* Cm, long long ldc,
                int M, int N, int K, int mode) {
  if (!h) return -1;
  if (!A || !B || !Cm || M < 128 || N < 64 || K < 16 || M % 128 || N % 64 || K % 16 || lda % 2 || ldb % 2 || ldc % 2)
    DGP_FAIL(h, -1, "dgp_gemm_nt: M %% 128, N %% 64, K %% 16 and even leading dimensions required");
  if (mode < -1 || mode > 1) DGP_FAIL(h, -1, "dgp_gemm_nt: mode must be -1, 0 or 1");
  CK(h, cudaSetDevice(h->device));
  CUtensorMap ta, tb;
  int rc;
  if ((rc = make_map(h, &ta, const_cast<double*>(A), M, K, lda))) return rc;
  if ((rc = make_map(h, &tb, const_cast<double*>(B), N, K, ldb))) return rc;
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.mode = M_GENERIC; g.nb = M / 128; g.n = M;
  g.aux0 = N / 64; g.aux1 = K / 16; g.aux2 = 0;
  g.ntiles = (M / 128) * (N / 64);
  g.C = Cm; g.ldc = ldc; g.sign = (mode == -1) ? -1.0 : 1.0;
  if (mode == 0) rc = launch_gemm<INIT_ZERO, EPI_STORE>(h, ta, tb, g);
  else rc = launch_gemm<INIT_LOAD, EPI_STORE>(h, ta, tb, g);
  if (rc) return rc;
  CK(h, cudaStreamSynchronize(h->stream));
  return 0;
}

// ------------------------------------------------------------------ accessors
int dgp_get_alpha(dgp_handle h, double* alpha_out, int out_on_device) {
  if (!h) return -1;
  if (!h->factorized || !alpha_out) DGP_FAIL(h, -1, "dgp_get_alpha: no factorisation (needs dgp_nlml_grad or dgp_factorize)");
  CK(h, cudaSetDevice(h->device));
  CK(h, cudaMemcpyAsync(alpha_out, h->alpha, (size_t)h->n * 8, out_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, h->stream));
  CK(h, cudaStreamSynchronize(h->stream));
  return 0;
}

int dgp_get_chol(dgp_handle h, double* L_out, int out_on_device) {
  if (!h) return -1;
  if (!h->factorized || !L_out) DGP_FAIL(h, -1, "dgp_get_chol: no factorisation");
  CK(h, cudaSetDevice(h->device));
  return copy_out(h, L_out, h->bufL, h->n, h->n, h->npad, out_on_device);
}

int dgp_set_debug_kinv(dgp_handle h, int enable) { if (!h) return -1; h->debug_kinv = enable != 0; return 0; }

int dgp_get_kinv(dgp_handle h, double* Kinv_out, int out_on_device) {
  if (!h) return -1;
  if (!h->factorized || !h->debug_kinv || h->pending_grad != 1 || !Kinv_out)
    DGP_FAIL(h, -1, "dgp_get_kinv: needs dgp_set_debug_kinv(1) + dgp_nlml_grad");
  CK(h, cudaSetDevice(h->device));
  return copy_out(h, Kinv_out, h->bufA, h->n, h->n, h->npad, out_on_device);
}

int dgp_get_uinv(dgp_handle h, double* U_out, int out_on_device) {
  if (!h) return -1;
  if (!h->factorized || h->pending_grad < 1 || !U_out)
    DGP_FAIL(h, -1, "dgp_get_uinv: needs a successful dgp_nlml_grad or dgp_factorize");
  CK(h, cudaSetDevice(h->device));
  return copy_out(h, U_out, h->bufU, h->n, h->n, h->npad, out_on_device);
}

// T = L^-1 sits in the lower triangle of bufA after dgp_factorize (the last merge level is transposed there too); the upper
// triangle holds the inverse's scratch, which the copy replaces with zeros
int dgp_get_linv(dgp_handle h, double* T_out, int out_on_device) {
  if (!h) return -1;
  if (!h->have_T || !T_out) DGP_FAIL(h, -1, "dgp_get_linv: needs a successful dgp_factorize (dgp_nlml* leave Ky^-1 there)");
  CK(h, cudaSetDevice(h->device));
  int rc = copy_out(h, T_out, h->bufA, h->n, h->n, h->npad, out_on_device);
  if (rc) return rc;
  const int n = h->n;
  if (out_on_device) {
    k_zero_strict_upper<<<n, 256, 0, h->stream>>>(T_out, n, n);
    h->launches++;
    CK(h, cudaGetLastError());
    CK(h, cudaStreamSynchronize(h->stream));
  } else {
    for (int i = 0; i + 1 < n; i++) memset(T_out + (size_t)i * n + i + 1, 0, (size_t)(n - i - 1) * 8);
  }
  return 0;
}

long long dgp_launch_count(dgp_handle h) { return h ? h->launches : 0; }
int dgp_set_timing(dgp_handle h, int enable) { if (!h) return -1; h->timing = enable != 0; return 0; }
int dgp_last_timing(dgp_handle h, double* ms4) {
  if (!h || !ms4) return -1;
  for (int i = 0; i < 4; i++) ms4[i] = h->last_ms[i];
  return 0;
}

}  // extern "C"

#include "dgp_batch.cuh"
