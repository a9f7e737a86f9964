// Latency-bound and memory-bound companions of the DMMA tile engine: diagonal-block factorisation
// (with the triangular inverse produced by the same elimination), feature-table / residual
// preparation, covariance panels and rectangles, blocked forward substitution, triangular GEMV,
// transposition and the deterministic final reductions.
#pragma once
#include "dgp_cov.cuh"

namespace dgp {

// device scalar block written by the kernels below and copied back to the host
enum { SC_LOGDET = 0, SC_INFO = 1, SC_QUAD = 2, SC_NLML = 3, SC_GRAD = 8 };  // grad at [SC_GRAD, SC_GRAD + ntheta)
constexpr int SC_SIZE = SC_GRAD + DGP_MAX_THETA;

// ------------------------------------------------------------------ features, residual, scalars
// Xw[i] = feature row of point i (copy / log-warp / gate columns, src/rating_gp/models/kernels.py:307-382),
// mean[i] = m(x_i) (ConstantMean, or PowerLawTransform src/rating_gp/models/gpytorch.py:28-40),
// r[i] = y[i] - mean[i] when y != nullptr.  Rows >= n are zero.
__device__ __forceinline__ void features_body(const dgp_spec& spec, const double* __restrict__ theta,
                                              const double* __restrict__ X, const double* __restrict__ y, double* __restrict__ Xw,
                                              double* __restrict__ r, double* __restrict__ mean_out, int n, int npad,
                                              double* __restrict__ scal, int i) {
  if (scal != nullptr && i < SC_SIZE) scal[i] = 0.0;
  if (i >= npad) return;
  double row[DGP_XS];
#pragma unroll
  for (int c = 0; c < DGP_XS; c++) row[c] = 0.0;
  double m = 0.0;
  if (i < n) {
    const double* x = X + (size_t)i * spec.ndim;
    for (int c = 0; c < spec.ncols; c++) {
      const dgp_col& sc = spec.col[c];
      const double v = (sc.kind >= DGP_COL_SINP) ? 0.0 : x[sc.src];
      if (sc.kind == DGP_COL_SINP) { row[c] = sinpi(row[sc.src] / theta[sc.theta]); continue; }  // src: feature column
      if (sc.kind == DGP_COL_COSP) { row[c] = cospi(row[sc.src] / theta[sc.theta]); continue; }
      if (sc.kind == DGP_COL_COPY) row[c] = v;
      else if (sc.kind == DGP_COL_LOG) row[c] = log(v + sc.aux);
      else row[c] = 1.0 / (1.0 + exp(sc.aux * (v - theta[sc.theta])));
    }
    if (spec.mean_kind == DGP_MEAN_CONST) m = theta[spec.mean_theta[0]];
    else if (spec.mean_kind == DGP_MEAN_POWERLAW)
      m = theta[spec.mean_theta[0]] + theta[spec.mean_theta[1]] * log(x[spec.mean_col] - theta[spec.mean_theta[2]]);
  }
#pragma unroll
  for (int c = 0; c < DGP_XS; c++) Xw[(size_t)i * DGP_XS + c] = row[c];
  if (mean_out != nullptr) mean_out[i] = m;
  if (r != nullptr) r[i] = (i < n && y != nullptr) ? y[i] - m : 0.0;
}

__global__ void k_features(const __grid_constant__ dgp_spec spec, const double* __restrict__ theta,
                           const double* __restrict__ X, const double* __restrict__ y, double* __restrict__ Xw,
                           double* __restrict__ r, double* __restrict__ mean_out, int n, int npad,
                           double* __restrict__ scal) {
  features_body(spec, theta, X, y, Xw, r, mean_out, n, npad, scal, blockIdx.x * blockDim.x + threadIdx.x);
}

// ------------------------------------------------------------------ batched companions (dgp_batch_*)
// Per-site sizes of a batch.  Per-site arrays are slabs indexed by the site: matrices [site][ld][ld], per-point vectors
// [site][ld], feature tables [site][ld][DGP_XS], inputs [site][ld][DGP_MAX_COLS], theta [site][DGP_MAX_THETA],
// scalar blocks [site][SC_SIZE].  The kernels below are the single-site bodies with the site taken from the grid.
struct SiteDims {
  int count, nbmax;
  long long ld;
  int n[DGP_BATCH_MAX], nb[DGP_BATCH_MAX];
  int tile0[DGP_BATCH_MAX + 1];   // prefix of nb (nb + 1) lower 128 x 64 tiles per site (gradient contraction)
};

// grid = (ceil(ld / 256), sites)
__global__ void k_features_b(const __grid_constant__ dgp_spec spec, const __grid_constant__ SiteDims sd,
                             const double* __restrict__ theta, const double* __restrict__ X, const double* __restrict__ y,
                             double* __restrict__ Xw, double* __restrict__ r, double* __restrict__ scal) {
  const int st = blockIdx.y;
  const size_t v = (size_t)st * sd.ld;
  features_body(spec, theta + st * DGP_MAX_THETA, X + v * DGP_MAX_COLS, y + v, Xw + v * DGP_XS, r + v, nullptr, sd.n[st],
                sd.nb[st] * 128, scal + (size_t)st * SC_SIZE, blockIdx.x * blockDim.x + threadIdx.x);
}

// ------------------------------------------------------------------ covariance rectangle
// out[i, j] = k(xa_i, xb_j) (+ noise on the global diagonal when `diag_noise`), i < ra_pad, j in this
// CTA's 128-column block.  Entries outside (na, nb_) are identity padding when `ident_pad`, else 0.
// Optionally accumulates dot[cblock][i] = sum_j out[i, j] * vec[j] (posterior mean partials).
// grid = (ra_pad / 32, ncol_blocks), block = 256 threads, each thread 16 entries.
__device__ __forceinline__ void cov_rect_body(const dgp_spec& spec, const double* __restrict__ theta,
           const double* __restrict__ XwA, const double* __restrict__ XwB, const double* __restrict__ noise,
           double jitter, double* __restrict__ out, long long ld, int na, int nb_, int diag_noise, int ident_pad,
           const double* __restrict__ vec, double* __restrict__ dot, int dot_ld, int bx, int by) {
  __shared__ CovC cc;
  __shared__ double xa[32 * DGP_XS];    // row points, row-major (broadcast side)
  __shared__ double xbT[DGP_XS * 128];  // column points, column-major (per-thread side)
  __shared__ double red[32][9];
  const int t = threadIdx.x;
  const int r0 = bx * 32, c0 = by * 128;
  cov_compile(&cc, spec, theta, jitter, t, 256);
  for (int e = t; e < 32 * DGP_XS; e += 256) xa[e] = XwA[(size_t)r0 * DGP_XS + e];
  for (int e = t; e < 128 * DGP_XS; e += 256) xbT[(e % DGP_XS) * 128 + e / DGP_XS] = XwB[(size_t)c0 * DGP_XS + e];
  __syncthreads();
  const int lc = t & 127, half = t >> 7;  // thread: column lc, rows half*16 .. +16 (the same rows for the whole warp)
  const int gc = c0 + lc;
  const double vj = (vec != nullptr) ? vec[gc] : 0.0;
#pragma unroll 1
  for (int rr0 = 0; rr0 < 16; rr0 += 8) {
    double val[8];
    cov_vals<8>(&cc, xbT, 128, lc, xa + (half * 16 + rr0) * DGP_XS, val);
#pragma unroll
    for (int u = 0; u < 8; u++) {
      const int lr = half * 16 + rr0 + u, gr = r0 + lr;
      double v = val[u];
      if (gr < na && gc < nb_) {
        if (diag_noise && gr == gc) v += noise[gr] + cc.extra_noise;
      } else {
        v = (ident_pad && gr == gc) ? 1.0 : 0.0;
      }
      if (out != nullptr) out[(size_t)gr * ld + gc] = v;
      if (dot != nullptr) {
        double s = v * vj;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if ((t & 31) == 0) red[lr][(t >> 5) & 3] = s;
      }
    }
  }
  if (dot != nullptr) {
    __syncthreads();
    if (t < 32) dot[(size_t)by * dot_ld + r0 + t] = (red[t][0] + red[t][1]) + (red[t][2] + red[t][3]);
  }
}

__global__ void __launch_bounds__(256)
k_cov_rect(const __grid_constant__ dgp_spec spec, const double* __restrict__ theta,
           const double* __restrict__ XwA, const double* __restrict__ XwB, const double* __restrict__ noise,
           double jitter, double* __restrict__ out, long long ld, int na, int nb_, int diag_noise, int ident_pad,
           const double* __restrict__ vec, double* __restrict__ dot, int dot_ld) {
  cov_rect_body(spec, theta, XwA, XwB, noise, jitter, out, ld, na, nb_, diag_noise, ident_pad, vec, dot, dot_ld, blockIdx.x,
                blockIdx.y);
}

// Matrices of more than this many block columns are written by the standalone generator ahead of the factorisation
// (both engines: which kernel generates a tile decides how its first update rounds).
constexpr int DGP_PREGEN_MIN_NB = 8;

// lower-triangle blocks of block columns [ob, ob + gridDim.y) of the work matrix (noise on the diagonal, identity padding),
// rows from block ob down: grid = (4 (nb - ob), width).  The standalone generator of the pre-generation schedule.
__global__ void __launch_bounds__(256)
k_cov_lower(const __grid_constant__ dgp_spec spec, const double* __restrict__ theta, const double* __restrict__ Xw,
            const double* __restrict__ noise, double jitter, double* __restrict__ A, long long ld, int n, int ob) {
  if ((int)blockIdx.x / 4 < (int)blockIdx.y) return;   // above the diagonal block
  const size_t o = (size_t)ob * 128;
  cov_rect_body(spec, theta, Xw + o * DGP_XS, Xw + o * DGP_XS, noise + o, jitter, A + o * ld + o, ld, n - (int)o, n - (int)o, 1, 1,
                nullptr, nullptr, 0, blockIdx.x, blockIdx.y);
}

// block column 0 of every site's work matrix (noise on the diagonal, identity padding): grid = (4 nbmax, 1, sites)
__global__ void __launch_bounds__(256)
k_cov_col0_b(const __grid_constant__ dgp_spec spec, const __grid_constant__ SiteDims sd, const double* __restrict__ theta,
             const double* __restrict__ Xw, const double* __restrict__ noise, const double* __restrict__ jitv,
             double* __restrict__ A) {
  const int st = blockIdx.z;
  if ((int)blockIdx.x >= 4 * sd.nb[st]) return;
  const size_t v = (size_t)st * sd.ld;
  cov_rect_body(spec, theta + st * DGP_MAX_THETA, Xw + v * DGP_XS, Xw + v * DGP_XS, noise + v, jitv[st], A + v * sd.ld, sd.ld,
                sd.n[st], sd.n[st], 1, 1, nullptr, nullptr, 0, blockIdx.x, 0);
}

// ... and the lower-triangle blocks of block columns >= 1 of the sites with more than `min_nb` block columns (DGP_PREGEN_MIN_NB): grid = (4 nbmax, nbmax - 1, sites)
__global__ void __launch_bounds__(256)
k_cov_lower_b(const __grid_constant__ dgp_spec spec, const __grid_constant__ SiteDims sd, const double* __restrict__ theta,
              const double* __restrict__ Xw, const double* __restrict__ noise, const double* __restrict__ jitv,
              double* __restrict__ A, int min_nb) {
  const int st = blockIdx.z, nbi = sd.nb[st], col = 1 + (int)blockIdx.y;
  if (nbi <= min_nb || col >= nbi || (int)blockIdx.x >= 4 * nbi || (int)blockIdx.x / 4 < col) return;
  const size_t v = (size_t)st * sd.ld;
  cov_rect_body(spec, theta + st * DGP_MAX_THETA, Xw + v * DGP_XS, Xw + v * DGP_XS, noise + v, jitv[st], A + v * sd.ld, sd.ld,
                sd.n[st], sd.n[st], 1, 1, nullptr, nullptr, 0, blockIdx.x, col);
}

// ------------------------------------------------------------------ forward substitution step
// z_s = Linv_s r_s ; r_i -= L[i, s] z_s for block rows i > s.  grid = nb - s, block = 256.
__global__ void __launch_bounds__(256)
k_fwd_step(const double* __restrict__ L, long long ld, const double* __restrict__ DI, double* __restrict__ r,
           double* __restrict__ z, int s) {
  __shared__ double rs[128];
  __shared__ double zs[128];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid < 128) rs[tid] = r[s * 128 + tid];
  __syncthreads();
  const double* D = DI + (size_t)s * 128 * 128;
  for (int row = warp; row < 128; row += 8) {
    double acc = 0.0;
    for (int k = lane; k <= row; k += 32) acc = fma(D[row * 128 + k], rs[k], acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) zs[row] = acc;
  }
  __syncthreads();
  if (blockIdx.x == 0) {
    if (tid < 128) z[s * 128 + tid] = zs[tid];
    return;
  }
  const int i = s + blockIdx.x;
  for (int row = warp; row < 128; row += 8) {
    const double* lp = L + (size_t)(i * 128 + row) * ld + s * 128;
    double acc = 0.0;
#pragma unroll
    for (int k = lane; k < 128; k += 32) acc = fma(lp[k], zs[k], acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) r[i * 128 + row] -= acc;
  }
}

// ------------------------------------------------------------------ alpha = U z  (U = L^-T upper triangular)
// one warp per row, grid = npad / 8, block = 256
__device__ __forceinline__ void upper_gemv_body(const double* __restrict__ U, long long ld, const double* __restrict__ z,
                                                double* __restrict__ out, int npad, int bx) {
  const int row = bx * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= npad) return;
  const double* up = U + (size_t)row * ld;
  double a0 = 0.0, a1 = 0.0;
  int k = (row & ~31) + lane;
  for (; k + 32 < npad; k += 64) {
    a0 = fma(up[k], z[k], a0);
    a1 = fma(up[k + 32], z[k + 32], a1);
  }
  if (k < npad) a0 = fma(up[k], z[k], a0);
  double acc = a0 + a1;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) out[row] = acc;
}
__global__ void __launch_bounds__(256)
k_upper_gemv(const double* __restrict__ U, long long ld, const double* __restrict__ z, double* __restrict__ out, int npad) {
  upper_gemv_body(U, ld, z, out, npad, blockIdx.x);
}
// grid = (ld / 8, sites)
__global__ void __launch_bounds__(256)
k_upper_gemv_b(const __grid_constant__ SiteDims sd, const double* __restrict__ U, const double* __restrict__ z,
               double* __restrict__ out) {
  const int st = blockIdx.y;
  const size_t v = (size_t)st * sd.ld;
  upper_gemv_body(U + v * sd.ld, sd.ld, z + v, out + v, sd.nb[st] * 128, blockIdx.x);
}

// ------------------------------------------------------------------ z = U^T r  (U upper triangular), two stages
// stage 1: grid = (nb, nb); CTA (cb, rb) with rb <= cb sums rows of row block rb for the 128 columns of block cb
// into part[rb][col]; stage 2 adds the row-block partials in a fixed order.
__device__ __forceinline__ void upperT_gemv_part_body(const double* __restrict__ U, long long ld, const double* __restrict__ r,
                                                      double* __restrict__ part, long long ldp, int cb, int rb) {
  if (rb > cb) return;
  __shared__ double rs[128];
  __shared__ double hs[128];
  const int tid = threadIdx.x, col = tid & 127, half = tid >> 7;
  if (tid < 128) rs[tid] = r[rb * 128 + tid];
  __syncthreads();
  const double* up = U + (size_t)(rb * 128 + half * 64) * ld + cb * 128 + col;
  double a0 = 0.0, a1 = 0.0, a2 = 0.0, a3 = 0.0;
#pragma unroll 4
  for (int i = 0; i < 64; i += 4) {
    a0 = fma(up[(size_t)(i + 0) * ld], rs[half * 64 + i + 0], a0);
    a1 = fma(up[(size_t)(i + 1) * ld], rs[half * 64 + i + 1], a1);
    a2 = fma(up[(size_t)(i + 2) * ld], rs[half * 64 + i + 2], a2);
    a3 = fma(up[(size_t)(i + 3) * ld], rs[half * 64 + i + 3], a3);
  }
  const double acc = (a0 + a1) + (a2 + a3);
  if (half == 1) hs[col] = acc;
  __syncthreads();
  if (half == 0) part[(size_t)rb * ldp + cb * 128 + col] = acc + hs[col];
}
__global__ void __launch_bounds__(256)
k_upperT_gemv_part(const double* __restrict__ U, long long ld, const double* __restrict__ r, double* __restrict__ part,
                   long long ldp) {
  upperT_gemv_part_body(U, ld, r, part, ldp, blockIdx.x, blockIdx.y);
}
// grid = (nbmax, nbmax, sites); part: [site][nbmax][ld]
__global__ void __launch_bounds__(256)
k_upperT_gemv_part_b(const __grid_constant__ SiteDims sd, const double* __restrict__ U, const double* __restrict__ r,
                     double* __restrict__ part) {
  const int st = blockIdx.z;
  if ((int)blockIdx.x >= sd.nb[st]) return;
  const size_t v = (size_t)st * sd.ld;
  upperT_gemv_part_body(U + v * sd.ld, sd.ld, r + v, part + v * sd.nbmax, sd.ld, blockIdx.x, blockIdx.y);
}

__device__ __forceinline__ void upperT_gemv_sum_body(const double* __restrict__ part, long long ldp, double* __restrict__ z,
                                                     int npad, int j) {
  if (j >= npad) return;
  double s = 0.0;
  for (int rb = 0; rb <= (j >> 7); rb++) s += part[(size_t)rb * ldp + j];
  z[j] = s;
}
__global__ void __launch_bounds__(256)
k_upperT_gemv_sum(const double* __restrict__ part, long long ldp, double* __restrict__ z, int npad) {
  upperT_gemv_sum_body(part, ldp, z, npad, blockIdx.x * 256 + threadIdx.x);
}
// grid = (ceil(ld / 256), sites)
__global__ void __launch_bounds__(256)
k_upperT_gemv_sum_b(const __grid_constant__ SiteDims sd, const double* __restrict__ part, double* __restrict__ z) {
  const int st = blockIdx.y;
  const size_t v = (size_t)st * sd.ld;
  upperT_gemv_sum_body(part + v * sd.nbmax, sd.ld, z + v, sd.nb[st] * 128, blockIdx.x * 256 + threadIdx.x);
}

// ------------------------------------------------------------------ T21 = U12^T for every pair of one merge level
// Pair p merges block ranges [o, o+h) and [o+h, o+2h), o = 2 h p.  grid.x = pairs * (4h)^2 tiles of 32x32; pr0 = first pair.
__device__ __forceinline__ void transpose_pairs_body(const double* __restrict__ U, double* __restrict__ T, long long ld, int hb,
                                                     int npad, int bx, int pr0) {
  __shared__ double tile[32][33];
  const int per = 16 * hb * hb;
  const int pr = pr0 + bx / per, rem = bx % per;
  const int ty32 = rem / (4 * hb), tx32 = rem % (4 * hb);
  const int r0 = pr * 2 * hb * 128 + ty32 * 32, c0 = (pr * 2 * hb + hb) * 128 + tx32 * 32;
  if (c0 >= npad) return;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) tile[r][tx] = U[(size_t)(r0 + r) * ld + c0 + tx];
  __syncthreads();
  for (int r = ty; r < 32; r += 8) T[(size_t)(c0 + r) * ld + r0 + tx] = tile[tx][r];
}
__global__ void __launch_bounds__(256)
k_transpose_pairs(const double* __restrict__ U, double* __restrict__ T, long long ld, int hb, int npad, int pr0) {
  transpose_pairs_body(U, T, ld, hb, npad, blockIdx.x, pr0);
}
// grid = (max over sites of pairs * 16 hb^2, sites); per site the pairs [pr0, pr0 + cnt) of this launch (cnt = 0: none)
struct PairRange { short pr0[DGP_BATCH_MAX], cnt[DGP_BATCH_MAX]; };
__global__ void __launch_bounds__(256)
k_transpose_pairs_b(const __grid_constant__ SiteDims sd, const __grid_constant__ PairRange pr, const double* __restrict__ U,
                    double* __restrict__ T, int hb) {
  const int st = blockIdx.y, nb = sd.nb[st];
  if ((int)blockIdx.x >= pr.cnt[st] * 16 * hb * hb) return;
  const size_t m = (size_t)st * sd.ld * sd.ld;
  transpose_pairs_body(U + m, T + m, sd.ld, hb, nb * 128, blockIdx.x, pr.pr0[st]);
}

// ------------------------------------------------------------------ final reductions (deterministic order)
// block b < ntheta: grad[b] = sum_tiles part[tile][b] (+ mean-parameter terms -J' alpha)
// block ntheta:     quad = z'z ; nlml = 1/2 quad + logdet + n/2 log 2 pi
__device__ __forceinline__ void finish_body(const dgp_spec& spec, const double* __restrict__ theta, const double* __restrict__ part,
         int ntiles, const double* __restrict__ z, const double* __restrict__ alpha, const double* __restrict__ X,
         int n, int npad, double* __restrict__ scal, int want_grad, int b) {
  __shared__ double red[256];
  const int tid = threadIdx.x;
  double s = 0.0;
  if (b == spec.ntheta) {
    for (int i = tid; i < npad; i += 256) s = fma(z[i], z[i], s);
  } else if (want_grad) {
    for (int t = tid; t < ntiles; t += 256) s += part[(size_t)t * DGP_MAX_THETA + b];
    int mk = -1;
    for (int k = 0; k < 3; k++)
      if ((spec.mean_kind == DGP_MEAN_CONST && k == 0 && spec.mean_theta[0] == b) ||
          (spec.mean_kind == DGP_MEAN_POWERLAW && spec.mean_theta[k] == b)) mk = k;
    if (mk >= 0) {
      double pb = 0.0, pc = 0.0;
      if (spec.mean_kind == DGP_MEAN_POWERLAW) { pb = theta[spec.mean_theta[1]]; pc = theta[spec.mean_theta[2]]; }
      for (int i = tid; i < n; i += 256) {
        double j = 1.0;  // d mean / d param
        if (spec.mean_kind == DGP_MEAN_POWERLAW && mk > 0) {
          const double u = X[(size_t)i * spec.ndim + spec.mean_col] - pc;
          j = (mk == 1) ? log(u) : -pb / u;
        }
        s = fma(-alpha[i], j, s);
      }
    }
  }
  red[tid] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (tid < o) red[tid] += red[tid + o];
    __syncthreads();
  }
  if (tid == 0) {
    if (b == spec.ntheta) {
      scal[SC_QUAD] = red[0];
      scal[SC_NLML] = 0.5 * red[0] + scal[SC_LOGDET] + 0.5 * (double)n * 1.8378770664093453;
    } else {
      scal[SC_GRAD + b] = want_grad ? red[0] : 0.0;
    }
  }
}
__global__ void __launch_bounds__(256)
k_finish(const __grid_constant__ dgp_spec spec, const double* __restrict__ theta, const double* __restrict__ part,
         int ntiles, const double* __restrict__ z, const double* __restrict__ alpha, const double* __restrict__ X,
         int n, int npad, double* __restrict__ scal, int want_grad) {
  finish_body(spec, theta, part, ntiles, z, alpha, X, n, npad, scal, want_grad, blockIdx.x);
}
// grid = (ntheta + 1, sites); part: [site][nbmax (nbmax + 1)][DGP_MAX_THETA]
__global__ void __launch_bounds__(256)
k_finish_b(const __grid_constant__ dgp_spec spec, const __grid_constant__ SiteDims sd, const double* __restrict__ theta,
           const double* __restrict__ part, const double* __restrict__ z, const double* __restrict__ alpha,
           const double* __restrict__ X, double* __restrict__ scal, int want_grad) {
  const int st = blockIdx.y, nb = sd.nb[st];
  const size_t v = (size_t)st * sd.ld;
  finish_body(spec, theta + st * DGP_MAX_THETA, part + (size_t)st * sd.nbmax * (sd.nbmax + 1) * DGP_MAX_THETA, nb * (nb + 1),
              z + v, alpha + v, X + v * DGP_MAX_COLS, sd.n[st], nb * 128, scal + (size_t)st * SC_SIZE, want_grad, blockIdx.x);
}

// ------------------------------------------------------------------ prediction reductions
// mu[i] = mean[i] + sum_cb dot[cb][i] ;  var[i] = k(x*_i, x*_i) - sum_cb vpart[cb][i]
__device__ __forceinline__ void pred_finish_body(const dgp_spec& spec, const double* __restrict__ theta,
              const double* __restrict__ Xws, const double* __restrict__ mean, const double* __restrict__ dot,
              int ndot, const double* __restrict__ vpart, int nvpart, int ldp, int m, double* __restrict__ mu,
              double* __restrict__ var, int i) {
  __shared__ CovC cc;
  cov_compile(&cc, spec, theta, 0.0, threadIdx.x, 256);
  __syncthreads();
  if (i >= m) return;
  double s = mean[i];
  for (int b = 0; b < ndot; b++) s += dot[(size_t)b * ldp + i];
  mu[i] = s;
  if (var != nullptr) {
    double xi[DGP_XS];
#pragma unroll
    for (int c = 0; c < DGP_XS; c++) xi[c] = Xws[(size_t)i * DGP_XS + c];
    double v = 0.0;
    for (int b = 0; b < nvpart; b++) v += vpart[(size_t)b * ldp + i];
    var[i] = cov_entry(&cc, xi, xi) - v;
  }
}
__global__ void __launch_bounds__(256)
k_pred_finish(const __grid_constant__ dgp_spec spec, const double* __restrict__ theta,
              const double* __restrict__ Xws, const double* __restrict__ mean, const double* __restrict__ dot,
              int ndot, const double* __restrict__ vpart, int nvpart, int ldp, int m, double* __restrict__ mu,
              double* __restrict__ var) {
  pred_finish_body(spec, theta, Xws, mean, dot, ndot, vpart, nvpart, ldp, m, mu, var, blockIdx.x * 256 + threadIdx.x);
}

// ------------------------------------------------------------------ batched prediction (dgp_batch_predict)
// One chunk of rows of every site's grid per launch.  Chunk slabs: inputs [site][chunk][DGP_MAX_COLS], features
// [site][chunk][DGP_XS], means / mu / var [site][chunk], Kx [site][chunk][ld], mean partials [site][nbmax][chunk], variance
// partials [site][2 nbmax][chunk]; the training side is the batch's slabs (SiteDims).  m[s] = rows of site s in this chunk
// (0: nothing to do), var[s] = 1: its variance is wanted.  The bodies are those of the single-site prediction.
struct PredChunk {
  int m[DGP_BATCH_MAX];
  int var[DGP_BATCH_MAX];
};

// grid = (chunk / 256, sites)
__global__ void k_pred_features_b(const __grid_constant__ dgp_spec spec, const __grid_constant__ PredChunk pc,
                                  const double* __restrict__ theta, const double* __restrict__ Xs, double* __restrict__ Xws,
                                  double* __restrict__ means, int chunk) {
  const int st = blockIdx.y, m = pc.m[st];
  if (m == 0) return;
  const size_t v = (size_t)st * chunk;
  features_body(spec, theta + st * DGP_MAX_THETA, Xs + v * DGP_MAX_COLS, nullptr, Xws + v * DGP_XS, nullptr, means + v, m,
                (m + 127) / 128 * 128, nullptr, blockIdx.x * blockDim.x + threadIdx.x);
}

// cross covariance Kx[s] = K(x*, X_s) of the chunk (only where the variance is wanted) fused with the mean partials
// dot[s][cb][i] = sum_{j in block cb} Kx[s][i, j] alpha_s[j].  grid = (chunk / 32, nbmax, sites)
__global__ void __launch_bounds__(256)
k_cov_rect_pred_b(const __grid_constant__ dgp_spec spec, const __grid_constant__ SiteDims sd, const __grid_constant__ PredChunk pc,
                  const double* __restrict__ theta, const double* __restrict__ Xws, const double* __restrict__ Xw,
                  const double* __restrict__ noise, const double* __restrict__ alpha, double* __restrict__ Kx,
                  double* __restrict__ dot, int chunk) {
  const int st = blockIdx.z, m = pc.m[st];
  if (m == 0 || (int)blockIdx.x >= (m + 127) / 128 * 4 || (int)blockIdx.y >= sd.nb[st]) return;
  const size_t v = (size_t)st * sd.ld, c = (size_t)st * chunk;
  cov_rect_body(spec, theta + st * DGP_MAX_THETA, Xws + c * DGP_XS, Xw + v * DGP_XS, noise + v, 0.0,
                pc.var[st] ? Kx + c * sd.ld : nullptr, sd.ld, m, sd.n[st], 0, 0, alpha + v, dot + c * sd.nbmax, chunk,
                blockIdx.x, blockIdx.y);
}

// grid = (chunk / 256, sites)
__global__ void __launch_bounds__(256)
k_pred_finish_b(const __grid_constant__ dgp_spec spec, const __grid_constant__ SiteDims sd, const __grid_constant__ PredChunk pc,
                const double* __restrict__ theta, const double* __restrict__ Xws, const double* __restrict__ means,
                const double* __restrict__ dot, const double* __restrict__ vpart, double* __restrict__ mu,
                double* __restrict__ var, int chunk) {
  const int st = blockIdx.y, m = pc.m[st], nb = sd.nb[st];
  if (m == 0) return;
  const size_t c = (size_t)st * chunk;
  pred_finish_body(spec, theta + st * DGP_MAX_THETA, Xws + c * DGP_XS, means + c, dot + c * sd.nbmax, nb,
                   vpart + c * 2 * sd.nbmax, 2 * nb, chunk, m, mu + c, pc.var[st] ? var + c : nullptr,
                   blockIdx.x * 256 + threadIdx.x);
}

}  // namespace dgp

namespace dgp {
// In-place factorisation: block column s of L, staged by the panel solve in P[rows][128], goes back into the matrix.
// grid = (row blocks below the diagonal block), block = 256.
__global__ void __launch_bounds__(256)
k_copy_panel(const double* __restrict__ P, double* __restrict__ A, long long ld, int s) {
  const size_t row0 = (size_t)(s + 1 + blockIdx.x) * 128;
  for (int e = threadIdx.x; e < 128 * 64; e += 256) {
    const int r = e >> 6, c2 = (e & 63) * 2;
    const double2 v = *reinterpret_cast<const double2*>(P + (row0 + r) * 128 + c2);
    *reinterpret_cast<double2*>(A + (row0 + r) * ld + (size_t)s * 128 + c2) = v;
  }
}

// zero the strict upper triangle of a dense row-major n x n matrix (leading dimension ld); grid = n rows, block = 256
__global__ void __launch_bounds__(256) k_zero_strict_upper(double* __restrict__ A, long long ld, int n) {
  double* row = A + (size_t)blockIdx.x * ld;
  for (int c = blockIdx.x + 1 + threadIdx.x; c < n; c += 256) row[c] = 0.0;
}

// Column panel [c0, c0 + w) of the rows >= r0 of A  <->  contiguous buffer P[rows][w]  (dir = 0: pack, 1: unpack).
// grid = (rows / 8), block = 256; w multiple of 2.
__global__ void __launch_bounds__(256)
k_pack_panel(double* __restrict__ A, long long ld, long long r0, long long c0, int w, double* __restrict__ P, int dir) {
  const int half = w >> 1;
  for (int e = threadIdx.x; e < 8 * half; e += 256) {
    const long long r = (long long)blockIdx.x * 8 + e / half;
    const int c2 = (e % half) * 2;
    double2* a = reinterpret_cast<double2*>(A + (r0 + r) * ld + c0 + c2);
    double2* p = reinterpret_cast<double2*>(P + r * w + c2);
    if (dir == 0) *p = *a; else *a = *p;
  }
}

// out[s, i] += mu[i]  (rows s < S, cols i < m), grid = (ceil(m/256), S)
__global__ void __launch_bounds__(256) k_add_rowvec(double* __restrict__ out, long long ld, const double* __restrict__ mu, int m) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < m) out[(size_t)blockIdx.y * ld + i] += mu[i];
}
}  // namespace dgp

namespace dgp {
// ------------------------------------------------------------------ base normals on the device
// Standard normal number e of the stream keyed by `seed`: Philox4x32-10 on counter (e >> 1, 0), key = seed, gives
// two 53-bit uniforms u1, u2 in (0, 1); z = sqrt(-2 ln u1) * (e odd ? sin : cos)(2 pi u2)   (Box-Muller).
// tests/test_gpu_parity.py restates the generator in numpy.
__device__ __forceinline__ double philox_normal(unsigned long long seed, unsigned long long e) {
  unsigned int c0 = (unsigned int)(e >> 1), c1 = (unsigned int)(e >> 33), c2 = 0u, c3 = 0u;
  unsigned int k0 = (unsigned int)seed, k1 = (unsigned int)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; r++) {
    const unsigned int hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const unsigned int hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  const unsigned long long a = ((unsigned long long)c1 << 32) | c0, b = ((unsigned long long)c3 << 32) | c2;
  const double u1 = ((double)(a >> 11) + 0.5) * (1.0 / 9007199254740992.0);
  const double u2 = ((double)(b >> 11) + 0.5) * (1.0 / 9007199254740992.0);
  const double rad = sqrt(-2.0 * log(u1));
  double sn, cs;
  sincospi(2.0 * u2, &sn, &cs);
  return rad * ((e & 1ull) ? sn : cs);
}

// Z[s, i] = normal number s * m + i, rows s < S, cols i < m of a [*, ld] matrix.  grid = (ceil(m / 256), S)
__global__ void __launch_bounds__(256)
k_fill_normals(double* __restrict__ Z, long long ld, int m, unsigned long long seed) {
  const int i = blockIdx.x * 256 + threadIdx.x;
  if (i < m) Z[(size_t)blockIdx.y * ld + i] = philox_normal(seed, (unsigned long long)blockIdx.y * (unsigned long long)m + i);
}

// ------------------------------------------------------------------ flux post-processing of the draws
// out[s, g] = sum_{i in [start[g], start[g+1])} w[i] * T(draw[s, i]),  T(z) = exp(z * scale + mean) (log pipelines,
// clipped below at 1e-6 like the reference's inverse transform), z * scale + mean clipped at 0 (standard pipeline), or affine:
// concentration_to_flux + resample("YE").sum() of src/loadest_gp/utils.py:14-56,89 without moving the draws.
// grid = (groups, ceil(S / 8)), block = 256: one warp per (draw, group).
__global__ void __launch_bounds__(256)
k_flux_reduce(const double* __restrict__ D, long long ld, const double* __restrict__ w, const int* __restrict__ start,
              int ngroups, int S, double mean, double scale, int log_transform, double* __restrict__ out) {
  const int g = blockIdx.x, s = blockIdx.y * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (s >= S) return;
  const double* row = D + (size_t)s * ld;
  double acc = 0.0;
  for (int i = start[g] + lane; i < start[g + 1]; i += 32) {
    double v = fma(row[i], scale, mean);
    if (log_transform == 1) v = fmax(exp(v), 1e-6);
    else if (log_transform == 2) v = fmax(v, 0.0);
    acc = fma(w[i], v, acc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) out[(size_t)s * ngroups + g] = acc;
}

// ------------------------------------------------------------------ gradient of a linear functional of the posterior mean
// F(theta) = sum_p c_p mu(x*_p),  mu = m(x*) + K*x alpha:
//   dF/dtheta_k = sum_{p,j} c_p alpha_j dk(x*_p, x_j)/dtheta_k - sum_{i,j} gamma_i alpha_j dK(x_i, x_j)/dtheta_k,
//   gamma = Ky^-1 Kx* c  (adjoint of the solve).  Both sums are rank-1-weighted contractions of dK/dtheta:
// k_wgrad: part[cta][t] = sgn * sum_{i in rows, j in cols of this 128x64 tile} wa_i wb_j dk(xa_i, xb_j)/dtheta_t.
// grid = (col blocks of 64, row blocks of 128), block = 128 (thread = row); wa / wb are zero on padding.
// (bx, by) = (column block, row block) of the CTA, ncb = column blocks: part index by * ncb + bx.
__device__ __forceinline__ void wgrad_body(const dgp_spec& spec, const double* __restrict__ theta, const double* __restrict__ XwA,
                                           const double* __restrict__ XwB, const double* __restrict__ wa,
                                           const double* __restrict__ wb, double sgn, double* __restrict__ part, int bx, int by,
                                           int ncb) {
  __shared__ CovC cc;
  __shared__ double xaT[DGP_XS * 128];
  __shared__ double xb[64 * DGP_XS];
  __shared__ double wbs[64];
  __shared__ double red[4 * DGP_MAX_TERMS * NSLOT];
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  const size_t r0 = (size_t)by * 128, c0b = (size_t)bx * 64;
  cov_compile(&cc, spec, theta, 0.0, t, 128);
  for (int e = t; e < 128 * DGP_XS; e += 128) xaT[(e % DGP_XS) * 128 + e / DGP_XS] = XwA[r0 * DGP_XS + e];
  for (int e = t; e < 64 * DGP_XS; e += 128) xb[e] = XwB[c0b * DGP_XS + e];
  if (t < 64) wbs[t] = wb[c0b + t];
  __syncthreads();
  const double wi = wa[r0 + t];
  for (int term = 0; term < cc.nterms; term++) {
    double sl[NSLOT];
#pragma unroll
    for (int k = 0; k < NSLOT; k++) sl[k] = 0.0;
    const TermC& tc = cc.t[term];
#pragma unroll 1
    for (int c0 = 0; c0 < 64; c0 += 4) {
      double w[4];
#pragma unroll
      for (int v = 0; v < 4; v++) w[v] = wi * wbs[c0 + v];
      term_grad_accum_v<4>(tc, xaT, 128, t, xb + c0 * DGP_XS, w, sl);
    }
#pragma unroll
    for (int k = 0; k < NSLOT; k++) {
      double v = sl[k];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) red[(warp * DGP_MAX_TERMS + term) * NSLOT + k] = v;
    }
  }
  __syncthreads();
  if (t < DGP_MAX_THETA) {
    double s = 0.0;
    if (t < cc.ntheta)
      for (int term = 0; term < cc.nterms; term++)
        for (int k = 0; k < NSLOT; k++)
          if (term_slot_theta(cc.t[term], k) == t)
            for (int w4 = 0; w4 < 4; w4++) s += red[(w4 * DGP_MAX_TERMS + term) * NSLOT + k];
    part[((size_t)by * ncb + bx) * DGP_MAX_THETA + t] = sgn * s;
  }
}
__global__ void __launch_bounds__(128)
k_wgrad(const __grid_constant__ dgp_spec spec, const double* __restrict__ theta, const double* __restrict__ XwA,
        const double* __restrict__ XwB, const double* __restrict__ wa, const double* __restrict__ wb, double sgn,
        double* __restrict__ part) {
  wgrad_body(spec, theta, XwA, XwB, wa, wb, sgn, part, blockIdx.x, blockIdx.y, gridDim.x);
}

// ------------------------------------------------------------------ NLML gradient contraction as its own pass
// part[tile][t] = -1/2 sum_{(i, j) in lower tile} wgt_ij (alpha_i alpha_j - Kinv_ij) dK_ij/dtheta_t  (+ -1/2 tr W on the
// learned-noise slot), wgt = 2 below the diagonal, 1 on it.  Same tiling as the LAUUM launch that wrote Kinv
// (128 x 64 lower tiles, tile -> (i, c) triangular), one thread per row, 4 columns side by side.  Unlike the fused
// epilogue this runs with every warp of the SM on FP64 ALU work, so the pipe is not shared with DMMA issue.
#ifndef DGP_GC_V
#define DGP_GC_V 4   // entries a thread evaluates side by side in the gradient contraction
#endif
#ifndef DGP_GC_BLOCKS
#define DGP_GC_BLOCKS 4
#endif
// one row of a 128 x 64 tile of W = alpha alpha' - Ky^-1 against d(term)/d(parameters), 4 entries side by side
template <class S>
__device__ __forceinline__ void grad_row(const TermC& tc, const double* __restrict__ xaT, int t, const double* __restrict__ xb,
                                         const double* __restrict__ al, const double* __restrict__ krow, double ai, int grow,
                                         int c0b, bool row_live, double (&sl)[NSLOT]) {
  if (!row_live) return;
#pragma unroll 1
  for (int c0 = 0; c0 < 64; c0 += DGP_GC_V) {
    if (c0b + c0 > grow) break;  // strictly above the diagonal from here on
    double w[DGP_GC_V];
#pragma unroll
    for (int v2 = 0; v2 < DGP_GC_V; v2 += 2) {
      const double2 kk = *reinterpret_cast<const double2*>(krow + c0 + v2);
      const double kv[2] = {kk.x, kk.y};
#pragma unroll
      for (int e = 0; e < 2; e++) {
        const int gcol = c0b + c0 + v2 + e;
        const double wgt = (gcol < grow) ? 2.0 : (gcol == grow ? 1.0 : 0.0);
        w[v2 + e] = wgt * (ai * al[c0 + v2 + e] - kv[e]);
      }
    }
    term_grad_accum_s<DGP_GC_V, S>(tc, xaT, 128, t, xb + c0 * DGP_XS, w, sl);
  }
}

__device__ __forceinline__ void grad_contract_body(const dgp_spec& spec, const double* __restrict__ theta, const double* __restrict__ Xw,
                const double* __restrict__ alpha, const double* __restrict__ Kinv, long long ld, int n,
                double* __restrict__ part, int tile) {
  __shared__ CovC cc;
  __shared__ double xaT[DGP_XS * 128];
  __shared__ double xb[64 * DGP_XS];
  __shared__ double al[64];
  __shared__ double red[4 * DGP_MAX_TERMS * NSLOT + 4];
  const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
  int ib = (int)sqrt((double)(4 * tile + 1));
  while (ib * ib > 4 * tile + 1) --ib;
  while ((ib + 1) * (ib + 1) <= 4 * tile + 1) ++ib;
  ib = (ib - 1) >> 1;
  const int cb = tile - ib * (ib + 1);
  const size_t r0 = (size_t)ib * 128, c0b = (size_t)cb * 64;
  cov_compile(&cc, spec, theta, 0.0, t, 128);
  for (int e = t; e < 128 * DGP_XS; e += 128) xaT[(e % DGP_XS) * 128 + e / DGP_XS] = Xw[r0 * DGP_XS + e];
  for (int e = t; e < 64 * DGP_XS; e += 128) xb[e] = Xw[c0b * DGP_XS + e];
  if (t < 64) al[t] = alpha[c0b + t];
  __syncthreads();
  const int grow = (int)r0 + t;
  const double ai = alpha[grow];
  const double* krow = Kinv + (size_t)grow * ld + c0b;
  double trw = 0.0;
  const bool row_live = grow < n;
  // trace of W on the diagonal entries of this row (noise / jitter parameter), once per row
  if (row_live && grow >= (int)c0b && grow < (int)c0b + 64) trw = ai * al[grow - (int)c0b] - krow[grow - (int)c0b];
  for (int term = 0; term < cc.nterms; term++) {
    double sl[NSLOT];
#pragma unroll
    for (int k = 0; k < NSLOT; k++) sl[k] = 0.0;
    const TermC& tc = cc.t[term];
    // the shape switch is taken once per term and row, around the whole row of the tile: inside a specialisation the
    // slots the shape does not have stay compile-time zeros instead of 17 live accumulators
    DGP_SHAPE_SWITCH(tc.shape, (grad_row<S>(tc, xaT, t, xb, al, krow, ai, grow, (int)c0b, row_live, sl)))
#pragma unroll
    for (int k = 0; k < NSLOT; k++) {
      double v = sl[k];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) red[(warp * DGP_MAX_TERMS + term) * NSLOT + k] = v;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) trw += __shfl_xor_sync(0xffffffffu, trw, o);
  if (lane == 0) red[4 * DGP_MAX_TERMS * NSLOT + warp] = trw;
  __syncthreads();
  if (t < cc.ntheta) {
    double s = 0.0;
    for (int term = 0; term < cc.nterms; term++)
      for (int k = 0; k < NSLOT; k++)
        if (term_slot_theta(cc.t[term], k) == t)
          for (int w4 = 0; w4 < 4; w4++) s += red[(w4 * DGP_MAX_TERMS + term) * NSLOT + k];
    if (t == cc.noise_idx)
      for (int w4 = 0; w4 < 4; w4++) s += red[4 * DGP_MAX_TERMS * NSLOT + w4];
    part[(size_t)tile * DGP_MAX_THETA + t] = -0.5 * s;
  }
}
__global__ void __launch_bounds__(128, DGP_GC_BLOCKS)
k_grad_contract(const __grid_constant__ dgp_spec spec, const double* __restrict__ theta, const double* __restrict__ Xw,
                const double* __restrict__ alpha, const double* __restrict__ Kinv, long long ld, int n,
                double* __restrict__ part) {
  grad_contract_body(spec, theta, Xw, alpha, Kinv, ld, n, part, blockIdx.x);
}
// grid = sd.tile0[sites] tiles of all sites (prefix lookup); part: [site][nbmax (nbmax + 1)][DGP_MAX_THETA]
__global__ void __launch_bounds__(128, DGP_GC_BLOCKS)
k_grad_contract_b(const __grid_constant__ dgp_spec spec, const __grid_constant__ SiteDims sd, const double* __restrict__ theta,
                  const double* __restrict__ Xw, const double* __restrict__ alpha, const double* __restrict__ Kinv,
                  double* __restrict__ part) {
  int st = 0;
#pragma unroll 1
  for (int i = 1; i < sd.count; i++) if ((int)blockIdx.x >= sd.tile0[i]) st = i;
  const size_t v = (size_t)st * sd.ld;
  grad_contract_body(spec, theta + st * DGP_MAX_THETA, Xw + v * DGP_XS, alpha + v, Kinv + v * sd.ld, sd.ld, sd.n[st],
                     part + (size_t)st * sd.nbmax * (sd.nbmax + 1) * DGP_MAX_THETA, (int)blockIdx.x - sd.tile0[st]);
}

// v[j] = sum_p c[p] Kx[p, j]   (p < mpad), grid = npad / 256
__device__ __forceinline__ void colsum_weighted_body(const double* __restrict__ Kx, long long ld, const double* __restrict__ c,
                                                     int mpad, double* __restrict__ v, int npad, int j) {
  if (j >= npad) return;
  double s = 0.0;
  for (int p = 0; p < mpad; p++) s = fma(c[p], Kx[(size_t)p * ld + j], s);
  v[j] = s;
}
__global__ void __launch_bounds__(256)
k_colsum_weighted(const double* __restrict__ Kx, long long ld, const double* __restrict__ c, int mpad, double* __restrict__ v) {
  colsum_weighted_body(Kx, ld, c, mpad, v, (int)ld, blockIdx.x * 256 + threadIdx.x);
}

// block b < ntheta: grad[b] = sum_parts part[.][b] + mean-parameter terms + learned-noise term; block ntheta: F = c'mu.
// out[0] = F, out[1 + b] = dF/dtheta_b.
__device__ __forceinline__ void mfg_finish_body(const dgp_spec& spec, const double* __restrict__ theta,
                                                const double* __restrict__ part, int nparts, const double* __restrict__ c,
                                                const double* __restrict__ mu, const double* __restrict__ Xs, int m,
                                                const double* __restrict__ gamma, const double* __restrict__ alpha,
                                                const double* __restrict__ X, int n, double* __restrict__ out, int b) {
  __shared__ double red[256];
  const int tid = threadIdx.x;
  double s = 0.0;
  if (b == spec.ntheta) {
    for (int p = tid; p < m; p += 256) s = fma(c[p], mu[p], s);
  } else {
    for (int i = tid; i < nparts; i += 256) s += part[(size_t)i * DGP_MAX_THETA + b];
    if (b == spec.noise_theta)
      for (int i = tid; i < n; i += 256) s = fma(-gamma[i], alpha[i], s);
    int mk = -1;
    for (int k = 0; k < 3; k++)
      if ((spec.mean_kind == DGP_MEAN_CONST && k == 0 && spec.mean_theta[0] == b) ||
          (spec.mean_kind == DGP_MEAN_POWERLAW && spec.mean_theta[k] == b)) mk = k;
    if (mk >= 0) {
      double pb = 0.0, pc = 0.0;
      if (spec.mean_kind == DGP_MEAN_POWERLAW) { pb = theta[spec.mean_theta[1]]; pc = theta[spec.mean_theta[2]]; }
      for (int i = tid; i < m + n; i += 256) {
        const bool test = i < m;
        const double* x = test ? Xs + (size_t)i * spec.ndim : X + (size_t)(i - m) * spec.ndim;
        double j = 1.0;  // d mean / d param
        if (spec.mean_kind == DGP_MEAN_POWERLAW && mk > 0) {
          const double u = x[spec.mean_col] - pc;
          j = (mk == 1) ? log(u) : -pb / u;
        }
        s = fma(test ? c[i] : -gamma[i - m], j, s);
      }
    }
  }
  red[tid] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (tid < o) red[tid] += red[tid + o];
    __syncthreads();
  }
  if (tid == 0) out[(b == spec.ntheta) ? 0 : 1 + b] = red[0];
}
__global__ void __launch_bounds__(256)
k_mfg_finish(const __grid_constant__ dgp_spec spec, const double* __restrict__ theta, const double* __restrict__ part,
             int nparts, const double* __restrict__ c, const double* __restrict__ mu, const double* __restrict__ Xs, int m,
             const double* __restrict__ gamma, const double* __restrict__ alpha, const double* __restrict__ X, int n,
             double* __restrict__ out) {
  mfg_finish_body(spec, theta, part, nparts, c, mu, Xs, m, gamma, alpha, X, n, out, blockIdx.x);
}

// ------------------------------------------------------------------ batched adjoint of the posterior mean
// (dgp_batch_mean_functional_grad).  Per site s with m[s] > 0: the chunk slabs of the prediction hold its points (Xs, Xws,
// mu: [site][chunk]..., Kx: [site][chunk][ld]), c / v / gamma are [site][chunk] / [site][ld] / [site][ld], and its partials
// [site][pstride] are laid out as those of dgp_mean_functional_grad for ITS OWN sizes: mpad = 128 ceil(m / 128) and
// npad = 128 nb, (mpad / 128 + nb) (npad / 64) tiles, the first mpad / 128 row blocks c x alpha, the rest -gamma x alpha.
// The bodies and the order of every sum are the single-site ones, so the results are bit-identical to it.
struct MfgTab {
  int m[DGP_BATCH_MAX];
  int tile0[DGP_BATCH_MAX + 1];   // prefix of the per-site tile counts (mpad / 128 + nb) (npad / 64)
};

// v[s][j] = sum_{p < mpad_s} c[s][p] Kx[s][p, j], j < npad_s;  grid = (ceil(ld / 256), sites)
__global__ void __launch_bounds__(256)
k_colsum_weighted_b(const __grid_constant__ SiteDims sd, const __grid_constant__ MfgTab mt, const double* __restrict__ Kx,
                    const double* __restrict__ c, double* __restrict__ v, int chunk) {
  const int st = blockIdx.y;
  const size_t cc = (size_t)st * chunk;
  colsum_weighted_body(Kx + cc * sd.ld, sd.ld, c + cc, (mt.m[st] + 127) / 128 * 128, v + (size_t)st * sd.ld, sd.nb[st] * 128,
                       blockIdx.x * 256 + threadIdx.x);
}

// both weighted contractions of every site in one launch: grid = mt.tile0[sites] (prefix lookup, no empty CTAs)
__global__ void __launch_bounds__(128)
k_wgrad_b(const __grid_constant__ dgp_spec spec, const __grid_constant__ SiteDims sd, const __grid_constant__ MfgTab mt,
          const double* __restrict__ theta, const double* __restrict__ Xws, const double* __restrict__ Xw,
          const double* __restrict__ c, const double* __restrict__ gamma, const double* __restrict__ alpha,
          double* __restrict__ part, int chunk, long long pstride) {
  int st = 0;
#pragma unroll 1
  for (int i = 1; i < sd.count; i++) if ((int)blockIdx.x >= mt.tile0[i]) st = i;
  const int t = (int)blockIdx.x - mt.tile0[st], ncb = sd.nb[st] * 2, mb = (mt.m[st] + 127) / 128;
  const size_t v = (size_t)st * sd.ld, cc = (size_t)st * chunk;
  const double* th = theta + st * DGP_MAX_THETA;
  double* pt = part + (size_t)st * pstride;
  if (t < mb * ncb) {
    wgrad_body(spec, th, Xws + cc * DGP_XS, Xw + v * DGP_XS, c + cc, alpha + v, 1.0, pt, t % ncb, t / ncb, ncb);
  } else {
    const int u = t - mb * ncb;
    wgrad_body(spec, th, Xw + v * DGP_XS, Xw + v * DGP_XS, gamma + v, alpha + v, -1.0, pt + (size_t)mb * ncb * DGP_MAX_THETA,
               u % ncb, u / ncb, ncb);
  }
}

// grid = (ntheta + 1, sites); out: [site][1 + DGP_MAX_THETA]
__global__ void __launch_bounds__(256)
k_mfg_finish_b(const __grid_constant__ dgp_spec spec, const __grid_constant__ SiteDims sd, const __grid_constant__ MfgTab mt,
               const double* __restrict__ theta, const double* __restrict__ part, const double* __restrict__ c,
               const double* __restrict__ mu, const double* __restrict__ Xs, const double* __restrict__ gamma,
               const double* __restrict__ alpha, const double* __restrict__ X, double* __restrict__ out, int chunk,
               long long pstride) {
  const int st = blockIdx.y, m = mt.m[st], nb = sd.nb[st];
  if (m == 0) return;
  const size_t v = (size_t)st * sd.ld, cc = (size_t)st * chunk;
  mfg_finish_body(spec, theta + st * DGP_MAX_THETA, part + (size_t)st * pstride, ((m + 127) / 128 + nb) * 2 * nb, c + cc, mu + cc,
                  Xs + cc * DGP_MAX_COLS, m, gamma + v, alpha + v, X + v * DGP_MAX_COLS, sd.n[st],
                  out + (size_t)st * (1 + DGP_MAX_THETA), blockIdx.x);
}
}  // namespace dgp
