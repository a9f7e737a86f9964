/* dgp.h -- C ABI of libdgp.so, the B200 exact-GP engine behind discontinuum's Marginal* engines.
 *
 * The reference (thodson-usgs/discontinuum) has NO FFI: its hot path is gpytorch/linear_operator
 * calls made from Python.  Each entry point below replaces the library calls made at the cited
 * reference lines (paths relative to the reference's src/):
 *
 *   dgp_set_train      <- tensors built in MarginalGPyTorch.fit, discontinuum/engines/gpytorch.py:219-235
 *                         and the model's build_model (loadest_gp/models/gpytorch.py:48-58,
 *                         rating_gp/models/gpytorch.py:64-79)
 *   dgp_covmat         <- ExactGPModel.forward -> covar_module(x)  (loadest_gp/models/gpytorch.py:71-76,
 *                         rating_gp/models/gpytorch.py:256-265, rating_gp/models/kernels.py:242-382)
 *   dgp_nlml           <- mll(output, train_y), discontinuum/engines/gpytorch.py:318,353
 *   dgp_nlml_grad      <- the same + objective.backward(), discontinuum/engines/gpytorch.py:353,384
 *   dgp_factorize      <- the eval-mode caches GPyTorch builds on the first prediction
 *                         (discontinuum/engines/gpytorch.py:618-622)
 *   dgp_predict        <- MarginalGPyTorch.__gpytorch_predict, discontinuum/engines/gpytorch.py:599-626
 *   dgp_sample         <- f_preds.sample(...), discontinuum/engines/gpytorch.py:578-580
 *   dgp_batch_sample_ex <- per site of nwqn-loadest-example.py:156-157: the joint draws and their annual flux,
 *                         loadest_gp/utils.py:14-56,89 (concentration_to_flux + resample("YE").sum()), for a whole group of
 *                         sites in one launch sequence on the batch handle's factorisation; its workspace is a grow-only
 *                         sampling arena on the handle (dgp_batch_sample_bytes)
 *
 * Conventions: plain pointers and sizes only.  All matrices are float64, row-major.  Every call
 * returns an int status: 0 = ok; > 0 = LAPACK-style info (1-based index of the first non-positive
 * pivot met by the Cholesky factorisation); < 0 = bad argument or CUDA error, text available from
 * dgp_last_error().  A handle owns one CUDA stream-ordered workspace sized at dgp_create; it is
 * not thread-safe, use one handle per host thread / per concurrent site.  There is no CPU
 * fallback: without a CUDA device dgp_create fails.
 */
#ifndef DGP_H
#define DGP_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DGP_ABI_VERSION 2

#define DGP_MAX_TERMS 8    /* additive terms of the covariance                        */
#define DGP_MAX_FACTORS 3  /* stationary factors multiplied inside one term           */
#define DGP_MAX_FDIMS 4    /* ARD dimensions of one factor                            */
#define DGP_MAX_COLS 8     /* columns of the per-point feature table                  */
#define DGP_MAX_THETA 48   /* natural hyper-parameters (kernel + mean + learned noise) */

/* stationary factor kinds (GPyTorch semantics, SURVEY Appendix A.2) */
enum { DGP_RBF = 0, DGP_MATERN32 = 1, DGP_MATERN52 = 2, DGP_PERIODIC = 3 };
/* multiplicative gate of a term: g(h)g(h') or (1-g(h))(1-g(h')), g = 1/(1+exp(a(h-b))) */
enum { DGP_GATE_NONE = 0, DGP_GATE_SIGMOID = 1, DGP_GATE_INV_SIGMOID = 2 };
/* feature-table column kinds.  A DGP_COL_GATE column may only be a term's gate_col: no factor dimension may read it,
 * because its value depends on theta[b] and a factor's gradient has no place for that dependence. */
enum { DGP_COL_COPY = 0, DGP_COL_LOG = 1 /* log(x + eps) */, DGP_COL_GATE = 2 /* g(x; a, theta[b]) */ };
/* mean functions */
enum { DGP_MEAN_ZERO = 0, DGP_MEAN_CONST = 1, DGP_MEAN_POWERLAW = 2 /* a + b log(x - c) */ };
/* dgp_set_train / dgp_batch_set_train reject (< 0, with a message) a spec with any kind outside the enums above (column,
 * factor, gate, mean), any theta index or column out of range, or a factor dimension on a DGP_COL_GATE column. */

typedef struct {
  int32_t kind;                 /* DGP_COL_*                                          */
  int32_t src;                  /* source column of X                                 */
  int32_t theta;                /* theta index of the gate switch point (GATE), else -1 */
  int32_t pad_;
  double aux;                   /* eps (LOG) or sharpness a (GATE)                    */
} dgp_col;

typedef struct {
  int32_t kind;                 /* DGP_RBF ... DGP_PERIODIC                           */
  int32_t ndims;                /* active dims (PERIODIC: 1)                          */
  int32_t col[DGP_MAX_FDIMS];   /* feature-table columns                              */
  int32_t ls[DGP_MAX_FDIMS];    /* theta index of the lengthscale of each dim
                                   (PERIODIC: ls[0] is GPyTorch's un-squared lengthscale) */
  int32_t period;               /* theta index of the period (PERIODIC) else -1       */
  int32_t pad_;
} dgp_factor;

typedef struct {
  int32_t scale;                /* theta index of the outputscale, -1 -> 1            */
  int32_t gate;                 /* DGP_GATE_*                                         */
  int32_t gate_col;             /* feature-table column holding g (kind DGP_COL_GATE) */
  int32_t nfactors;
  dgp_factor factor[DGP_MAX_FACTORS];
} dgp_term;

typedef struct {
  int32_t abi;                  /* DGP_ABI_VERSION                                    */
  int32_t ndim;                 /* columns of X                                       */
  int32_t ncols;                /* feature-table columns                              */
  int32_t nterms;
  int32_t ntheta;               /* length of theta / grad                             */
  int32_t noise_theta;          /* theta index of the learned homoskedastic noise, -1 = none */
  int32_t mean_kind;            /* DGP_MEAN_*                                         */
  int32_t mean_col;             /* X column the mean reads (POWERLAW)                 */
  int32_t mean_theta[4];        /* theta indices: CONST {c}; POWERLAW {a, b, c}       */
  dgp_col col[DGP_MAX_COLS];
  dgp_term term[DGP_MAX_TERMS];
} dgp_spec;

typedef struct dgp_handle_s* dgp_handle;

/* Create an engine on CUDA device `device` for up to max_n training points and prediction chunks
 * of up to max_m points (0 -> default).  Allocates every workspace (3 padded n x n float64 panels +
 * prediction chunk); later calls allocate nothing.  stream: a cudaStream_t to run on, or NULL to
 * let the handle create its own non-blocking stream.  Exception: the first gradient evaluation of a training set of
 * at least 8192 padded points (n rounded up to 128) forms Ky^-1 on the INT8 tensor cores and allocates its residue
 * buffers then, kept until destroy: 16 max_pad^2 + 2048 max_pad + 4 max_pad B (max_pad = max_n rounded up to 128).  If
 * that allocation fails the evaluation returns an error. */
int dgp_create(dgp_handle* out, int device, int max_n, int max_m, void* stream);

int dgp_destroy(dgp_handle h);
const char* dgp_last_error(dgp_handle h); /* h may be NULL: error of a failed dgp_create */
int dgp_abi_version(void);
/* Device bytes allocated by dgp_create; the INT8 LAUUM's residue buffers (16 max_pad^2 + 2052 max_pad B, allocated by the
 * first gradient evaluation of a training set of >= 8192 padded points) are not included. */
size_t dgp_workspace_bytes(int max_n, int max_m);

/* Training set of one site.  X[n, ndim], y[n], noise[n] (fixed per-point noise variances).
 * on_device != 0: pointers are device memory on the handle's device; else host memory. */
int dgp_set_train(dgp_handle h, const dgp_spec* spec, const double* X, const double* y,
                  const double* noise, int n, int on_device);

/* Dense K(X, X; theta) WITHOUT noise, n x n row-major, into K_out (parity/debug entry). */
int dgp_covmat(dgp_handle h, const double* theta, double* K_out, int out_on_device);
/* Cross covariance K(Xs, X; theta), m x n row-major (parity/debug entry). */
int dgp_cross_covmat(dgp_handle h, const double* theta, const double* Xs, int m, int xs_on_device,
                     double* K_out, int out_on_device);

/* NLML = 1/2 r'Ky^-1 r + sum log L_ii + n/2 log 2pi with Ky = K + diag(noise) + (theta[noise_theta]
 * + jitter) I and r = y - mean(X).  theta: host array [ntheta] of NATURAL parameter values. */
int dgp_nlml(dgp_handle h, const double* theta, double jitter, double* nlml_out);

/* NLML and its gradient w.r.t. every natural parameter (kernel, mean, learned noise):
 * -1/2 tr((alpha alpha' - Ky^-1) dK/dtheta), -J'alpha, -1/2 tr W.  grad_out: host [ntheta]. */
int dgp_nlml_grad(dgp_handle h, const double* theta, double jitter, double* nlml_out, double* grad_out);

/* Asynchronous pair for multi-site overlap: launch enqueues the whole evaluation and the
 * device-to-host copy of the results on the handle's stream; wait blocks on that stream. */
int dgp_nlml_grad_launch(dgp_handle h, const double* theta, double jitter);
int dgp_nlml_grad_wait(dgp_handle h, double* nlml_out, double* grad_out);
/* Non-blocking poll of the evaluation in flight: 1 = finished (dgp_nlml_grad_wait returns at once), 0 = still
 * running, < 0 = error / nothing in flight.  Lets a host thread that drives many sites (the reference's
 * `fexec.map` over sites, examples/nwqn-loadest-example/nwqn-loadest-example.py:156-157) serve them in completion
 * order instead of in a fixed round. */
int dgp_nlml_grad_ready(dgp_handle h);

/* Factorise at theta and keep L, L^-1 and alpha resident for dgp_predict / dgp_sample. */
int dgp_factorize(dgp_handle h, const double* theta, double jitter, double* nlml_out);

/* Posterior mean m(x*) + K*x alpha and LATENT variance k** - |L^-1 Kx*|^2 at Xs[m, ndim]
 * (host adds the likelihood-noise rule and clamp of SURVEY A.5).  var_out may be NULL. */
int dgp_predict(dgp_handle h, const double* Xs, int m, int on_device, double* mu_out, double* var_out);

/* Adjoint of the posterior mean: F = sum_p c[p] mu(Xs[p]) and dF/dtheta[ntheta] (natural parameters, including mean
 * and learned-noise parameters) at the theta of the last dgp_nlml_grad / dgp_factorize.  Replaces the autograd pass
 * through two eval-mode predictions in the rating-curve monotonicity penalty (rating_gp/models/gpytorch.py:126-187):
 * once the active set is fixed the penalty is such a functional.  Host pointers; m <= prediction chunk. */
int dgp_mean_functional_grad(dgp_handle h, const double* Xs, int m, const double* c, double* val_out,
                             double* grad_out);

/* Joint latent posterior draws out[S, m] = mu* + Z[S, m] Lpost' with Lpost the exact Cholesky
 * factor of K** - K*x Ky^-1 Kx* (+ jitter I).  Z: caller-supplied standard normals. */
int dgp_sample(dgp_handle h, const double* Xs, int m, const double* Z, int S, double jitter,
               double* out, int on_device);

/* Extended sampling entry.
 *  - Z == NULL: the base normals are generated on the device, Z[s, i] = standard normal number s*m + i of the
 *    Philox4x32-10 stream keyed by `seed` (Box-Muller; generator documented in csrc/dgp_panel.cuh), so the S x m
 *    matrix never crosses PCIe.
 *  - red != NULL: instead of the draws, out[S, ngroups] receives, for every draw, the grouped sums
 *      sum_{i in [group_start[g], group_start[g+1])} weight[i] * T(draw[s, i]),  T(z) = exp(z*y_scale + y_mean) or affine,
 *    i.e. concentration_to_flux + annual resample-sum of src/loadest_gp/utils.py:14-56,89 applied on the device
 *    (weight[i] = flow_i * dt * 1e-3, groups = calendar years of a time-sorted grid).  weight / group_start: host. */
typedef struct {
  double y_mean, y_scale;       /* target pipeline: model space -> original units                 */
  int32_t log_transform;        /* 1: exp, clipped below at 1e-6 (LogStandardPipeline); 2: affine clipped at 0
                                   (StandardPipeline); 0: affine                                     */
  int32_t ngroups;
  const double* weight;         /* [m]                                                              */
  const int32_t* group_start;   /* [ngroups + 1], non-decreasing indices into the grid              */
} dgp_flux_reduce;
int dgp_sample_ex(dgp_handle h, const double* Xs, int m, const double* Z, unsigned long long seed, int S,
                  double jitter, const dgp_flux_reduce* red, double* out, int on_device);

/* Workspace of dgp_sample / dgp_sample_ex / dgp_dist_*: sized ahead of time for grids of up to max_m_sample points, max_S
 * draws and max_groups flux groups, so that those calls allocate nothing (dgp_sample_ex: 8 (m n + m^2) B + O(m); the
 * dgp_dist_* term is that of world 1, the largest: dgp_dist_arena_bytes(h, m, S, 1, 0), about 4 m^2 B + O(m)).  Without it
 * the first call that needs more grows the workspace once and keeps it.  max_m_sample = 0 releases it. */
int dgp_reserve(dgp_handle h, int max_m_sample, int max_S, int max_groups);

/* Distributed joint posterior sampling: the per-rank half of a panel-cyclic Cholesky of the m x m posterior covariance
 * (the exchange step of SURVEY 8e).  Panel p (panel_cols / 128 block columns) belongs to rank p mod world, and only its
 * owner stores it: the rows from the panel's diagonal down (the lower trapezoid of its columns), so the posterior
 * covariance takes about 4 mpad^2 / world bytes per rank.  The handle's workspace holds those slabs, two receive slots
 * [mpad, panel_cols] for broadcast panels, Z and the staging buffers: dgp_dist_arena_bytes(h, m, S, world, rank) bytes
 * (0 on bad arguments or without training data), allocated by dgp_dist_begin unless dgp_reserve made room.  The caller
 * owns the collectives and the exchanged DEVICE buffers (row-major float64):
 *   VT   [rows_per_rank * world, npad]  V' = Kx T'; every rank fills its row shard, the caller all-gathers
 *   pack [mpad, panel_cols]             rows below a factored panel's diagonal blocks, broadcast from its owner
 *                                       (passed per call: the caller may double-buffer it)
 *   Od   [Spad, mpad]                   partial draws, all-reduced (sum) by the caller
 *   mu   [mpad]                         posterior mean, each rank fills its rows (zeros elsewhere): all-reduce (sum)
 * dgp_dist_dims -> {mpad, npad, Spad, panel_cols, npanels, rows_per_rank}.  Rank r's V' shard is rows
 * [r rows_per_rank, (r + 1) rows_per_rank); dgp_dist_vt_rows clamps both ends to mpad, so a shard may be empty: when world
 * is large for mb = mpad / 128 (world 3 with mb 1, world 8 with mb 41) the last ranks' shards lie at or past mpad, and
 * vt_rows on them succeeds and does nothing.  A rank that owns no panel is valid too.  Call order per rank:
 *   begin -> vt_rows(my shard) -> [all_gather VT, all_reduce mu] -> sigma ->
 *   for p: (owner: panel_factor) -> [broadcast pack] -> (others: panel_unpack) -> trail(p, p+1, npanels-1)
 *          (look-ahead: trail(p, p+1, p+1) first, factor panel p+1 on a side stream while trail(p, p+2, ...) runs)
 *   -> draws_partial -> [all_reduce Od] -> finish(out host [S, m]) or finish_ex -> end.
 * Everything is enqueued on the handle's stream (pass the stream the collectives are ordered against to dgp_create).
 * Z: host base normals [S, m] or NULL for the Philox stream `seed` (identical on every rank). */
typedef struct dgp_dist_s* dgp_dist;
int dgp_dist_dims(dgp_handle h, int m, int S, int world, long long* dims6);
int dgp_dist_begin(dgp_handle h, const double* Xs, int m, int S, const double* Z, unsigned long long seed, double jitter,
                   int rank, int world, double* VT, double* Od, double* mu, dgp_dist* out);
int dgp_dist_vt_rows(dgp_dist d, int row0, int row1);
int dgp_dist_sigma(dgp_dist d);
int dgp_dist_panel_factor(dgp_dist d, int p, double* pack, void* stream);
int dgp_dist_panel_unpack(dgp_dist d, int p, double* pack);
int dgp_dist_trail(dgp_dist d, int p, int j_first, int j_last);
int dgp_dist_draws_partial(dgp_dist d);
int dgp_dist_finish(dgp_dist d, double* out);  /* > 0: first non-positive pivot met on THIS rank's panels */
/* dgp_dist_finish with the grouped flux reduction of dgp_sample_ex (red != NULL: out host [S, ngroups], computed on the
 * device from this rank's all-reduced draws; the checks on red are dgp_sample_ex's).  red == NULL: dgp_dist_finish. */
int dgp_dist_finish_ex(dgp_dist d, const dgp_flux_reduce* red, double* out);
int dgp_dist_end(dgp_dist d);
size_t dgp_dist_arena_bytes(dgp_handle h, int m, int S, int world, int rank);

/* Parity accessors (valid after dgp_nlml* / dgp_factorize): alpha[n]; L[n, n] lower triangular. */
int dgp_get_alpha(dgp_handle h, double* alpha_out, int out_on_device);
int dgp_get_chol(dgp_handle h, double* L_out, int out_on_device);
/* Ky^-1 [n, n] (lower triangle valid), materialised only when debug_kinv was enabled. */
int dgp_set_debug_kinv(dgp_handle h, int enable);
int dgp_get_kinv(dgp_handle h, double* Kinv_out, int out_on_device);
/* T = L^-1 [n, n], lower triangular (zeros above the diagonal): the inverse the variance and sampling products use.  Valid
 * after a successful dgp_factorize only (dgp_nlml_grad overwrites it with Ky^-1); fails with a message otherwise. */
int dgp_get_linv(dgp_handle h, double* T_out, int out_on_device);
/* U = L^-T [n, n], upper triangular: the operand of the LAUUM that forms Ky^-1.  Valid after dgp_nlml_grad or
 * dgp_factorize; fails with a message otherwise. */
int dgp_get_uinv(dgp_handle h, double* U_out, int out_on_device);

/* Utility: the FP64 tensor-pipe tile engine as a plain product on device pointers,
 * C[M, N] = A[M, K] B[N, K]' (mode 0), C += A B' (mode 1), C -= A B' (mode -1).
 * M % 128 == 0, N % 64 == 0, K % 16 == 0; row-major with leading dimensions lda/ldb/ldc. */
int dgp_gemm_nt(dgp_handle h, const double* A, long long lda, const double* B, long long ldb, double* C,
                long long ldc, int M, int N, int K, int mode);

/* ---------------------------------------------------------------------------------------------------------------
 * Batched, variable-size multi-site evaluation: up to DGP_BATCH_MAX_SITES independent sites that share one covariance
 * spec (an NWQN-style batch of loadest-gp sites, a set of rating-gp gauges) evaluated by ONE launch sequence.  Replaces
 * the reference's one-worker-per-site map, examples/nwqn-loadest-example/nwqn-loadest-example.py:156-157 (fexec.map over
 * sites, each running MarginalGPyTorch.fit, discontinuum/engines/gpytorch.py:346-444) and the per-gauge loop of
 * docs/source/notebooks/rating-gp-demo.ipynb.  Every kernel launch of the single-site schedule covers all sites (tile
 * index -> (site, tile) through a per-launch prefix table), so the latency-bound panel chain is paid once per block step
 * for the whole batch.  Sites of different n are end-aligned; per site the arithmetic is that of dgp_nlml_grad (and of
 * dgp_factorize + dgp_predict), bit for bit.  Workspace (3 max_sites x max_n^2 float64 + O(max_sites max_n)) is allocated
 * at create.  The first dgp_batch_predict on a handle adds the prediction slabs, once: 8 max_sites x 1024 x (max_pad +
 * 3 max_pad / 128 + 19) B on the device (max_pad = max_n rounded up to 128; the cross covariance of 1024 grid rows per
 * site) and 80 max_sites x 1024 B of pinned host memory.  Every other call allocates nothing, and handles that never
 * predict keep the create-time footprint.  The first dgp_batch_nlml_grad with a site of at least 8192 padded points
 * adds the residue buffers of the INT8 LAUUM once, for one site at a time: 16 max_pad^2 + 2052 max_pad B.  Host pointers
 * throughout. */
#define DGP_BATCH_MAX_SITES 32
typedef struct dgp_batch_s* dgp_batch;
int dgp_batch_create(dgp_batch* out, int device, int max_sites, int max_n, void* stream);
int dgp_batch_destroy(dgp_batch b);
const char* dgp_batch_last_error(dgp_batch b); /* b may be NULL: error of a failed dgp_batch_create */
/* Device bytes allocated by dgp_batch_create (the prediction slabs of the first dgp_batch_predict and the INT8 LAUUM's
 * residue buffers of the first gradient evaluation with a site of >= 8192 padded points are not included). */
size_t dgp_batch_workspace_bytes(int max_sites, int max_n);
/* Training sets of nsites sites: n[s] points each, X[s][n[s], ndim], y[s][n[s]], noise[s][n[s]] (host arrays of host pointers). */
int dgp_batch_set_train(dgp_batch b, const dgp_spec* spec, int nsites, const int* n, const double* const* X,
                        const double* const* y, const double* const* noise);
/* NLML and gradient of every site.  theta[nsites][ntheta] natural parameters, jitter[nsites] (NULL: 0);
 * nlml_out[nsites], grad_out[nsites][ntheta], info_out[nsites] (LAPACK-style, 0 = ok) may each be NULL.
 * Returns the number of sites with info != 0, or < 0 (bad argument / CUDA error). */
int dgp_batch_nlml_grad(dgp_batch b, const double* theta, const double* jitter, double* nlml_out, double* grad_out,
                        int* info_out);
/* Asynchronous form: launch enqueues the evaluation and the device-to-host copy of the results; ready polls (1 / 0 / < 0);
 * wait blocks and returns like dgp_batch_nlml_grad. */
int dgp_batch_nlml_grad_launch(dgp_batch b, const double* theta, const double* jitter);
int dgp_batch_nlml_grad_ready(dgp_batch b);
int dgp_batch_nlml_grad_wait(dgp_batch b, double* nlml_out, double* grad_out, int* info_out);
/* Factorise every site of the batch at theta[nsites][ntheta] (+ jitter[nsites], NULL: 0) and keep, per site, L^-1 and
 * alpha resident for dgp_batch_predict (the batch form of dgp_factorize).  nlml_out[nsites], info_out[nsites] may be NULL.
 * Returns the number of sites with info != 0, or < 0. */
int dgp_batch_factorize(dgp_batch b, const double* theta, const double* jitter, double* nlml_out, int* info_out);
/* Posterior mean m(x*) + K*x alpha and LATENT variance k** - |L^-1 Kx*|^2 of every site on its own grid:
 * m[s] points Xs[s][m[s], ndim] -> mu_out[s][m[s]], var_out[s][m[s]] (host pointers; var_out == NULL or var_out[s] == NULL:
 * mean only; m[s] == 0: site skipped).  The variance of a site needs its successful dgp_batch_factorize since the last
 * dgp_batch_set_train / dgp_batch_nlml_grad; the mean alone needs a successful dgp_batch_factorize or dgp_batch_nlml_grad
 * of the site (as dgp_predict); fails (< 0) otherwise.  Grids are walked in chunks of 1024 rows, each chunk
 * of all sites in one launch sequence; the results equal dgp_predict's bit for bit. */
int dgp_batch_predict(dgp_batch b, const int* m, const double* const* Xs, double* const* mu_out, double* const* var_out);
/* Batch form of dgp_mean_functional_grad: for every site s with m[s] > 0, F_s = sum_p c[s][p] mu_s(Xs[s][p]) and
 * dF_s/dtheta_s (natural parameters, including mean and learned-noise parameters) at the theta of the site's last
 * successful dgp_batch_nlml_grad or dgp_batch_factorize.  m[s] <= 1024; m[s] == 0: site skipped (val 0, grad zeros).
 * val_out[nsites], grad_out[nsites][ntheta] (host).  Results equal dgp_mean_functional_grad of a per-site handle bit for bit.
 * Fails (< 0) on NULL pointers, m[s] > 1024, a site with m[s] > 0 whose last evaluation did not succeed (or none since
 * dgp_batch_set_train), and while an evaluation is in flight.  Each step is one launch over all sites.  The first call on a
 * handle adds the adjoint slabs, once: 8 max_sites x (1024 + max_pad (3 + max_pad / 128) + (8 + max_pad / 128)
 * (max_pad / 64) 48 + 49) B on the device, next to the prediction slabs (which it also uses and allocates if
 * dgp_batch_predict has not), and 8 max_sites x 1073 B of pinned host memory.  Later calls allocate nothing. */
int dgp_batch_mean_functional_grad(dgp_batch b, const int* m, const double* const* Xs, const double* const* c,
                                   double* val_out, double* grad_out);
/* Batch form of dgp_sample_ex.  For every site s with m[s] > 0: S joint latent draws of the posterior on Xs[s][m[s], ndim]
 * (out[s][S, m[s]]) or, with red != NULL and red[s] != NULL, their grouped sums (out[s][S, red[s]->ngroups]).  Z == NULL:
 * the normals of site s are the Philox4x32-10 stream keyed by seed[s] (dgp_sample_ex's numbering); else Z[s][S, m[s]] host
 * normals (seed may then be NULL).  jitter[s] (NULL: 0) is added to the diagonal of site s's posterior covariance.
 * info_out[nsites]: LAPACK-style, 0 = ok (and 0 for skipped sites); a site whose posterior covariance is not positive
 * definite gets info > 0 and does not affect the others.  Per site the draws, sums and info equal those of dgp_sample_ex
 * on a handle factorised at the same training set, theta and jitter, bit for bit.  Each step is one launch over all
 * sampled sites: normals, per 1024-row chunk the cross covariance and V' = Kx T', Sigma* = K** + jitter I - V'V', the
 * in-place posterior Cholesky (end-aligned like the training factorisation), the draws, the mean, the grouped sums.
 * Needs a successful dgp_batch_factorize of every sampled site since the last dgp_batch_set_train / dgp_batch_nlml_grad;
 * reads T = L^-1, alpha and the training features and writes nothing later factorisations, predictions or evaluations
 * read.  Fails (< 0) on NULL pointers, m[s] < 0, S < 1, a malformed red[s] (the checks of dgp_sample_ex), a sampled site
 * without that factorisation, and while an evaluation is in flight.  Returns the number of sampled sites with info != 0.
 * Workspace: a grow-only sampling arena on the handle (freed at destroy, allocated only when a call needs more than the
 * largest before) of, per sampled site, in doubles, with mld = the largest m[s] of the call rounded up to 128, ld = the
 * largest training n of the batch rounded up to 128, Spad = S rounded up to 128:
 *   mld^2 + mld ld + 2 Spad mld + 2 128 mld + 9 mld + 105 (+ mld + S ng + (ng + 1) / 2 when any site reduces, ng = the
 *   largest ngroups), every slab rounded up to 256 B
 * (1.9 GB per site at m = 10 958, n <= 8 000, S = 1000).  The prediction slabs of dgp_batch_predict are used (and
 * allocated if no prediction has). */
int dgp_batch_sample_ex(dgp_batch b, const int* m, const double* const* Xs, int S, const double* const* Z,
                        const unsigned long long* seed, const double* jitter, const dgp_flux_reduce* const* red,
                        double* const* out, int* info_out);
/* Device bytes of the sampling arena a dgp_batch_sample_ex call with these m[] / S / red[] needs (0 for a malformed call or
 * one that samples no site). */
size_t dgp_batch_sample_bytes(dgp_batch b, const int* m, int S, const dgp_flux_reduce* const* red);
/* Parity accessor: alpha of one site after an evaluation. */
int dgp_batch_get_alpha(dgp_batch b, int site, double* alpha_out);
long long dgp_batch_launch_count(dgp_batch b);
/* Device time (ms) of the last evaluation: factorisation / inverse / LAUUM + gradient / rest. */
int dgp_batch_set_timing(dgp_batch b, int enable);
int dgp_batch_last_timing(dgp_batch b, double* ms4);

/* Counters for bench.py: kernels launched by this handle since creation. */
long long dgp_launch_count(dgp_handle h);
/* Device time (ms, CUDA events on the handle's stream) of the last dgp_nlml / dgp_nlml_grad /
 * dgp_factorize, split as potrf / trtri / lauum+grad / rest. */
int dgp_last_timing(dgp_handle h, double* ms4);
int dgp_set_timing(dgp_handle h, int enable);

#ifdef __cplusplus
}
#endif
#endif /* DGP_H */
