"""The factorisation schedule of libdgp at every size class where it changes its launches, against a float64 GPU reference.

Above n = 1300 the engine's correctness rests on the schedule of `potrf_core`, `factor_panel`, `trtri_advance` and
`eager_hook` (csrc/dgp_api.cu), which switches launches at fixed sizes.  With `sms` SMs (`slots = 2 sms` CTA slots) and
nb = ceil(n / 128) block columns:

  switch                                                        condition (dgp_api.cu)        first nb (148 SMs)
  ------------------------------------------------------------  ----------------------------  ------------------
  panel solve (TRSM) on full 128-row tiles                       4 (nb - s - 1) > 2 sms        76   (n >= 9601)
  inverse merges released during the factorisation               nb <= EAGER_INV_MAX_NB = 96   97 is the first without
  first-column trailing update on full tiles                     2 (nb - pe) > slots           153  (n >= 19457)
  ragged last panel / strip, `pe & 7` advance points, ragged     nb mod 4, nb mod 8, nb not a power of two
    merge levels

`sizes(sms)` derives one n per class from the device's SM count and asserts that it lands there.  On a 148-SM B200 they are
9601 (nb 76: first full-tile TRSM, eager inverse, one valid row in the last block, half a last strip), 11000 (nb 86: last
panel of 2 columns), 12288 (nb 96: last eager size), 12289 (nb 97: first size without eager release, top merge level
[0, 64) | [64, 97)), 14000 (nb 110) and 19457 (nb 153: first-column update on full tiles, last panel and strip of one
column).  The sites are loadest sites at theta1; one rating gauge at the first lazy size adds the gate, learned-noise and
power-law-mean gradient.

The reference is the oracle (oracle/gp_oracle.py) on CUDA tensors: cuSOLVER / cuBLAS in float64, which share no code with
libdgp.  test_gpu_reference_matches_cpu_oracle pins it to the CPU oracle at n = 2048.  Per size:
  * backward errors, which bound what rounding allows whatever the conditioning (LAPACK's test ratios; its own suite
    accepts 30, these tests accept 1, and print cuSOLVER's ratio beside the engine's):
      DPOT01  ||Ky - L L'||_1 / (n ||Ky||_1 eps)                      L of nlml_grad and of the NLML-only path
      DPOT03  ||I - Ky Kinv||_1 / (n ||Ky||_1 ||Kinv||_1 eps)         Kinv = the LAUUM output, symmetrised from its lower tiles
      DTRT01  ||L T - I||_1 / (n ||L||_1 ||T||_1 eps)                 T = L^-1 of factorize, L of the same call
  * forward errors at max(the spec tests' tolerance, 20 kappa_1 eps), kappa_1 = ||Ky||_1 ||Ky^-1||_1: NLML (both paths),
    alpha, the gradient per component (test_spec_generic's rule and floor), mu* and var* on a 3000-point grid (two
    prediction chunks of 2048 rows).
test_sampler_posterior_factor holds the in-place posterior Cholesky of dgp_sample to the same DPOT01 bar at mb = 9, the
first full-tile TRSM size and the first full-tile first-column size; test_batch_matches_per_site_across_eager_limit holds
the batch engine, which releases the inverse eagerly at every size, bit for bit to per-site handles on both sides of the
single-site limit.
"""
import time

import numpy as np
import pytest
import torch

import helpers as H
from helpers import orc
from discontinuum_b200 import capi, models, synthetic
from test_spec_generic import GRAD_FLOOR, TOL_G_ABS, TOL_G_REL, TOL_NLML, TOL_VEC

pytestmark = pytest.mark.gpu

EAGER_INV_MAX_NB = 96   # csrc/dgp_api.cu: a single site releases the inverse merges during the factorisation up to here
PANEL_BLOCKS, STRIP_BLOCKS = 4, 8   # csrc/dgp_api.cu
EPS = float(np.finfo(np.float64).eps)
RATIO_MAX = 1.0
KAPPA_FACTOR = 20.0
GRID_M = 3000
GRID_SHIFT = {"loadest": np.array([0.0004, 0.01]), "rating": np.array([0.0004, 0.001])}
DEV = "cuda"


def _nb(n):
    return (n + 127) // 128


def _switches(sms):
    """first nb of the full-tile panel solve and of the full-tile first-column trailing update (dgp_api.cu)"""
    nb_trsm = next(nb for nb in range(2, 4 * sms) if 4 * (nb - 1) > 2 * sms)        # s = 0: m = nb - 1
    nb_col0 = next(nb for nb in range(2, 4 * sms) if 2 * (nb - PANEL_BLOCKS) > 2 * sms)  # first panel: pe = 4
    return nb_trsm, nb_col0


def _pow2(x):
    return x & (x - 1) == 0


def sizes(sms):
    """label -> (n, what it reaches, predicate on nb that must hold)"""
    nb_trsm, nb_col0 = _switches(sms)
    return {
        "trsm_full": (128 * (nb_trsm - 1) + 1, "first full-tile TRSM, eager inverse, 1 valid row in the last block",
                      lambda nb: nb == nb_trsm and nb <= EAGER_INV_MAX_NB and nb % STRIP_BLOCKS == 4),
        "panel2": (11000, "last panel of 2 block columns, full-tile TRSM, eager inverse",
                   lambda nb: nb_trsm < nb < EAGER_INV_MAX_NB and nb % PANEL_BLOCKS == 2 and not _pow2(nb)),
        "eager_last": (128 * EAGER_INV_MAX_NB, "last size with eager inverse release",
                       lambda nb: nb == EAGER_INV_MAX_NB and nb >= nb_trsm),
        "lazy_first": (128 * EAGER_INV_MAX_NB + 1, "first size without eager release, ragged top merge level",
                       lambda nb: nb == EAGER_INV_MAX_NB + 1 and nb < nb_col0),
        "lazy_110": (14000, "no eager release, nb not a power of two, ragged last strip",
                     lambda nb: EAGER_INV_MAX_NB < nb < nb_col0 and not _pow2(nb) and nb % STRIP_BLOCKS != 0),
        "col0_full": (128 * (nb_col0 - 1) + 1, "first full-tile first-column update, last panel and strip of 1 column",
                      lambda nb: nb == nb_col0 and nb % PANEL_BLOCKS == 1 and nb % STRIP_BLOCKS == 1),
    }


CASES = [("loadest", lab) for lab in ("trsm_full", "panel2", "eager_last", "lazy_first", "lazy_110", "col0_full")] + \
        [("rating", "lazy_first")]


@pytest.fixture(scope="module")
def size_table(cuda_device):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    tab = sizes(sms)
    for lab, (n, what, ok) in tab.items():
        assert ok(_nb(n)), (lab, n, _nb(n), sms, what)
    return tab


# ------------------------------------------------------------------------------------------------------------------
# float64 reference (the oracle on whatever device its inputs live on)
# ------------------------------------------------------------------------------------------------------------------
def _site(model, n):
    if model == "loadest":
        X, y, noise = synthetic.loadest_site(n, 1000)
        return X, y, noise, H.loadest_theta1(), models.loadest_spec(2)
    X, y, noise = synthetic.rating_gauge(n, 7)
    b_lo, b_hi = models.stage_quantile_bounds(X[:, 1])
    return X, y, noise, H.rating_theta1(b_lo, b_hi), models.rating_spec(b_lo, b_hi)


def _model(model):
    """(cov, mean, nat(theta tensor), learned extra noise of nat or None)"""
    if model == "loadest":
        return orc.loadest_cov, orc.loadest_mean, H.loadest_nat_from_theta, lambda nat: None
    return orc.rating_cov, orc.rating_mean, H.rating_nat_from_theta, lambda nat: nat["noise"]


def _n1(A):
    return float(torch.linalg.matrix_norm(A, ord=1))


class Reference:
    """Ky, its Cholesky factor L, Ky^-1, alpha, NLML and the gradient of one site, in float64 on `device`.  The gradient is
    nlml_grad_closed_form's trace formula -1/2 sum_ij W_ij dK_ij / dtheta - alpha' dm / dtheta (W = alpha alpha' - Ky^-1),
    taken by autograd over row blocks of at most `block` rows so that the graph stays a few GB at n = 19 457."""

    def __init__(self, model, X, y, noise, theta, device, block=1024):
        self.cov, self.mean, self.nat_of, self.extra_of = _model(model)
        self.X, y, noise = (torch.tensor(a, device=device) for a in (X, y, noise))
        self.theta = torch.tensor(theta, device=device)
        self.n = n = self.X.shape[0]
        with torch.no_grad():
            nat = self.nat_of(self.theta)
            self.Ky = self.cov(self.X, self.X, nat)
            extra = self.extra_of(nat)
            self.Ky.diagonal().add_(noise if extra is None else noise + extra)
            r = y - self.mean(self.X, nat)
            self.L = torch.linalg.cholesky(self.Ky)
            self.alpha = torch.cholesky_solve(r[:, None], self.L)[:, 0]
            self.nlml = float(0.5 * (r @ self.alpha) + torch.log(torch.diagonal(self.L)).sum() + 0.5 * n * orc.LOG2PI)
            self.Kinv = torch.cholesky_inverse(self.L)
        th = self.theta.clone().requires_grad_(True)
        grad = torch.zeros_like(th)
        for i0 in range(0, n, block):
            i1 = min(n, i0 + block)
            nat = self.nat_of(th)
            W = self.alpha[i0:i1, None] * self.alpha[None, :] - self.Kinv[i0:i1]
            s = -0.5 * (W * self.cov(self.X[i0:i1], self.X, nat)).sum()
            extra = self.extra_of(nat)
            if extra is not None:
                s = s - 0.5 * torch.diagonal(W[:, i0:i1]).sum() * extra.reshape(())
            grad += torch.autograd.grad(s, th)[0]
        s = -(self.alpha * self.mean(self.X, self.nat_of(th))).sum()
        grad += torch.autograd.grad(s, th)[0]
        self.grad = grad.cpu().numpy()

    def kappa1(self):
        return _n1(self.Ky) * _n1(self.Kinv)

    def predict(self, Xs):
        """posterior mean and latent variance at Xs[m, d] (host array) from this reference's L and alpha"""
        Xs = torch.tensor(Xs, device=self.X.device)
        with torch.no_grad():
            nat = self.nat_of(self.theta)
            Kx = self.cov(Xs, self.X, nat)
            mu = self.mean(Xs, nat) + Kx @ self.alpha
            V = torch.linalg.solve_triangular(self.L, Kx.T, upper=False)
            kss = orc._diag_cov(self.cov, Xs, nat)
            return mu.cpu().numpy(), (kss - (V * V).sum(0)).cpu().numpy()


# ------------------------------------------------------------------------------------------------------------------
# LAPACK test ratios
# ------------------------------------------------------------------------------------------------------------------
def dpot01(Ky, L):
    """||Ky - L L'||_1 / (n ||Ky||_1 eps)"""
    R = torch.mm(L, L.T)
    R -= Ky
    return _n1(R) / (Ky.shape[0] * _n1(Ky) * EPS)


def dpot03(Ky, Kinv):
    """||I - Ky Kinv||_1 / (n ||Ky||_1 ||Kinv||_1 eps)"""
    R = torch.mm(Ky, Kinv)
    R.neg_().diagonal().add_(1.0)
    return _n1(R) / (Ky.shape[0] * _n1(Ky) * _n1(Kinv) * EPS)


def dtrt01(L, T):
    """||L T - I||_1 / (n ||L||_1 ||T||_1 eps)"""
    R = torch.mm(L, T)
    R.diagonal().sub_(1.0)
    return _n1(R) / (L.shape[0] * _n1(L) * _n1(T) * EPS)


def _sym_from_lower(A):
    """the lower triangle of A mirrored into its upper triangle"""
    S = torch.tril(A)
    S += torch.tril(A, -1).T
    return S


def _rel(got, want):
    got, want = np.asarray(got), np.asarray(want)
    return float(np.max(np.abs(got - want)) / np.max(np.abs(want)))


def _grad_err(got, want, rel):
    """max over components of |g - o| / (rel |o| + TOL_G_ABS max|o|): <= 1 passes (test_spec_generic's rule)"""
    return float(np.max(np.abs(got - want) / (rel * np.abs(want) + TOL_G_ABS * np.max(np.abs(want)))))


def _free():
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------------------------
# the reference itself
# ------------------------------------------------------------------------------------------------------------------
def test_gpu_reference_matches_cpu_oracle(cuda_device):
    """The GPU reference (this file's blocked trace formula included) against the CPU oracle's nlml_grad_closed_form at
    n = 2048: K, NLML and the gradient to 1e-12 relative.  alpha may differ by up to kappa_1 eps where that is larger: two
    backward-stable Cholesky solves can differ by that much, and two CPU LAPACK builds already differ by 9e-13 in alpha at
    n = 1024."""
    n = 2048
    X, y, noise, theta, _ = _site("loadest", n)
    ref = Reference("loadest", X, y, noise, theta, DEV)
    Xt, yt, nt = (torch.tensor(a) for a in (X, y, noise))
    nat = H.loadest_nat_from_theta(theta)
    v, g, a, _ = orc.nlml_grad_closed_form(orc.loadest_cov, orc.loadest_mean, nat, Xt, yt, nt)
    g = H.loadest_theta_from_nat({k: t.numpy() for k, t in g.items()})
    K_cpu = orc.loadest_cov(Xt, Xt, nat)
    K_gpu = ref.Ky.cpu()
    K_gpu.diagonal().sub_(nt)
    err = {"K": _rel(K_gpu.numpy(), K_cpu.numpy()), "nlml": abs(ref.nlml - float(v)) / abs(float(v)),
           "alpha": _rel(ref.alpha.cpu().numpy(), a.numpy()), "grad": _rel(ref.grad, g)}
    kappa = ref.kappa1()
    print(f"\nGPU reference vs CPU oracle, n = 2048, kappa1 = {kappa:.2e}: " + " ".join(f"{k}={e:.1e}" for k, e in err.items()))
    lim = {"K": 1e-12, "nlml": 1e-12, "alpha": max(1e-12, kappa * EPS), "grad": 1e-12}
    assert all(err[k] <= lim[k] for k in err), (err, lim)


def test_linv_accessor(cuda_device):
    """dgp_get_linv: T = L^-1 after factorize, to the host or into a CUDA tensor, zeros above the diagonal; refused before
    any evaluation and after nlml_grad / nlml (which leave other contents where T was); `out` of the wrong shape refused.
    Also: Engine.sample refuses a CUDA grid with host normals."""
    n = 300
    X, y, noise, theta, spec = _site("loadest", n)
    eng = capi.Engine(max_n=n, max_m=256)
    eng.set_train(spec.to_c(), X, y, noise)
    with pytest.raises(capi.DgpError, match="dgp_get_linv"):
        eng.linv()
    eng.factorize(theta)
    T = eng.linv()
    Td = eng.linv(out=torch.empty((n, n), dtype=torch.float64, device=DEV))
    assert np.array_equal(Td.cpu().numpy(), T)
    assert np.all(np.triu(T, 1) == 0.0)
    L = eng.chol()
    assert np.array_equal(eng.chol(out=torch.empty((n, n), dtype=torch.float64, device=DEV)).cpu().numpy(), L)
    assert np.max(np.abs(T @ L - np.eye(n))) <= 1e-10
    with pytest.raises(ValueError):
        eng.linv(out=torch.empty((n, n + 1), dtype=torch.float64, device=DEV))
    for call in (eng.nlml_grad, eng.nlml):
        call(theta)
        with pytest.raises(capi.DgpError, match="dgp_get_linv"):
            eng.linv()
    # sample: the grid on the GPU with host normals is refused before anything is launched
    with pytest.raises(ValueError, match="Z is not"):
        eng.sample(torch.tensor(X[:8], device=DEV), np.zeros((2, 8)))
    eng.close()


# ------------------------------------------------------------------------------------------------------------------
# single site: every size class
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model,label", CASES)
def test_single_site_schedule(cuda_device, size_table, model, label):
    n, what, _ = size_table[label]
    t0 = time.time()
    X, y, noise, theta, spec = _site(model, n)
    # every n x n tensor and the engine are released in `finally`, so that a failing size does not hold ~15 GB into the next
    ref = eng = A = B = L = T = Ki = None
    try:
        ref = Reference(model, X, y, noise, theta, DEV)
        kappa = ref.kappa1()
        fwd = KAPPA_FACTOR * kappa * EPS
        tol_nlml, tol_vec, tol_g = max(TOL_NLML, fwd), max(TOL_VEC, fwd), max(TOL_G_REL, fwd)
        assert np.all(np.abs(ref.grad) >= GRAD_FLOOR * np.max(np.abs(ref.grad))), ref.grad
        ratio, err = {}, {}
        with torch.no_grad():
            ratio["dpot01_cusolver"] = dpot01(ref.Ky, ref.L)
            ratio["dpot03_cusolver"] = dpot03(ref.Ky, ref.Kinv)
            T_ref = torch.linalg.solve_triangular(ref.L, torch.eye(n, dtype=torch.float64, device=DEV), upper=False)
            ratio["dtrt01_cusolver"] = dtrt01(ref.L, T_ref)
            del T_ref
        eng = capi.Engine(max_n=n, max_m=2048)
        eng.set_train(spec.to_c(), X, y, noise)
        A = torch.empty((n, n), dtype=torch.float64, device=DEV)
        B = torch.empty((n, n), dtype=torch.float64, device=DEV)
        # NLML + gradient, with the LAUUM output kept
        eng.set_debug_kinv(True)
        val, grad, info = eng.nlml_grad(theta)
        assert info == 0
        err["nlml"] = abs(val - ref.nlml) / abs(ref.nlml)
        err["alpha"] = _rel(eng.alpha(), ref.alpha.cpu().numpy())
        err["grad"] = _grad_err(grad, ref.grad, tol_g)
        err["grad_rel"] = float(np.max(np.abs(grad - ref.grad) / np.abs(ref.grad)))
        with torch.no_grad():
            L = eng.chol(out=A)
            assert torch.count_nonzero(torch.triu(L, 1)) == 0, "L has entries above the diagonal"
            ratio["dpot01"] = dpot01(ref.Ky, L)
            Ki = _sym_from_lower(eng.kinv(out=B))
            ratio["dpot03"] = dpot03(ref.Ky, Ki)
            Ki = None
        # NLML-only path (forward substitution in the panel chain)
        val0, info0 = eng.nlml(theta)
        assert info0 == 0
        err["nlml_only"] = abs(val0 - ref.nlml) / abs(ref.nlml)
        with torch.no_grad():
            ratio["dpot01_nlml_only"] = dpot01(ref.Ky, eng.chol(out=A))
        # factorise for prediction: T = L^-1 (its last merge level transposed) and the posterior on two prediction chunks
        _, infof = eng.factorize(theta)
        assert infof == 0
        with torch.no_grad():
            L, T = eng.chol(out=A), eng.linv(out=B)
            assert torch.count_nonzero(torch.triu(L, 1)) == 0
            ratio["dtrt01"] = dtrt01(L, T)
        Xs = synthetic.daily_grid(X, GRID_M) + GRID_SHIFT[model]
        mu, var = eng.predict(Xs)
        mu_r, var_r = ref.predict(Xs)
        err["mu"] = _rel(mu, mu_r)
        err["var"] = _rel(var, var_r)
    finally:
        if eng is not None:
            eng.close()
        ref = A = B = L = T = Ki = None
        _free()
    print(f"\n{model} {label} n={n} nb={_nb(n)} kappa1={kappa:.2e} fwd_tol={fwd:.1e} ({time.time() - t0:.1f} s; {what})\n  "
          + " ".join(f"{k}={v:.2e}" for k, v in ratio.items()) + "\n  " + " ".join(f"{k}={v:.2e}" for k, v in err.items()))
    lim = {"nlml": tol_nlml, "nlml_only": tol_nlml, "alpha": tol_vec, "mu": tol_vec, "var": tol_vec, "grad": 1.0,
           "grad_rel": np.inf}
    bad = {k: v for k, v in err.items() if not v <= lim[k]}
    bad.update({k: v for k, v in ratio.items() if not v <= RATIO_MAX})
    assert not bad, (model, label, n, bad)


# ------------------------------------------------------------------------------------------------------------------
# posterior factor of the sampler
# ------------------------------------------------------------------------------------------------------------------
SAMPLER_N, SAMPLER_JITTER = 2000, 1e-6


def _sampler_m(label, sms):
    nb_trsm, nb_col0 = _switches(sms)
    return {"mb9": 1100, "trsm_full": 128 * (nb_trsm - 1) + 1, "col0_full": 128 * (nb_col0 - 1) + 1}[label]


@pytest.mark.parametrize("label", ["mb9", "trsm_full", "col0_full"])
def test_sampler_posterior_factor(cuda_device, size_table, label):
    """dgp_sample factors Sigma* = K** + jitter I - V'V (m x m) in place.  With y = 0 and a zero constant mean, mu* = 0
    exactly, and Z = [I_m; 0] makes the draws [Lpost'; mu*]: the last row must be exactly zero, Lpost lower triangular, and
    ||Sigma - Lpost Lpost'||_1 / (m (||K**||_1 + ||V'V||_1) eps) <= 1 with Sigma formed by cuBLAS from the engine's own
    T = L^-1 (so that forming V is not counted against the Cholesky)."""
    m = _sampler_m(label, torch.cuda.get_device_properties(0).multi_processor_count)
    assert label != "mb9" or _nb(m) == 9
    t0 = time.time()
    n = SAMPLER_N
    X, _, noise = synthetic.loadest_site(n, 1005)
    y = np.zeros(n)
    theta = H.loadest_theta1()
    theta[0] = 0.0
    # the m x m tensors and the engine are released in `finally`, so that a failing size does not hold them into the next
    eng = T = Z = D = V = VtV = S = None
    try:
        eng = capi.Engine(max_n=n, max_m=2048)
        eng.set_train(models.loadest_spec(2).to_c(), X, y, noise)
        _, info = eng.factorize(theta)
        assert info == 0
        T = eng.linv(out=torch.empty((n, n), dtype=torch.float64, device=DEV))
        Xs = synthetic.daily_grid(X, m) + GRID_SHIFT["loadest"]
        Z = torch.zeros((m + 1, m), dtype=torch.float64, device=DEV)
        Z[:m].diagonal().fill_(1.0)
        D, info = eng.sample(Xs, Z, jitter=SAMPLER_JITTER)
        Z = None
        assert info == 0
        assert torch.count_nonzero(D[m]) == 0, "mu* is not exactly zero: the draws are not Lpost'"
        D = D[:m]
        assert torch.count_nonzero(torch.tril(D, -1)) == 0, "Lpost has entries above the diagonal"
        with torch.no_grad():
            nat = H.loadest_nat_from_theta(torch.tensor(theta, device=DEV))
            Xt, Xst = torch.tensor(X, device=DEV), torch.tensor(Xs, device=DEV)
            V = T @ orc.loadest_cov(Xst, Xt, nat).T        # [n, m]
            T = None
            VtV = V.T @ V
            V = None
            S = orc.loadest_cov(Xst, Xst, nat)
            nK, nV = _n1(S), _n1(VtV)
            S.diagonal().add_(SAMPLER_JITTER)
            S -= VtV
            VtV = None
            S -= torch.mm(D.T, D)   # Lpost Lpost'
            ratio = _n1(S) / (m * (nK + nV) * EPS)
    finally:
        if eng is not None:
            eng.close()
        T = Z = D = V = VtV = S = None
        _free()
    print(f"\nsampler {label} n={n} m={m} mb={_nb(m)} dpot01={ratio:.2e} ({time.time() - t0:.1f} s)")
    assert ratio <= RATIO_MAX, (label, m, ratio)


# ------------------------------------------------------------------------------------------------------------------
# batch engine across the single-site eager limit
# ------------------------------------------------------------------------------------------------------------------
def test_batch_matches_per_site_across_eager_limit(cuda_device, size_table):
    """Sites of sizes {first lazy, first full-tile TRSM, 3000} (leading dimension 12 416 on 148 SMs) in one batch handle:
    NLML, gradient and alpha, then factorize + predict, equal per-site handles bit for bit, although the batch releases the
    inverse during the factorisation at every size and a single site above EAGER_INV_MAX_NB block columns does not."""
    ns = (size_table["lazy_first"][0], size_table["trsm_full"][0], 3000)
    assert _nb(ns[0]) > EAGER_INV_MAX_NB >= _nb(ns[1])
    spec = models.loadest_spec(2)
    sites = [synthetic.loadest_site(n, 3000 + k) for k, n in enumerate(ns)]
    thetas = np.stack([H.loadest_theta1() * (1.0 + 0.01 * k) for k in range(len(ns))])
    grids = [synthetic.daily_grid(s[0], GRID_M) + GRID_SHIFT["loadest"] for s in sites]
    b = capi.BatchEngine(max_sites=len(ns), max_n=max(ns))
    try:
        b.set_train(spec.to_c(), sites)
        val, grad, info = b.nlml_grad(thetas)
        assert np.all(info == 0)
        alphas = [b.alpha(k) for k in range(len(ns))]
        fval, finfo = b.factorize(thetas)
        assert np.all(finfo == 0)
        out = b.predict(grids)
    finally:   # the batch workspace (3 x 3 x 12 416^2 doubles) is not held past a failure
        b.close()
        _free()
    for k, (X, y, noise) in enumerate(sites):
        eng = capi.Engine(max_n=X.shape[0], max_m=2048)
        try:
            eng.set_train(spec.to_c(), X, y, noise)
            v, g, i = eng.nlml_grad(thetas[k])
            assert i == 0 and val[k] == v and np.array_equal(grad[k], g), (k, val[k] - v, grad[k] - g)
            a = eng.alpha()
            assert np.array_equal(alphas[k], a), (k, np.max(np.abs(alphas[k] - a)))
            fv, fi = eng.factorize(thetas[k])
            assert fi == 0 and fval[k] == fv, (k, fval[k] - fv)
            mu, var = eng.predict(grids[k])
        finally:
            eng.close()
            _free()
        assert np.array_equal(out[k][0], mu), (k, np.max(np.abs(out[k][0] - mu)))
        assert np.array_equal(out[k][1], var), (k, np.max(np.abs(out[k][1] - var)))
