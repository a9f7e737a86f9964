"""CPU oracle for discontinuum's exact-GP marginal-likelihood path (TEST INFRASTRUCTURE ONLY).

This file is a float64 torch restatement, on the CPU, of what the reference computes on its
hot path when GPyTorch takes the exact-Cholesky branch (n <= max_cholesky_size).  It is the
checker for the CUDA engine: only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
--impl reference legs may import it.  The product package never does.  Every function that takes data tensors creates
its tensors on their device, so the same code also runs on CUDA tensors: tests/test_factor_schedule.py uses it that way
as a float64 GPU reference (cuSOLVER / cuBLAS underneath) at sizes the CPU cannot reach in a test.  The initial-value
and fixed-noise constructors (`*_init_raw`, `loadest_noise`) take no tensors and build theirs on the CPU.

PARITY STATUS.  Two layers, pinned differently:
  * what the REFERENCE owns (which kernels act on which dimensions with which priors, constraints and initial values; the
    sigmoid gate, its inversion and the log warp of rating_gp/models/kernels.py; PowerLawTransform and its clamps; the noise
    model; the objective as engines/gpytorch.py:318,353 forms it; the whole optimiser loop of engines/gpytorch.py:162-458;
    the module tree whose parameter paths are the checkpoint keys) is pinned by OUTPUTS OF THE REFERENCE'S OWN CODE RUN HERE:
    oracle/make_reference_golden.py imports the unmodified model and engine modules from /root/reference/src, executes
    them on a small stand-in for the gpytorch API (oracle/gpytorch_standin) and writes tests/golden/ref_models.json
    (covariance matrices, means, objectives, latent posteriors at two parameter sets per model; 30-iteration objective
    trajectories of MarginalGPyTorch.fit for loadest Adam / AdamW and rating Adam, one with the monotonic-rating penalty).  tests/test_reference_golden.py holds
    this oracle (<= 1e-10 / 1e-8), the checkpoint key mapping and, on the GPU, the CUDA engine and MarginalB200.fit to them.
  * the THIRD-PARTY layer underneath (gpytorch / linear_operator: unpinned in /root/reference/pyproject.toml:19-25, not
    installable in this image or on the GPU box; the reference's own tests assert no numbers on this path,
    tests/test_loadest_gp.py:77-85, tests/test_rating_gp.py:32-65) stays "parity unpinned" in the strict sense: its kernel,
    constraint, prior and marginal-likelihood formulas are restated from gpytorch's documentation (SURVEY Appendix A) both
    here and in the stand-in.  They are checked by (i) 40-digit mpmath known-answer vectors (oracle/make_golden.py ->
    tests/golden/kat_*.json), (ii) analytic n=1 / n=2 closed forms, (iii) autograd-vs-closed-form gradient agreement,
    (iv) scikit-learn's independent exact-GP implementation (tests/test_oracle_vs_sklearn.py) and (v)
    tests/test_vs_gpytorch.py, which compares oracle and engine with the real library wherever it is importable (skipped
    here).

What each function follows (paths relative to /root/reference/src):
  loadest_cov / loadest_mean      loadest_gp/models/gpytorch.py:61-128 (covar_module :71, mean :70)
  rating_cov / rating_mean        rating_gp/models/gpytorch.py:205-372, rating_gp/models/kernels.py:242-382
  loadest_* / rating_* priors     the *_prior arguments at the lines above
  objective                       gpytorch ExactMarginalLogLikelihood as called at
                                  discontinuum/engines/gpytorch.py:318,353 (SURVEY Appendix A.1)
  predict                         discontinuum/engines/gpytorch.py:599-626 (exact form of fast_pred_var)
  sample                          discontinuum/engines/gpytorch.py:551-593 with supplied base normals
"""
from __future__ import annotations

import math
from typing import Callable, Dict, Tuple

import torch

DT = torch.float64
LOG2PI = math.log(2.0 * math.pi)


# ----------------------------------------------------------------------------------------
# constraints (gpytorch.constraints semantics, SURVEY A.1)
# ----------------------------------------------------------------------------------------
def softplus(x):
    return torch.nn.functional.softplus(x)


def inv_softplus(y):
    y = torch.as_tensor(y, dtype=DT)
    return y + torch.log(-torch.expm1(-y))


def interval(raw, lo, hi):
    return lo + (hi - lo) * torch.sigmoid(raw)


def inv_interval(v, lo, hi):
    v = torch.as_tensor(v, dtype=DT)
    u = (v - lo) / (hi - lo)
    return torch.log(u) - torch.log1p(-u)


# ----------------------------------------------------------------------------------------
# priors (log densities on the transformed value)
# ----------------------------------------------------------------------------------------
def lp_halfnormal(x, s):
    return (math.log(2.0) - 0.5 * LOG2PI - math.log(s) - x * x / (2.0 * s * s)).sum()


def lp_normal(x, mu, s):
    return (-0.5 * LOG2PI - math.log(s) - (x - mu) ** 2 / (2.0 * s * s)).sum()


def lp_gamma(x, a, b):
    return (a * math.log(b) + (a - 1.0) * torch.log(x) - b * x - math.lgamma(a)).sum()


# ----------------------------------------------------------------------------------------
# stationary factors
# ----------------------------------------------------------------------------------------
def _scaled_dist(X1, X2, cols, ls):
    """Euclidean distance of x/ls over `cols`, clamped like gpytorch's covar_dist."""
    d2 = torch.zeros(X1.shape[0], X2.shape[0], dtype=DT, device=X1.device)
    for c, l in zip(cols, ls):
        diff = (X1[:, c, None] - X2[None, :, c]) / l
        d2 = d2 + diff * diff
    return d2


def k_rbf(X1, X2, cols, ls):
    return torch.exp(-0.5 * _scaled_dist(X1, X2, cols, ls))


def k_matern(X1, X2, cols, ls, nu):
    d2 = _scaled_dist(X1, X2, cols, ls)
    r = torch.sqrt(torch.clamp_min(d2, 1e-30))
    if nu == 1.5:
        a = math.sqrt(3.0) * r
        return (1.0 + a) * torch.exp(-a)
    if nu == 2.5:
        a = math.sqrt(5.0) * r
        return (1.0 + a + a * a / 3.0) * torch.exp(-a)
    raise ValueError(nu)


def k_periodic(X1, X2, col, period, lam):
    diff = (X1[:, col, None] - X2[None, :, col]) * (math.pi / period)
    return torch.exp(-2.0 * torch.sin(diff) ** 2 / lam)


# ----------------------------------------------------------------------------------------
# loadest-gp  (x = (t, q1, ..., q_{d-1}))
# ----------------------------------------------------------------------------------------
LOADEST_RAW_ORDER = ("mean_c", "s1", "lam", "period", "l1", "s2", "l2", "s3", "l3")


def loadest_init_raw(d: int = 2) -> Dict[str, torch.Tensor]:
    """GPyTorch initial values: every raw parameter 0 (-> softplus(0) = 0.6931...)."""
    z = lambda k=1: torch.zeros(k, dtype=DT)
    return {"mean_c": z(), "s1": z(), "lam": z(), "period": z(), "l1": z(),
            "s2": z(), "l2": z(d - 1), "s3": z(), "l3": z(d)}


def loadest_natural(raw):
    nat = {k: softplus(v) for k, v in raw.items() if k != "mean_c"}
    nat["mean_c"] = raw["mean_c"]
    return nat


def loadest_raw_from_natural(nat):
    raw = {k: inv_softplus(v).reshape(-1) for k, v in nat.items() if k != "mean_c"}
    raw["mean_c"] = torch.as_tensor(nat["mean_c"], dtype=DT).reshape(-1)
    return raw


def loadest_cov(X1, X2, nat):
    d = X1.shape[1]
    seasonal = nat["s1"] * k_periodic(X1, X2, 0, nat["period"], nat["lam"]) \
        * k_matern(X1, X2, [0], [nat["l1"]], 2.5)
    flow = nat["s2"] * k_rbf(X1, X2, list(range(1, d)), list(nat["l2"]))
    resid = nat["s3"] * k_matern(X1, X2, list(range(d)), list(nat["l3"]), 1.5)
    return seasonal + flow + resid


def loadest_mean(X, nat):
    return nat["mean_c"].expand(X.shape[0])


def loadest_log_prior(nat):
    lp = lp_halfnormal(nat["s1"], 1.0) + lp_normal(nat["period"], 1.0, 0.01)
    lp = lp + lp_halfnormal(nat["s2"], 2.0) + lp_gamma(nat["l2"], 2.0, 3.0)
    lp = lp + lp_halfnormal(nat["s3"], 0.2) + lp_gamma(nat["l3"], 2.0, 10.0)
    return lp


def loadest_noise(n):
    """Fixed noise 0.1**2 per point, no learned noise (loadest_gp/models/gpytorch.py:50-54)."""
    return torch.full((n,), 0.1 ** 2, dtype=DT)


# ----------------------------------------------------------------------------------------
# rating-gp  (x = (t, h), h in [1, 2])
# ----------------------------------------------------------------------------------------
RATING_SHARPNESS = 20.0
RATING_EPS = 1e-6


def rating_init_raw(b_lo, b_hi, gate_b=None, pl_a=0.0, pl_b=1.3, pl_c=0.5):
    """All positive raw parameters 0; the reference's random draws (PowerLawTransform a, b, c at
    rating_gp/models/gpytorch.py:31-36, SigmoidKernel b at kernels.py:276) replaced by constants."""
    z = lambda: torch.zeros(1, dtype=DT)
    if gate_b is None:
        gate_b = 0.5 * (b_lo + b_hi)
    raw = {k: z() for k in (
        "noise", "shiftA_s", "shiftA_lh", "shiftA_lt", "shiftB_s", "shiftB_lh", "shiftB_lt",
        "bend_s", "bend_lh", "bend_lt", "base_s", "base_l", "per_s", "per_period", "per_lam", "per_l")}
    raw["gate_b"] = inv_interval(gate_b, b_lo, b_hi).reshape(1)
    raw["pl_a"] = torch.tensor([pl_a], dtype=DT)
    raw["pl_b"] = torch.tensor([pl_b], dtype=DT)
    raw["pl_c"] = torch.tensor([pl_c], dtype=DT)
    return raw


def rating_natural(raw, b_lo, b_hi):
    nat = {}
    for k, v in raw.items():
        if k in ("pl_a", "pl_b", "pl_c"):
            nat[k] = v
        elif k == "gate_b":
            nat[k] = interval(v, b_lo, b_hi)
        elif k == "noise":
            nat[k] = softplus(v) + 1e-4
        else:
            nat[k] = softplus(v)
    return nat


def rating_project_(raw, h_min):
    """In-place projections done by every forward (rating_gp/models/gpytorch.py:39,259)."""
    with torch.no_grad():
        raw["pl_b"].clamp_(1.2, 2.5)
        raw["pl_c"].clamp_(max=float(h_min) - 1e-6)
    return raw


def _gate(h, b):
    return 1.0 / (1.0 + torch.exp(RATING_SHARPNESS * (h - b)))


def rating_cov(X1, X2, nat):
    W1 = torch.stack([X1[:, 0], torch.log(X1[:, 1] + RATING_EPS)], dim=1)
    W2 = torch.stack([X2[:, 0], torch.log(X2[:, 1] + RATING_EPS)], dim=1)
    g1, g2 = _gate(X1[:, 1], nat["gate_b"]), _gate(X2[:, 1], nat["gate_b"])
    lower = g1[:, None] * g2[None, :]
    upper = (1.0 - g1)[:, None] * (1.0 - g2)[None, :]

    def shift(p):
        return nat[p + "_s"] * k_matern(W1, W2, [1], [nat[p + "_lh"]], 2.5) \
            * k_matern(W1, W2, [0], [nat[p + "_lt"]], 1.5)

    bend = nat["bend_s"] * k_matern(W1, W2, [1], [nat["bend_lh"]], 2.5) \
        * k_matern(W1, W2, [0], [nat["bend_lt"]], 2.5)
    base = nat["base_s"] * k_matern(W1, W2, [1], [nat["base_l"]], 2.5)
    per = nat["per_s"] * k_periodic(W1, W2, 0, nat["per_period"], nat["per_lam"]) \
        * k_matern(W1, W2, [0], [nat["per_l"]], 2.5)
    return lower * (shift("shiftA") + shift("shiftB")) + upper * bend + base + per


def rating_mean(X, nat):
    return nat["pl_a"] + nat["pl_b"] * torch.log(X[:, 1] - nat["pl_c"])


def rating_log_prior(nat):
    lp = lp_halfnormal(nat["noise"], 0.03) + lp_normal(nat["gate_b"], 0.0, 1.0)
    lp = lp + lp_halfnormal(nat["shiftA_s"], 0.6) + lp_gamma(nat["shiftA_lt"], 3.0, 1.0) + lp_gamma(nat["shiftA_lh"], 3.0, 2.0)
    lp = lp + lp_halfnormal(nat["shiftB_s"], 0.3) + lp_gamma(nat["shiftB_lt"], 1.0, 7.0) + lp_gamma(nat["shiftB_lh"], 3.0, 1.0)
    lp = lp + lp_halfnormal(nat["bend_s"], 0.6) + lp_gamma(nat["bend_lh"], 3.0, 2.0) + lp_gamma(nat["bend_lt"], 4.0, 2.0)
    lp = lp + lp_halfnormal(nat["base_s"], 1.0) + lp_gamma(nat["base_l"], 4.0, 4.0)
    lp = lp + lp_halfnormal(nat["per_s"], 0.2) + lp_normal(nat["per_period"], 1.0, 0.05) + lp_gamma(nat["per_lam"], 9.0, 10.0)
    return lp


# ----------------------------------------------------------------------------------------
# marginal likelihood, gradient, prediction, sampling (model independent)
# ----------------------------------------------------------------------------------------
def nlml_from_K(Ky, r):
    """NLML = 1/2 r' Ky^-1 r + sum log L_ii + n/2 log 2pi ;  also returns (L, alpha)."""
    L = torch.linalg.cholesky(Ky)
    alpha = torch.cholesky_solve(r[:, None], L)[:, 0]
    n = r.shape[0]
    val = 0.5 * (r @ alpha) + torch.log(torch.diagonal(L)).sum() + 0.5 * n * LOG2PI
    return val, L, alpha


def nlml(cov: Callable, mean: Callable, nat, X, y, noise, extra_noise=None):
    K = cov(X, X, nat)
    d = noise if extra_noise is None else noise + extra_noise
    Ky = K + torch.diag(d)
    return nlml_from_K(Ky, y - mean(X, nat))[0]


def nlml_grad_closed_form(cov, mean, nat_leaf: Dict[str, torch.Tensor], X, y, noise, extra_key=None):
    """dNLML/d(natural theta) by the trace identity  -1/2 sum_ij W_ij dK_ij/dtheta,
    W = alpha alpha' - Ky^-1 (SURVEY Appendix B) -- the formula the CUDA engine implements.
    d/d(mean parameters) = -J' alpha;  d/d(extra noise) = -1/2 tr W."""
    leaves = {k: v.detach().clone().requires_grad_(True) for k, v in nat_leaf.items()}
    n = X.shape[0]
    with torch.no_grad():
        K = cov(X, X, leaves)
        d = noise.clone()
        if extra_key is not None:
            d = d + leaves[extra_key]
        Ky = K + torch.diag(d)
        r = y - mean(X, leaves)
        val, L, alpha = nlml_from_K(Ky, r)
        Kinv = torch.cholesky_inverse(L)
        W = torch.outer(alpha, alpha) - Kinv
    K2 = cov(X, X, leaves)
    if extra_key is not None:
        K2 = K2 + torch.diag(leaves[extra_key].expand(n))
    surrogate = -0.5 * (W * K2).sum() - (alpha * mean(X, leaves)).sum()
    names = list(leaves)
    grads = torch.autograd.grad(surrogate, [leaves[k] for k in names], allow_unused=True)
    out = {k: (g if g is not None else torch.zeros_like(leaves[k])) for k, g in zip(names, grads)}
    return val, out, alpha, L


def nlml_grad_autograd(cov, mean, nat_leaf, X, y, noise, extra_key=None):
    """Independent path: autograd straight through Cholesky (what the reference's backward does)."""
    leaves = {k: v.detach().clone().requires_grad_(True) for k, v in nat_leaf.items()}
    d = noise if extra_key is None else noise + leaves[extra_key]
    Ky = cov(X, X, leaves) + torch.diag(d)
    val = nlml_from_K(Ky, y - mean(X, leaves))[0]
    names = list(leaves)
    grads = torch.autograd.grad(val, [leaves[k] for k in names], allow_unused=True)
    return val.detach(), {k: (g if g is not None else torch.zeros_like(leaves[k])) for k, g in zip(names, grads)}


def objective(model: str, raw: Dict[str, torch.Tensor], X, y, noise, b_lo=None, b_hi=None):
    """The reference's training objective  -[log N(y|m,Ky) + sum log prior] / n
    (discontinuum/engines/gpytorch.py:353; SURVEY A.1).  Differentiable w.r.t. raw."""
    n = X.shape[0]
    if model == "loadest":
        nat = loadest_natural(raw)
        val = nlml(loadest_cov, loadest_mean, nat, X, y, noise)
        lp = loadest_log_prior(nat)
    elif model == "rating":
        nat = rating_natural(raw, b_lo, b_hi)
        val = nlml(rating_cov, rating_mean, nat, X, y, noise, extra_noise=nat["noise"])
        lp = rating_log_prior(nat)
    else:
        raise ValueError(model)
    return (val - lp) / n


def predict(cov, mean, nat, X, y, noise, Xs, extra_noise=None, min_variance=1e-10,
            add_fixed_noise_if_same_size=True) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """Posterior mean and variance at Xs (discontinuum/engines/gpytorch.py:599-626, SURVEY A.5).

    Returns (mu, var_observed, var_latent).  var_observed follows `likelihood(model(x))`:
    learned extra noise is always added; the fixed training noise only when m == n."""
    n, m = X.shape[0], Xs.shape[0]
    d = noise if extra_noise is None else noise + extra_noise
    Ky = cov(X, X, nat) + torch.diag(d)
    r = y - mean(X, nat)
    L = torch.linalg.cholesky(Ky)
    alpha = torch.cholesky_solve(r[:, None], L)[:, 0]
    Ksx = cov(Xs, X, nat)
    mu = mean(Xs, nat) + Ksx @ alpha
    V = torch.linalg.solve_triangular(L, Ksx.T, upper=False)
    kss = torch.diagonal(cov(Xs, Xs, nat)) if m <= 4096 else _diag_cov(cov, Xs, nat)
    var_lat = kss - (V * V).sum(0)
    var_obs = var_lat.clone()
    if extra_noise is not None:
        var_obs = var_obs + extra_noise
    if add_fixed_noise_if_same_size and m == n:
        var_obs = var_obs + noise
    return mu, torch.clamp_min(var_obs, min_variance), var_lat


def monotonic_penalty(cov, mean, nat, X, y, noise, x_grid, stage_dim=1, fd_eps=1e-3, extra_noise=None):
    """rating_gp/models/gpytorch.py:126-187: mean over the grid of clamp(-(mu(x + eps e_stage) - mu(x)) / eps, min=0),
    mu = eval-mode posterior mean; differentiable w.r.t. nat through the solve (what the reference's autograd does)."""
    mu = predict(cov, mean, nat, X, y, noise, x_grid, extra_noise)[0]
    xp = x_grid.clone()
    xp[:, stage_dim] = x_grid[:, stage_dim] + fd_eps
    mu_plus = predict(cov, mean, nat, X, y, noise, xp, extra_noise)[0]
    d = (mu_plus - mu) / fd_eps
    return torch.clamp(-d, min=0.0).mean()


def monotonic_grid(X, grid_size=64, time_dim=0, stage_dim=1):
    """The reference's random penalty grid (rating_gp/models/gpytorch.py:139-158): time uniform, stage log-uniform,
    both drawn in float32 from torch's global generator (time first)."""
    import numpy as np

    x_min, x_max = np.asarray(X).min(axis=0), np.asarray(X).max(axis=0)
    u_time = torch.rand((grid_size,), dtype=torch.float32)
    time_grid = u_time * (x_max[time_dim] - x_min[time_dim]) + x_min[time_dim]
    eps = 1e-6
    log_xmin, log_xmax = float(np.log(x_min[stage_dim] + eps)), float(np.log(x_max[stage_dim] + eps))
    u_stage = torch.rand((grid_size,), dtype=torch.float32)
    stage_grid = torch.exp(u_stage * (log_xmax - log_xmin) + log_xmin)
    cols = [None, None]
    cols[time_dim], cols[stage_dim] = time_grid, stage_grid
    return torch.stack(cols, dim=1).to(DT)


def _diag_cov(cov, Xs, nat, chunk=2048):
    out = []
    for i in range(0, Xs.shape[0], chunk):
        out.append(torch.diagonal(cov(Xs[i:i + chunk], Xs[i:i + chunk], nat)))
    return torch.cat(out)


def posterior_cov(cov, nat, X, noise, Xs, extra_noise=None):
    d = noise if extra_noise is None else noise + extra_noise
    L = torch.linalg.cholesky(cov(X, X, nat) + torch.diag(d))
    V = torch.linalg.solve_triangular(L, cov(Xs, X, nat).T, upper=False)
    return cov(Xs, Xs, nat) - V.T @ V


def sample(cov, mean, nat, X, y, noise, Xs, Z, extra_noise=None, jitter=0.0):
    """Latent posterior draws mu + L_post Z for supplied base normals Z[S, m]
    (discontinuum/engines/gpytorch.py:578-580; exact Cholesky root, SURVEY A.5)."""
    mu, _, _ = predict(cov, mean, nat, X, y, noise, Xs, extra_noise)
    S = posterior_cov(cov, nat, X, noise, Xs, extra_noise)
    S = 0.5 * (S + S.T)
    Lp = torch.linalg.cholesky(S + jitter * torch.eye(S.shape[0], dtype=DT, device=S.device))
    return mu[None, :] + Z @ Lp.T, Lp


# ----------------------------------------------------------------------------------------
# PyMC variant (loadest_gp/models/pymc.py:37-88, SURVEY A.6): PyMC's own kernel formulas
# ----------------------------------------------------------------------------------------
def pymc_loadest_cov(X1, X2, v):
    """eta_per^2 Periodic(period, ls_psmooth) Matern52(ls_pdecay) + eta_trend^2 ExpQuad(t) + eta_cov^2 ExpQuad(q)
    + eta_res^2 Matern32(t, q), with pm.gp.cov semantics: Periodic = exp(-sin^2(pi |d| / T) / (2 ls^2)),
    ExpQuad = exp(-|d|^2 / (2 ls^2)), Matern as GPyTorch's."""
    d = X1.shape[1]
    t1, t2 = X1[:, 0:1], X2[:, 0:1]
    dt = (t1 - t2.T).abs()
    per = torch.exp(-torch.sin(math.pi * dt / v["period"]) ** 2 / (2.0 * v["ls_psmooth"] ** 2))
    seasonal = v["eta_per"] ** 2 * per * k_matern(X1, X2, [0], v["ls_pdecay"], 2.5)
    trend = v["eta_trend"] ** 2 * k_rbf(X1, X2, [0], v["ls_trend"])
    covs = v["eta_covariates"] ** 2 * k_rbf(X1, X2, list(range(1, d)), v["ls_covariates"])
    res = v["eta_res"] ** 2 * k_matern(X1, X2, list(range(d)), v["ls_res"], 1.5)
    return seasonal + trend + covs + res


def pymc_loadest_neg_logp(v, X, y, sigma=0.1, jitter=1e-6):
    """-(log N(y | 0, K + (sigma^2 + jitter) I) + sum log prior), the quantity pm.find_MAP minimises (no Jacobian)."""
    n = X.shape[0]
    Ky = pymc_loadest_cov(X, X, v) + (sigma ** 2 + jitter) * torch.eye(n, dtype=DT, device=X.device)
    val = nlml_from_K(Ky, y)[0]
    lp = lp_halfnormal(v["eta_per"], 1.0).sum() + lp_gamma(v["ls_pdecay"], 10.0, 1.0).sum() + lp_normal(v["period"], 1.0, 0.05).sum()
    lp = lp + lp_gamma(v["ls_psmooth"], 4.0, 3.0).sum() + (-math.log(1.5) - v["eta_trend"] / 1.5).sum()
    lp = lp + lp_gamma(v["ls_trend"], 4.0, 1.0).sum() + lp_halfnormal(v["eta_covariates"], 2.0).sum()
    lp = lp + lp_gamma(v["ls_covariates"], 2.0, 3.0).sum() + (-math.log(0.2) - v["eta_res"] / 0.2).sum()
    lp = lp + lp_gamma(v["ls_res"], 2.0, 10.0).sum()
    return val - lp


# ----------------------------------------------------------------------------------------
# reference optimiser loop restated (discontinuum/engines/gpytorch.py:266-444), used by the
# fit-trajectory parity tests and the CPU baseline
# ----------------------------------------------------------------------------------------
def fit_adam(model, raw, X, y, noise, iterations=100, lr=0.05, b_lo=None, b_hi=None,
             optimizer="adam", scheduler=True, patience=60, h_min=None, penalty_weight=0.0, grid_size=64):
    params = [v.requires_grad_(True) for v in raw.values()]
    if optimizer == "adam":
        opt = torch.optim.Adam(params, lr=lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-4)
    else:
        opt = torch.optim.AdamW(params, lr=lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2)
    sch = None
    if scheduler:
        sch = torch.optim.lr_scheduler.ReduceLROnPlateau(
            opt, mode="min", factor=0.7, patience=max(20, patience // 2), threshold=1e-4,
            threshold_mode="rel", min_lr=1e-6, cooldown=10)
    history = []
    for _ in range(iterations):
        opt.zero_grad(set_to_none=True)
        if model == "rating":
            rating_project_(raw, h_min)
        obj = objective(model, raw, X, y, noise, b_lo, b_hi)
        if penalty_weight > 0.0 and model == "rating":  # engines/gpytorch.py:371-373 with the rating-gp callback
            nat = rating_natural(raw, b_lo, b_hi)
            grid = monotonic_grid(X.numpy(), grid_size)
            obj = obj + penalty_weight * monotonic_penalty(rating_cov, rating_mean, nat, X, y, noise, grid,
                                                           extra_noise=nat["noise"])
        obj.backward()
        torch.nn.utils.clip_grad_norm_(params, max_norm=1.0)
        opt.step()
        history.append(float(obj.detach()))
        if sch is not None:
            sch.step(history[-1])
    return raw, history
