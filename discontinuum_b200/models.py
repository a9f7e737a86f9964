"""Covariance / mean / likelihood definitions of the reference's two model packages, restated as
CovSpec trees for the CUDA tile generator.

  loadest_spec  <- src/loadest_gp/models/gpytorch.py:48-128  (ExactGPModel: seasonal + covariates + residual,
                   ConstantMean, fixed noise 0.1**2, no learned noise; cov_trend is defined there but unused)
  rating_spec   <- src/rating_gp/models/gpytorch.py:64-79,205-372 and src/rating_gp/models/kernels.py:242-382
                   (sigmoid-gated shift kernels, inverted-gate bend kernel, base + periodic, all on log-warped
                   stage; power-law mean; fixed per-point noise + learned homoskedastic noise)
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional

import numpy as np

from . import capi
from .spec import CovSpec, Factor

LOADEST_FIXED_NOISE = 0.1 ** 2
RATING_DEFAULT_NOISE = 0.1 ** 2
RATING_SHARPNESS = 20.0     # SigmoidKernel.a, src/rating_gp/models/kernels.py:271
RATING_LOG_EPS = 1e-6       # LogWarpKernel eps, src/rating_gp/models/kernels.py:368
RATING_MIN_NOISE = 1e-4     # GreaterThan(1e-4) default of gpytorch's HomoskedasticNoise


def loadest_spec(ndim: int = 2) -> CovSpec:
    """x = (time, covariates...).  K = s1 Per(t) M52(t) + s2 RBF_ard(q) + s3 M32_ard(t, q)."""
    if ndim < 2:
        raise ValueError("loadest-gp needs time + at least one covariate")
    s = CovSpec(ndim=ndim)
    cols = [s.col_copy(d) for d in range(ndim)]
    c = s.param("mean.constant", ("none",), None)
    s1 = s.param("seasonal.outputscale", prior=("halfnormal", 1.0))
    lam = s.param("seasonal.periodic.lengthscale")
    per = s.param("seasonal.periodic.period_length", prior=("normal", 1.0, 0.01))
    l1 = s.param("seasonal.matern52.lengthscale")
    s2 = s.param("covariates.outputscale", prior=("halfnormal", 2.0))
    l2 = [s.param(f"covariates.rbf.lengthscale.{d}", prior=("gamma", 2.0, 3.0)) for d in range(ndim - 1)]
    s3 = s.param("residual.outputscale", prior=("halfnormal", 0.2))
    l3 = [s.param(f"residual.matern32.lengthscale.{d}", prior=("gamma", 2.0, 10.0)) for d in range(ndim)]
    s.term(s1, [Factor(capi.PERIODIC, [cols[0]], [lam], per), Factor(capi.MATERN52, [cols[0]], [l1])])
    s.term(s2, [Factor(capi.RBF, cols[1:], l2)])
    s.term(s3, [Factor(capi.MATERN32, cols, l3)])
    s.mean_kind, s.mean_theta = capi.MEAN_CONST, (c,)
    return s


def rating_spec(b_lo: float, b_hi: float, gate_b_init: Optional[float] = None, pl_a: float = 0.0, pl_b: float = 1.3,
                pl_c: float = 0.5) -> CovSpec:
    """x = (time, stage in [1, 2]).  b_lo / b_hi: 10 % / 90 % stage quantiles bounding the switch point
    (src/rating_gp/models/gpytorch.py:221-235).  The reference draws gate_b, pl_a, pl_b, pl_c at random
    (gpytorch.py:31-36, kernels.py:276); callers pass the draws, defaults are deterministic."""
    s = CovSpec(ndim=2)
    t = s.col_copy(0)
    hw = s.col_log(1, RATING_LOG_EPS)
    a = s.param("powerlaw.a", ("none",), init_raw=pl_a)
    b = s.param("powerlaw.b", ("none",), init_raw=pl_b)
    c = s.param("powerlaw.c", ("none",), init_raw=pl_c)
    noise = s.param("likelihood.second_noise", ("greater_than", RATING_MIN_NOISE), ("halfnormal", 0.03), group="likelihood")
    gb = s.param("sigmoid.b", ("interval", float(b_lo), float(b_hi)), ("normal", 0.0, 1.0))
    if gate_b_init is None:
        gate_b_init = 0.5 * (b_lo + b_hi)
    from .spec import inverse_transform
    s.params[gb].init_raw = inverse_transform(s.params[gb], gate_b_init)
    g = s.col_gate(1, RATING_SHARPNESS, gb)

    def shift(name, eta, tp, sp):
        sc = s.param(f"{name}.outputscale", prior=("halfnormal", eta))
        lh = s.param(f"{name}.stage_matern52.lengthscale", prior=("gamma",) + sp)
        lt = s.param(f"{name}.time_matern32.lengthscale", prior=("gamma",) + tp)
        s.term(sc, [Factor(capi.MATERN52, [hw], [lh]), Factor(capi.MATERN32, [t], [lt])], capi.GATE_SIGMOID, g)

    shift("shiftA", 0.6, (3.0, 1.0), (3.0, 2.0))
    shift("shiftB", 0.3, (1.0, 7.0), (3.0, 1.0))
    sc = s.param("bend.outputscale", prior=("halfnormal", 0.6))
    lh = s.param("bend.stage_matern52.lengthscale", prior=("gamma", 3.0, 2.0))
    lt = s.param("bend.time_matern52.lengthscale", prior=("gamma", 4.0, 2.0))
    s.term(sc, [Factor(capi.MATERN52, [hw], [lh]), Factor(capi.MATERN52, [t], [lt])], capi.GATE_INV_SIGMOID, g)
    sc = s.param("base.outputscale", prior=("halfnormal", 1.0))
    lb = s.param("base.stage_matern52.lengthscale", prior=("gamma", 4.0, 4.0))
    s.term(sc, [Factor(capi.MATERN52, [hw], [lb])])
    sc = s.param("periodic.outputscale", prior=("halfnormal", 0.2))
    pp = s.param("periodic.period_length", prior=("normal", 1.0, 0.05))
    pl = s.param("periodic.lengthscale", prior=("gamma", 9.0, 10.0))
    pm = s.param("periodic.time_matern52.lengthscale")
    s.term(sc, [Factor(capi.PERIODIC, [t], [pl], pp), Factor(capi.MATERN52, [t], [pm])])
    s.mean_kind, s.mean_col, s.mean_theta = capi.MEAN_POWERLAW, 1, (a, b, c)
    s.noise_theta = noise
    return s


def stage_quantile_bounds(stage: np.ndarray):
    """np.quantile(stage, 0.10 / 0.90) as at src/rating_gp/models/gpytorch.py:221-223."""
    return float(np.quantile(stage, 0.10)), float(np.quantile(stage, 0.90))


# ----------------------------------------------------------------------------------------------
# model classes: the reference's  class Model(DataMixin, PlotMixin, Marginal<Engine>)  pattern
# (src/loadest_gp/models/gpytorch.py:24-58, src/rating_gp/models/gpytorch.py:43-202) with the
# engine base swapped for MarginalB200.  Plot mixins are the reference's own and are not rebuilt.
# ----------------------------------------------------------------------------------------------
import torch  # noqa: E402

from .data import LogStandardPipeline, TimePipeline, UnitPipeline  # noqa: E402
from .engine import JITTERS, DataMixin, MarginalB200, ModelConfig  # noqa: E402
from .spec import GPModule  # noqa: E402


def annual_flux_groups(time, flow, target_pipeline):
    """(weight[m], group_start[G + 1], years[G], log_transform) of the annual-flux reduction over a strictly increasing
    time grid: weight = flow * dt * 1e-3 (concentration_to_flux, src/loadest_gp/utils.py:14-56), groups = calendar years
    (resample(time="YE").sum(), utils.py:89), log_transform the dgp_flux_reduce kind of the target pipeline."""
    time = np.asarray(time).astype("datetime64[ns]")
    if np.any(np.diff(time) <= np.timedelta64(0, "ns")):
        raise ValueError("sample_annual_flux needs a strictly increasing time grid")
    dts = np.unique(np.diff(time).astype("timedelta64[ns]").astype(np.int64))
    if dts.shape[0] != 1:
        import warnings

        warnings.warn("Time delta is not constant", UserWarning, stacklevel=3)
    dt_s = float(dts[0]) * 1e-9
    weight = np.asarray(flow, dtype=np.float64) * dt_s * 1e-3
    years = time.astype("datetime64[Y]").astype(np.int64) + 1970
    uniq, first = np.unique(years, return_index=True)
    group_start = np.concatenate([first, [time.shape[0]]]).astype(np.int32)
    log_t = 1 if isinstance(target_pipeline, LogStandardPipeline) else 2  # exp clipped at 1e-6 | affine clipped at 0 (data.py pipelines)
    return weight, group_start, uniq, log_t


@dataclass
class FluxSpec:
    """The annual-flux reduction of one site's posterior draws on `grid` (model-space inputs [m, ndim]): the dgp_flux_reduce
    of LoadestGPMarginalB200.sample_annual_flux.  years[G] labels the groups."""
    grid: np.ndarray
    weight: np.ndarray
    group_start: np.ndarray
    years: np.ndarray
    y_mean: float
    y_scale: float
    log_transform: int

    @classmethod
    def from_series(cls, grid, time, flow, target_pipeline) -> "FluxSpec":
        """From the grid, its time stamps and flow (original units) and the fitted target pipeline of the site."""
        weight, group_start, years, log_t = annual_flux_groups(time, flow, target_pipeline)
        grid = np.ascontiguousarray(grid, dtype=np.float64)
        if grid.shape[0] != weight.shape[0]:
            raise ValueError("FluxSpec: grid, time and flow must have the same length")
        return cls(grid, weight, group_start, years, float(target_pipeline.mean_), float(target_pipeline.scale_), log_t)

    def reduce(self) -> dict:
        """The `flux` dict of Engine.sample_ex / BatchEngine.sample."""
        return dict(y_mean=self.y_mean, y_scale=self.y_scale, log_transform=self.log_transform, weight=self.weight,
                    group_start=self.group_start)


class LoadestDataMixin(DataMixin):
    """src/loadest_gp/models/base.py:7-19."""

    def build_datamanager(self, model_config: Optional[ModelConfig] = None):
        self._build_datamanager({"time": TimePipeline, "flow": LogStandardPipeline}, model_config)


class RatingDataMixin(DataMixin):
    """src/rating_gp/models/base.py:7-19."""

    def build_datamanager(self, model_config: Optional[ModelConfig] = None):
        self._build_datamanager({"time": TimePipeline, "stage": UnitPipeline}, model_config)


class LoadestGPMarginalB200(LoadestDataMixin, MarginalB200):
    """Gaussian-process LOADEST model on the B200 engine (src/loadest_gp/models/gpytorch.py:24-58)."""

    def __init__(self, model_config: Optional[ModelConfig] = None):
        if model_config is None:
            model_config = ModelConfig()
        super().__init__(model_config=model_config)
        self.build_datamanager(model_config)

    def build_model(self, X, y, y_unc=None) -> GPModule:
        self.fixed_noise = np.full(y.shape[0], LOADEST_FIXED_NOISE)
        return GPModule(loadest_spec(X.shape[1]))

    def sample_annual_flux(self, covariates, n: int = 1000, seed: int = 0, flow_key: str = "flow", time_key: str = "time"):
        """Annual flux (kg / year) of `n` joint posterior draws over a regular (e.g. daily) grid, reduced on the GPU:
        draws -> concentration (inverse target pipeline) -> concentration * flow * dt * 1e-3 (src/loadest_gp/utils.py:
        14-56) -> sum per calendar year (`flux.resample(time="YE").sum()`, utils.py:89).  The n x m draw matrix and its
        base normals never leave the device.  Returns (years[G], flux[n, G])."""
        from .data import _cov_dict
        from .engine import JITTERS, NotPSDError

        if not self.is_fitted:
            raise RuntimeError("The model hasn't been fitted yet, call .fit().")
        cov = _cov_dict(covariates)
        weight, group_start, uniq, log_t = annual_flux_groups(cov[time_key], cov[flow_key], self.dm.target_pipeline)
        tp = self.dm.target_pipeline
        Xnew = np.ascontiguousarray(self.dm.Xnew(covariates), dtype=np.float64)
        self._ensure_factorized(Xnew)
        for jit in JITTERS:
            flux, info = self._engine.sample_ex(Xnew, n, Z=None, seed=seed, jitter=jit,
                                                flux=dict(y_mean=float(tp.mean_), y_scale=float(tp.scale_), log_transform=log_t,
                                                          weight=weight, group_start=group_start))
            if info == 0 and np.all(np.isfinite(flux)):
                return uniq, flux
        raise NotPSDError("posterior covariance not positive definite")


class RatingGPMarginalB200(RatingDataMixin, MarginalB200):
    """Stage-discharge rating-curve GP on the B200 engine (src/rating_gp/models/gpytorch.py:43-265)."""

    def __init__(self, model_config: Optional[ModelConfig] = None):
        if model_config is None:
            model_config = ModelConfig()
        super().__init__(model_config=model_config)
        self.build_datamanager(model_config)

    def build_model(self, X, y, y_unc=None) -> GPModule:
        assert X.shape[1] == 2, "Only two dimensions supported"
        self.fixed_noise = np.asarray(y_unc, dtype=np.float64) if y_unc is not None else np.full(y.shape[0], RATING_DEFAULT_NOISE)
        b_lo, b_hi = stage_quantile_bounds(X[:, 1])
        # same random initial draws as the reference (gpytorch.py:31-36, kernels.py:276)
        a = float(torch.randn(1)); b = float(torch.randn(1) + 1.3); c = float(torch.rand(1))
        gb = b_lo + float(torch.rand(1)) * (b_hi - b_lo)
        gb = min(max(gb, b_lo + 1e-9 * (b_hi - b_lo)), b_hi - 1e-9 * (b_hi - b_lo))
        return GPModule(rating_spec(b_lo, b_hi, gate_b_init=gb, pl_a=a, pl_b=b, pl_c=c))

    def project_parameters(self, X_all: np.ndarray):
        """b clamped to [1.2, 2.5], c <= min(stage) - 1e-6, in place on every forward (gpytorch.py:39,259)."""
        with torch.no_grad():
            raw = self.model.raw
            raw["powerlaw__b"].clamp_(1.2, 2.5)
            raw["powerlaw__c"].clamp_(max=float(X_all[:, 1].min()) - 1e-6)

    def fit(self, covariates, target, target_unc=None, iterations=100, optimizer=None, learning_rate=None,
            early_stopping=False, patience=60, scheduler=True, resume=False, monotonic_penalty_weight: float = 0.0,
            grid_size: int = 64, monotonic_penalty_interval: int = 1, penalty_generator: Optional[torch.Generator] = None,
            **kw):
        """src/rating_gp/models/gpytorch.py:81-202: optional penalty on negative dQ/dStage of the posterior mean over a
        random (time uniform, stage log-uniform) grid, every `monotonic_penalty_interval` iterations.  The grids are drawn
        from torch's global generator, or from `penalty_generator`."""
        if monotonic_penalty_weight <= 0:
            return super().fit(covariates=covariates, target=target, target_unc=target_unc, iterations=iterations,
                               optimizer=optimizer, learning_rate=learning_rate, early_stopping=early_stopping,
                               patience=patience, scheduler=scheduler, resume=resume, **kw)
        # dgp_mean_functional_grad takes the 2 x grid_size penalty points in one prediction chunk
        self.max_predict_chunk = max(self.max_predict_chunk, -(-2 * int(grid_size) // 128) * 128)
        step = {"i": 0}

        def penalty_callback():
            step["i"] += 1
            if monotonic_penalty_interval > 1 and (step["i"] % monotonic_penalty_interval) != 0:
                return torch.zeros((), dtype=torch.float64)
            grid = monotonic_penalty_grid(self.dm.X, grid_size, generator=penalty_generator)
            pen = _MonotonicPenalty.apply(self.model.natural(), self, grid, 1e-3)
            if monotonic_penalty_interval > 1:
                pen = pen * float(monotonic_penalty_interval)
            return pen

        return super().fit(covariates=covariates, target=target, target_unc=target_unc, iterations=iterations,
                           optimizer=optimizer, learning_rate=learning_rate, early_stopping=early_stopping,
                           patience=patience, scheduler=scheduler, resume=resume, penalty_callback=penalty_callback,
                           penalty_weight=float(monotonic_penalty_weight), **kw)


def monotonic_penalty_grid(X: np.ndarray, grid_size: int = 64, time_dim: int = 0, stage_dim: int = 1,
                           generator: Optional[torch.Generator] = None) -> np.ndarray:
    """The reference's random grid (rating_gp/models/gpytorch.py:139-158): float32 draws from torch's global generator
    (or from `generator`), time uniform over the training range (drawn first), stage log-uniform."""
    x_min, x_max = X.min(axis=0), X.max(axis=0)
    u_time = torch.rand((grid_size,), dtype=torch.float32, generator=generator)
    time_grid = u_time * (x_max[time_dim] - x_min[time_dim]) + x_min[time_dim]
    eps = 1e-6
    log_xmin, log_xmax = float(np.log(x_min[stage_dim] + eps)), float(np.log(x_max[stage_dim] + eps))
    u_stage = torch.rand((grid_size,), dtype=torch.float32, generator=generator)
    stage_grid = torch.exp(u_stage * (log_xmax - log_xmin) + log_xmin)
    cols = [None, None]
    cols[time_dim], cols[stage_dim] = time_grid, stage_grid
    return torch.stack(cols, dim=1).to(torch.float64).numpy()


class _MonotonicPenalty(torch.autograd.Function):
    """mean_p clamp(-(mu(x_p + eps e_stage) - mu(x_p)) / eps, 0) on the GPU engine.  With the active set fixed the
    penalty is a linear functional c'mu of the posterior mean; its gradient w.r.t. natural theta comes from
    dgp_mean_functional_grad (adjoint of the solve), replacing the reference's autograd through two predictions."""

    @staticmethod
    def forward(ctx, nat: torch.Tensor, owner: "RatingGPMarginalB200", grid: np.ndarray, fd_eps: float, stage_dim: int = 1):
        th = nat.detach().cpu().numpy().astype(np.float64)
        eng = owner._engine
        if getattr(owner, "_last_theta", None) is None or not np.array_equal(owner._last_theta, th):
            for jit in JITTERS:  # the factorisation of this theta must be resident (normally left by _NLML.forward)
                val, _, info = eng.nlml_grad(th, jit)
                if info == 0 and np.isfinite(val):
                    break
            owner._last_theta = th.copy()
        G = grid.shape[0]
        plus = grid.copy()
        plus[:, stage_dim] += fd_eps
        pts = np.ascontiguousarray(np.concatenate([grid, plus], axis=0))
        mu, _ = eng.predict(pts, want_var=False)
        d = (mu[G:] - mu[:G]) / fd_eps
        active = d < 0.0
        c = np.zeros(2 * G)
        c[:G][active] = 1.0 / (G * fd_eps)
        c[G:][active] = -1.0 / (G * fd_eps)
        val, grad = eng.mean_functional_grad(pts, c)
        ctx.grad = torch.from_numpy(grad.copy())
        return torch.tensor(float(np.maximum(-d, 0.0).mean()), dtype=torch.float64)

    @staticmethod
    def backward(ctx, g):
        return g * ctx.grad, None, None, None, None


LoadestGP = LoadestGPMarginalB200
RatingGP = RatingGPMarginalB200
