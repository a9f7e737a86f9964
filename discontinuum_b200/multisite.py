"""Multi-site batch: the B200 counterpart of the reference's `fexec.map(map_retrieval, sites)`
(examples/nwqn-loadest-example/nwqn-loadest-example.py:38-128,156-159).

Sites are independent GPs: nothing is exchanged while fitting.  One process per GPU (torchrun); sites are
assigned to ranks by longest-processing-time-first on the cost iterations * n^3; inside a rank the sites are fitted in
groups on one batch handle (dgp_batch_*): every optimiser iteration of a group is ONE launch sequence that evaluates
NLML + gradient of all its sites, so the latency-bound panel chain is paid once per block step for the whole group.
The only collective is the final gather.
"""
from __future__ import annotations

import time
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import capi
from .engine import JITTERS, MIN_VARIANCE
from .models import LOADEST_FIXED_NOISE, loadest_spec, monotonic_penalty_grid
from .spec import GPModule


def assign_sites(costs: Sequence[float], world: int) -> List[List[int]]:
    """Greedy LPT: sites sorted by decreasing cost, each to the least-loaded rank.  Deterministic on every rank."""
    order = sorted(range(len(costs)), key=lambda i: (-float(costs[i]), i))
    load = [0.0] * world
    out: List[List[int]] = [[] for _ in range(world)]
    for i in order:
        r = min(range(world), key=lambda k: (load[k], k))
        out[r].append(i)
        load[r] += float(costs[i])
    return out


def site_cost(n: int, iterations: int, m_predict: int = 0) -> float:
    """flop model of one site: iterations * n^3 (NLML+grad) + factorise + n^2 per predicted point (SURVEY 8d)."""
    return float(iterations) * float(n) ** 3 + float(n) ** 3 + float(m_predict) * float(n) ** 2


def gather_results(local: Dict[int, dict], dist=None) -> Optional[Dict[int, dict]]:
    """All ranks -> rank 0.  `dist` is torch.distributed (initialised) or None for a single process."""
    if dist is None or not dist.is_initialized() or dist.get_world_size() == 1:
        return dict(local)
    bucket = [None] * dist.get_world_size() if dist.get_rank() == 0 else None
    dist.gather_object(local, bucket, dst=0)
    if dist.get_rank() != 0:
        return None
    merged: Dict[int, dict] = {}
    for part in bucket:
        merged.update(part)
    return merged


# ---------------------------------------------------------------- model kinds of a site batch
class LoadestKind:
    """loadest-gp sites (src/loadest_gp/models/gpytorch.py:48-128): fixed noise 0.1**2, nothing projected."""
    name = "loadest"

    def module(self, X, y, noise) -> GPModule:
        return GPModule(loadest_spec(X.shape[1]))

    def default_noise(self, n):
        return np.full(n, LOADEST_FIXED_NOISE)

    def project(self, module: GPModule, X: np.ndarray):
        pass

    def project_raw(self, raw: np.ndarray, modules, Xs):
        pass


class RatingKind:
    """rating-gp gauges (src/rating_gp/models/gpytorch.py:64-79,205-372): per-point noise from the measurement
    uncertainties plus a learned homoskedastic term, the power-law mean's random initial draws (in the reference's order:
    a, b, c, then the gate switch point) and its in-place projection on every forward (gpytorch.py:39,259)."""
    name = "rating"

    def module(self, X, y, noise) -> GPModule:
        from .models import rating_spec, stage_quantile_bounds

        b_lo, b_hi = stage_quantile_bounds(X[:, 1])
        a = float(torch.randn(1)); b = float(torch.randn(1) + 1.3); c = float(torch.rand(1))
        gb = b_lo + float(torch.rand(1)) * (b_hi - b_lo)
        gb = min(max(gb, b_lo + 1e-9 * (b_hi - b_lo)), b_hi - 1e-9 * (b_hi - b_lo))
        return GPModule(rating_spec(b_lo, b_hi, gate_b_init=gb, pl_a=a, pl_b=b, pl_c=c))

    def default_noise(self, n):
        from .models import RATING_DEFAULT_NOISE

        return np.full(n, RATING_DEFAULT_NOISE)

    def project(self, module: GPModule, X: np.ndarray):
        with torch.no_grad():
            module.raw["powerlaw__b"].clamp_(1.2, 2.5)
            module.raw["powerlaw__c"].clamp_(max=float(X[:, 1].min()) - 1e-6)

    def project_raw(self, raw: np.ndarray, modules, Xs):
        """The same projection on the [G, P] raw-parameter array of a group (Xs: the sites' training inputs)."""
        ib, ic = modules[0].spec.index("powerlaw.b"), modules[0].spec.index("powerlaw.c")
        raw[:, ib] = np.clip(raw[:, ib], 1.2, 2.5)
        raw[:, ic] = np.minimum(raw[:, ic], np.array([float(X[:, 1].min()) - 1e-6 for X in Xs]))


KINDS = {"loadest": LoadestKind, "rating": RatingKind}


def _kind(model):
    return KINDS[model]() if isinstance(model, str) else model


def observed_variance(spec, theta: np.ndarray, var_latent: np.ndarray, fixed_noise: np.ndarray, m: int) -> np.ndarray:
    """Variance of `likelihood(model(x))` in eval mode (SURVEY A.5), as MarginalB200._model_space_predict returns it:
    latent variance + learned noise, + the fixed training noise only when m == n_train, clamped at MIN_VARIANCE."""
    var = np.asarray(var_latent, dtype=np.float64)
    if spec.noise_theta >= 0:
        var = var + theta[spec.noise_theta]
    if m == fixed_noise.shape[0]:
        var = var + fixed_noise
    return np.maximum(var, MIN_VARIANCE)


# ---------------------------------------------------------------- vectorised host step of a group of sites
class GroupOptimizer:
    """The reference's per-site optimiser step (discontinuum/engines/gpytorch.py:266-315,353-420) for G sites at once:
    raw parameters, constraint / prior chain rule (GPModule.host_chain semantics), global-norm clipping at 1.0, Adam
    (lr, betas 0.9 / 0.999, eps 1e-8, weight_decay 1e-4 added to the gradient, torch.optim.Adam's arithmetic) on [G, P]
    numpy arrays, and one torch ReduceLROnPlateau per site (its own state machine, driven by a one-element dummy
    optimiser whose learning rate is read back).  tests/test_multisite.py checks it against torch.optim.Adam."""

    def __init__(self, modules: Sequence[GPModule], lr: float = 0.05, scheduler: bool = True, patience: int = 60,
                 weight_decay: float = 1e-4):
        self.modules = list(modules)
        G, P = len(self.modules), len(self.modules[0].spec.params)
        tabs = [m._tables() for m in self.modules]
        self.kind, self.lb, self.lo, self.hi, self.pk, self.pa, self.pb, self.pc = (np.stack([t[k] for t in tabs]) for k in range(8))
        self.raw = np.array([[float(r.detach()) for r in m.raw_list()] for m in self.modules], dtype=np.float64)
        self.m = np.zeros((G, P))
        self.v = np.zeros((G, P))
        self.steps = np.zeros(G, dtype=np.int64)
        self.lr = np.full(G, float(lr))
        self.wd = float(weight_decay)
        self.sched = None
        if scheduler:
            self.sched = []
            for _ in range(G):
                dummy = torch.optim.SGD([torch.zeros(1, requires_grad=True)], lr=float(lr))
                self.sched.append(torch.optim.lr_scheduler.ReduceLROnPlateau(
                    dummy, mode="min", factor=0.7, patience=max(20, patience // 2), threshold=1e-4, threshold_mode="rel",
                    min_lr=1e-6, cooldown=10))

    def pull(self, g: Optional[int] = None):
        """raw parameters of the torch modules -> the arrays (after a projection changed them)."""
        for k in ([g] if g is not None else range(len(self.modules))):
            self.raw[k] = [float(r.detach()) for r in self.modules[k].raw_list()]

    def push(self):
        with torch.no_grad():
            for k, mod in enumerate(self.modules):
                for p, v in zip(mod.raw_list(), self.raw[k]):
                    p.fill_(float(v))

    def chain(self):
        """(natural[G, P], d natural / d raw, sum log prior [G], d sum log prior / d natural) -- GPModule.host_chain."""
        raw, kind = self.raw, self.kind
        sig = 1.0 / (1.0 + np.exp(-raw))
        sp = np.where(raw > 20.0, raw, np.log1p(np.exp(np.minimum(raw, 20.0))))
        nat = np.where(kind == 1, sp + self.lb, np.where(kind == 2, self.lo + (self.hi - self.lo) * sig, raw))
        dnat = np.where(kind == 1, np.where(raw > 20.0, 1.0, sig), np.where(kind == 2, (self.hi - self.lo) * sig * (1.0 - sig), 1.0))
        pk, pa, pb, pc = self.pk, self.pa, self.pb, self.pc
        with np.errstate(divide="ignore", invalid="ignore"):
            lp = np.where(pk == 1, pc - nat * nat / (2.0 * pb * pb),
                          np.where(pk == 2, pc - (nat - pa) ** 2 / (2.0 * pb * pb),
                                   np.where(pk == 3, pc + (pa - 1.0) * np.log(nat) - pb * nat, 0.0)))
            dlp = np.where(pk == 1, -nat / (pb * pb),
                           np.where(pk == 2, -(nat - pa) / (pb * pb),
                                    np.where(pk == 3, (pa - 1.0) / nat - pb, 0.0)))
        return nat, dnat, lp.sum(axis=1), dlp

    def step(self, graw: np.ndarray, objective: np.ndarray, active: np.ndarray):
        """clip_grad_norm_(1.0) + NaN guard + Adam + scheduler for the sites in `active` (bool [G])."""
        g = np.array(graw, dtype=np.float64)
        coef = 1.0 / (np.sqrt(np.sum(g * g, axis=1)) + 1e-6)
        scale = np.where(coef >= 1.0, 1.0, coef)      # (a NaN norm scales the row to NaN, as torch's clamp does)
        g = g * scale[:, None]
        g = np.where(np.isnan(g).any(axis=1)[:, None], np.nan_to_num(g, nan=0.0, posinf=0.0, neginf=0.0), g)
        a = np.asarray(active, dtype=bool)
        b1, b2, eps = 0.9, 0.999, 1e-8
        self.steps[a] += 1
        g = g + self.wd * self.raw
        m = self.m + (g - self.m) * (1.0 - b1)
        v = self.v * b2 + (1.0 - b2) * g * g
        t = np.maximum(self.steps, 1).astype(np.float64)
        bc1, bc2 = 1.0 - b1 ** t, 1.0 - b2 ** t
        denom = np.sqrt(v) / np.sqrt(bc2)[:, None] + eps
        new = self.raw - (self.lr / bc1)[:, None] * (m / denom)
        am = a[:, None]
        self.m, self.v, self.raw = np.where(am, m, self.m), np.where(am, v, self.v), np.where(am, new, self.raw)
        if self.sched is not None:
            for k in np.nonzero(a)[0]:
                self.sched[k].step(float(objective[k]))
                self.lr[k] = self.sched[k].optimizer.param_groups[0]["lr"]


@dataclass
class _Site:
    idx: int
    X: np.ndarray
    y: np.ndarray
    noise: np.ndarray
    module: GPModule
    history: List[float] = field(default_factory=list)
    failed: Optional[str] = None
    bad_streak: int = 0
    # early stopping (MarginalB200.fit's rule) and the monotonicity penalty
    best: float = float("inf")
    patience_counter: int = 0
    stopped_at: Optional[int] = None
    good_iters: int = 0
    penalty_gen: Optional[torch.Generator] = None
    penalty: Optional[float] = None


def _groups(order: List[int], group: int) -> List[List[int]]:
    return [order[i:i + group] for i in range(0, len(order), group)]


def _predict_group(batch: capi.BatchEngine, grp: List[_Site], want: List[bool], predict: Dict[int, np.ndarray], kind,
                   res_of: Dict[int, dict]):
    """Prediction of a group through its own batch handle (whose training set is the group's): factorise every site at its
    fitted theta (dgp_batch_factorize), climb psd_safe_cholesky's jitter ladder only for the wanted sites that failed -- the
    others are re-factorised unchanged and keep their bits -- and predict every wanted site's grid in one dgp_batch_predict.
    Sites not wanted (not in `predict`, or failed while fitting) are factorised at their last theta, results unused."""
    G = len(grp)
    grids: List[Optional[np.ndarray]] = [None] * G
    thetas = []
    for k, s in enumerate(grp):
        if want[k]:
            grids[k] = np.ascontiguousarray(predict[s.idx], dtype=np.float64)
            kind.project(s.module, np.concatenate([s.X, grids[k]], axis=0))
        with torch.no_grad():
            thetas.append(s.module.natural().numpy().astype(np.float64))
        if want[k]:
            res_of[s.idx]["theta"] = thetas[k]
    thetas = np.ascontiguousarray(np.stack(thetas))
    jit = np.full(G, JITTERS[0])
    _, info = batch.factorize(thetas, jit)
    bad = np.array(want) & (info != 0)
    for j in JITTERS[1:]:
        if not bad.any():
            break
        jit[bad] = j
        _, i2 = batch.factorize(thetas, jit)
        info = np.where(bad, i2, info)
        bad &= i2 != 0
    for k in np.nonzero(bad)[0]:
        res_of[grp[k].idx]["failed"] = f"prediction: not positive definite after jitter {JITTERS[-1]:g} (info={int(info[k])})"
        grids[k] = None
    if all(g is None for g in grids):
        return
    out = batch.predict(grids)
    for k, s in enumerate(grp):
        if grids[k] is None:
            continue
        mu, var = out[k]
        res = res_of[s.idx]
        res["mu"], res["var_latent"] = mu, var
        res["var"] = observed_variance(s.module.spec, thetas[k], var, s.noise, grids[k].shape[0])


@dataclass
class PenaltyConfig:
    """The rating-gp monotonicity penalty of a driver fit (RatingGP.fit's monotonic_penalty_weight / grid_size /
    monotonic_penalty_interval); site `idx` draws its grids from torch.Generator().manual_seed(seed + idx)."""
    weight: float
    grid_size: int = 64
    interval: int = 1
    seed: int = 0
    fd_eps: float = 1e-3


_MIN_IMPROVEMENT = 1e-6   # MarginalB200.fit's early-stopping threshold


class _GroupRun:
    """One group of sites on one batch handle: `launch()` enqueues the next optimiser iteration's NLML + gradient evaluation of
    the whole group, `finish()` collects it and takes the host step.  Two of these in flight on one GPU fill each other's
    latency-bound stretches (measured: +1 % for two groups of n ~ 7k sites, +8 % for two groups of n ~ 2-3k sites)."""

    def __init__(self, grp, batch, kind, iterations, lr, scheduler, patience, st, timed, early_stopping=False, penalty=None):
        self.grp, self.batch, self.kind, self.left, self.st = grp, batch, kind, int(iterations), st
        self.iterations, self.patience, self.early_stopping, self.pen = int(iterations), int(patience), bool(early_stopping), penalty
        if penalty is not None:
            for s in grp:
                s.penalty_gen = torch.Generator().manual_seed(int(penalty.seed) + int(s.idx))
        self.G = len(grp)
        batch.set_train(grp[0].module.spec.to_c(), [(s.X, s.y, s.noise) for s in grp])
        batch.set_timing(timed)
        self.timed = timed
        self.opt = GroupOptimizer([s.module for s in grp], lr=lr, scheduler=scheduler, patience=patience)
        self.ns = np.array([s.X.shape[0] for s in grp], dtype=np.float64)
        self.inflight = False

    @property
    def done(self):
        return self.left <= 0 and not self.inflight

    def launch(self):
        if self.left <= 0:
            return False
        self.alive = np.array([s.failed is None and s.stopped_at is None for s in self.grp])
        if not self.alive.any():
            self.left = 0
            return False
        stopped = np.array([s.stopped_at is not None for s in self.grp])
        kept = self.opt.raw[stopped].copy()      # a stopped site keeps its last parameters as they are
        self.kind.project_raw(self.opt.raw, self.opt.modules, [s.X for s in self.grp])
        self.opt.raw[stopped] = kept
        self.nat, self.dnat, self.lp, self.dlp = self.opt.chain()
        self.theta = np.ascontiguousarray(self.nat)
        self.batch.nlml_grad_launch(self.theta)
        self.inflight = True
        return True

    def finish(self):
        st, grp, G, alive, theta = self.st, self.grp, self.G, self.alive, self.theta
        val, grad, info = self.batch.nlml_grad_wait()
        self.inflight = False
        self.left -= 1
        st["evals"] += 1
        st["site_evals"] += G
        st["wasted_site_evals"] += int(G - alive.sum())   # stopped / failed sites still evaluated with their group
        if self.timed:
            st["gpu_eval_ms"] += sum(self.batch.last_timing())
        bad = alive & ((info != 0) | ~np.isfinite(val))
        if bad.any():   # jitter ladder, per site; the others are re-evaluated unchanged and keep their numbers
            jit = np.zeros(G)
            for j in JITTERS[1:]:
                jit[bad] = j
                v2, g2, i2 = self.batch.nlml_grad(theta, jit)
                st["retries"] += 1
                fixed = bad & (i2 == 0) & np.isfinite(v2)
                val[fixed], grad[fixed], info[fixed] = v2[fixed], g2[fixed], 0
                bad &= ~fixed
                if not bad.any():
                    break
        t0 = time.perf_counter()
        obj = (val - self.lp) / self.ns
        ok = alive & ~bad & np.isfinite(obj)
        if self.pen is None:
            graw = (grad - self.dlp) * self.dnat / self.ns[:, None]
        else:
            t1 = time.perf_counter()
            wpen, dpen = self._penalty(ok)
            st["penalty_s"] += time.perf_counter() - t1
            t0 += time.perf_counter() - t1
            obj = obj + wpen
            graw = ((grad - self.dlp) / self.ns[:, None] + dpen) * self.dnat
            ok &= np.isfinite(obj)
        for k, s in enumerate(grp):
            if not alive[k]:
                continue
            if ok[k]:
                s.bad_streak = 0
                s.history.append(float(obj[k]))
            else:
                s.bad_streak += 1
                if s.bad_streak > 10:
                    s.failed = f"more than 10 consecutive bad objectives (info={int(info[k])})"
        self.opt.step(np.where(ok[:, None], graw, 0.0), obj, ok)
        if self.early_stopping:   # MarginalB200.fit: bad iterations neither count nor reset the counter
            for k in np.nonzero(ok)[0]:
                s = grp[k]
                if s.history[-1] < s.best - _MIN_IMPROVEMENT:
                    s.best, s.patience_counter = s.history[-1], 0
                else:
                    s.patience_counter += 1
                if s.patience_counter >= self.patience:
                    s.stopped_at = self.iterations - self.left
        st["host_step_s"] += time.perf_counter() - t0
        if self.left <= 0:
            self.opt.push()

    def _penalty(self, ok):
        """(w pen [G], w d pen / d natural theta [G, P]) of the sites whose evaluation is good (zeros elsewhere and between
        penalty iterations): RatingGP.fit's _MonotonicPenalty for the whole group, with one mean-only dgp_batch_predict of
        every site's [grid; grid + eps e_stage] at the evaluated theta and one dgp_batch_mean_functional_grad of c'mu with
        the active set fixed.  Every `interval`-th good iteration of a site, scaled by the interval."""
        pen, G, gs, eps = self.pen, self.G, int(self.pen.grid_size), float(self.pen.fd_eps)
        wpen, dpen = np.zeros(G), np.zeros((G, self.theta.shape[1]))
        pts: List[Optional[np.ndarray]] = [None] * G
        for k, s in enumerate(self.grp):
            if not ok[k]:
                continue
            s.good_iters += 1
            if pen.interval > 1 and s.good_iters % pen.interval != 0:
                continue
            grid = monotonic_penalty_grid(s.X, gs, generator=s.penalty_gen)
            plus = grid.copy()
            plus[:, 1] += eps
            pts[k] = np.ascontiguousarray(np.concatenate([grid, plus], axis=0))
        if all(p is None for p in pts):
            return wpen, dpen
        out = self.batch.predict(pts, want_var=False)
        cs: List[Optional[np.ndarray]] = [None] * G
        for k, s in enumerate(self.grp):
            if pts[k] is None:
                continue
            mu = out[k][0]
            d = (mu[gs:] - mu[:gs]) / eps
            active = d < 0.0
            c = np.zeros(2 * gs)
            c[:gs][active] = 1.0 / (gs * eps)
            c[gs:][active] = -1.0 / (gs * eps)
            cs[k] = c
            s.penalty = float(np.maximum(-d, 0.0).mean())
            wpen[k] = pen.weight * (s.penalty * pen.interval)
        _, g = self.batch.mean_functional_grad(pts, cs)
        for k in range(G):
            if pts[k] is not None:
                dpen[k] = pen.weight * (g[k] * pen.interval)
        return wpen, dpen


def fit_sites_local(sites: Dict[int, tuple], iterations: int = 100, device: int = 0, group: int = 16,
                    predict: Optional[Dict[int, np.ndarray]] = None, lr: float = 0.05, scheduler: bool = True,
                    patience: int = 60, model="loadest", stats: Optional[dict] = None, concurrency: Optional[int] = None,
                    lanes: int = 2, early_stopping: bool = False, monotonic_penalty_weight: float = 0.0, grid_size: int = 64,
                    monotonic_penalty_interval: int = 1, penalty_seed: int = 0) -> Dict[int, dict]:
    """Fit one GP per site on this rank.  sites: {index: (X, y[, noise])} in model space; model: "loadest", "rating" or a
    kind object (see LoadestKind).  Returns {index: {"theta", "objective", "history", "failed", "n", "mu", "var",
    "var_latent"}} ("var" follows `likelihood(model(x))` like MarginalB200.predict).

    Sites are sorted by size and fitted in groups of up to `group` on batch handles (capi.BatchEngine): every iteration of a
    group is a single launch sequence that evaluates NLML + gradient of the whole group (dgp_batch_nlml_grad), one
    device-to-host copy of the G results, and one vectorised host step (GroupOptimizer).  The latency-bound panel chain,
    which dominated when every site ran its own launch sequence, is paid once per block step for the group.  `lanes` groups
    are in flight at a time, each on its own handle (the largest remaining group next to the smallest, so that memory stays
    bounded and the pair finishes together); a rank with a single group's worth of sites splits it.  Results do not depend on
    `lanes`: every site sees the same sequence of evaluations.  Evaluations that fail (info != 0 or a non-finite value) climb
    psd_safe_cholesky's jitter ladder per site; a site whose objective stays bad for more than 10 consecutive iterations is
    marked failed, as MarginalB200.fit gives up.
    The sites of a finished group that have a grid in `predict` are factorised and predicted on the group's own handle
    (dgp_batch_factorize + dgp_batch_predict: every site's numbers equal a per-site capi.Engine factorize + predict bit for bit).
    `early_stopping` applies MarginalB200.fit's rule per site (best objective, improvement 1e-6, stop when `patience`
    good iterations in a row did not improve it; bad iterations neither count nor reset): a stopped site is frozen at its
    last parameters ("stopped_at": the iteration it stopped after, else None) and a group ends when every site has stopped
    or failed.  Stopped and failed sites are still evaluated with their group until it ends.
    `monotonic_penalty_weight` > 0 (rating kind only) adds RatingGP.fit's penalty on negative dQ/dstage of the posterior
    mean over a random grid of `grid_size` points (<= 512: grid and shifted grid share one 1024-row chunk), drawn by site
    `idx` from torch.Generator().manual_seed(penalty_seed + idx), every `monotonic_penalty_interval`-th good iteration
    and scaled by the interval; its gradient comes from dgp_batch_mean_functional_grad.  "penalty" holds the last
    (unweighted) value.  Neither depends on `lanes`, on the group a site lands in, or on the rank.
    `concurrency` selects the round-1 per-handle pipelines instead (fit_sites_local_per_handle), which has neither."""
    pen = None
    if monotonic_penalty_weight > 0.0:
        if getattr(_kind(model), "name", None) != "rating":
            raise ValueError("monotonic_penalty_weight applies to rating gauges only (model='rating')")
        if not 1 <= int(grid_size) <= capi.BATCH_PREDICT_CHUNK // 2:
            raise ValueError(f"grid_size must be in [1, {capi.BATCH_PREDICT_CHUNK // 2}]: the grid and its shifted copy share "
                             f"one {capi.BATCH_PREDICT_CHUNK}-row chunk")
        if int(monotonic_penalty_interval) < 1:
            raise ValueError("monotonic_penalty_interval must be >= 1")
        pen = PenaltyConfig(float(monotonic_penalty_weight), int(grid_size), int(monotonic_penalty_interval), int(penalty_seed))
    if concurrency is not None:
        if early_stopping or pen is not None:
            raise ValueError("early_stopping and the monotonicity penalty need the batch driver (concurrency=None)")
        return fit_sites_local_per_handle(sites, iterations=iterations, device=device, concurrency=concurrency or 4,
                                          predict=predict, lr=lr, scheduler=scheduler, patience=patience)
    kind = _kind(model)
    t_start = time.perf_counter()
    st = {"groups": 0, "evals": 0, "gpu_eval_ms": 0.0, "fit_wall_s": 0.0, "predict_s": 0.0, "host_step_s": 0.0, "retries": 0,
          "lanes": 1, "penalty_s": 0.0, "site_evals": 0, "wasted_site_evals": 0}
    results: Dict[int, dict] = {}
    if not sites:
        if stats is not None:
            stats.update(st, wall_s=0.0)
        return results
    state: Dict[int, _Site] = {}
    for idx in sorted(sites):   # modules are built in index order: the rating kind draws from torch's global generator
        tup = sites[idx]
        X, y = np.ascontiguousarray(tup[0], dtype=np.float64), np.ascontiguousarray(tup[1], dtype=np.float64)
        noise = np.ascontiguousarray(tup[2], dtype=np.float64) if len(tup) > 2 and tup[2] is not None else kind.default_noise(y.shape[0])
        state[idx] = _Site(idx, X, y, noise, kind.module(X, y, noise))
    order = sorted(state, key=lambda i: (-state[i].X.shape[0], i))
    group = max(1, min(int(group), capi.BATCH_MAX_SITES))
    lanes = max(1, int(lanes))
    if lanes > 1 and len(order) >= 2 * lanes:   # enough sites for `lanes` groups at a time: never leave a lane empty
        group = min(group, -(-len(order) // lanes))
    pending = _groups(order, group)              # largest sites first
    lanes = min(lanes, len(pending)) if iterations > 0 else 1
    st["lanes"] = lanes
    n_max = state[order[0]].X.shape[0]
    handles: List[capi.BatchEngine] = []

    def close_group(grp, batch: Optional[capi.BatchEngine] = None):
        """Results of a finished group; its predictions run on the group's batch handle (idle now: the other lane's group keeps
        the GPU busy meanwhile), or on a handle of its own when the group was never fitted (iterations <= 0)."""
        t0 = time.perf_counter()
        res_of = {}
        for s in grp:
            with torch.no_grad():
                theta = s.module.natural().numpy().astype(np.float64)
            res_of[s.idx] = {"theta": theta, "history": s.history, "objective": s.history[-1] if s.history else None,
                             "failed": s.failed, "n": int(s.X.shape[0]), "stopped_at": s.stopped_at}
            if pen is not None:
                res_of[s.idx]["penalty"] = s.penalty
        want = [predict is not None and s.idx in predict and s.failed is None for s in grp]
        if any(want):
            own = batch is None
            if own:
                batch = capi.BatchEngine(max_sites=len(grp), max_n=max(s.X.shape[0] for s in grp), device=device)
            try:
                if own:
                    batch.set_train(grp[0].module.spec.to_c(), [(s.X, s.y, s.noise) for s in grp])
                _predict_group(batch, grp, want, predict, kind, res_of)
            finally:
                if own:
                    batch.close()
        for s in grp:
            results[s.idx] = res_of[s.idx]
        st["predict_s"] += time.perf_counter() - t0

    try:
        if iterations <= 0:
            for members in pending:
                st["groups"] += 1
                close_group([state[i] for i in members])
        else:
            for _ in range(lanes):
                handles.append(capi.BatchEngine(max_sites=min(group, len(order)), max_n=n_max, device=device))
            runs: List[Optional[_GroupRun]] = [None] * lanes

            def next_group(lane):
                if not pending:
                    return None
                members = pending.pop(0) if lane == 0 else pending.pop()   # lane 0 from the large end, the others from the small end
                st["groups"] += 1
                return _GroupRun([state[i] for i in members], handles[lane], kind, iterations, lr, scheduler, patience, st,
                                 stats is not None, early_stopping, pen)

            # rolling: every lane always has an evaluation in flight (wait -> host step -> launch the next one), so the GPU
            # works on one group while the host steps the other
            t_loop, p_before = time.perf_counter(), st["predict_s"]
            for lane in range(lanes):
                runs[lane] = next_group(lane)
                if runs[lane] is not None:
                    runs[lane].launch()
            while any(r is not None for r in runs):
                for lane, r in enumerate(runs):
                    if r is None:
                        continue
                    if r.inflight:
                        r.finish()
                    if r.left > 0 and not r.launch() and r.left <= 0:
                        r.opt.push()             # (every site of the group has failed: nothing left to evaluate)
                    if r.done:
                        close_group(r.grp, r.batch)
                        runs[lane] = next_group(lane)
                        if runs[lane] is not None:
                            runs[lane].launch()
            st["fit_wall_s"] = (time.perf_counter() - t_loop) - (st["predict_s"] - p_before)
    finally:
        for b in handles:
            b.close()
    if stats is not None:
        stats.update(st, wall_s=time.perf_counter() - t_start)
    return results


# ---------------------------------------------------------------- round-1 path: one handle and launch sequence per site
@dataclass
class _SiteState:
    idx: int
    X: np.ndarray
    y: np.ndarray
    noise: np.ndarray
    module: GPModule
    engine: capi.Engine
    opt: torch.optim.Optimizer
    sched: Optional[torch.optim.lr_scheduler.ReduceLROnPlateau]
    chain: Optional[tuple] = None  # GPModule.host_chain() of the evaluation in flight
    history: List[float] = field(default_factory=list)
    failed: Optional[str] = None


def _finish_step(s: _SiteState):
    """Host side of one optimiser step (discontinuum/engines/gpytorch.py:353-420) once the GPU results are back: the
    constraint / prior chain rule in closed form (GPModule.host_chain, no autograd graph), clipping, Adam, scheduler."""
    val, grad, info = s.engine.nlml_grad_wait()
    nat, dnat, lp, dlp = s.chain
    if info != 0 or not np.isfinite(val):
        for jit in JITTERS[1:]:
            val, grad, info = s.engine.nlml_grad(nat, jit)
            if info == 0 and np.isfinite(val):
                break
        else:
            s.failed = f"not positive definite (info={info})"
            return
    n = s.X.shape[0]
    obj = (val - lp) / n
    graw = (grad - dlp) * dnat / n
    coef = 1.0 / (float(np.sqrt(np.sum(graw * graw))) + 1e-6)   # clip_grad_norm_(max_norm=1.0)
    if not coef >= 1.0:
        graw = graw * coef
    if np.isnan(graw).any():
        graw = np.nan_to_num(graw, nan=0.0, posinf=0.0, neginf=0.0)
    for p, gv in zip(s.module.raw_list(), graw):
        p.grad = torch.tensor([gv], dtype=torch.float64)
    s.opt.step()
    s.history.append(float(obj))
    if s.sched is not None:
        s.sched.step(s.history[-1])


_COMPLETION_ORDER = True  # serve sites as their evaluations finish (False: fixed round, blocking on each in turn)


def _open_site(idx, tup, device, lr, scheduler, patience, pool: Optional[List[capi.Engine]] = None) -> _SiteState:
    X, y = np.ascontiguousarray(tup[0], dtype=np.float64), np.ascontiguousarray(tup[1], dtype=np.float64)
    noise = np.ascontiguousarray(tup[2], dtype=np.float64) if len(tup) > 2 else np.full(y.shape[0], LOADEST_FIXED_NOISE)
    module = GPModule(loadest_spec(X.shape[1]))
    eng = None
    if pool:  # reuse the workspace of a finished (larger) site: no cudaMalloc / cudaFree (a device-wide sync) mid-batch
        k = next((i for i, e in enumerate(pool) if e.max_n >= X.shape[0]), None)
        if k is not None:
            eng = pool.pop(k)
    if eng is None:
        eng = capi.Engine(max_n=X.shape[0], max_m=2048, device=device)
    eng.set_train(module.spec.to_c(), X, y, noise)
    opt = torch.optim.Adam(module.raw_list(), lr=lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-4, fused=True)
    sch = None
    if scheduler:
        sch = torch.optim.lr_scheduler.ReduceLROnPlateau(opt, mode="min", factor=0.7, patience=max(20, patience // 2),
                                                         threshold=1e-4, threshold_mode="rel", min_lr=1e-6, cooldown=10)
    return _SiteState(idx, X, y, noise, module, eng, opt, sch)


def _launch_step(s: _SiteState):
    s.opt.zero_grad(set_to_none=True)
    s.chain = s.module.host_chain()
    s.engine.nlml_grad_launch(np.ascontiguousarray(s.chain[0]))


def _close_site(s: _SiteState, predict, pool: Optional[List[capi.Engine]] = None) -> dict:
    with torch.no_grad():
        theta = s.module.natural().numpy().astype(np.float64)
    res = {"theta": theta, "history": s.history, "objective": s.history[-1] if s.history else None, "failed": s.failed,
           "n": int(s.X.shape[0])}
    if predict is not None and s.idx in predict and s.failed is None:
        for jit in JITTERS:
            _, info = s.engine.factorize(theta, jit)
            if info == 0:
                break
        else:
            res["failed"] = f"prediction: not positive definite after jitter {JITTERS[-1]:g} (info={info})"
        if res["failed"] is None:
            mu, var = s.engine.predict(predict[s.idx])
            res["mu"], res["var_latent"] = mu, var
            res["var"] = observed_variance(s.module.spec, theta, var, s.noise, predict[s.idx].shape[0])
    if pool is not None:
        pool.append(s.engine)
    else:
        s.engine.close()
    return res


def fit_sites_local_per_handle(sites: Dict[int, tuple], iterations: int = 100, device: int = 0, concurrency: int = 4,
                               predict: Optional[Dict[int, np.ndarray]] = None, lr: float = 0.05, scheduler: bool = True,
                               patience: int = 60) -> Dict[int, dict]:
    """Round-1 driver, kept for comparison and as the reference of the bit-identity tests: `concurrency` loadest sites in
    flight, each a pipeline of its own on its own libdgp handle and streams (dgp_nlml_grad_launch / _ready / _wait), served
    in completion order."""
    results: Dict[int, dict] = {}
    queue = sorted(sites, key=lambda i: -sites[i][0].shape[0])  # largest first: later sites fit the pooled workspaces
    active: List[_SiteState] = []
    pool: List[capi.Engine] = []

    def refill():
        while queue and len(active) < max(1, concurrency):
            s = _open_site(queue[0], sites[queue.pop(0)], device, lr, scheduler, patience, pool)
            if iterations > 0:
                _launch_step(s)
            active.append(s)

    refill()
    while active:
        served = False
        for s in list(active):
            if iterations > 0 and _COMPLETION_ORDER and not s.engine.nlml_grad_ready():
                continue
            served = True
            if iterations > 0:
                _finish_step(s)
            if s.failed is None and len(s.history) < iterations:
                _launch_step(s)
                continue
            active.remove(s)
            results[s.idx] = _close_site(s, predict, pool)
            refill()
        if not served:
            time.sleep(0)  # nothing finished yet: yield, then poll again
    for e in pool:
        e.close()
    return results


def fit_sites(sites: Dict[int, tuple], iterations: int = 100, predict: Optional[Dict[int, np.ndarray]] = None,
              group: int = 16, dist=None, device: int = 0, model="loadest", stats: Optional[dict] = None,
              concurrency: Optional[int] = None, lanes: int = 2, early_stopping: bool = False, patience: int = 60,
              monotonic_penalty_weight: float = 0.0, grid_size: int = 64, monotonic_penalty_interval: int = 1,
              penalty_seed: int = 0) -> Optional[Dict[int, dict]]:
    """Shard `sites` (every rank holds the same dict, or at least the same keys and sizes) over the ranks of
    `dist`, fit this rank's share, gather everything on rank 0.  The fit options are fit_sites_local's."""
    world = dist.get_world_size() if dist is not None and dist.is_initialized() else 1
    rank = dist.get_rank() if world > 1 else 0
    keys = sorted(sites)
    costs = [site_cost(sites[k][0].shape[0], iterations, predict[k].shape[0] if predict and k in predict else 0) for k in keys]
    mine = [keys[i] for i in assign_sites(costs, world)[rank]]
    local = fit_sites_local({k: sites[k] for k in mine}, iterations=iterations, device=device, group=group,
                            predict={k: predict[k] for k in mine} if predict else None, model=model, stats=stats,
                            concurrency=concurrency, lanes=lanes, early_stopping=early_stopping, patience=patience,
                            monotonic_penalty_weight=monotonic_penalty_weight, grid_size=grid_size,
                            monotonic_penalty_interval=monotonic_penalty_interval, penalty_seed=penalty_seed)
    return gather_results(local, dist)


# ---------------------------------------------------------------- sharded prediction grid (SURVEY 8e)
def shard_rows(m: int, world: int) -> List[tuple]:
    """Contiguous row ranges [start, stop) of an m-point grid, one per rank, sizes differing by at most one."""
    base, rem = divmod(int(m), int(world))
    out, start = [], 0
    for r in range(world):
        stop = start + base + (1 if r < rem else 0)
        out.append((start, stop))
        start = stop
    return out


def predict_sharded(engine, Xs: np.ndarray, dist=None, want_var: bool = True):
    """Posterior mean / latent variance over a grid sharded across ranks.  Every rank holds the same factorisation
    (fitted redundantly or loaded from the same checkpoint: `engine.factorize` was called with the same theta) and
    predicts its contiguous slice; the only collective is the final all_gather of 16 m bytes.  `engine` is a
    capi.Engine (anything with .predict(Xs, want_var) -> (mu, var)).  Returns (mu[m], var[m]) on every rank."""
    Xs = np.ascontiguousarray(Xs, dtype=np.float64)
    m = Xs.shape[0]
    world = dist.get_world_size() if dist is not None and dist.is_initialized() else 1
    rank = dist.get_rank() if world > 1 else 0
    lo, hi = shard_rows(m, world)[rank]
    if hi > lo:
        mu, var = engine.predict(Xs[lo:hi], want_var)
    else:
        mu, var = np.empty(0), (np.empty(0) if want_var else None)
    if world == 1:
        return mu, var
    parts = [None] * world
    dist.all_gather_object(parts, (np.asarray(mu), None if var is None else np.asarray(var)))
    mu_all = np.concatenate([p[0] for p in parts])
    var_all = np.concatenate([p[1] for p in parts]) if want_var else None
    return mu_all, var_all


# ---------------------------------------------------------------- joint posterior draws over a sharded grid (SURVEY 8e)
def panel_owner(p: int, world: int) -> int:
    """Panel-cyclic distribution of the posterior covariance's block columns."""
    return p % world


def sample_sharded(engine, Xs: np.ndarray, S: int, dist=None, seed: int = 0, jitter: float = 0.0, Z: Optional[np.ndarray] = None,
                   stats: Optional[dict] = None):
    """Exact joint posterior draws [S, m] with the m x m posterior-covariance Cholesky distributed over the ranks of
    `dist` (torch.distributed, NCCL).  Every rank holds the same training factorisation (`engine.factorize` at the same
    theta) and calls this with the same arguments; every rank returns (draws, info).

    Exchange steps (the only collectives): all_gather of V' (m x n), all_reduce of the mean, one broadcast of the
    sub-diagonal rows of each factored panel from its owner, all_reduce of the partial draws.  Look-ahead: the owner of
    panel p+1 updates that panel first, factors it on a high-priority side stream and broadcasts it while every rank
    is still applying panel p to the rest of its columns.  The engine must have been created on torch's current CUDA
    stream (`capi.Engine(stream=torch.cuda.current_stream().cuda_stream)`); with a private engine stream the kernels and
    collectives are ordered through host synchronisation instead (correct, no overlap)."""
    Xs = np.ascontiguousarray(Xs, dtype=np.float64)
    m = Xs.shape[0]
    world = dist.get_world_size() if dist is not None and dist.is_initialized() else 1
    rank = dist.get_rank() if world > 1 else 0
    dims = engine.dist_dims(m, S, world)
    dev = torch.device("cuda", engine.device)
    f64 = dict(dtype=torch.float64, device=dev)
    rpr = dims["rows_per_rank"]
    VT = torch.zeros((rpr * world, dims["npad"]), **f64)
    packs = [torch.empty((dims["mpad"], dims["panel_cols"]), **f64) for _ in range(2)]
    Od = torch.empty((dims["Spad"], dims["mpad"]), **f64)
    mu = torch.empty((dims["mpad"],), **f64)
    T = torch.cuda.current_stream(dev)
    shared_stream = engine.stream != 0 and engine.stream == T.cuda_stream
    side = torch.cuda.Stream(device=dev, priority=-1) if shared_stream else None  # look-ahead stream

    def fence():  # engine on a private stream: order kernels and collectives through the host instead
        if not shared_stream:
            torch.cuda.synchronize(dev)

    pw_blocks, mb, npanels = dims["panel_cols"] // 128, dims["mpad"] // 128, dims["npanels"]

    def rows_below(p):
        return (mb - min((p + 1) * pw_blocks, mb)) * 128

    if stats is not None:   # bytes each collective moves (payload of the buffer it is called on), for the bench line
        stats.update(world=world, npanels=npanels, all_gather_VT_bytes=int(VT.numel()) * 8 if world > 1 else 0,
                     all_reduce_mu_bytes=int(mu.numel()) * 8 if world > 1 else 0,
                     broadcast_panel_bytes=sum(rows_below(p) for p in range(npanels)) * dims["panel_cols"] * 8 if world > 1 else 0,
                     all_reduce_draws_bytes=int(Od.numel()) * 8 if world > 1 else 0)
    tok = engine.dist_begin(Xs, S, Z, seed, jitter, rank, world, VT, Od, mu)
    try:
        engine.dist_call("vt_rows", tok, rank * rpr, min((rank + 1) * rpr, dims["mpad"]))
        if world > 1:
            fence()
            dist.all_gather_into_tensor(VT, VT[rank * rpr:(rank + 1) * rpr].clone())
            dist.all_reduce(mu)
            fence()
        engine.dist_call("sigma", tok)
        # p = -1 bootstraps panel 0; iteration p leaves panel p+1 factored and in place on every rank
        for p in range(-1, npanels - 1):
            nxt = p + 1
            owner = panel_owner(nxt, world)
            buf = packs[nxt % 2]
            rows = rows_below(nxt)
            work = None
            if owner == rank:
                if p >= 0:
                    engine.dist_call("trail", tok, p, nxt, nxt)          # panel p -> panel p+1 first
                if side is not None:
                    side.wait_event(T.record_event())
                    engine.dist_call("panel_factor", tok, nxt, buf.data_ptr(), side.cuda_stream)
                else:
                    engine.dist_call("panel_factor", tok, nxt, buf.data_ptr(), None)
            if world > 1 and rows > 0:
                if side is not None:
                    if owner != rank:
                        side.wait_event(T.record_event())              # the receive buffer is free once T got here
                    with torch.cuda.stream(side):
                        work = dist.broadcast(buf[:rows], src=owner, async_op=True)
                else:
                    fence()
                    dist.broadcast(buf[:rows], src=owner)
                    fence()
            if p >= 0:
                engine.dist_call("trail", tok, p, nxt + 1, npanels - 1)  # ... then the rest, overlapping the above
            if work is not None:
                work.wait()                                                # T waits for the broadcast
            elif side is not None and owner == rank:
                T.wait_stream(side)
            if owner != rank and rows > 0:
                engine.dist_call("panel_unpack", tok, nxt, buf.data_ptr())
        engine.dist_call("draws_partial", tok)
        if world > 1:
            fence()
            dist.all_reduce(Od)
            fence()
        out = np.empty((S, m))
        info = engine.dist_call("finish", tok, out.ctypes.data)
        if world > 1:
            t = torch.tensor([info if info > 0 else 2 ** 31 - 1], dtype=torch.int64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)  # first failing pivot over all ranks
            info = 0 if int(t) == 2 ** 31 - 1 else int(t)
        return out, info
    finally:
        engine.dist_call("end", tok)
