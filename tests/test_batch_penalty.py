"""Rating-gp monotonicity penalty and early stopping in the multi-site batch driver, and the batched adjoint of the posterior
mean behind the penalty (dgp_batch_mean_functional_grad).

CPU: the driver against the oracle's restatement of the reference loop, through an oracle-backed stand-in for the batch
handle (penalised trajectories, independence from lanes and group sizes, the early-stopping rule, argument checks).
GPU: every site of a batch gets exactly the numbers of a per-site handle (value and gradient, bit for bit) for ragged sizes,
point counts across the chunk's 128-row blocks, per-site jitter and a fixture spec; mean-only prediction after an
evaluation; the state rules; the launch count; and the driver against orc.fit_adam, RatingGP.fit and LoadestGP.fit."""
import numpy as np
import pytest
import torch

import helpers as H
from discontinuum_b200 import capi, models, multisite, synthetic
from discontinuum_b200.spec import CovSpec, Factor, GPModule
from helpers import orc

CHUNK = capi.BATCH_PREDICT_CHUNK


# ---------------------------------------------------------------------------------------------------- CPU stand-ins
class _OracleRatingBatch:
    """capi.BatchEngine's surface as fit_sites_local drives it for rating gauges, served by the CPU oracle: nlml_grad (autograd
    through the Cholesky), mean-only predict and mean_functional_grad (autograd of c'mu through orc.predict) at the theta of
    the last evaluation."""

    def __init__(self, max_sites, max_n, device=0):
        self.inflight = None

    def set_train(self, spec_c, sites):
        self.sites = [(torch.tensor(X), torch.tensor(y), torch.tensor(nz)) for X, y, nz in sites]
        self.theta = None

    def set_timing(self, on):
        pass

    def last_timing(self):
        return [0.0, 0.0, 0.0, 0.0]

    def _eval(self, theta):
        G = len(self.sites)
        val, grad, info = np.zeros(G), np.zeros((G, theta.shape[1])), np.zeros(G, dtype=np.int32)
        for k, (X, y, nz) in enumerate(self.sites):
            v, g = orc.nlml_grad_autograd(orc.rating_cov, orc.rating_mean, H.rating_nat_from_theta(theta[k]), X, y, nz,
                                          extra_key="noise")
            val[k], grad[k] = float(v), H.rating_theta_from_nat({n: t.numpy() for n, t in g.items()})
        self.theta = theta
        return val, grad, info

    def nlml_grad_launch(self, theta, jitter=None):
        assert self.inflight is None, "one evaluation in flight per handle"
        self.inflight = np.array(theta)

    def nlml_grad_wait(self):
        theta, self.inflight = self.inflight, None
        return self._eval(theta)

    def nlml_grad(self, theta, jitter=None):
        return self._eval(np.array(theta))

    def _mu(self, k, nat, pts):
        X, y, nz = self.sites[k]
        return orc.predict(orc.rating_cov, orc.rating_mean, nat, X, y, nz, torch.tensor(pts), extra_noise=nat["noise"])[0]

    def predict(self, grids, want_var=True):
        assert not want_var and self.inflight is None and len(grids) == len(self.sites)
        out = []
        for k, g in enumerate(grids):
            out.append((None, None) if g is None else (self._mu(k, H.rating_nat_from_theta(self.theta[k]), g).numpy(), None))
        return out

    def mean_functional_grad(self, points, c):
        assert self.inflight is None
        G = len(self.sites)
        val, grad = np.zeros(G), np.zeros((G, self.theta.shape[1]))
        for k, (p, cv) in enumerate(zip(points, c)):
            if p is None:
                continue
            leaves = {n: t.detach().clone().requires_grad_(True) for n, t in H.rating_nat_from_theta(self.theta[k]).items()}
            F = torch.tensor(cv) @ self._mu(k, leaves, p)
            gs = torch.autograd.grad(F, list(leaves.values()), allow_unused=True)
            val[k] = float(F.detach())
            grad[k] = [0.0 if g is None else float(g) for g in gs]
        return val, grad

    def close(self):
        pass


def _gauges(ns, seed0=40):
    """rating gauges; every other one with the discharge falling with stage, so that the penalty has work to do"""
    out = {}
    for i, n in enumerate(ns):
        X, y, noise = synthetic.rating_gauge(n, seed0 + i)
        out[i] = (X, -y if i % 2 else y, noise)
    return out


def _reference_penalised(sites, iterations, weight, grid_size, penalty_seed, init_seed):
    """orc.fit_adam per gauge with the driver's initial draws (all gauges in index order from torch's generator seeded with
    init_seed) and penalty grids (torch's generator seeded with penalty_seed + idx right before the fit)."""
    torch.manual_seed(init_seed)
    draws = {}
    for i in sorted(sites):
        a = float(torch.randn(1)); b = float(torch.randn(1) + 1.3); c = float(torch.rand(1)); u = float(torch.rand(1))
        draws[i] = (a, b, c, u)
    out = {}
    for i in sorted(sites):
        X, y, noise = sites[i]
        a, b, c, u = draws[i]
        b_lo, b_hi = models.stage_quantile_bounds(X[:, 1])
        raw = orc.rating_init_raw(b_lo, b_hi, gate_b=b_lo + u * (b_hi - b_lo), pl_a=a, pl_b=b, pl_c=c)
        torch.manual_seed(penalty_seed + i)
        _, hist = orc.fit_adam("rating", raw, torch.tensor(X), torch.tensor(y), torch.tensor(noise), iterations=iterations,
                               b_lo=b_lo, b_hi=b_hi, h_min=float(X[:, 1].min()), penalty_weight=weight, grid_size=grid_size)
        out[i] = hist
    return out


def test_penalised_driver_matches_reference_loop(monkeypatch):
    monkeypatch.setattr(capi, "BatchEngine", _OracleRatingBatch)
    sites = _gauges((40, 28, 33))
    iters = 6
    torch.manual_seed(1)
    res = multisite.fit_sites_local(sites, iterations=iters, model="rating", group=3, monotonic_penalty_weight=0.5,
                                    grid_size=16, penalty_seed=11)
    torch.manual_seed(1)
    plain = multisite.fit_sites_local(sites, iterations=iters, model="rating", group=3)
    want = _reference_penalised(sites, iters, 0.5, 16, 11, 1)
    active = 0
    for i in sites:
        r = res[i]
        assert r["failed"] is None and len(r["history"]) == iters and r["stopped_at"] is None
        assert H.relerr(r["history"], want[i]) <= 1e-10, (i, r["history"], want[i])
        assert r["penalty"] is not None and r["penalty"] >= 0.0 and "penalty" not in plain[i]
        active += r["penalty"] > 0.0 and r["history"] != plain[i]["history"]
    assert active > 0   # the penalty was active and changed at least one trajectory


def test_penalised_driver_independent_of_lanes_and_groups(monkeypatch):
    monkeypatch.setattr(capi, "BatchEngine", _OracleRatingBatch)
    sites = _gauges((36, 30, 26, 41, 22), 60)
    runs = []
    for lanes, group in ((1, 16), (2, 16), (3, 2), (1, 1)):
        torch.manual_seed(2)
        runs.append(multisite.fit_sites_local(sites, iterations=4, model="rating", group=group, lanes=lanes,
                                              monotonic_penalty_weight=0.5, grid_size=12, monotonic_penalty_interval=2,
                                              penalty_seed=5))
    for r in runs[1:]:
        for i in sites:
            assert r[i]["history"] == runs[0][i]["history"] and np.array_equal(r[i]["theta"], runs[0][i]["theta"])
            assert r[i]["penalty"] == runs[0][i]["penalty"]


class _QuadKind:
    """Sites whose NLML is n |theta - target|^2 over two positive parameters without priors: Adam reaches the minimum of a
    near target within a few iterations and then stalls (early stopping), and keeps improving toward a far one."""
    name = "quad"

    def module(self, X, y, noise):
        s = CovSpec(ndim=1)
        c = s.col_copy(0)
        sc, ls = s.param("s"), s.param("l")
        s.term(sc, [Factor(capi.RBF, [c], [ls])])
        return GPModule(s)

    def default_noise(self, n):
        return np.full(n, 0.01)

    def project(self, module, X):
        pass

    def project_raw(self, raw, modules, Xs):
        pass


class _QuadBatch:
    def __init__(self, max_sites, max_n, device=0):
        self.inflight = None

    def set_train(self, spec_c, sites):
        self.targets = [np.array([y[0], y[1]]) for _, y, _ in sites]
        self.ns = [X.shape[0] for X, _, _ in sites]

    def set_timing(self, on):
        pass

    def _eval(self, theta):
        d = theta - np.stack(self.targets)
        n = np.array(self.ns, dtype=np.float64)
        return n * np.sum(d * d, axis=1), 2.0 * n[:, None] * d, np.zeros(len(self.ns), dtype=np.int32)

    def nlml_grad_launch(self, theta, jitter=None):
        self.inflight = np.array(theta)

    def nlml_grad_wait(self):
        theta, self.inflight = self.inflight, None
        return self._eval(theta)

    def nlml_grad(self, theta, jitter=None):
        return self._eval(np.array(theta))

    def close(self):
        pass


def _stop_rule(history, patience):
    best, counter = float("inf"), 0
    for i, h in enumerate(history):
        if h < best - 1e-6:
            best, counter = h, 0
        else:
            counter += 1
        if counter >= patience:
            return i + 1
    return None


def test_early_stopping_is_a_prefix_of_the_full_run(monkeypatch):
    monkeypatch.setattr(capi, "BatchEngine", _QuadBatch)
    n = 8
    X = np.zeros((n, 1))
    sites = {0: (X, np.array([6.0, 5.0] + [0.0] * (n - 2))),      # far: still improving at the end
             1: (X, np.array([0.75, 0.70] + [0.0] * (n - 2))),    # near: stalls and stops
             2: (X, np.array([0.9, 0.5] + [0.0] * (n - 2)))}
    kw = dict(iterations=60, model=_QuadKind(), scheduler=False, patience=5)
    full = multisite.fit_sites_local(sites, **kw)
    runs = [multisite.fit_sites_local(sites, early_stopping=True, lanes=lanes, group=group, **kw)
            for lanes, group in ((1, 16), (2, 1))]
    stopped = 0
    for es in runs:
        for i in sites:
            k = _stop_rule(full[i]["history"], 5)
            assert es[i]["stopped_at"] == k, (i, es[i]["stopped_at"], k)
            if k is None:
                assert es[i]["history"] == full[i]["history"] and np.array_equal(es[i]["theta"], full[i]["theta"])
                continue
            stopped += 1
            assert es[i]["history"] == full[i]["history"][:k]
            short = multisite.fit_sites_local({i: sites[i]}, **dict(kw, iterations=k))   # its last parameters, not its best
            assert np.array_equal(es[i]["theta"], short[i]["theta"])
    assert full[0]["stopped_at"] is None and _stop_rule(full[0]["history"], 5) is None   # one site runs to the end ...
    assert stopped > 0                                                                   # ... and at least one stops


def test_driver_argument_checks(monkeypatch):
    monkeypatch.setattr(capi, "BatchEngine", _OracleRatingBatch)
    g = _gauges((20,))
    lo = {0: synthetic.loadest_site(20, 3)[:2]}
    with pytest.raises(ValueError, match="rating"):
        multisite.fit_sites_local(lo, iterations=2, monotonic_penalty_weight=0.5)
    with pytest.raises(ValueError, match="grid_size"):
        multisite.fit_sites_local(g, iterations=2, model="rating", monotonic_penalty_weight=0.5, grid_size=513)
    with pytest.raises(ValueError, match="monotonic_penalty_interval"):
        multisite.fit_sites_local(g, iterations=2, model="rating", monotonic_penalty_weight=0.5, monotonic_penalty_interval=0)
    with pytest.raises(ValueError, match="batch driver"):
        multisite.fit_sites_local(lo, iterations=2, concurrency=2, early_stopping=True)
    with pytest.raises(ValueError):
        multisite.fit_sites(g, iterations=2, model="rating", concurrency=2, monotonic_penalty_weight=0.5)
    res = multisite.fit_sites_local(g, iterations=2, model="rating", monotonic_penalty_weight=0.5, grid_size=512)
    assert len(res[0]["history"]) == 2


def test_penalty_grid_generator():
    X = synthetic.rating_gauge(50, 1)[0]
    a = models.monotonic_penalty_grid(X, 8, generator=torch.Generator().manual_seed(4))
    torch.manual_seed(4)
    b = models.monotonic_penalty_grid(X, 8)
    assert np.array_equal(a, b)


# ---------------------------------------------------------------------------------------------------- GPU
def _points(X, m, seed):
    """m points over the record (time uniform, stage / covariate from the record, nudged)"""
    if m == 0:
        return None
    rng = np.random.default_rng(seed)
    g = synthetic.daily_grid(X, m)
    g[:, 1:] += 1e-3 * rng.uniform(size=(m, X.shape[1] - 1))
    return np.ascontiguousarray(g)


def _weights(m, seed):
    return None if m == 0 else np.random.default_rng(seed).standard_normal(m)


def _per_site_mfg(spec, site, theta, pts, c, jitter, factorize):
    X, y, noise = site
    eng = capi.Engine(max_n=X.shape[0], max_m=CHUNK)
    eng.set_train(spec.to_c(), X, y, noise)
    if factorize:
        _, info = eng.factorize(theta, jitter)
    else:
        _, _, info = eng.nlml_grad(theta, jitter)
    assert info == 0
    mu, _ = eng.predict(pts, want_var=False)
    val, grad = eng.mean_functional_grad(pts, c)
    eng.close()
    return val, grad, mu


def _check_mfg(spec, sites, thetas, ms, jit=None, seed=0):
    G = len(sites)
    b = capi.BatchEngine(max_sites=G, max_n=max(s[0].shape[0] for s in sites))
    b.set_train(spec.to_c(), sites)
    pts = [_points(s[0], m, seed + k) for k, (s, m) in enumerate(zip(sites, ms))]
    cs = [_weights(m, seed + 100 + k) for k, m in enumerate(ms)]
    for factorize in (False, True):
        if factorize:
            _, info = b.factorize(thetas, jit)
        else:
            _, _, info = b.nlml_grad(thetas, jit)
            with pytest.raises(capi.DgpError, match="factorize"):
                b.predict(pts)          # the variance still needs a factorisation
        assert np.all(info == 0)
        mean_only = b.predict(pts, want_var=False)
        val, grad = b.mean_functional_grad(pts, cs)
        for k, s in enumerate(sites):
            if ms[k] == 0:
                assert val[k] == 0.0 and not grad[k].any() and mean_only[k] == (None, None)
                continue
            v, g, mu = _per_site_mfg(spec, s, thetas[k], pts[k], cs[k], 0.0 if jit is None else float(jit[k]), factorize)
            assert np.array_equal(mean_only[k][0], mu), (factorize, k, np.max(np.abs(mean_only[k][0] - mu)))
            assert val[k] == v and np.array_equal(grad[k], g), (factorize, k, val[k] - v, np.max(np.abs(grad[k] - g)))
    b.close()


@pytest.mark.gpu
def test_batch_mfg_rating_ragged(cuda_device):
    ns = (129, 300, 1300, 640, 200, 257)
    ms = (1, 127, 1024, 0, 128, 500)
    sites = [synthetic.rating_gauge(n, 70 + k) for k, n in enumerate(ns)]
    spec = models.rating_spec(1.0, 2.0)
    thetas = np.stack([H.rating_theta1(*models.stage_quantile_bounds(X[:, 1])) * (1.0 + 0.01 * k)
                       for k, (X, _, _) in enumerate(sites)])
    _check_mfg(spec, sites, thetas, ms, jit=np.array([0.0, 1e-6, 0.0, 1e-4, 3e-5, 0.0]))


@pytest.mark.gpu
def test_batch_mfg_loadest_ragged(cuda_device):
    ns = (1300, 129, 513, 384, 700)
    ms = (1024, 128, 0, 129, 1)
    sites = [synthetic.loadest_site(n, 800 + k) for k, n in enumerate(ns)]
    thetas = np.stack([H.loadest_theta1() * (1.0 + 0.02 * k) for k in range(len(ns))])
    _check_mfg(models.loadest_spec(2), sites, thetas, ms, seed=5)


@pytest.mark.gpu
def test_batch_mfg_fixture_spec(cuda_device):
    import test_spec_generic as tsg

    spec, theta = tsg.FIXTURES["F4"]()
    ns = (37, 300, 700)
    sites = [tsg._data(spec, theta, n, 900 + n) for n in ns]
    thetas = np.stack([theta * (1.0 + 0.02 * k) for k in range(len(ns))])
    b = capi.BatchEngine(max_sites=3, max_n=700)
    b.set_train(spec.to_c(), sites)
    _, _, info = b.nlml_grad(thetas)
    assert np.all(info == 0)
    pts = [tsg._grid(s[0], m, 5, 950 + k)[0] for k, (s, m) in enumerate(zip(sites, (300, 1024, 129)))]
    cs = [_weights(p.shape[0], 960 + k) for k, p in enumerate(pts)]
    val, grad = b.mean_functional_grad(pts, cs)
    for k, s in enumerate(sites):
        v, g, _ = _per_site_mfg(spec, s, thetas[k], pts[k], cs[k], 0.0, False)
        assert val[k] == v and np.array_equal(grad[k], g), (k, np.max(np.abs(grad[k] - g)))
    b.close()


@pytest.mark.gpu
def test_batch_mfg_state_rules_and_launches(cuda_device):
    spec = models.loadest_spec(2)
    ns = (300, 500, 260)
    sites = [synthetic.loadest_site(n, 4000 + k) for k, n in enumerate(ns)]
    thetas = np.stack([H.loadest_theta1()] * 3)
    X, y, noise = sites[1]
    noise = noise.copy()
    noise[200:] = -3.0      # indefinite from row 200 on: this site's evaluation fails
    sites[1] = (X, y, noise)
    pts = [_points(s[0], 200, k) for k, s in enumerate(sites)]
    cs = [_weights(200, 10 + k) for k in range(3)]
    b = capi.BatchEngine(max_sites=3, max_n=500)
    b.set_train(spec.to_c(), sites)
    with pytest.raises(capi.DgpError, match="no successful evaluation"):
        b.mean_functional_grad(pts, cs)                     # nothing evaluated since set_train
    _, _, info = b.nlml_grad(thetas)
    assert info[0] == 0 and info[1] != 0 and info[2] == 0
    with pytest.raises(capi.DgpError, match="site 1"):
        b.mean_functional_grad(pts, cs)                     # the failed site
    with pytest.raises(capi.DgpError, match="site 1"):
        b.predict([None, pts[1], None], want_var=False)
    val, _ = b.mean_functional_grad([pts[0], None, pts[2]], [cs[0], None, cs[2]])
    assert val[1] == 0.0 and val[0] != 0.0
    big = _points(sites[0][0], CHUNK + 1, 3)
    with pytest.raises(capi.DgpError, match="m = 1025"):
        b.mean_functional_grad([big, None, None], [_weights(CHUNK + 1, 4), None, None])
    b.nlml_grad_launch(thetas)
    with pytest.raises(capi.DgpError, match="in flight"):
        b.mean_functional_grad([pts[0], None, None], [cs[0], None, None])
    b.nlml_grad_wait()
    b.set_train(spec.to_c(), [sites[0], sites[2]])
    with pytest.raises(capi.DgpError, match="no successful evaluation"):
        b.mean_functional_grad([pts[0], None], [cs[0], None])
    b.close()
    # one call costs the same launches for 1 and for 16 sites
    per = {}
    for G in (1, 16):
        gs = [synthetic.loadest_site(150 + 37 * k, 5000 + k) for k in range(G)]
        bb = capi.BatchEngine(max_sites=G, max_n=max(s[0].shape[0] for s in gs))
        bb.set_train(spec.to_c(), gs)
        bb.nlml_grad(np.stack([H.loadest_theta1()] * G))
        l0 = bb.launches
        bb.mean_functional_grad([_points(s[0], 300, k) for k, s in enumerate(gs)], [_weights(300, k) for k in range(G)])
        per[G] = bb.launches - l0
        bb.close()
    assert per[1] == per[16], per


@pytest.mark.gpu
def test_fit_sites_penalty_matches_reference_loop(cuda_device):
    sites = _gauges((150, 260, 200, 330), 20)
    torch.manual_seed(0)
    res = multisite.fit_sites(sites, iterations=8, model="rating", group=4, monotonic_penalty_weight=0.5, grid_size=64,
                              penalty_seed=3)
    want = _reference_penalised(sites, 8, 0.5, 64, 3, 0)
    for i in sites:
        assert res[i]["failed"] is None and res[i]["penalty"] is not None
        assert H.relerr(res[i]["history"], want[i]) <= 1e-6, (i, H.relerr(res[i]["history"], want[i]))


def _rating_raw_data(n, seed):
    rng = np.random.default_rng(seed)
    days = np.sort(rng.uniform(0, 3650, n))
    time = np.datetime64("2005-01-01") + (days * 86400e9).astype("timedelta64[ns]")
    stage = rng.lognormal(1.0, 0.5, n)
    q = 3.0 * (stage - 0.5 * stage.min()) ** 1.6 * np.exp(0.03 * rng.standard_normal(n))
    gse = rng.choice(np.array([1.02, 1.05, 1.08]), n)
    return {"time": time, "stage": stage}, q, gse


@pytest.mark.gpu
def test_fit_sites_penalty_interval_matches_rating_gp_fit(cuda_device):
    cov, q, gse = _rating_raw_data(180, 5)
    torch.manual_seed(7)
    m = models.RatingGP()
    m.fit(cov, q, target_unc=gse, iterations=10, monotonic_penalty_weight=0.5, grid_size=64, monotonic_penalty_interval=3,
          penalty_generator=torch.Generator().manual_seed(9 + 4))
    torch.manual_seed(7)
    res = multisite.fit_sites({4: (m.X, m.y, m.fixed_noise)}, iterations=10, model="rating", monotonic_penalty_weight=0.5,
                              grid_size=64, monotonic_penalty_interval=3, penalty_seed=9)
    assert res[4]["failed"] is None
    assert H.relerr(res[4]["history"], m.history) <= 1e-6, H.relerr(res[4]["history"], m.history)


@pytest.mark.gpu
def test_fit_sites_early_stopping_matches_loadest_gp_fit(cuda_device):
    sites, want = {}, {}
    for i, n in enumerate((150, 230)):
        rng = np.random.default_rng(30 + i)
        days = np.sort(rng.uniform(0, 3650, n))
        time = np.datetime64("2005-01-01") + (days * 86400e9).astype("timedelta64[ns]")
        flow = np.exp(rng.standard_normal(n))
        conc = np.exp(0.5 * np.log(flow) + 0.3 * np.sin(2 * np.pi * days / 365.25) + 0.2 * rng.standard_normal(n))
        m = models.LoadestGP()
        m.fit({"time": time, "flow": flow}, conc, iterations=400, early_stopping=True, patience=4)
        sites[i] = (m.X, m.y)
        want[i] = m.history
    res = multisite.fit_sites(sites, iterations=400, early_stopping=True, patience=4)
    stopped = 0
    for i in sites:
        got = res[i]
        assert got["failed"] is None
        stopped += got["stopped_at"] is not None
        assert len(got["history"]) == len(want[i]) and got["stopped_at"] == (len(want[i]) if len(want[i]) < 400 else None)
        assert H.relerr(got["history"], want[i]) <= 1e-6
    assert stopped > 0
