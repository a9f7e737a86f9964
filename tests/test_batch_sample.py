"""Batched joint posterior sampling (dgp_batch_sample_ex / BatchEngine.sample): every sampled site of a batch must get
exactly the draws, flux sums and info a per-site handle gives it (dgp_factorize + dgp_sample_ex), bit for bit, for ragged
sizes, grids that end anywhere in a chunk, supplied and device normals, per-site jitter, all reductions and a failing site;
sampling must leave the handle's factorisation intact; and the multi-site driver's annual flux must equal a per-site
factorise (same training ladder) + sample_ex (posterior ladder, seed sample_seed + idx) at the returned theta.
The driver's logic is also checked on the CPU, through a numpy stand-in for the batch handle."""
import numpy as np
import pytest
import torch

import helpers as H
from discontinuum_b200 import capi, models, multisite, synthetic
from discontinuum_b200.data import LogStandardPipeline, StandardPipeline
from discontinuum_b200.engine import JITTERS
from test_multisite import _OracleBatch

gpu = pytest.mark.gpu
GRID_LENGTHS = (1, 127, 128, 129, 1025, 2049, 3000)


def _loadest(ns, seed0):
    sites = [synthetic.loadest_site(n, seed0 + k) for k, n in enumerate(ns)]
    thetas = np.stack([H.loadest_theta1() * (1.0 + 0.01 * k) for k in range(len(ns))])
    return sites, thetas


def _ref(spec, site, theta, grid, S, seed=0, Z=None, jitter=0.0, flux=None, train_jitter=0.0):
    """per-site reference: a handle factorised at theta, then sample_ex"""
    X, y, noise = site
    eng = capi.Engine(max_n=X.shape[0], max_m=2048)
    eng.set_train(spec.to_c(), X, y, noise)
    _, info = eng.factorize(theta, train_jitter)
    assert info == 0
    out, info = eng.sample_ex(grid, S, Z=Z, seed=seed, jitter=jitter, flux=flux)
    eng.close()
    return out, info


def _flux(m, k, kind):
    """weights, groups (some empty, some past the grid's start) and a reduction kind for a grid of m points"""
    rng = np.random.default_rng(100 + k)
    w = np.exp(rng.standard_normal(m)) * 86.4
    cuts = np.sort(rng.integers(0, m + 1, size=4))
    gs = np.concatenate([[0], cuts[:2], cuts[1:2], cuts[2:], [m]]).astype(np.int32)   # one empty group
    return dict(y_mean=0.3 + 0.1 * k, y_scale=0.8, log_transform=kind, weight=w, group_start=gs)


# ---------------------------------------------------------------- GPU: bit identity against per-site handles
@gpu
@pytest.mark.parametrize("ns", [(300, 450, 700, 129, 1100), (1100, 31, 640, 513, 512, 90, 257)])
@pytest.mark.parametrize("S", [1, 7, 130])
def test_batch_sample_ragged_bit_identical(cuda_device, ns, S):
    spec = models.loadest_spec(2)
    sites, thetas = _loadest(ns, 5000)
    G = len(ns)
    grids = [synthetic.daily_grid(s[0], GRID_LENGTHS[(k + S) % len(GRID_LENGTHS)]) for k, s in enumerate(sites)]
    grids[2] = None                                            # one site skipped
    seeds = [1000 * S + 17 * k for k in range(G)]
    jit = np.array([1e-8 * (k % 3) for k in range(G)])         # per-site posterior jitter
    b = capi.BatchEngine(max_sites=G, max_n=max(ns))
    b.set_train(spec.to_c(), sites)
    _, info = b.factorize(thetas)
    assert np.all(info == 0)
    dev = b.sample(grids, S, seeds=seeds, jitter=jit)
    Zs = [None if g is None else H.philox_normals(seeds[k] + 1, S * g.shape[0]).reshape(S, g.shape[0])
          for k, g in enumerate(grids)]
    sup = b.sample(grids, S, Z=Zs, jitter=jit)
    for k in range(G):
        if grids[k] is None:
            assert dev[k] == (None, 0) and sup[k] == (None, 0)
            continue
        want, i = _ref(spec, sites[k], thetas[k], grids[k], S, seed=seeds[k], jitter=jit[k])
        assert dev[k][1] == i == 0 and np.array_equal(dev[k][0], want), (k, np.max(np.abs(dev[k][0] - want)))
        want, i = _ref(spec, sites[k], thetas[k], grids[k], S, Z=Zs[k], jitter=jit[k])
        assert sup[k][1] == i == 0 and np.array_equal(sup[k][0], want), (k, np.max(np.abs(sup[k][0] - want)))
    # the device normals are helpers.philox_normals (numpy's sin / cos may differ from sincospi in the last bits)
    k = 0
    zref = H.philox_normals(seeds[k], S * grids[k].shape[0]).reshape(S, -1)
    viaz = b.sample([grids[0]] + [None] * (G - 1), S, Z=[zref] + [None] * (G - 1), jitter=jit)[0][0]
    assert np.max(np.abs(viaz - dev[0][0])) <= 1e-9 * max(1.0, np.max(np.abs(dev[0][0])))
    b.close()


@gpu
def test_batch_sample_flux_reduction_bit_identical(cuda_device):
    spec = models.loadest_spec(2)
    ns = (600, 300, 1100, 450)
    sites, thetas = _loadest(ns, 5100)
    grids = [synthetic.daily_grid(s[0], m) for s, m in zip(sites, (2049, 365, 1500, 129))]
    flux = [_flux(g.shape[0], k, kind) for k, (g, kind) in enumerate(zip(grids, (1, 2, 0, 1)))]
    flux[3] = None                                             # raw draws next to reduced sites
    seeds = [5, 6, 7, 8]
    b = capi.BatchEngine(max_sites=4, max_n=max(ns))
    b.set_train(spec.to_c(), sites)
    b.factorize(thetas)
    out = b.sample(grids, 64, seeds=seeds, flux=flux)
    for k in range(4):
        want, i = _ref(spec, sites[k], thetas[k], grids[k], 64, seed=seeds[k], flux=flux[k])
        assert out[k][1] == i == 0 and out[k][0].shape == want.shape and np.array_equal(out[k][0], want), k
    b.close()


@gpu
def test_batch_sample_isolated_failure(cuda_device):
    """duplicated grid points: Sigma* is singular at jitter 0 for that site only"""
    spec = models.loadest_spec(2)
    ns = (400, 700, 300)
    sites, thetas = _loadest(ns, 5200)
    grids = [synthetic.daily_grid(s[0], m) for s, m in zip(sites, (900, 500, 1300))]
    grids[1] = np.ascontiguousarray(np.concatenate([grids[1], grids[1][:40]], axis=0))
    b = capi.BatchEngine(max_sites=3, max_n=max(ns))
    b.set_train(spec.to_c(), sites)
    b.factorize(thetas)
    out = b.sample(grids, 9, seeds=[1, 2, 3])
    _, i1 = _ref(spec, sites[1], thetas[1], grids[1], 9, seed=2)
    assert out[1][1] > 0 and out[1][1] == i1
    alone = b.sample([grids[0], None, grids[2]], 9, seeds=[1, 2, 3])
    for k in (0, 2):
        want, i = _ref(spec, sites[k], thetas[k], grids[k], 9, seed=k + 1)
        assert out[k][1] == 0 and np.array_equal(out[k][0], want) and np.array_equal(alone[k][0], want)
    b.close()


@gpu
def test_batch_sample_config4_sizes_and_launches(cuda_device):
    """BASELINE config 4 sizes, 10 958-point daily grids, S = 1000 with the flux reduction; one call for 4 sites costs the same
    launches as the call for one site"""
    spec = models.loadest_spec(2)
    ns = (2565, 4100, 3333, 2048)
    sites, thetas = _loadest(ns, 5300)
    grids = [synthetic.daily_grid(s[0], 10958) for s in sites]
    flux = [_flux(10958, k, 1) for k in range(4)]
    b = capi.BatchEngine(max_sites=4, max_n=max(ns))
    b.set_train(spec.to_c(), sites)
    b.factorize(thetas)
    l0 = b.launches
    out = b.sample(grids, 1000, seeds=[11, 12, 13, 14], flux=flux)
    per4 = b.launches - l0
    for k in range(4):
        want, i = _ref(spec, sites[k], thetas[k], grids[k], 1000, seed=11 + k, flux=flux[k])
        assert out[k][1] == i == 0 and np.array_equal(out[k][0], want), k
    b.close()
    b1 = capi.BatchEngine(max_sites=1, max_n=ns[1])
    b1.set_train(spec.to_c(), sites[1:2])
    b1.factorize(thetas[1:2])
    l0 = b1.launches
    b1.sample(grids[1:2], 1000, seeds=[12], flux=flux[1:2])
    per1 = b1.launches - l0
    b1.close()
    print(f"launches of one sample call: G = 4: {per4}, G = 1: {per1}")
    assert abs(per4 - per1) <= 4


@gpu
def test_batch_sample_state_refusals_and_splitting(cuda_device):
    spec = models.loadest_spec(2)
    ns = (500, 300, 800)
    sites, thetas = _loadest(ns, 5400)
    grids = [synthetic.daily_grid(s[0], m) for s, m in zip(sites, (700, 1100, 260))]
    flux = [_flux(g.shape[0], k, 1) for k, g in enumerate(grids)]
    b = capi.BatchEngine(max_sites=3, max_n=max(ns))
    b.set_train(spec.to_c(), sites)
    with pytest.raises(capi.DgpError, match="not factorised"):
        b.sample(grids, 4)
    b.factorize(thetas)
    before = b.predict(grids)
    one = b.sample(grids, 33, seeds=[4, 5, 6], flux=flux)
    after = b.predict(grids)
    for k in range(3):
        assert np.array_equal(before[k][0], after[k][0]) and np.array_equal(before[k][1], after[k][1])
    # one site per call gives the same bits
    split = b.sample(grids, 33, seeds=[4, 5, 6], flux=flux, max_bytes=1)
    for k in range(3):
        assert np.array_equal(one[k][0], split[k][0]) and one[k][1] == split[k][1] == 0
    # the arena grew to what dgp_batch_sample_bytes reports for the largest call so far
    need = b.sample_bytes([g.shape[0] for g in grids], 33, flux)
    assert need > 0 and b.lib.dgp_batch_sample_bytes(b._h, None, 33, None) == 0
    got = b.sample_bytes([g.shape[0] for g in grids], 33, flux)
    assert got == need
    with pytest.raises(capi.DgpError, match="S = 0"):
        b.sample(grids, 0)
    bad = dict(flux[0], group_start=np.array([0, 5, 3, 700], dtype=np.int32))
    with pytest.raises(capi.DgpError, match="non-decreasing"):
        b.sample(grids, 4, flux=[bad, None, None])
    b.nlml_grad_launch(thetas)
    with pytest.raises(capi.DgpError, match="in flight"):
        b.sample(grids, 4)
    b.nlml_grad_wait()
    with pytest.raises(capi.DgpError, match="not factorised"):
        b.sample(grids, 4)
    b.close()


@gpu
def test_batch_sample_arena_bytes(cuda_device):
    """dgp_batch_sample_bytes equals the arena a fresh handle grows to (the formula of dgp.h)"""
    spec = models.loadest_spec(2)
    ns = (900, 400)
    sites, thetas = _loadest(ns, 5500)
    grids = [synthetic.daily_grid(s[0], m) for s, m in zip(sites, (1300, 600))]
    b = capi.BatchEngine(max_sites=2, max_n=900)
    b.set_train(spec.to_c(), sites)
    b.factorize(thetas)
    need = b.sample_bytes([1300, 600], 50)
    free0 = torch.cuda.mem_get_info()[0]
    b.sample(grids, 50)
    free1 = torch.cuda.mem_get_info()[0]
    mld, ld, Spad = 1408, 1024, 128
    doubles = 2 * (mld * mld + mld * ld + 2 * Spad * mld + 256 * mld + 9 * mld) + 2 * 105
    assert abs(need - 8 * doubles) <= 8 * 32 * 11      # every slab rounded up to 256 B
    # the prediction slabs come first on a handle that never predicted; the arena is the rest
    pred = 8 * 2 * 1024 * (1024 + 3 * 8 + 19)
    assert free0 - free1 >= need and free0 - free1 <= need + pred + (64 << 20)
    b.close()


# ---------------------------------------------------------------- GPU: the driver against per-site handles
def _flux_spec(grid, k, kind=1):
    f = _flux(grid.shape[0], k, kind)
    return models.FluxSpec(grid, f["weight"], f["group_start"], np.arange(f["group_start"].shape[0] - 1), f["y_mean"],
                           f["y_scale"], kind)


@gpu
def test_driver_annual_flux_matches_per_site(cuda_device):
    spec = models.loadest_spec(2)
    ns = (700, 300, 520, 129, 900)
    sites = {i: synthetic.loadest_site(n, 5600 + i)[:2] for i, n in enumerate(ns)}
    predict = {i: synthetic.daily_grid(sites[i][0], 400 + 100 * i) for i in (0, 2, 3)}
    annual = {i: _flux_spec(synthetic.daily_grid(sites[i][0], 1000 + 37 * i), i) for i in (0, 1, 3, 4)}
    base = multisite.fit_sites_local(sites, iterations=3, group=16, predict=predict)
    runs = {}
    for lanes, group in ((1, 16), (2, 16), (1, 3), (2, 3)):
        runs[(lanes, group)] = multisite.fit_sites_local(sites, iterations=3, group=group, lanes=lanes, predict=predict,
                                                         annual_flux=annual, draws=64, sample_seed=40)
    res = runs[(1, 16)]
    for i, (X, y) in sites.items():
        r = res[i]
        assert r["failed"] is None and "flux_failed" not in r
        if i in predict:
            assert np.array_equal(r["mu"], base[i]["mu"]) and np.array_equal(r["var"], base[i]["var"])
        if i not in annual:
            assert "annual_flux" not in r
            continue
        eng = capi.Engine(max_n=X.shape[0])
        eng.set_train(spec.to_c(), X, y, np.full(X.shape[0], models.LOADEST_FIXED_NOISE))
        for j in JITTERS:
            if eng.factorize(r["theta"], j)[1] == 0:
                break
        for j in JITTERS:
            want, info = eng.sample_ex(annual[i].grid, 64, seed=40 + i, jitter=j, flux=annual[i].reduce())
            if info == 0 and np.all(np.isfinite(want)):
                break
        eng.close()
        assert np.array_equal(r["annual_flux"], want) and np.array_equal(r["flux_years"], annual[i].years), i
        for key, other in runs.items():
            assert np.array_equal(other[i]["annual_flux"], r["annual_flux"]), (key, i)


# ---------------------------------------------------------------- CPU: the driver's logic on a numpy stand-in
def _standin_draws(grid, S, seed, jitter, red):
    """what the stand-in computes: a squared-exponential posterior covariance over the grid's first column"""
    t = grid[:, 0]
    K = np.exp(-0.5 * (t[:, None] - t[None, :]) ** 2 / 0.3 ** 2) + (1e-6 + jitter) * np.eye(t.shape[0])
    L = np.linalg.cholesky(K)
    Z = H.philox_normals(seed, S * t.shape[0]).reshape(S, t.shape[0])
    D = Z @ L.T
    if red is None:
        return D
    v = D * red["y_scale"] + red["y_mean"]
    v = np.maximum(np.exp(v), 1e-6) if red["log_transform"] == 1 else (np.maximum(v, 0.0) if red["log_transform"] == 2 else v)
    gs = red["group_start"]
    return np.stack([(v[:, gs[g]:gs[g + 1]] * red["weight"][gs[g]:gs[g + 1]]).sum(axis=1) for g in range(gs.shape[0] - 1)], axis=1)


class _SamplingBatch(_OracleBatch):
    """_OracleBatch plus factorize / predict / sample.  A site's posterior is not positive definite below the jitter
    FAIL_BELOW[n] (n = its training size); calls are recorded."""
    FAIL_BELOW = {}
    calls = []

    def factorize(self, theta, jitter=None):
        G = len(self.sites)
        return np.zeros(G), np.zeros(G, dtype=np.int32)

    def predict(self, grids, want_var=True):
        return [(None, None) if g is None else (np.zeros(g.shape[0]), np.ones(g.shape[0])) for g in grids]

    def sample(self, grids, S, seeds=None, Z=None, jitter=None, flux=None, max_bytes=None):
        out = []
        for k, g in enumerate(grids):
            if g is None:
                out.append((None, 0))
                continue
            n = self.sites[k][0].shape[0]
            type(self).calls.append((n, float(jitter[k]), int(seeds[k])))
            if jitter[k] < self.FAIL_BELOW.get(n, -1.0):
                out.append((np.full((S, flux[k]["group_start"].shape[0] - 1), np.nan), 1))
                continue
            out.append((_standin_draws(g, S, seeds[k], jitter[k], flux[k]), 0))
        return out


def test_driver_annual_flux_logic_on_standin(monkeypatch):
    monkeypatch.setattr(capi, "BatchEngine", _SamplingBatch)
    ns = [24 + 5 * i for i in range(6)]
    sites = {i: synthetic.loadest_site(n, 700 + i)[:2] for i, n in enumerate(ns)}
    annual = {i: _flux_spec(synthetic.daily_grid(sites[i][0], 30 + 3 * i), i, kind=(1, 2, 0)[i % 3]) for i in (0, 1, 2, 4, 5)}
    predict = {i: synthetic.daily_grid(sites[i][0], 20) for i in (0, 3)}
    _SamplingBatch.FAIL_BELOW = {ns[1]: JITTERS[2], ns[4]: 1.0}   # site 1: fails at the first two jitters; site 4: always
    runs = {}
    for lanes, group in ((1, 16), (2, 16), (1, 2), (3, 2)):
        _SamplingBatch.calls = []
        runs[(lanes, group)] = multisite.fit_sites_local(sites, iterations=2, group=group, lanes=lanes, predict=predict,
                                                         annual_flux=annual, draws=8, sample_seed=90)
        calls = list(_SamplingBatch.calls)
        # only the failing sites come back, each at the next jitter; every site draws from its own stream
        for i in annual:
            mine = [c for c in calls if c[0] == ns[i]]
            want_j = JITTERS[:3] if i == 1 else (JITTERS if i == 4 else JITTERS[:1])
            assert [c[1] for c in mine] == list(want_j) and all(c[2] == 90 + i for c in mine), (i, mine)
        assert not [c for c in calls if c[0] == ns[3]]
    res = runs[(1, 16)]
    for i in sites:
        r = res[i]
        if i == 4:
            assert "annual_flux" not in r and "not positive definite" in r["flux_failed"] and r["failed"] is None
            continue
        if i not in annual:
            assert "annual_flux" not in r and "flux_failed" not in r
            continue
        jit = JITTERS[2] if i == 1 else JITTERS[0]
        want = _standin_draws(annual[i].grid, 8, 90 + i, jit, annual[i].reduce())
        assert "flux_failed" not in r and np.array_equal(r["annual_flux"], want), i
        assert np.array_equal(r["flux_years"], annual[i].years)
        for key, other in runs.items():
            assert np.array_equal(other[i]["annual_flux"], r["annual_flux"]), (key, i)
    assert "mu" in res[0] and "mu" in res[3]
    with pytest.raises(ValueError, match="annual_flux"):
        multisite.fit_sites_local(sites, iterations=2, concurrency=2, annual_flux=annual)


def test_site_cost_sampling_term():
    assert multisite.site_cost(4000, 100, 2000) == 100 * 4000.0 ** 3 + 4000.0 ** 3 + 2000 * 4000.0 ** 2
    m, n, S = 10958.0, 8000.0, 1000
    extra = multisite.site_cost(8000, 100, 0, 10958, S) - multisite.site_cost(8000, 100)
    assert extra == pytest.approx(m * m * n + m ** 3 / 3 + 2 * m * m * S, rel=1e-12)


@pytest.mark.parametrize("pipe", [LogStandardPipeline, StandardPipeline])
def test_flux_spec_daily_axis_matches_sample_annual_flux_rule(pipe):
    """FluxSpec.from_series on a daily axis gives the weights, groups, labels and reduction kind that
    LoadestGPMarginalB200.sample_annual_flux computed inline before the grouping moved into annual_flux_groups"""
    time = np.datetime64("2001-03-05") + np.arange(1500).astype("timedelta64[D]")
    flow = np.exp(np.sin(np.arange(1500) / 50.0))
    p = pipe().fit(np.exp(np.random.default_rng(0).standard_normal(50)))
    fs = models.FluxSpec.from_series(np.zeros((1500, 2)), time, flow, p)
    # the former inline code of sample_annual_flux
    t = np.asarray(time).astype("datetime64[ns]")
    dt_s = float(np.unique(np.diff(t).astype("timedelta64[ns]").astype(np.int64))[0]) * 1e-9
    weight = np.asarray(flow, dtype=np.float64) * dt_s * 1e-3
    years = t.astype("datetime64[Y]").astype(np.int64) + 1970
    uniq, first = np.unique(years, return_index=True)
    group_start = np.concatenate([first, [t.shape[0]]]).astype(np.int32)
    assert np.array_equal(fs.weight, weight) and np.array_equal(fs.weight, flow * 86400.0 * 1e-3)
    assert np.array_equal(fs.group_start, group_start) and fs.group_start.dtype == np.int32
    assert fs.years.tolist() == uniq.tolist() == [2001, 2002, 2003, 2004, 2005]
    assert fs.group_start.tolist() == [0, 302, 667, 1032, 1398, 1500]
    assert fs.log_transform == (1 if pipe is LogStandardPipeline else 2)
    assert fs.y_mean == float(p.mean_) and fs.y_scale == float(p.scale_)
    with pytest.raises(ValueError, match="strictly increasing"):
        models.FluxSpec.from_series(np.zeros((3, 2)), time[[0, 2, 1]], flow[:3], p)
