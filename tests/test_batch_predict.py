"""Batched factorisation and posterior prediction (dgp_batch_factorize / dgp_batch_predict): every site of a batch must get
exactly the numbers a per-site handle gives it (dgp_factorize + dgp_predict) -- nlml, info, mean and latent variance, bit for
bit -- for ragged sizes, grids that end anywhere in a chunk, both models, per-site jitter and failing sites; and the
multi-site driver's predictions must equal a per-site factorise (same jitter ladder) + predict at the returned theta."""
import numpy as np
import pytest
import torch

import helpers as H
from discontinuum_b200 import capi, models, multisite, synthetic
from discontinuum_b200.engine import JITTERS

pytestmark = pytest.mark.gpu

CHUNK = capi.BATCH_PREDICT_CHUNK
GRID_LENGTHS = (2 * CHUNK + 1, 1, 127, 128, 129, 3000)


def _per_site(spec, site, theta, grid, jitter=0.0):
    X, y, noise = site
    eng = capi.Engine(max_n=X.shape[0], max_m=2048)
    eng.set_train(spec.to_c(), X, y, noise)
    val, info = eng.factorize(theta, jitter)
    mu = var = None
    if info == 0 and grid is not None:
        mu, var = eng.predict(grid)
    eng.close()
    return val, info, mu, var


def _check_group(b, spec, sites, thetas, grids, jit=None):
    """batch factorize + predict (full and mean-only) against per-site handles, np.array_equal throughout"""
    val, info = b.factorize(thetas, jit)
    out = b.predict(grids)
    mean_only = b.predict(grids, want_var=False)
    for k, site in enumerate(sites):
        v, i, mu, var = _per_site(spec, site, thetas[k], grids[k], 0.0 if jit is None else float(jit[k]))
        assert info[k] == i, (k, info[k], i)
        if i != 0:
            continue
        assert val[k] == v, (k, val[k], v)
        if grids[k] is None:
            assert out[k] == (None, None) and mean_only[k] == (None, None)
            continue
        assert np.array_equal(out[k][0], mu), (k, np.max(np.abs(out[k][0] - mu)))
        assert np.array_equal(out[k][1], var), (k, np.max(np.abs(out[k][1] - var)))
        assert mean_only[k][1] is None and np.array_equal(mean_only[k][0], out[k][0])
    return val, info, out


def _loadest(ns, seed0):
    sites = [synthetic.loadest_site(n, seed0 + k) for k, n in enumerate(ns)]
    thetas = np.stack([H.loadest_theta1() * (1.0 + 0.01 * k) for k in range(len(ns))])
    return sites, thetas


@pytest.mark.parametrize("ns", [(300,), (300, 450, 700, 129, 1100), (1100, 31, 640, 513, 512, 90, 257)])
def test_batch_predict_bit_identical_loadest(cuda_device, ns):
    spec = models.loadest_spec(2)
    sites, thetas = _loadest(ns, 2000)
    grids = [synthetic.daily_grid(s[0], GRID_LENGTHS[k % len(GRID_LENGTHS)]) for k, s in enumerate(sites)]
    b = capi.BatchEngine(max_sites=len(ns), max_n=max(ns))
    b.set_train(spec.to_c(), sites)
    val, info, _ = _check_group(b, spec, sites, thetas, grids)
    assert np.all(info == 0)
    # again at other hyper-parameters (slabs reused), some sites skipped
    grids2 = [g if k % 2 == 0 else None for k, g in enumerate(grids)]
    _check_group(b, spec, sites, thetas * 1.03, grids2)
    b.close()


def test_batch_predict_config4_sizes_and_launches(cuda_device):
    """BASELINE config 4 sizes with their 10 958-point daily grids; one predict call of the group costs the same launches
    as the same call for one site."""
    spec = models.loadest_spec(2)
    ns = (2565, 4100, 3333, 2048)
    sites, thetas = _loadest(ns, 3000)
    grids = [synthetic.daily_grid(s[0], 10958) for s in sites]
    b = capi.BatchEngine(max_sites=4, max_n=max(ns))
    b.set_train(spec.to_c(), sites)
    _check_group(b, spec, sites, thetas, grids)
    l0 = b.launches
    b.predict(grids)
    per4 = b.launches - l0
    b.close()
    b1 = capi.BatchEngine(max_sites=1, max_n=ns[0])
    b1.set_train(spec.to_c(), sites[:1])
    b1.factorize(thetas[:1])
    l0 = b1.launches
    b1.predict(grids[:1])
    per1 = b1.launches - l0
    b1.close()
    print(f"launches of one predict: G = 4: {per4}, G = 1: {per1}")
    assert abs(per4 - per1) <= 4 and per4 <= 4 * -(-10958 // CHUNK)


def test_batch_predict_rating_gauges(cuda_device):
    """rating-gp: per-point noise, learned noise, power-law mean"""
    ns = (200, 1000, 600)
    sites = [synthetic.rating_gauge(n, 7 + k) for k, n in enumerate(ns)]
    spec = models.rating_spec(1.0, 2.0)
    thetas = np.stack([H.rating_theta1(*models.stage_quantile_bounds(X[:, 1])) for X, _, _ in sites])
    grids = [synthetic.daily_grid(s[0], m) for s, m in zip(sites, (3000, 129, 2 * CHUNK + 1))]
    b = capi.BatchEngine(max_sites=3, max_n=1000)
    b.set_train(spec.to_c(), sites)
    _, info, _ = _check_group(b, spec, sites, thetas, grids)
    assert np.all(info == 0)
    b.close()


def test_batch_predict_per_site_jitter_and_failing_site(cuda_device):
    spec = models.loadest_spec(2)
    ns = (300, 500, 260)
    sites, thetas = _loadest(ns, 4000)
    X, y, noise = sites[1]
    noise = noise.copy()
    noise[200:] = -3.0  # indefinite from row 200 on
    sites[1] = (X, y, noise)
    grids = [synthetic.daily_grid(s[0], m) for s, m in zip(sites, (1500, 700, 129))]
    b = capi.BatchEngine(max_sites=3, max_n=500)
    b.set_train(spec.to_c(), sites)
    val, info = b.factorize(thetas)
    assert info[0] == 0 and info[2] == 0 and 200 < info[1] <= 500
    assert info[1] == _per_site(spec, sites[1], thetas[1], None)[1]
    with pytest.raises(capi.DgpError):
        b.predict(grids)
    _check_group(b, spec, sites, thetas, [grids[0], None, grids[2]])
    jit = np.array([1e-6, 3.5, 0.0])
    _, info2, _ = _check_group(b, spec, sites, thetas, grids, jit)
    assert np.all(info2 == 0)
    b.close()


def test_batch_predict_state(cuda_device):
    """predict needs a factorisation since the last set_train / nlml_grad; factorize + predict leave nlml_grad exact"""
    spec = models.loadest_spec(2)
    ns = (700, 300)
    sites, thetas = _loadest(ns, 4500)
    grids = [synthetic.daily_grid(s[0], 300) for s in sites]
    b = capi.BatchEngine(max_sites=2, max_n=700)
    b.set_train(spec.to_c(), sites)
    with pytest.raises(capi.DgpError, match="factorize"):
        b.predict(grids)
    _check_group(b, spec, sites, thetas, grids)
    val, grad, info = b.nlml_grad(thetas)
    for k, (X, y, noise) in enumerate(sites):
        eng = capi.Engine(max_n=X.shape[0], max_m=128)
        eng.set_train(spec.to_c(), X, y, noise)
        v, g, i = eng.nlml_grad(thetas[k])
        assert info[k] == i == 0 and val[k] == v and np.array_equal(grad[k], g)
        assert np.array_equal(b.alpha(k), eng.alpha())
        eng.close()
    with pytest.raises(capi.DgpError, match="factorize"):
        b.predict(grids)
    b.factorize(thetas)
    b.predict(grids)
    b.set_train(spec.to_c(), sites)
    with pytest.raises(capi.DgpError, match="factorize"):
        b.predict(grids)
    with pytest.raises(ValueError):
        b.predict(grids[:1])
    b.close()


def _reference(spec_c, obs_spec, X, y, noise, theta, grid):
    """the per-site path: psd_safe_cholesky's ladder on a capi.Engine, then predict and the observed-variance rule"""
    eng = capi.Engine(max_n=X.shape[0], max_m=2048)
    eng.set_train(spec_c, X, y, noise)
    for jit in JITTERS:
        _, info = eng.factorize(theta, jit)
        if info == 0:
            break
    else:
        eng.close()
        return None
    mu, var = eng.predict(grid)
    eng.close()
    return mu, var, multisite.observed_variance(obs_spec, theta, var, noise, grid.shape[0])


def _assert_driver_matches(res, sites, grids, spec_of, skip=()):
    for i, (X, y, noise) in sites.items():
        if i in skip:
            continue
        r = res[i]
        assert r["failed"] is None, (i, r["failed"])
        spec = spec_of(X)
        want = _reference(spec.to_c(), spec, X, y, noise, r["theta"], grids[i])
        assert want is not None
        assert np.array_equal(r["mu"], want[0]) and np.array_equal(r["var_latent"], want[1])
        assert np.array_equal(r["var"], want[2])


def test_driver_predicts_through_the_batch_handle_loadest(cuda_device):
    ns = (700, 450, 300, 129, 260)
    sites = {i: synthetic.loadest_site(n, 6000 + i) for i, n in enumerate(ns)}
    X, y, noise = sites[2]
    noise = noise.copy()
    noise[150:] = -3.0   # fails every evaluation: marked failed after 11 iterations, no prediction
    sites[2] = (X, y, noise)
    grids = {i: synthetic.daily_grid(sites[i][0], m) for i, m in zip(sites, (1500, 129, 400, 2 * CHUNK + 1, 64))}
    spec_of = lambda X: models.loadest_spec(2)  # noqa: E731
    out = {}
    for lanes in (1, 2):
        res = multisite.fit_sites_local(sites, iterations=12, group=2, lanes=lanes, predict=grids)
        assert res[2]["failed"] is not None and "mu" not in res[2]
        _assert_driver_matches(res, sites, grids, spec_of, skip=(2,))
        out[lanes] = res
    for i in sites:
        if i != 2:
            assert np.array_equal(out[1][i]["mu"], out[2][i]["mu"]) and np.array_equal(out[1][i]["var"], out[2][i]["var"])
    # no fit: the initial parameters, one handle per group; the indefinite site fails the whole jitter ladder
    res0 = multisite.fit_sites_local(sites, iterations=0, group=2, predict=grids)
    assert res0[2]["failed"].startswith("prediction: not positive definite") and "mu" not in res0[2]
    _assert_driver_matches(res0, sites, grids, spec_of, skip=(2,))
    # sites without a grid get no prediction
    res1 = multisite.fit_sites_local(sites, iterations=0, group=2, predict={0: grids[0]})
    assert "mu" in res1[0] and all("mu" not in res1[i] for i in (1, 3, 4))


def test_driver_predicts_through_the_batch_handle_rating(cuda_device):
    ns = (150, 260, 200)
    sites = {i: synthetic.rating_gauge(n, 30 + i) for i, n in enumerate(ns)}
    grids = {i: synthetic.daily_grid(sites[i][0], m) for i, m in zip(sites, (1100, 120, 300))}

    def spec_of(X):
        return models.rating_spec(*models.stage_quantile_bounds(X[:, 1]))

    for lanes, iters in ((2, 4), (1, 4), (1, 0)):
        torch.manual_seed(0)
        res = multisite.fit_sites_local(sites, iterations=iters, group=2, lanes=lanes, predict=grids, model="rating")
        _assert_driver_matches(res, sites, grids, spec_of)
