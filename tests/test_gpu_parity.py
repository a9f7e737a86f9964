"""GPU parity tests proper: everything goes through the C ABI (libdgp.so via ctypes) and is compared with the
mpmath golden vectors, with the CPU oracle on the same seeded inputs, and -- at BASELINE.json's full sizes --
through size-independent properties.  Tolerance of the north star: <= 1e-6 relative in float64 (observed ~1e-11)."""
import io
import json
import os

import numpy as np
import pytest
import torch

import helpers as H
from helpers import orc
from discontinuum_b200 import capi, models, synthetic

pytestmark = pytest.mark.gpu
RTOL = 1e-6  # north-star tolerance for NLML, gradients, predictive mean and variance
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _engine(spec, X, y, noise, max_m=256):
    eng = capi.Engine(max_n=X.shape[0], max_m=max_m)
    eng.set_train(spec.to_c(), X, y, noise)
    return eng


def _oracle(model, theta, X, y, noise):
    Xt, yt, nt = torch.tensor(X), torch.tensor(y), torch.tensor(noise)
    if model == "loadest":
        nat = H.loadest_nat_from_theta(theta, X.shape[1])
        v, g, a, L = orc.nlml_grad_closed_form(orc.loadest_cov, orc.loadest_mean, nat, Xt, yt, nt)
        return float(v), H.loadest_theta_from_nat({k: t.numpy() for k, t in g.items()}), a.numpy(), L.numpy(), nat
    nat = H.rating_nat_from_theta(theta)
    v, g, a, L = orc.nlml_grad_closed_form(orc.rating_cov, orc.rating_mean, nat, Xt, yt, nt, extra_key="noise")
    return float(v), H.rating_theta_from_nat({k: t.numpy() for k, t in g.items()}), a.numpy(), L.numpy(), nat


def _grad_close(got, want, rtol=RTOL):
    assert np.max(np.abs(got - want)) <= rtol * np.max(np.abs(want)), (got, want)


@pytest.mark.parametrize("fname", ["kat_loadest.json", "kat_rating.json"])
def test_golden_vectors_through_cabi(cuda_device, fname):
    with open(os.path.join(GOLD, fname)) as f:
        cases = json.load(f)
    for case in cases:
        X, y, noise, theta = (np.array(case[k]) for k in ("X", "y", "noise", "theta"))
        if case["model"] == "loadest":
            spec = models.loadest_spec(2)
        else:
            spec = models.rating_spec(1.0, 2.0)  # bounds only constrain the raw value; theta is passed in natural space
        eng = _engine(spec, X, y, noise)
        assert np.max(np.abs(eng.covmat(theta) - np.array(case["K"]))) < 1e-14
        val, info = eng.nlml(theta)
        assert info == 0 and abs(val - case["nlml"]) <= 1e-12 * max(1.0, abs(case["nlml"]))
        val2, grad, info = eng.nlml_grad(theta)
        assert info == 0 and abs(val2 - val) <= 1e-13 * max(1.0, abs(val))  # nlml-only path: z by forward substitution; grad path: z = U'r
        gold = np.array(case["grad"])
        assert np.max(np.abs(grad - gold)) <= 1e-8 * max(1.0, np.max(np.abs(gold))), (case["n"], grad, gold)
        assert np.max(np.abs(eng.alpha() - np.array(case["alpha"]))) <= 1e-9 * np.max(np.abs(case["alpha"]))
        assert np.max(np.abs(np.tril(eng.chol()) - np.array(case["L"]))) < 1e-12
        eng.factorize(theta)
        mu, var = eng.predict(np.array(case["Xs"]))
        assert np.max(np.abs(mu - np.array(case["mu"]))) <= 1e-9 * max(1.0, np.max(np.abs(case["mu"])))
        assert np.max(np.abs(var - np.array(case["var_latent"]))) <= 1e-9
        eng.close()


@pytest.mark.parametrize("model,n,kind", [("loadest", 127, 0), ("loadest", 128, 1), ("loadest", 129, 0), ("loadest", 300, 1),
                                           ("loadest", 600, 0), ("loadest", 1000, 1), ("loadest", 1100, 1), ("loadest", 2000, 0),
                                           ("rating", 200, 0), ("rating", 1000, 1), ("rating", 2000, 1)])
def test_nlml_grad_alpha_chol_vs_oracle(cuda_device, model, n, kind):
    if model == "loadest":
        X, y, noise = synthetic.loadest_site(n, 1000 + n)
        spec = models.loadest_spec(2)
        theta = H.loadest_theta0() if kind == 0 else H.loadest_theta1()
    else:
        X, y, noise = synthetic.rating_gauge(n, 7)
        b_lo, b_hi = models.stage_quantile_bounds(X[:, 1])
        spec = models.rating_spec(b_lo, b_hi)
        theta = H.rating_theta0(b_lo, b_hi) if kind == 0 else H.rating_theta1(b_lo, b_hi)
    v, g, a, L, _ = _oracle(model, theta, X, y, noise)
    eng = _engine(spec, X, y, noise)
    val, grad, info = eng.nlml_grad(theta)
    assert info == 0
    assert abs(val - v) <= RTOL * abs(v)
    _grad_close(grad, g)
    assert np.max(np.abs(eng.alpha() - a)) <= RTOL * np.max(np.abs(a))
    Lg = eng.chol()
    assert np.max(np.abs(np.tril(Lg) - L)) <= RTOL * np.max(np.abs(L)) and np.max(np.abs(np.triu(Lg, 1))) == 0.0
    val0, info0 = eng.nlml(theta)
    assert info0 == 0 and abs(val0 - val) <= 1e-13 * max(1.0, abs(val))
    eng.close()


def test_loadest_three_covariate_dims(cuda_device):
    rng = np.random.default_rng(3)
    n = 400
    X = np.ascontiguousarray(np.stack([np.sort(rng.uniform(-5, 5, n)), rng.standard_normal(n), rng.standard_normal(n)], 1))
    y, noise = rng.standard_normal(n), np.full(n, 0.01)
    theta = np.array([0.1, 0.7, 1.0, 1.0, 2.0, 1.3, 0.5, 0.8, 0.2, 0.3, 0.4, 0.6])
    v, g, a, L, _ = _oracle("loadest", theta, X, y, noise)
    eng = _engine(models.loadest_spec(3), X, y, noise)
    val, grad, info = eng.nlml_grad(theta)
    assert info == 0 and abs(val - v) <= RTOL * abs(v)
    _grad_close(grad, g)
    eng.close()


def test_kinv_and_cross_covariance(cuda_device):
    n = 500
    X, y, noise = synthetic.loadest_site(n, 11)
    theta = H.loadest_theta1()
    _, _, _, L, nat = _oracle("loadest", theta, X, y, noise)
    eng = _engine(models.loadest_spec(2), X, y, noise)
    eng.set_debug_kinv(True)
    eng.nlml_grad(theta)
    Ki = torch.cholesky_inverse(torch.tensor(L)).numpy()
    assert np.max(np.abs(np.tril(eng.kinv()) - np.tril(Ki))) <= RTOL * np.max(np.abs(Ki))
    Xs = synthetic.daily_grid(X, 333)
    Kx = eng.cross_covmat(theta, Xs)
    assert np.max(np.abs(Kx - orc.loadest_cov(torch.tensor(Xs), torch.tensor(X), nat).numpy())) < 1e-14
    eng.close()


def test_predict_mean_variance_vs_oracle_multi_chunk(cuda_device):
    for model in ("loadest", "rating"):
        if model == "loadest":
            X, y, noise = synthetic.loadest_site(700, 21)
            spec, theta = models.loadest_spec(2), H.loadest_theta1()
            nat, cov, mean, en = H.loadest_nat_from_theta(theta), orc.loadest_cov, orc.loadest_mean, None
        else:
            X, y, noise = synthetic.rating_gauge(600, 9)
            b_lo, b_hi = models.stage_quantile_bounds(X[:, 1])
            spec, theta = models.rating_spec(b_lo, b_hi), H.rating_theta1(b_lo, b_hi)
            nat = H.rating_nat_from_theta(theta)
            cov, mean, en = orc.rating_cov, orc.rating_mean, nat["noise"]
        Xs = synthetic.daily_grid(X, 1000)  # 4 chunks of 256
        eng = _engine(spec, X, y, noise, max_m=256)
        _, info = eng.factorize(theta)
        assert info == 0
        mu, var = eng.predict(Xs)
        mu_o, _, var_o = orc.predict(cov, mean, nat, torch.tensor(X), torch.tensor(y), torch.tensor(noise), torch.tensor(Xs), extra_noise=en)
        assert np.max(np.abs(mu - mu_o.numpy())) <= RTOL * np.max(np.abs(mu_o.numpy()))
        assert np.max(np.abs(var - var_o.numpy())) <= RTOL * np.max(np.abs(var_o.numpy()))
        mu2, none = eng.predict(Xs, want_var=False)
        assert none is None and np.array_equal(mu2, mu)
        eng.close()


def test_sample_matches_oracle_given_same_normals(cuda_device):
    n, m, S = 300, 200, 64
    X, y, noise = synthetic.loadest_site(n, 31)
    theta = H.loadest_theta1()
    nat = H.loadest_nat_from_theta(theta)
    Xs = synthetic.daily_grid(X, m) + np.array([0.003, 0.01])
    Z = np.random.default_rng(0).standard_normal((S, m))
    eng = _engine(models.loadest_spec(2), X, y, noise)
    eng.factorize(theta)
    draws, info = eng.sample(Xs, Z, jitter=1e-8)
    assert info == 0
    want, _ = orc.sample(orc.loadest_cov, orc.loadest_mean, nat, torch.tensor(X), torch.tensor(y), torch.tensor(noise),
                         torch.tensor(Xs), torch.tensor(Z), jitter=1e-8)
    assert np.max(np.abs(draws - want.numpy())) <= 1e-5 * np.max(np.abs(want.numpy()))
    # moments: mean over draws -> posterior mean within Monte-Carlo error
    mu, var = eng.predict(Xs)
    assert np.max(np.abs(draws.mean(0) - mu)) < 6 * np.sqrt(np.max(var) / S) + 1e-6
    eng.close()


def test_sample_multi_chunk_in_place_factorisation(cuda_device):
    """m spans several prediction chunks and several panels of the in-place posterior Cholesky (ragged m, n)."""
    n, m, S = 450, 1100, 8
    X, y, noise = synthetic.loadest_site(n, 32)
    theta = H.loadest_theta1()
    nat = H.loadest_nat_from_theta(theta)
    Xs = synthetic.daily_grid(X, m) + np.array([0.0007, 0.01])
    Z = np.random.default_rng(1).standard_normal((S, m))
    eng = _engine(models.loadest_spec(2), X, y, noise, max_m=256)
    eng.factorize(theta)
    draws, info = eng.sample(Xs, Z, jitter=1e-6)
    assert info == 0
    want, _ = orc.sample(orc.loadest_cov, orc.loadest_mean, nat, torch.tensor(X), torch.tensor(y), torch.tensor(noise),
                         torch.tensor(Xs), torch.tensor(Z), jitter=1e-6)
    assert np.max(np.abs(draws - want.numpy())) <= 1e-5 * np.max(np.abs(want.numpy()))
    eng.close()


def test_sample_device_normals_and_fused_flux_reduction(cuda_device):
    """dgp_sample_ex: (i) Z = NULL draws equal the draws from the numpy restatement of the Philox stream;
    (ii) the grouped flux reduction equals concentration_to_flux + annual sums computed on the host from the draws."""
    n, m, S = 300, 730, 24
    X, y, noise = synthetic.loadest_site(n, 33)
    theta = H.loadest_theta1()
    Xs = synthetic.daily_grid(X, m) + np.array([0.0011, 0.0])
    eng = _engine(models.loadest_spec(2), X, y, noise)
    eng.factorize(theta)
    Z = H.philox_normals(1234567891011, S * m).reshape(S, m)
    assert abs(Z.mean()) < 0.03 and abs(Z.std() - 1.0) < 0.03
    want, info = eng.sample(Xs, Z, jitter=1e-8)
    got, info2 = eng.sample_ex(Xs, S, Z=None, seed=1234567891011, jitter=1e-8)
    assert info == 0 and info2 == 0
    assert np.max(np.abs(got - want)) <= 1e-9 * np.max(np.abs(want))
    # flux: weight = flow * dt * 1e-3, groups = "years" of 365 grid points, log-standard target pipeline
    rng = np.random.default_rng(2)
    w = np.exp(rng.standard_normal(m)) * 86400.0 * 1e-3
    gs = np.array([0, 365, 730], dtype=np.int32)
    y_mean, y_scale = 0.7, 1.3
    flux, info3 = eng.sample_ex(Xs, S, Z=Z, jitter=1e-8, flux=dict(y_mean=y_mean, y_scale=y_scale, log_transform=1,
                                                                 weight=w, group_start=gs))
    conc = np.clip(np.exp(want * y_scale + y_mean), 1e-6, None)
    ref = np.stack([(conc[:, a:b] * w[a:b]).sum(axis=1) for a, b in zip(gs[:-1], gs[1:])], axis=1)
    assert info3 == 0 and flux.shape == (S, 2)
    assert np.max(np.abs(flux - ref) / np.abs(ref)) <= 1e-10
    aff, _ = eng.sample_ex(Xs, S, Z=Z, jitter=1e-8, flux=dict(y_mean=y_mean, y_scale=y_scale, log_transform=0,
                                                            weight=w, group_start=gs))
    ref2 = np.stack([((want[:, a:b] * y_scale + y_mean) * w[a:b]).sum(axis=1) for a, b in zip(gs[:-1], gs[1:])], axis=1)
    assert np.max(np.abs(aff - ref2)) <= 1e-10 * np.max(np.abs(ref2))
    with pytest.raises(capi.DgpError):
        eng.sample_ex(Xs, S, Z=Z, flux=dict(y_mean=0.0, y_scale=1.0, weight=w, group_start=np.array([0, 800], dtype=np.int32)))
    eng.close()


@pytest.mark.parametrize("model", ["loadest", "rating"])
def test_mean_functional_gradient_vs_autograd(cuda_device, model):
    """dgp_mean_functional_grad: F = c'mu(X*) and dF/dtheta against torch autograd through the solve (oracle)."""
    n, m = 300, 100
    rng = np.random.default_rng(5)
    if model == "loadest":
        X, y, noise = synthetic.loadest_site(n, 41)
        spec, theta = models.loadest_spec(2), H.loadest_theta1()
        nat0 = H.loadest_nat_from_theta(theta)
        cov, mean, extra, to_theta = orc.loadest_cov, orc.loadest_mean, None, H.loadest_theta_from_nat
    else:
        X, y, noise = synthetic.rating_gauge(n, 7)
        b_lo, b_hi = models.stage_quantile_bounds(X[:, 1])
        spec, theta = models.rating_spec(b_lo, b_hi), H.rating_theta1(b_lo, b_hi)
        nat0 = H.rating_nat_from_theta(theta)
        cov, mean, extra, to_theta = orc.rating_cov, orc.rating_mean, "noise", H.rating_theta_from_nat
    Xs = synthetic.daily_grid(X, m) + np.array([0.004, 0.0])
    c = rng.standard_normal(m)
    eng = _engine(spec, X, y, noise)
    _, _, info = eng.nlml_grad(theta)
    assert info == 0
    val, grad = eng.mean_functional_grad(Xs, c)
    leaves = {k: v.detach().clone().requires_grad_(True) for k, v in nat0.items()}
    mu = orc.predict(cov, mean, leaves, torch.tensor(X), torch.tensor(y), torch.tensor(noise), torch.tensor(Xs),
                     leaves[extra] if extra else None)[0]
    F = (torch.tensor(c) * mu).sum()
    gs = torch.autograd.grad(F, list(leaves.values()), allow_unused=True)
    want = to_theta({k: (g if g is not None else torch.zeros_like(leaves[k])).numpy() for k, g in zip(leaves, gs)})
    assert abs(val - float(F.detach())) <= RTOL * abs(float(F.detach()))
    _grad_close(grad, want)
    # the same call after dgp_factorize (prediction state) gives the same numbers
    eng.factorize(theta)
    val2, grad2 = eng.mean_functional_grad(Xs, c)
    assert abs(val2 - val) <= 1e-12 * abs(val) and np.max(np.abs(grad2 - grad)) <= 1e-10 * np.max(np.abs(grad))
    eng.close()


def test_non_positive_definite_reports_info_and_jitter_repairs(cuda_device):
    """LAPACK-style info: 1-based index of the first non-positive pivot; jitter on the diagonal repairs it."""
    n = 300
    X, y, _ = synthetic.loadest_site(n, 41)
    noise = np.zeros(n)
    noise[200:] = -3.0  # k(x, x) = 2.2 < 3: rows >= 200 make the matrix indefinite
    eng = _engine(models.loadest_spec(2), X, y, noise)
    val, info = eng.nlml(H.loadest_theta1())
    assert 200 < info <= 300
    with pytest.raises(capi.DgpError, match="no factorisation"):
        eng.alpha()
    val2, info2 = eng.nlml(H.loadest_theta1(), jitter=3.5)
    assert info2 == 0 and np.isfinite(val2)
    eng.close()


def test_bad_arguments_raise(cuda_device):
    eng = capi.Engine(max_n=64)
    X, y, noise = synthetic.loadest_site(100, 1)
    with pytest.raises(capi.DgpError, match="max_n"):
        eng.set_train(models.loadest_spec(2).to_c(), X, y, noise)
    with pytest.raises(capi.DgpError, match="set_train"):
        eng.lib.dgp_nlml.restype = int
        eng._check(eng.lib.dgp_nlml(eng._h, H.loadest_theta1().ctypes.data, 0.0, None), "dgp_nlml")
    bad = models.loadest_spec(2).to_c()
    bad.nterms = 99
    with pytest.raises(capi.DgpError, match="nterms"):
        eng.set_train(bad, X[:50], y[:50], noise[:50])
    eng.close()


def test_tile_engine_many_tiles_regression(cuda_device):
    """Regression for the shared-memory WAR race (ring stage released before its fragment loads returned):
    it only showed with > 2 waves of co-resident CTAs and a wrapped ring (K >= 128)."""
    eng = capi.Engine(max_n=128)
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    for (M, N, K) in [(4096, 4096, 128), (4096, 4096, 512), (1024, 8192, 256)]:
        A = torch.randn(M, K, dtype=torch.float64, device=dev)
        B = torch.randn(N, K, dtype=torch.float64, device=dev)
        ref = A @ B.T
        for mode in (0, -1, 1):
            C0 = torch.randn(M, N, dtype=torch.float64, device=dev)
            Cm = C0.clone()
            torch.cuda.synchronize()
            eng.gemm_nt(A, B, Cm, mode)
            want = ref if mode == 0 else C0 + mode * ref
            assert float((Cm - want).abs().max()) < 1e-10
    eng.close()


def test_large_n_deterministic_and_consistent(cuda_device):
    n = 3584
    X, y, noise = synthetic.loadest_site(n, 51)
    eng = _engine(models.loadest_spec(2), X, y, noise)
    th = H.loadest_theta1()
    runs = [eng.nlml_grad(th) for _ in range(3)]
    assert all(r[2] == 0 for r in runs)
    assert runs[0][0] == runs[1][0] == runs[2][0]
    assert np.array_equal(runs[0][1], runs[1][1]) and np.array_equal(runs[0][1], runs[2][1])
    v, g, _, _, _ = _oracle("loadest", th, X, y, noise)
    assert abs(runs[0][0] - v) <= RTOL * abs(v)
    _grad_close(runs[0][1], g)
    eng.close()


def test_full_size_properties_n16384(cuda_device):
    """BASELINE config 3 size (the oracle cannot run here in seconds): size-independent checks.
    (i) directional derivative of NLML by central differences agrees with the analytic gradient;
    (ii) posterior mean at the training inputs equals y - noise * alpha (since K alpha = r - noise alpha);
    (iii) latent variance at training inputs lies in [0, noise]."""
    n = 16384
    X, y, noise = synthetic.loadest_site(n, 1000)
    eng = _engine(models.loadest_spec(2), X, y, noise, max_m=512)
    th = H.loadest_theta1()
    val, grad, info = eng.nlml_grad(th)
    assert info == 0 and np.isfinite(val)
    d = np.random.default_rng(0).standard_normal(th.shape[0]) * th * 1e-2
    d[0] = 1e-2
    eps = 1e-3
    vp, ip = eng.nlml(th + eps * d)
    vm, im = eng.nlml(th - eps * d)
    assert ip == 0 and im == 0
    fd = (vp - vm) / (2 * eps)
    assert abs(fd - grad @ d) <= 1e-5 * abs(grad @ d) + 1e-8 * abs(val), (fd, grad @ d)
    _, info = eng.factorize(th)
    assert info == 0
    alpha = eng.alpha()
    idx = np.arange(0, n, 37)[:400]
    mu, var = eng.predict(X[idx])
    assert np.max(np.abs(mu - (y[idx] - noise[idx] * alpha[idx]))) <= 1e-7 * max(1.0, np.max(np.abs(y)))
    assert np.all(var > -1e-9) and np.all(var <= noise[idx] + 1e-9)
    eng.close()


def test_async_launch_wait_two_sites(cuda_device):
    sites = [synthetic.loadest_site(n, 60 + n) for n in (900, 1400)]
    engs = [_engine(models.loadest_spec(2), *s) for s in sites]
    th = H.loadest_theta1()
    for e in engs:
        e.nlml_grad_launch(th)
    res = [e.nlml_grad_wait() for e in engs]
    for e, r in zip(engs, res):
        v, g, info = e.nlml_grad(th)
        assert info == 0 and r[0] == v and np.array_equal(r[1], g)
        e.close()


def test_ready_poll_then_wait(cuda_device):
    import time
    X, y, noise = synthetic.loadest_site(1100, 77)
    eng = _engine(models.loadest_spec(2), X, y, noise)
    th = H.loadest_theta1()
    want = eng.nlml_grad(th)
    eng.nlml_grad_launch(th)
    t0 = time.time()
    while not eng.nlml_grad_ready():
        assert time.time() - t0 < 30.0
    got = eng.nlml_grad_wait()
    assert got[2] == 0 and got[0] == want[0] and np.array_equal(got[1], want[1])
    with pytest.raises(capi.DgpError):
        eng.nlml_grad_ready()  # nothing in flight any more
    eng.close()


def test_diagonal_block_kernel_edge_sizes(cuda_device):
    """n around multiples of 32 and 128: ragged last diagonal block (identity padding) through the 32x32 sub-block kernel."""
    th = H.loadest_theta1()
    for n in (31, 33, 95, 161, 257, 383):
        X, y, noise = synthetic.loadest_site(n, 300 + n)
        eng = _engine(models.loadest_spec(2), X, y, noise)
        val, grad, info = eng.nlml_grad(th)
        v, g, a, L, _ = _oracle("loadest", th, X, y, noise)
        assert info == 0
        assert abs(val - v) <= RTOL * abs(v)
        _grad_close(grad, g)
        Lg = eng.chol()
        assert np.max(np.abs(np.tril(Lg) - L)) <= 1e-9 * np.max(np.abs(L))
        eng.close()


def _loadest_arrays(n, seed):
    rng = np.random.default_rng(seed)
    days = np.sort(rng.uniform(0, 3650, n))
    time = np.datetime64("2000-01-01") + (days * 86400e9).astype("timedelta64[ns]")
    flow = np.exp(1.0 + 0.8 * np.sin(2 * np.pi * days / 365.25) + 0.5 * rng.standard_normal(n))
    conc = np.exp(0.3 * np.log(flow) + 0.2 * np.cos(2 * np.pi * days / 365.25) + 0.2 * rng.standard_normal(n))
    return {"time": time, "flow": flow}, conc


def test_engine_fit_trajectory_matches_reference_loop_loadest(cuda_device):
    """MarginalB200.fit against the oracle's restatement of the reference loop (Adam lr .05 wd 1e-4, clip 1.0,
    ReduceLROnPlateau): same objective at every iteration."""
    cov, conc = _loadest_arrays(200, 0)
    m = models.LoadestGP()
    m.fit(cov, conc, iterations=12)
    assert m.is_fitted and len(m.history) == 12
    raw = orc.loadest_init_raw()
    _, hist = orc.fit_adam("loadest", raw, torch.tensor(m.X), torch.tensor(m.y), torch.tensor(m.fixed_noise), iterations=12)
    assert np.max(np.abs(np.array(m.history) - np.array(hist)) / np.abs(hist)) <= RTOL
    # surface: predict / predict_grid / sample / save / load / resume
    target, se = m.predict(cov)
    assert target.shape == (200,) and se.shape == (200,) and np.all(se >= 1.0) and np.all(target > 0)
    grid, index, covs = m.predict_grid("flow")
    assert grid.shape[1] == 18 and grid.shape[0] == index.shape[0] and covs.shape == (18,)
    sub = {k: v[:50] for k, v in cov.items()}
    sim = m.sample(sub, n=32, seed=1)
    assert sim.shape == (32, 50) and np.all(np.isfinite(sim)) and np.all(sim > 0)
    buf = io.BytesIO()
    m.save(buf)
    buf.seek(0)
    m2 = models.LoadestGP.load(buf, cov, conc)
    assert m2.is_fitted and m2._current_iteration == 11
    t2, _ = m2.predict(cov)
    assert np.allclose(t2, target, rtol=1e-10)
    m2.fit(cov, conc, iterations=15, resume=True)
    assert len(m2.history) == 4
    with pytest.raises(ValueError, match="Unsupported optimizer"):
        models.LoadestGP().fit(cov, conc, iterations=1, optimizer="sgd")
    # annual flux of joint draws, reduced on the device (src/loadest_gp/utils.py:14-56,89)
    days = np.arange(0, 800)
    daily = {"time": np.datetime64("2001-06-01") + days.astype("timedelta64[D]"),
             "flow": np.exp(1.0 + 0.8 * np.sin(2 * np.pi * days / 365.25))}
    years, flux = m.sample_annual_flux(daily, n=16, seed=77)
    assert list(years) == [2001, 2002, 2003] and flux.shape == (16, 3) and np.all(flux > 0)
    Xd = m.dm.Xnew(daily)
    Zs = H.philox_normals(77, 16 * 800).reshape(16, 800)
    draws, info = m._engine.sample(Xd, Zs, jitter=0.0)
    concd = np.asarray(m.dm.y_t(draws.reshape(-1))).reshape(16, 800)
    fl = concd * daily["flow"] * 86400.0 * 1e-3
    yr = daily["time"].astype("datetime64[Y]").astype(int) + 1970
    ref = np.stack([fl[:, yr == yv].sum(axis=1) for yv in years], axis=1)
    assert info == 0 and np.max(np.abs(flux - ref) / ref) <= 1e-9


def test_engine_fit_trajectory_matches_reference_loop_rating(cuda_device):
    rng = np.random.default_rng(5)
    n = 150
    days = np.sort(rng.uniform(0, 3650, n))
    time = np.datetime64("2005-01-01") + (days * 86400e9).astype("timedelta64[ns]")
    stage = rng.lognormal(1.0, 0.5, n)
    q = 3.0 * (stage - 0.5 * stage.min()) ** 1.6 * np.exp(0.03 * rng.standard_normal(n))
    gse = rng.choice(np.array([1.02, 1.05, 1.08]), n)
    torch.manual_seed(0)
    m = models.RatingGP()
    m.fit({"time": time, "stage": stage}, q, target_unc=gse, iterations=10)
    torch.manual_seed(0)
    a = float(torch.randn(1)); b = float(torch.randn(1) + 1.3); c = float(torch.rand(1)); u = float(torch.rand(1))
    b_lo, b_hi = models.stage_quantile_bounds(m.X[:, 1])
    raw = orc.rating_init_raw(b_lo, b_hi, gate_b=b_lo + u * (b_hi - b_lo), pl_a=a, pl_b=b, pl_c=c)
    _, hist = orc.fit_adam("rating", raw, torch.tensor(m.X), torch.tensor(m.y), torch.tensor(m.fixed_noise), iterations=10,
                           b_lo=b_lo, b_hi=b_hi, h_min=float(m.X[:, 1].min()))
    assert np.max(np.abs(np.array(m.history) - np.array(hist)) / np.abs(hist)) <= RTOL
    target, se = m.predict({"time": time, "stage": stage})
    assert target.shape == (n,) and np.all(np.isfinite(target)) and np.all(se >= 1.0)
    # monotonic rating penalty (src/rating_gp/models/gpytorch.py:126-202; reference test tests/test_rating_gp.py:52-65):
    # same random grids (torch global generator), same objective trajectory as autograd through two predictions
    torch.manual_seed(3)
    mp_ = models.RatingGP()
    mp_.fit({"time": time, "stage": stage}, q, target_unc=gse, iterations=8, monotonic_penalty_weight=0.5, grid_size=64)
    torch.manual_seed(3)
    a = float(torch.randn(1)); b = float(torch.randn(1) + 1.3); c = float(torch.rand(1)); u = float(torch.rand(1))
    raw = orc.rating_init_raw(b_lo, b_hi, gate_b=b_lo + u * (b_hi - b_lo), pl_a=a, pl_b=b, pl_c=c)
    _, histp = orc.fit_adam("rating", raw, torch.tensor(mp_.X), torch.tensor(mp_.y), torch.tensor(mp_.fixed_noise), iterations=8,
                            b_lo=b_lo, b_hi=b_hi, h_min=float(mp_.X[:, 1].min()), penalty_weight=0.5, grid_size=64)
    assert mp_.is_fitted and np.max(np.abs(np.array(mp_.history) - np.array(histp)) / np.abs(histp)) <= RTOL
    assert np.max(np.abs(np.array(histp) - np.array(hist[:8]))) > 0  # the penalty was active on this data


def test_engine_fit_adamw_matches_reference_loop(cuda_device):
    """optimizer="adamw" (gpytorch.py:271-288: AdamW, weight decay 1e-2) through the closed-form host path and fused AdamW."""
    cov, conc = _loadest_arrays(180, 11)
    m = models.LoadestGP()
    m.fit(cov, conc, iterations=10, optimizer="adamw")
    raw = orc.loadest_init_raw()
    _, hist = orc.fit_adam("loadest", raw, torch.tensor(m.X), torch.tensor(m.y), torch.tensor(m.fixed_noise), iterations=10,
                           optimizer="adamw")
    assert np.max(np.abs(np.array(m.history) - np.array(hist)) / np.abs(hist)) <= RTOL


def test_nlml_only_path_matches_nlml_grad(cuda_device):
    """The NLML-only path (forward substitution along the factorisation) gives the NLML of the NLML + gradient path
    (z = U'r after the triangular inverse)."""
    X, y, noise = synthetic.loadest_site(1300, 21)
    eng = _engine(models.loadest_spec(2), X, y, noise)
    th = np.array([0.05, 0.7, 1.0, 1.0, 2.0, 1.3, 0.5, 0.2, 0.3, 0.4])
    v, _, info = eng.nlml_grad(th)
    v0, info0 = eng.nlml(th)
    assert info == 0 and info0 == 0
    assert abs(v - v0) <= 1e-10 * abs(v)
    eng.close()


def test_engine_surface_with_xarray_stand_in(cuda_device, monkeypatch):
    """predict / predict_grid / sample return the reference's container types when xarray objects come in
    (engines/gpytorch.py:496-499,541-549,583-591); xarray itself is not installable here: tests/fake_xarray.py."""
    import fake_xarray as fx
    from discontinuum_b200 import data as dmod

    monkeypatch.setattr(dmod, "_xr", fx)
    cov, conc = _loadest_arrays(160, 3)
    ds = fx.Dataset({"flow": ("time", cov["flow"])}, coords={"time": cov["time"]})
    tgt = fx.DataArray(conc, coords={"time": cov["time"]}, dims=("time",), attrs={"units": "mg/L"}, name="conc")
    m = models.LoadestGP()
    m.fit(ds, tgt, iterations=5)
    ref = models.LoadestGP()
    ref.fit(cov, conc, iterations=5)
    target, se = m.predict(ds)
    t_ref, se_ref = ref.predict(cov)
    assert isinstance(target, fx.DataArray) and isinstance(se, fx.DataArray) and target.attrs == {"units": "mg/L"}
    assert np.allclose(target.values, t_ref, rtol=1e-12) and np.allclose(se.values, se_ref, rtol=1e-12)
    assert np.array_equal(target.coords["time"].values, cov["time"])
    grid = m.predict_grid("flow")
    assert isinstance(grid, fx.DataArray) and grid.dims == ("time", "flow") and grid.shape[1] == 18
    sub = fx.Dataset({"flow": ("time", cov["flow"][:30])}, coords={"time": cov["time"][:30]})
    sim = m.sample(sub, n=8, seed=2)
    assert isinstance(sim, fx.DataArray) and sim.dims == ("draw", "time") and sim.shape == (8, 30) and np.all(sim.values > 0)


def test_graft_smoke(cuda_device):
    import __graft_entry__ as ge

    ge.smoke()


def test_set_train_reuses_cleared_buffers_and_reserved_sampling_workspace(cuda_device):
    """dgp_set_train skips the 2 n^2 memset when the padded size is unchanged (the zero sub-blocks of L / U are only ever
    written with zeros), and dgp_reserve sizes the sampling workspace ahead of time: a handle that has seen other sites
    and other grid sizes must return exactly what a fresh handle returns."""
    th = H.loadest_theta1()
    spec = models.loadest_spec(2)
    a = synthetic.loadest_site(700, 91)
    b = synthetic.loadest_site(690, 92)     # same padded size (768): no memset between the two
    c = synthetic.loadest_site(300, 93)     # smaller padded size: buffers are cleared again
    Xs = synthetic.daily_grid(b[0], 500) + np.array([0.0005, 0.0])
    Z = np.random.default_rng(3).standard_normal((8, 500))
    fresh = {}
    for name, site in (("b", b), ("c", c)):
        e = _engine(spec, *site)
        fresh[name] = e.nlml_grad(th)
        if name == "b":
            e.factorize(th)
            fresh["Lb"] = e.chol()
            fresh["draws"] = e.sample(Xs, Z, jitter=1e-7)[0]
        e.close()
    eng = capi.Engine(max_n=700, max_m=256)
    eng.reserve(600, 16)
    eng.set_train(spec.to_c(), *a)
    eng.nlml_grad(th)
    eng.factorize(th)
    eng.sample(synthetic.daily_grid(a[0], 300), np.zeros((4, 300)), jitter=1e-7)   # a different grid size through the same arena
    eng.set_train(spec.to_c(), *b)
    got = eng.nlml_grad(th)
    assert got[2] == 0 and got[0] == fresh["b"][0] and np.array_equal(got[1], fresh["b"][1])
    eng.factorize(th)
    Lb = eng.chol()
    assert np.array_equal(Lb, fresh["Lb"]) and np.max(np.abs(np.triu(Lb, 1))) == 0.0
    assert np.array_equal(eng.sample(Xs, Z, jitter=1e-7)[0], fresh["draws"])
    eng.set_train(spec.to_c(), *c)
    got = eng.nlml_grad(th)
    assert got[2] == 0 and got[0] == fresh["c"][0] and np.array_equal(got[1], fresh["c"][1])
    eng.reserve(0)   # releases the workspace; the next call grows it again
    eng.set_train(spec.to_c(), *b)
    eng.factorize(th)
    assert np.array_equal(eng.sample(Xs, Z, jitter=1e-7)[0], fresh["draws"])
    eng.close()


def test_fit_aborts_on_device_fault_instead_of_counting_nan_iterations(cuda_device):
    """A bad-argument / CUDA error from libdgp (rc < 0 -> DgpError) must end fit() at once; only numerical failures are
    skipped like the reference does (engines/gpytorch.py:356-361)."""
    cov, conc = _loadest_arrays(120, 3)
    m = models.LoadestGP()
    m.fit(cov, conc, iterations=2)
    calls = {"n": 0}
    real = m._engine.nlml_grad

    def broken(theta, jitter=0.0):
        calls["n"] += 1
        raise capi.DgpError("dgp_nlml_grad failed (-2): injected CUDA error")

    m._engine.nlml_grad = broken
    with pytest.raises(capi.DgpError, match="injected"):
        m.fit(cov, conc, iterations=5, resume=True)
    assert calls["n"] == 1
    m._engine.nlml_grad = real
