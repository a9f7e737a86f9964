"""libdgp's covariance language against a spec-driven float64 reference (oracle/spec_oracle.py).

The shipped models reach the language through four specs whose terms, but one, all hit a specialised term shape.  The
fixtures below are built to reach the rest of it:

  path                                                       reached by
  ---------------------------------------------------------  --------------------------------------------------------
  run-time interpreter (ShapeRT): covmat, NLML + gradient,    F1 - F6 (test_fixture_vs_reference) and the batch engine
    prediction, sampling, mean-functional gradient, batch       (test_batch_fixture_vs_per_handle_and_reference)
  3-factor terms; factors of 3 and 4 dimensions               F1 (RBF x PER x M52, RBF on 3 dims), F2 / F5 (4 dims)
  periodic factor not first, or alone in its term             F1 (position 1), F2 / F3 (alone), F6
  sinpi fallback: no room for the sin / cos columns           F2 (7 columns), F3 (fifth pair), F5 (8 columns)
  sin / cos pair reuse; several periods in one spec           F3
  unit scale (scale = -1); learned noise with a non-zero mean F1; F4 (power-law mean + learned noise)
  power-law mean on column 2; two gate columns                F4
  tied parameters                                             F6
  limits: 8 terms, 48 theta, 8 columns                        F5
  each specialised shape against the interpreter              test_shape_matches_interpreter
  spec validation (column / gate / mean kinds, gate inputs)   test_set_train_rejects_*

Sizes 37, 300, 900 and 1300 reach the three ways the factorisation generates K: inside the single panel (n <= 512),
by first-touch INIT_COV trailing updates (n = 900: 8 block columns, not above DGP_PREGEN_MIN_NB) and by the standalone
k_cov_lower generator (n = 1300: 11 block columns).  The kernels of one nlml_grad of F1 were listed once with
torch.profiler on a B200: at 300 and 900, k_cov_rect writes the first block column and k_gemm<INIT_COV, ...> the rest
(1 and 3 launches); at 1300, two k_cov_lower strips and no INIT_COV launch.

GPU tests are marked one by one; the CPU tests pin the reference to the oracle's hand-written covariances.
"""
import numpy as np
import pytest
import torch

import helpers as H
from helpers import orc
from discontinuum_b200 import capi, models, synthetic
from discontinuum_b200 import pymc_variant as pv
from discontinuum_b200.spec import CovSpec, Factor
from oracle import spec_oracle as so

RBF, M32, M52, PER = capi.RBF, capi.MATERN32, capi.MATERN52, capi.PERIODIC

# tolerances (float64; the north star of the project is 1e-6 relative)
TOL_K = 1e-13        # covariance entries, relative to max |K|
TOL_NLML = 1e-10     # relative
TOL_VEC = 1e-9       # alpha, mu*, var*, relative to the max norm of the reference
TOL_DRAW = 1e-7      # posterior draws, relative to the max norm
TOL_G_REL, TOL_G_ABS = 1e-8, 1e-12   # gradient, per component: |g - o| <= rel |o| + abs max|o|
# Every used theta has |o_i| >= GRAD_FLOOR max|o|, so no component hides under the absolute term: one at the floor is still
# held to 1e-8 + 1e-12 / GRAD_FLOOR = 1e-6 relative.  The floor is not 1e-4 because the constant-mean component does not
# grow with n while the kernel and noise components do: at n = 900 - 1300 it sits 3e-6 - 7e-5 below the largest.
GRAD_FLOOR = 1e-6

# X columns: time-like, then positive columns (log warps, gate sources, the power-law mean), then centred ones
COLUMN_RANGES = [(0.0, 3.0), (1.0, 3.0), (1.5, 3.0), (-1.0, 1.0), (-1.0, 1.0), (-1.0, 1.0), (0.5, 2.5), (0.0, 1.0)]


class _Builder:
    """CovSpec plus the natural theta that goes with it."""

    def __init__(self, ndim):
        self.s = CovSpec(ndim=ndim)
        self.theta = []

    def p(self, name, value):
        self.theta.append(float(value))
        return self.s.param(name)

    def done(self):
        return self.s, np.array(self.theta)


def f1_interpreter_products():
    """3 COPY columns.  Every term runs the interpreter: PER(c0) x M52(c0, c1); unit-scale M32(c1) x M52(c0) (the reverse
    of SH_M52_M32); RBF(c1) x PER(c0) x M52(c2) (3 factors, periodic at position 1); RBF on 3 dims.  Constant mean, no
    learned noise.  Two periods: sin / cos pairs at columns 3-4 and 5-6."""
    b = _Builder(3)
    c = [b.s.col_copy(d) for d in range(3)]
    s0, lam0, per0 = b.p("t0.s", 0.8), b.p("t0.lam", 1.2), b.p("t0.per", 1.0)
    la, lb = b.p("t0.l0", 1.5), b.p("t0.l1", 0.9)
    b.s.term(s0, [Factor(PER, [c[0]], [lam0], per0), Factor(M52, [c[0], c[1]], [la, lb])])
    l1a, l1b = b.p("t1.l32", 0.7), b.p("t1.l52", 1.1)
    b.s.term(-1, [Factor(M32, [c[1]], [l1a]), Factor(M52, [c[0]], [l1b])])
    s2, l2r, lam2, per2, l2m = b.p("t2.s", 0.6), b.p("t2.lr", 1.1), b.p("t2.lam", 0.8), b.p("t2.per", 0.7), b.p("t2.lm", 1.0)
    b.s.term(s2, [Factor(RBF, [c[1]], [l2r]), Factor(PER, [c[0]], [lam2], per2), Factor(M52, [c[2]], [l2m])])
    s3, l3 = b.p("t3.s", 0.5), [b.p("t3.l0", 1.3), b.p("t3.l1", 1.0), b.p("t3.l2", 0.8)]
    b.s.term(s3, [Factor(RBF, c, l3)])
    b.s.mean_kind, b.s.mean_theta = capi.MEAN_CONST, (b.p("mean.c", 0.3),)
    return b.done()


def f2_no_room():
    """7 COPY columns: one free feature column, so no periodic factor gets its sin / cos pair (7 + 2 > 8) and both take
    the sinpi path.  PER(c0) alone; PER(c3) x M52(c3) is the specialised SH_PER_M52 in its sc_col < 0 branch; RBF on
    4 dims.  Zero mean, learned noise."""
    b = _Builder(7)
    c = [b.s.col_copy(d) for d in range(7)]
    s0, lam0, per0 = b.p("t0.s", 0.7), b.p("t0.lam", 1.0), b.p("t0.per", 0.9)
    b.s.term(s0, [Factor(PER, [c[0]], [lam0], per0)])
    s1, lam1, per1, l1 = b.p("t1.s", 0.5), b.p("t1.lam", 0.9), b.p("t1.per", 0.8), b.p("t1.l", 1.2)
    b.s.term(s1, [Factor(PER, [c[3]], [lam1], per1), Factor(M52, [c[3]], [l1])])
    s2 = b.p("t2.s", 0.9)
    l2 = [b.p("t2.l0", 1.0), b.p("t2.l1", 0.8), b.p("t2.l2", 1.1), b.p("t2.l3", 0.9)]
    b.s.term(s2, [Factor(RBF, [c[1], c[2], c[4], c[5]], l2)])
    b.s.noise_theta = b.p("noise", 0.02)
    return b.done()


def f3_periodic_pairs():
    """Columns COPY x0 (c0) and LOG x1 (c1), so ncols starts at 2.  Column arithmetic of the sin / cos pairs:
    PER(c0, p1) x M52(c0)  -> pair at 2-3, ncols 4;   PER(c0, p1), another lambda -> reuses 2-3;
    PER(c1, p2) x RBF(c1)  -> pair at 4-5, ncols 6 (on a log-warped column);   PER(c0, p3) -> pair at 6-7, ncols 8;
    PER(c1, p4)            -> 8 + 2 > 8: no room, sinpi fallback.  Constant mean, fixed noise only."""
    b = _Builder(2)
    c0, c1 = b.s.col_copy(0), b.s.col_log(1, 1e-6)
    p1 = b.p("p1", 1.0)
    s0, lam0, l0 = b.p("t0.s", 0.6), b.p("t0.lam", 1.1), b.p("t0.l", 1.4)
    b.s.term(s0, [Factor(PER, [c0], [lam0], p1), Factor(M52, [c0], [l0])])
    s1, lam1 = b.p("t1.s", 0.4), b.p("t1.lam", 0.6)
    b.s.term(s1, [Factor(PER, [c0], [lam1], p1)])
    s2, lam2, p2, l2 = b.p("t2.s", 0.5), b.p("t2.lam", 0.9), b.p("p2", 0.6), b.p("t2.l", 0.7)
    b.s.term(s2, [Factor(PER, [c1], [lam2], p2), Factor(RBF, [c1], [l2])])
    s3, lam3, p3 = b.p("t3.s", 0.3), b.p("t3.lam", 1.3), b.p("p3", 0.45)
    b.s.term(s3, [Factor(PER, [c0], [lam3], p3)])
    s4, lam4, p4 = b.p("t4.s", 0.35), b.p("t4.lam", 0.8), b.p("p4", 0.9)
    b.s.term(s4, [Factor(PER, [c1], [lam4], p4)])
    b.s.mean_kind, b.s.mean_theta = capi.MEAN_CONST, (b.p("mean.c", -0.2),)
    return b.done()


def _f4(gate_input=False):
    b = _Builder(3)
    c0, c1 = b.s.col_copy(0), b.s.col_log(1, 1e-6)
    g1 = b.s.col_gate(1, 6.0, b.p("gate1.b", 2.0))
    g2 = b.s.col_gate(2, 3.0, b.p("gate2.b", 2.2))
    s0, l0h, l0t = b.p("t0.s", 0.9), b.p("t0.lh", 0.6), b.p("t0.lt", 1.2)
    b.s.term(s0, [Factor(M52, [c1], [l0h]), Factor(M32, [c0], [l0t])], capi.GATE_SIGMOID, g1)
    s1, l1 = b.p("t1.s", 0.7), b.p("t1.l", 0.9)
    b.s.term(s1, [Factor(M52, [c0], [l1])], capi.GATE_INV_SIGMOID, g2)
    s2, l2h, l2t = b.p("t2.s", 0.5), b.p("t2.lh", 0.8), b.p("t2.lt", 1.5)
    b.s.term(s2, [Factor(RBF, [g1 if gate_input else c1, c0], [l2h, l2t])], capi.GATE_SIGMOID, g1)
    b.s.mean_kind, b.s.mean_col = capi.MEAN_POWERLAW, 2
    b.s.mean_theta = (b.p("pl.a", 0.2), b.p("pl.b", 0.8), b.p("pl.c", 1.0))
    b.s.noise_theta = b.p("noise", 0.01)
    return b.done()


def f4_gates_and_means():
    """COPY x0, LOG x1 and two gate columns (x1 with sharpness 6, x2 with sharpness 3).  SIGMOID on the first gate column
    for two terms (shared), INV_SIGMOID on the second; factors on the LOG column.  Power-law mean on X column 2, learned
    noise."""
    return _f4()


def f5_limits():
    """ndim = ncols = 8 (no room for any sin / cos pair), nterms = 8, ntheta = 48 with the learned noise at index 47 and
    18 entries used nowhere.  Every factor kind, every gate kind, a LOG and a GATE column, one 3-factor term, one 4-dim
    factor, constant mean."""
    b = _Builder(8)
    c = [b.s.col_copy(d) for d in range(6)]
    c.append(b.s.col_log(6, 0.1))
    g = b.s.col_gate(7, 6.0, b.p("gate.b", 0.5))
    s = [b.p(f"t{k}.s", v) for k, v in enumerate((0.5, 0.6, 0.4, 0.5, 0.3, 0.7, 0.4, 0.6))]
    b.s.term(s[0], [Factor(PER, [c[0]], [b.p("t0.lam", 1.0)], b.p("t0.per", 1.1)), Factor(M52, [c[0]], [b.p("t0.l", 1.5)])])
    b.s.term(s[1], [Factor(RBF, [c[1]], [b.p("t1.l", 0.9)])])
    b.s.term(s[2], [Factor(M32, [c[2], c[3]], [b.p("t2.l0", 1.2), b.p("t2.l1", 1.4)])])
    b.s.term(s[3], [Factor(M52, [c[4]], [b.p("t3.l0", 1.1)]), Factor(M32, [c[5]], [b.p("t3.l1", 1.3)]),
                    Factor(RBF, [c[6]], [b.p("t3.l2", 0.8)])])
    b.s.term(s[4], [Factor(RBF, c[0:4], [b.p(f"t4.l{d}", v) for d, v in enumerate((1.6, 1.0, 1.2, 1.5))])])
    b.s.term(s[5], [Factor(M52, [c[1], c[4]], [b.p("t5.l0", 1.0), b.p("t5.l1", 1.3)])], capi.GATE_SIGMOID, g)
    b.s.term(s[6], [Factor(PER, [c[5]], [b.p("t6.lam", 0.9)], b.p("t6.per", 0.8)), Factor(RBF, [c[2]], [b.p("t6.l", 1.1)])])
    b.s.term(s[7], [Factor(M32, [c[6]], [b.p("t7.l", 0.9)])], capi.GATE_INV_SIGMOID, g)
    b.s.mean_kind, b.s.mean_theta = capi.MEAN_CONST, (b.p("mean.c", 0.25),)
    while b.s.ntheta < capi.MAX_THETA - 1:
        b.p(f"unused.{b.s.ntheta}", 0.5 + 0.01 * b.s.ntheta)
    b.s.noise_theta = b.p("noise", 0.015)
    assert b.s.ntheta == capi.MAX_THETA and b.s.noise_theta == 47
    return b.done()


def f6_tied():
    """One lengthscale index L on both dims of RBF(c0, c1) and on M32(c2) of another term; the scale index sA on two
    terms.  Zero mean, no learned noise."""
    b = _Builder(3)
    c = [b.s.col_copy(d) for d in range(3)]
    sA, L = b.p("sA", 0.6), b.p("L", 1.1)
    b.s.term(sA, [Factor(RBF, [c[0], c[1]], [L, L])])
    sB, l2 = b.p("sB", 0.5), b.p("l2", 0.9)
    b.s.term(sB, [Factor(M32, [c[2]], [L]), Factor(M52, [c[0]], [l2])])
    lam, per = b.p("lam", 1.0), b.p("per", 0.8)
    b.s.term(sA, [Factor(PER, [c[1]], [lam], per)])
    return b.done()


FIXTURES = {"F1": f1_interpreter_products, "F2": f2_no_room, "F3": f3_periodic_pairs, "F4": f4_gates_and_means,
            "F5": f5_limits, "F6": f6_tied}


def _inputs(ndim, n, rng):
    X = np.stack([rng.uniform(*COLUMN_RANGES[d], n) for d in range(ndim)], 1)
    X[:, 0] = np.sort(X[:, 0])
    return np.ascontiguousarray(X)


def _data(spec, theta, n, seed):
    """X[n, ndim] over COLUMN_RANGES (column 0 sorted), fixed noise in [0.01, 0.02], and y drawn from the model itself
    with every scale, lengthscale and period moved by a random factor in [0.6, 1.5]: the misfit keeps the gradient
    components away from zero."""
    rng = np.random.default_rng(seed)
    X = _inputs(spec.ndim, n, rng)
    noise = 0.01 * (1.0 + rng.uniform(0.0, 1.0, n))
    kern = sorted({t.scale for t in spec.terms if t.scale >= 0} |
                  {i for t in spec.terms for f in t.factors for i in list(f.ls) + ([f.period] if f.kind == PER else [])})
    th2 = theta.copy()
    th2[kern] *= rng.uniform(0.6, 1.5, len(kern))
    ref = so.SpecModel(spec, X, np.zeros(n), noise)
    nat = ref.nat(th2)
    extra = float(ref.extra(nat)) if spec.noise_theta >= 0 else 0.0
    L = torch.linalg.cholesky(ref.cov(ref.X, ref.X, nat) + torch.diag(ref.noise + extra))
    y = ref.mean(ref.X, ref.nat(theta)) + L @ torch.tensor(rng.standard_normal(n))
    return X, y.numpy(), noise


def _grid(X, m, n_exact, seed):
    """m grid points: m - n_exact fresh points off the training set, then n_exact exact training inputs."""
    rng = np.random.default_rng(seed)
    fresh = _inputs(X.shape[1], m - n_exact, rng)
    idx = rng.choice(X.shape[0], n_exact, replace=False)
    return np.ascontiguousarray(np.concatenate([fresh, X[idx]])), idx


def _used_theta(spec):
    used = set()
    for kind, src, th, aux in spec.cols:
        if kind == capi.COL_GATE:
            used.add(th)
    for t in spec.terms:
        if t.scale >= 0:
            used.add(t.scale)
        for f in t.factors:
            used.update(f.ls)
            if f.kind == PER:
                used.add(f.period)
    used.update(spec.mean_theta[:{capi.MEAN_ZERO: 0, capi.MEAN_CONST: 1, capi.MEAN_POWERLAW: 3}[spec.mean_kind]])
    if spec.noise_theta >= 0:
        used.add(spec.noise_theta)
    return sorted(used)


def _grad_err(got, want):
    """max over components of |g - o| / (rel |o| + abs max|o|): <= 1 passes."""
    scale = TOL_G_REL * np.abs(want) + TOL_G_ABS * np.max(np.abs(want))
    return float(np.max(np.abs(got - want) / scale))


def _rel(got, want):
    return float(np.max(np.abs(np.asarray(got) - np.asarray(want))) / np.max(np.abs(want)))


# ------------------------------------------------------------------------------------------------------------------
# CPU: the reference against the oracle's hand-written models
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d", [2, 3])
def test_reference_matches_oracle_loadest(d):
    X, y, noise = synthetic.loadest_site(300, 5)
    if d == 3:
        X = np.concatenate([X, np.random.default_rng(0).standard_normal((300, 1))], 1)
        th = np.array([0.1, 0.7, 1.0, 1.0, 2.0, 1.3, 0.5, 0.8, 0.2, 0.3, 0.4, 0.6])
    else:
        th = H.loadest_theta1()
    Xt, tt = torch.tensor(X), torch.tensor(th)
    nat = H.loadest_nat_from_theta(th, d)
    spec = models.loadest_spec(d)
    want = orc.loadest_cov(Xt, Xt, nat)
    got = so.spec_cov(spec, Xt, Xt, tt)
    assert float((got - want).abs().max()) <= 1e-15 * float(want.abs().max())
    assert torch.equal(so.spec_mean(spec, Xt, tt), orc.loadest_mean(Xt, nat))


def test_reference_matches_oracle_rating():
    X, y, noise = synthetic.rating_gauge(300, 7)
    b_lo, b_hi = models.stage_quantile_bounds(X[:, 1])
    th = H.rating_theta1(b_lo, b_hi)
    Xt, tt = torch.tensor(X), torch.tensor(th)
    nat = H.rating_nat_from_theta(th)
    spec = models.rating_spec(b_lo, b_hi)
    want = orc.rating_cov(Xt, Xt, nat)
    got = so.spec_cov(spec, Xt, Xt, tt)
    assert float((got - want).abs().max()) <= 1e-15 * float(want.abs().max())
    assert float((so.spec_mean(spec, Xt, tt) - orc.rating_mean(Xt, nat)).abs().max()) == 0.0


def test_reference_matches_oracle_pymc():
    X, _, _ = synthetic.loadest_site(300, 6)
    Xt = torch.tensor(X)
    v = {x.name: torch.tensor(x.init, dtype=torch.float64).reshape(-1) * (1.0 + 0.1 * k)
         for k, x in enumerate(pv.loadest_pymc_vars(2))}
    want = orc.pymc_loadest_cov(Xt, Xt, v)
    got = so.spec_cov(pv.loadest_pymc_spec(2), Xt, Xt, pv.pymc_to_natural(v))
    assert float((got - want).abs().max()) <= 1e-15 * float(want.abs().max())


def test_reference_gradient_and_prediction_match_closed_form():
    """SpecModel's autograd-through-Cholesky gradient (learned noise as its own leaf) equals the oracle's trace-identity
    gradient of the rating model, and its prediction equals orc.predict with the rating callables."""
    X, y, noise = synthetic.rating_gauge(200, 8)
    b_lo, b_hi = models.stage_quantile_bounds(X[:, 1])
    th = H.rating_theta1(b_lo, b_hi)
    ref = so.SpecModel(models.rating_spec(b_lo, b_hi), X, y, noise)
    val, grad, alpha = ref.nlml_grad(th)
    nat = H.rating_nat_from_theta(th)
    v, g, a, _ = orc.nlml_grad_closed_form(orc.rating_cov, orc.rating_mean, nat, torch.tensor(X), torch.tensor(y),
                                           torch.tensor(noise), extra_key="noise")
    want = H.rating_theta_from_nat({k: t.numpy() for k, t in g.items()})
    assert abs(val - float(v)) <= 1e-12 * abs(float(v))
    assert np.max(np.abs(grad - want)) <= 1e-9 * np.max(np.abs(want))
    assert np.max(np.abs(alpha - a.numpy())) <= 1e-12 * np.max(np.abs(a.numpy()))
    Xs = synthetic.daily_grid(X, 50)
    mu, var = ref.predict(th, Xs)
    mu_o, _, var_o = orc.predict(orc.rating_cov, orc.rating_mean, nat, torch.tensor(X), torch.tensor(y), torch.tensor(noise),
                                 torch.tensor(Xs), extra_noise=nat["noise"])
    assert np.max(np.abs(mu - mu_o.numpy())) <= 1e-12 * np.max(np.abs(mu_o.numpy()))
    assert np.max(np.abs(var - var_o.numpy())) <= 1e-12 * np.max(np.abs(var_o.numpy()))


@pytest.mark.parametrize("name", sorted(FIXTURES))
def test_fixture_specs_are_valid_and_every_used_theta_matters(name):
    """Each fixture converts to a dgp_spec within the limits, and at n = 300 every theta it uses moves the NLML by at least
    GRAD_FLOOR of the largest component (so the per-component gradient check sees each of them); unused entries get 0."""
    spec, theta = FIXTURES[name]()
    cs = spec.to_c()
    assert cs.ntheta == theta.shape[0] and cs.ncols <= capi.MAX_COLS
    X, y, noise = _data(spec, theta, 300, 1)
    _, g, _ = so.SpecModel(spec, X, y, noise).nlml_grad(theta)
    used = _used_theta(spec)
    assert np.all(np.abs(g[used]) >= GRAD_FLOOR * np.max(np.abs(g))), (name, g)
    unused = np.setdiff1d(np.arange(theta.shape[0]), used)
    assert np.all(g[unused] == 0.0)


# ------------------------------------------------------------------------------------------------------------------
# GPU: every entry point of the single-site engine against the reference
# ------------------------------------------------------------------------------------------------------------------
CASES = [(f, n) for f in sorted(FIXTURES) for n in (37, 300, 900)] + [(f, 1300) for f in ("F1", "F3", "F5")]
MFG_FIXTURES = ("F1", "F4", "F5")
SAMPLE_FIXTURES = ("F1", "F3", "F4")


@pytest.mark.gpu
@pytest.mark.parametrize("name,n", CASES)
def test_fixture_vs_reference(cuda_device, name, n):
    spec, theta = FIXTURES[name]()
    X, y, noise = _data(spec, theta, n, 100 + n)
    ref = so.SpecModel(spec, X, y, noise)
    eng = capi.Engine(max_n=n, max_m=256)
    eng.set_train(spec.to_c(), X, y, noise)
    err = {}
    # covariance and cross covariance
    Kw = ref.K(theta)
    err["K"] = _rel(eng.covmat(theta), Kw)
    Xs, idx = _grid(X, 1030, 10, 200 + n)
    err["Kx"] = _rel(eng.cross_covmat(theta, Xs), ref.K(theta, Xs))
    # NLML, gradient, alpha; the NLML-only path
    v, g, a = ref.nlml_grad(theta)
    val, grad, info = eng.nlml_grad(theta)
    assert info == 0
    err["nlml"] = abs(val - v) / abs(v)
    err["grad"] = _grad_err(grad, g)
    used = _used_theta(spec)
    err["grad_rel"] = float(np.max(np.abs(grad[used] - g[used]) / np.abs(g[used])))
    err["floor"] = float(np.min(np.abs(g[used])) / np.max(np.abs(g)))
    err["alpha"] = _rel(eng.alpha(), a)
    assert np.all(np.abs(g[used]) >= GRAD_FLOOR * np.max(np.abs(g))), g
    unused = np.setdiff1d(np.arange(theta.shape[0]), used)
    assert np.all(grad[unused] == 0.0), grad[unused]
    val0, info0 = eng.nlml(theta)
    assert info0 == 0
    err["nlml_only"] = abs(val0 - val) / abs(val)
    # factorize + predict on 1030 points (5 chunks of 256, the last ragged), 10 of them exact training inputs
    _, info = eng.factorize(theta)
    assert info == 0
    mu, var = eng.predict(Xs)
    mu_w, var_w = ref.predict(theta, Xs)
    err["mu"] = _rel(mu, mu_w)
    err["var"] = _rel(var, var_w)
    learned = theta[spec.noise_theta] if spec.noise_theta >= 0 else 0.0
    assert np.all(var[-10:] <= noise[idx] + learned + 1e-12) and np.all(var[-10:] > -1e-12)
    if name in MFG_FIXTURES:
        m = 200
        c = np.random.default_rng(n).standard_normal(m)
        F, gF = eng.mean_functional_grad(Xs[:m], c)
        Fw, gFw = ref.mean_functional_grad(theta, Xs[:m], c)
        err["mfg_F"] = abs(F - Fw) / abs(Fw)
        err["mfg_grad"] = _grad_err(gF, gFw)
    if name in SAMPLE_FIXTURES:
        m, S = 200, 16
        Z = np.random.default_rng(7 + n).standard_normal((S, m))
        draws, info = eng.sample(Xs[:m], Z, jitter=1e-6)
        assert info == 0
        err["draws"] = _rel(draws, ref.sample(theta, Xs[:m], Z, jitter=1e-6))
    eng.close()
    print(f"\n{name} n={n} " + " ".join(f"{k}={v:.2e}" for k, v in err.items()))
    lim = {"K": TOL_K, "Kx": TOL_K, "nlml": TOL_NLML, "nlml_only": TOL_NLML, "alpha": TOL_VEC, "mu": TOL_VEC,
           "var": TOL_VEC, "mfg_F": TOL_VEC, "draws": TOL_DRAW, "grad": 1.0, "mfg_grad": 1.0, "grad_rel": np.inf, "floor": np.inf}
    bad = {k: v for k, v in err.items() if not v <= lim[k]}
    assert not bad, (name, n, bad)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(FIXTURES))
def test_batch_fixture_vs_per_handle_and_reference(cuda_device, name):
    """Batch engine, 3 ragged sites: NLML + gradient and factorise + predict equal the per-handle path bit for bit, and
    each site's gradient matches the reference."""
    spec, theta = FIXTURES[name]()
    ns = (37, 300, 700)
    sites = [_data(spec, theta, n, 500 + n) for n in ns]
    thetas = np.stack([theta * (1.0 + 0.02 * k) for k in range(len(ns))])
    grids = [_grid(s[0], 300 + 97 * k, 5, 600 + k)[0] for k, s in enumerate(sites)]
    b = capi.BatchEngine(max_sites=len(ns), max_n=max(ns))
    b.set_train(spec.to_c(), sites)
    val, grad, info = b.nlml_grad(thetas)
    assert np.all(info == 0)
    fval, finfo = b.factorize(thetas)
    assert np.all(finfo == 0)
    out = b.predict(grids)
    for k, (X, y, noise) in enumerate(sites):
        eng = capi.Engine(max_n=X.shape[0], max_m=2048)
        eng.set_train(spec.to_c(), X, y, noise)
        v, g, i = eng.nlml_grad(thetas[k])
        assert i == 0 and val[k] == v and np.array_equal(grad[k], g), (k, grad[k] - g)
        fv, fi = eng.factorize(thetas[k])
        assert fi == 0 and fval[k] == fv
        mu, var = eng.predict(grids[k])
        assert np.array_equal(out[k][0], mu) and np.array_equal(out[k][1], var), k
        eng.close()
        _, gw, _ = so.SpecModel(spec, X, y, noise).nlml_grad(thetas[k])
        assert _grad_err(grad[k], gw) <= 1.0, (k, _grad_err(grad[k], gw))
    b.close()


# ------------------------------------------------------------------------------------------------------------------
# GPU: each specialised term shape against the same function through the run-time interpreter
# ------------------------------------------------------------------------------------------------------------------
CONST_X = 0.7   # value of the extra X column every training and grid point holds


def _shape_pair(shape):
    """(spec that hits `shape`, twin that computes the same function through ShapeRT, theta of each).  X = (x0, x1, const).  2-factor shapes whose factors differ are swapped; the
    others get two extra dims on COPY columns of the constant column (z = 0 exactly), taking a factor from 1 to 3 or
    from 2 to 4 dims.  The dummy lengthscales are the last two theta entries of the twin."""
    kinds = {"RBF1": (RBF, 1), "RBF2": (RBF, 2), "M32_1": (M32, 1), "M32_2": (M32, 2), "M52_1": (M52, 1),
             "M52_2": (M52, 2)}

    def build(twin):
        s = CovSpec(ndim=3)
        c0, c1 = s.col_copy(0), s.col_copy(1)
        th = []

        def p(v):
            th.append(v)
            return s.param(f"p{len(th)}")

        sc = p(0.8)
        dummy = []
        if twin and shape not in ("PER_M52", "M52_M32"):
            dummy = [s.col_copy(2), s.col_copy(2)]
        if shape in kinds:
            kind, nd = kinds[shape]
            cols, ls = [c0, c1][:nd], [p(1.1), p(0.8)][:nd]
            facs = [Factor(kind, cols, ls)]
        elif shape == "PER_M52":
            facs = [Factor(PER, [c0], [p(0.9)], p(1.0)), Factor(M52, [c0], [p(1.3)])]
        elif shape == "M52_M32":
            facs = [Factor(M52, [c1], [p(0.9)]), Factor(M32, [c0], [p(1.2)])]
        else:  # M52_M52
            facs = [Factor(M52, [c1], [p(0.9)]), Factor(M52, [c0], [p(1.2)])]
        s.term(sc, facs)
        s.mean_kind, s.mean_theta = capi.MEAN_CONST, (p(0.1),)
        s.noise_theta = p(0.01)
        if twin:
            if dummy:
                f0 = facs[0]
                f0.cols, f0.ls = list(f0.cols) + dummy, list(f0.ls) + [p(0.5), p(2.0)]
            else:
                s.terms[0].factors = facs[::-1]
        return s, np.array(th)

    a, tha = build(False)
    b, thb = build(True)
    return a, b, tha, thb


SHAPES = ("PER_M52", "RBF1", "M32_2", "M52_1", "M52_M32", "M52_M52", "RBF2", "M32_1", "M52_2")


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES)
def test_shape_matches_interpreter(cuda_device, shape):
    a, b, tha, thb = _shape_pair(shape)
    P = tha.shape[0]
    for n in (300, 1300):
        X, y, noise = _data(a, tha, n, 900 + n)   # a does not read column 2: y does not depend on it
        X[:, 2] = CONST_X
        Xs, _ = _grid(X, 700, 10, 901)
        Xs[:, 2] = CONST_X
        c = np.random.default_rng(n).standard_normal(200)
        res = []
        for spec, th in ((a, tha), (b, thb)):
            eng = capi.Engine(max_n=n, max_m=256)
            eng.set_train(spec.to_c(), X, y, noise)
            K = eng.covmat(th)
            val, grad, info = eng.nlml_grad(th)
            assert info == 0
            eng.factorize(th)
            mu, var = eng.predict(Xs)
            F, gF = eng.mean_functional_grad(Xs[:200], c)
            eng.close()
            res.append((K, val, grad, mu, var, F, gF))
        (K, val, grad, mu, var, F, gF), (K2, val2, grad2, mu2, var2, F2, gF2) = res
        assert np.all(grad2[P:] == 0.0) and np.all(gF2[P:] == 0.0), (grad2[P:], gF2[P:])
        err = {"K": _rel(K2, K), "nlml": abs(val2 - val) / abs(val), "grad": _rel(grad2[:P], grad),
               "mu": _rel(mu2, mu), "var": _rel(var2, var), "F": abs(F2 - F) / abs(F), "mfg_grad": _rel(gF2[:P], gF)}
        print(f"\n{shape} n={n} " + " ".join(f"{k}={v:.2e}" for k, v in err.items()))
        assert err["K"] <= 1e-12 and all(v <= 1e-10 for v in err.values()), (shape, n, err)


# ------------------------------------------------------------------------------------------------------------------
# spec validation (check_spec, shared by both engines).  Nothing here evaluates a spec: set_train must refuse it.
# ------------------------------------------------------------------------------------------------------------------
def _invalid_specs():
    out = []
    for kind in (3, 99, 100, 101, -1):
        s = f1_interpreter_products()[0].to_c()
        s.col[1].kind = kind
        out.append((f"col_kind_{kind}", s, "col 1 kind"))
    for gate in (3, -1):
        s = f4_gates_and_means()[0].to_c()
        s.term[1].gate = gate
        out.append((f"gate_{gate}", s, "term 1 gate kind"))
    for mk in (3, -1):
        s = f1_interpreter_products()[0].to_c()
        s.mean_kind = mk
        out.append((f"mean_kind_{mk}", s, "mean kind"))
    out.append(("gate_input", _f4(gate_input=True)[0].to_c(), "term 2 factor 0 dim 0 reads gate column 2"))
    return out


INVALID = _invalid_specs()


@pytest.mark.gpu
@pytest.mark.parametrize("case", [c[0] for c in INVALID])
def test_set_train_rejects_invalid_spec(cuda_device, case):
    _, spec, msg = next(c for c in INVALID if c[0] == case)
    X = _inputs(spec.ndim, 40, np.random.default_rng(3))
    y, noise = np.zeros(40), np.full(40, 0.01)
    eng = capi.Engine(max_n=64, max_m=64)
    with pytest.raises(capi.DgpError, match=msg):
        eng.set_train(spec, X, y, noise)
    eng.close()
    b = capi.BatchEngine(max_sites=2, max_n=64)
    with pytest.raises(capi.DgpError, match=msg):
        b.set_train(spec, [(X, y, noise), (X[:20], y[:20], noise[:20])])
    b.close()
