"""The split Cholesky factorisation of libdgp: above a size rule the lower-right quadrant of the training matrix receives the
updates of all panels left of the split as one exact INT8 product (syrk_i8, csrc/dgp_api.cu; the kernels of
csrc/dgp_lauum8.cuh), both engines alike.

CPU: the size rule syrk_split(nb), restated from the constants of dgp_api.cu, at every boundary (the smallest split size,
the largest size the INT32 accumulators allow, the split a whole strip, the sizes of the benchmark's workloads).
GPU: against the float64 GPU reference of test_factor_schedule, for loadest sites just below and at the rule, a ragged size
above it (nb mod 8 != 0) and one rating gauge: DPOT01 <= 1 for the L of nlml_grad, and forward errors of NLML, alpha and
the gradient within max(the spec tests' tolerance, 20 kappa_1 eps); the NLML-only path and factorize give the same L as
nlml_grad above the rule; a batch with sites on both sides of the rule (one of them ragged and off the strip grid of the
end-aligned batch, one indefinite) equals per-site handles bit for bit, for nlml_grad, factorize + predict, and the failing
site's info.
"""
import os
import re

import numpy as np
import pytest
import torch

import helpers as H
import test_factor_schedule as F
from discontinuum_b200 import capi, synthetic, models
from test_spec_generic import TOL_G_REL, TOL_NLML, TOL_VEC

API = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "discontinuum_b200", "csrc", "dgp_api.cu")
LAUUM8 = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "discontinuum_b200", "csrc", "dgp_lauum8.cuh")


def _const(path, name):
    return int(re.search(r"\b%s = (\d+)" % name, open(path).read()).group(1))


SYRK_MIN_NB = _const(API, "SYRK_MIN_NB")
SYRK_NUM, SYRK_DEN = _const(API, "SYRK_NUM"), _const(API, "SYRK_DEN")
STRIP_BLOCKS = _const(API, "STRIP_BLOCKS")
L8_MAX_NPAD = _const(LAUUM8, "L8_MAX_NPAD")


def syrk_split(nb):
    """the rule of dgp_api.cu: SYRK_NUM / SYRK_DEN of the block columns, rounded to the nearest whole strip, or 0"""
    if nb < SYRK_MIN_NB or 128 * nb > L8_MAX_NPAD:
        return 0
    return (SYRK_NUM * nb + SYRK_DEN * STRIP_BLOCKS // 2) // (SYRK_DEN * STRIP_BLOCKS) * STRIP_BLOCKS


def _nb(n):
    return (n + 127) // 128


# ------------------------------------------------------------------------------------------------------------------
# CPU: the size rule
# ------------------------------------------------------------------------------------------------------------------
def test_rule_boundaries():
    assert syrk_split(SYRK_MIN_NB - 1) == 0 and syrk_split(SYRK_MIN_NB) > 0
    max_nb = L8_MAX_NPAD // 128
    assert syrk_split(max_nb) > 0 and syrk_split(max_nb + 1) == 0
    for nb in range(SYRK_MIN_NB, max_nb + 1):
        hs = syrk_split(nb)
        assert hs % STRIP_BLOCKS == 0 and 0 < hs < nb, (nb, hs)
        assert abs(hs - SYRK_NUM * nb / SYRK_DEN) <= STRIP_BLOCKS / 2, (nb, hs)
        # the product's planes fit the LAUUM's residue buffer, the INT32 accumulators cannot overflow
        assert (nb - hs) * nb <= nb * nb and 128 * hs * 127 ** 2 < 2 ** 31
    # the workloads of bench.py: the n = 16 384 headline and config 5 (n = 32 768) split; no config-4 site (n <= 8000) does
    assert syrk_split(_nb(16384)) == 48 and syrk_split(_nb(32768)) == 96
    assert all(syrk_split(_nb(n)) == 0 for n in range(2000, 8001))


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
# (model, n): loadest just below and at the rule, ragged above it, one rating gauge above it
ACC_CASES = [("loadest", 128 * (SYRK_MIN_NB - 1)), ("loadest", 128 * SYRK_MIN_NB),
             ("loadest", 128 * (SYRK_MIN_NB + 5) - 40), ("rating", 128 * (SYRK_MIN_NB + 1) - 7)]


@pytest.mark.gpu
@pytest.mark.parametrize("model,n", ACC_CASES)
def test_split_factorisation_accuracy(cuda_device, model, n):
    nb = _nb(n)
    assert (syrk_split(nb) > 0) == (nb >= SYRK_MIN_NB)
    X, y, noise, theta, spec = F._site(model, n)
    ref = eng = A = B = L = L0 = None
    try:
        ref = F.Reference(model, X, y, noise, theta, F.DEV)
        kappa = ref.kappa1()
        fwd = F.KAPPA_FACTOR * kappa * F.EPS
        tol_nlml, tol_vec, tol_g = max(TOL_NLML, fwd), max(TOL_VEC, fwd), max(TOL_G_REL, fwd)
        eng = capi.Engine(max_n=n, max_m=256)
        eng.set_train(spec.to_c(), X, y, noise)
        val, grad, info = eng.nlml_grad(theta)
        assert info == 0
        err = {"nlml": abs(val - ref.nlml) / abs(ref.nlml), "alpha": F._rel(eng.alpha(), ref.alpha.cpu().numpy()),
               "grad": F._grad_err(grad, ref.grad, tol_g)}
        A = torch.empty((n, n), dtype=torch.float64, device=F.DEV)
        B = torch.empty((n, n), dtype=torch.float64, device=F.DEV)
        with torch.no_grad():
            L = eng.chol(out=A)
            assert torch.count_nonzero(torch.triu(L, 1)) == 0
            dpot01 = F.dpot01(ref.Ky, L)
            dpot01_ref = F.dpot01(ref.Ky, ref.L)
        if nb >= SYRK_MIN_NB:
            # the NLML-only path (forward substitution in the panel chain) and factorize run the same split
            val0, info0 = eng.nlml(theta)
            assert info0 == 0
            L0 = eng.chol(out=B)
            assert torch.equal(L0, L), "the NLML-only path factors differently"
            _, infof = eng.factorize(theta)
            assert infof == 0
            assert torch.equal(eng.chol(out=B), L), "factorize factors differently"
            err["nlml_only"] = abs(val0 - ref.nlml) / abs(ref.nlml)
    finally:
        if eng is not None:
            eng.close()
        ref = A = B = L = L0 = None
        F._free()
    print(f"\n{model} n={n} nb={nb} split={syrk_split(nb)} kappa1={kappa:.2e} dpot01={dpot01:.2e} "
          f"(cusolver {dpot01_ref:.2e}) " + " ".join(f"{k}={v:.2e}" for k, v in err.items()))
    lim = {"nlml": tol_nlml, "nlml_only": tol_nlml, "alpha": tol_vec, "grad": 1.0}
    assert dpot01 <= F.RATIO_MAX, dpot01
    bad = {k: v for k, v in err.items() if not v <= lim[k]}
    assert not bad, (model, n, bad)


@pytest.mark.gpu
def test_batch_across_rule_matches_per_site(cuda_device):
    """Sites {at the rule, ragged above it, below it, indefinite above it} in one batch: the end-aligned batch puts the
    ragged site's split off the global strip grid.  NLML, gradient, alpha and info of nlml_grad, then factorize + predict,
    equal per-site handles bit for bit."""
    ns = (128 * SYRK_MIN_NB, 128 * (SYRK_MIN_NB + 5) - 40, 128 * (SYRK_MIN_NB - 9) + 3, 128 * (SYRK_MIN_NB + 2))
    nbmax = max(_nb(n) for n in ns)
    offs = [(nbmax - _nb(n)) // 4 * 4 for n in ns]
    assert any((o + syrk_split(_nb(n))) % STRIP_BLOCKS for o, n in zip(offs, ns) if syrk_split(_nb(n)))
    spec = models.loadest_spec(2)
    sites = [synthetic.loadest_site(n, 5100 + k) for k, n in enumerate(ns)]
    X, y, noise = sites[3]
    noise = noise.copy()
    fail_row = 128 * (syrk_split(_nb(ns[3])) + 3) + 17   # inside the quadrant, right of the split
    noise[fail_row:] = -3.0
    sites[3] = (X, y, noise)
    thetas = np.stack([H.loadest_theta1() * (1.0 + 0.01 * k) for k in range(len(ns))])
    grids = [synthetic.daily_grid(s[0], 2500) + F.GRID_SHIFT["loadest"] for s in sites]
    b = capi.BatchEngine(max_sites=len(ns), max_n=max(ns))
    try:
        b.set_train(spec.to_c(), sites)
        val, grad, info = b.nlml_grad(thetas)
        assert np.all(info[:3] == 0) and fail_row < info[3] <= ns[3], info
        alphas = [b.alpha(k) for k in range(3)]
        fval, finfo = b.factorize(thetas)
        assert np.all(finfo[:3] == 0) and finfo[3] == info[3]
    finally:
        b.close()
        F._free()
    # the prediction, from a batch of the sites that factorise
    b = capi.BatchEngine(max_sites=3, max_n=max(ns[:3]))
    try:
        b.set_train(spec.to_c(), sites[:3])
        pval, pinfo = b.factorize(thetas[:3])
        assert np.all(pinfo == 0) and np.array_equal(pval, fval[:3])
        out = b.predict(grids[:3])
    finally:
        b.close()
        F._free()
    for k, (X, y, noise) in enumerate(sites):
        eng = capi.Engine(max_n=X.shape[0], max_m=2048)
        try:
            eng.set_train(spec.to_c(), X, y, noise)
            v, g, i = eng.nlml_grad(thetas[k])
            assert i == info[k], (k, i, info[k])
            if k == 3:
                continue
            assert val[k] == v and np.array_equal(grad[k], g), (k, val[k] - v, grad[k] - g)
            assert np.array_equal(alphas[k], eng.alpha()), k
            fv, fi = eng.factorize(thetas[k])
            assert fi == 0 and fval[k] == fv, (k, fval[k] - fv)
            mu, var = eng.predict(grids[k])
        finally:
            eng.close()
            F._free()
        assert np.array_equal(out[k][0], mu), (k, np.max(np.abs(out[k][0] - mu)))
        assert np.array_equal(out[k][1], var), (k, np.max(np.abs(out[k][1] - var)))
