"""Ky^-1 on the INT8 tensor cores (csrc/dgp_lauum8.cuh): the modular (Ozaki scheme II) LAUUM of both engines.

CPU: the constants of the header (moduli, CRT weights, M), the operand width b(npad) against the bounds that make the
products exact, a Python-integer restatement of the conversion and the CRT reconstruction, and the header's own host
functions (l8_bits, l8_residue, l8_round, l8_crt, compiled by nvcc) against exact Python arithmetic on random, extreme,
tie and sticky-bit inputs.
GPU: kinv() of nlml_grad at n = 16 384 and at the size rule equals, bit for bit, the exactly rounded product of the
engine's own U (uinv()) converted in Python integers, on sampled entries of the diagonal blocks, the first and last row
blocks and the last valid row; batch handles with sites on both sides of the size rule (loadest sites, rating gauges)
equal per-site handles bit for bit.
"""
import math
import os
import random
import re
import shutil
import subprocess
import tempfile
from fractions import Fraction

import numpy as np
import pytest

HDR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "discontinuum_b200", "csrc", "dgp_lauum8.cuh")
API = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "discontinuum_b200", "csrc", "dgp_api.cu")


def _header():
    src = open(HDR).read()
    mods = [(int(m), int(inv), int(hi, 16), int(lo, 16)) for m, inv, hi, lo in
            re.findall(r"return \{(\d+), (\d+), (0x[0-9a-f]+)ull, (0x[0-9a-f]+)ull\}", src)]
    mhi, mlo = re.search(r"L8_M_HI = (0x[0-9a-f]+)ull, L8_M_LO = (0x[0-9a-f]+)ull", src).groups()
    max_npad = int(re.search(r"L8_MAX_NPAD = (\d+)", src).group(1))
    return mods, (int(mhi, 16) << 64) | int(mlo, 16), max_npad


MODS, M, MAX_NPAD = _header()
MS = [m for m, _, _, _ in MODS]
MIN_NPAD = int(re.search(r"L8_MIN_NPAD = (\d+)", open(API).read()).group(1))


def bits(npad):
    """csrc l8_bits: the largest b with 2 npad 2^(2b-2) < M."""
    b = 2
    while (2 * npad) << (2 * (b + 1) - 2) < M:
        b += 1
    return b


def convert_row(row, b):
    """k_l8_convert: scale exponent s and the integers A' = round_half_even(u 2^s) of one row."""
    mx = max(abs(x) for x in row)
    if mx == 0.0:
        return 0, [0] * len(row)
    e = math.frexp(mx)[1]
    s = b - 1 - e
    return s, [round(Fraction(x) * Fraction(2) ** s) for x in row]


def sym_residue(a, m):
    r = a % m
    return r - m if r > m // 2 else r


def crt(res):
    """k_l8_recon: the integer with these symmetric residues, |x| < M / 2."""
    x = 0
    for (m, inv, hi, lo), y in zip(MODS, res):
        x = (x + ((y * inv) % m) * ((hi << 64) | lo)) % M
    return x - M if x > M // 2 else x


def test_moduli_and_crt_constants():
    assert len(MODS) == 16 and all(m % 2 == 1 and m <= 255 for m in MS)
    for i in range(16):
        for j in range(i):
            assert math.gcd(MS[i], MS[j]) == 1, (MS[i], MS[j])
    assert M == math.prod(MS)
    for m, inv, hi, lo in MODS:
        assert (hi << 64) | lo == M // m and (inv * (M // m)) % m == 1


def test_operand_width_bounds():
    assert bits(16384) == 55 and bits(32768) == 55
    # INT32 accumulators: npad 127^2 < 2^31 up to the limit and not one block beyond it
    assert MAX_NPAD % 128 == 0 and MAX_NPAD * 127 ** 2 < 2 ** 31 <= (MAX_NPAD + 128) * 127 ** 2
    assert 128 <= MIN_NPAD <= MAX_NPAD
    for npad in range(128, MAX_NPAD + 1, 128):
        b = bits(npad)
        # |A'| <= 2^(b-1): |C'| <= npad 2^(2b-2) < M / 2, and b is the largest such width
        assert 2 * npad * 2 ** (2 * b - 2) < M <= 2 * npad * 2 ** (2 * b)


def test_conversion_and_reconstruction_exact():
    rng = random.Random(7)
    npad = 16384
    b = bits(npad)
    half = (M - 1) // 2
    extremes = [0, 1, -1, half, -half, half - 1, -(half - 1), M // 4, -(M // 4)]
    for x in extremes + [rng.randrange(-half, half + 1) for _ in range(2000)]:
        assert crt([sym_residue(x, m) for m in MS]) == x
    # rows of doubles over many binades, with zeros and ties: the dot product of the integers is recovered exactly
    for t in range(40):
        k = 64
        r1 = [rng.choice([0.0, rng.uniform(-1, 1) * 2.0 ** rng.randint(-60, 3)]) for _ in range(k)]
        r2 = [rng.uniform(-1, 1) * 2.0 ** rng.randint(-30, 0) for _ in range(k)]
        r2[0] = 0.5 + 2.0 ** -53
        s1, a1 = convert_row(r1, b)
        s2, a2 = convert_row(r2, b)
        assert all(abs(v) <= 2 ** (b - 1) for v in a1 + a2)
        assert all(-127 <= sym_residue(v, m) <= 127 for v in a1 for m in MS)
        exact = sum(x * y for x, y in zip(a1, a2))
        prods = [sum(sym_residue(x, m) * sym_residue(y, m) for x, y in zip(a1, a2)) for m in MS]
        assert all(abs(p) < 2 ** 31 for p in prods)
        assert crt([sym_residue(p, m) for p, m in zip(prods, MS)]) == exact


HOST_PROG = r"""
#include <cstdio>
#include <cstring>
#include "dgp_lauum8.cuh"
using namespace dgp;
static unsigned long long bits_of(double d) { unsigned long long u; memcpy(&u, &d, 8); return u; }
int main() {
  char op;
  while (scanf(" %c", &op) == 1) {
    if (op == 'b') { long long npad; scanf("%lld", &npad); printf("%d\n", l8_bits(npad)); }
    else if (op == 'r') { unsigned long long a; int neg, j; scanf("%llu %d %d", &a, &neg, &j); printf("%d\n", l8_residue(a, neg != 0, j)); }
    else if (op == 'd') { unsigned long long hi, lo; int sc; scanf("%llu %llu %d", &hi, &lo, &sc);
                          printf("%llu\n", bits_of(l8_round(((u128)hi << 64) | lo, sc))); }
    else if (op == 'c') { int y[L8_NMOD], sc; for (int j = 0; j < L8_NMOD; j++) scanf("%d", &y[j]); scanf("%d", &sc);
                          printf("%llu\n", bits_of(l8_crt(y, sc))); }
  }
  return 0;
}
"""


def _fbits(v):
    return int(np.array([v], dtype=np.float64).view(np.uint64)[0])


def _scaled(x, sc):
    """x 2^sc rounded once to double (Python's int division rounds correctly)."""
    return x / (1 << -sc) if sc < 0 else float(x << sc)


def test_header_host_functions_exact():
    """l8_bits, l8_residue, l8_round and l8_crt as compiled from the header, against exact Python arithmetic: ties to
    even and the sticky bit of l8_round, symmetric residues up to 2^58, CRT at +-(M - 1) / 2 and at sign boundaries."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not (os.path.exists(nvcc) or shutil.which(nvcc)):
        pytest.skip("nvcc not available")
    rng = random.Random(11)
    cases, want = [], []
    for npad in (128, 1024, 8192, 16384, 32768, MAX_NPAD):
        cases.append("b %d" % npad); want.append(str(bits(npad)))
    for _ in range(3000):
        a = rng.getrandbits(rng.randint(1, 58)) if rng.random() < 0.9 else (1 << 58)
        neg, j = rng.randint(0, 1), rng.randrange(16)
        cases.append("r %d %d %d" % (a, neg, j)); want.append(str(sym_residue(-a if neg else a, MS[j])))
    mags = [0, 1, (1 << 53) + 1, (1 << 64) - 1, 1 << 64, ((1 << 53) + 1) << 60 | 1 << 59, (((1 << 53) + 1) << 60 | 1 << 59) + 1,
            ((1 << 53) + 3) << 60 | 1 << 59, (((1 << 53) + 1) << 11) | 1 << 10, ((((1 << 53) + 1) << 11) | 1 << 10) + 1,
            (M - 1) // 2]
    mags += [rng.getrandbits(rng.randint(1, 124)) for _ in range(3000)]
    for x in mags:
        sc = rng.randint(-200, 0)
        cases.append("d %d %d %d" % (x >> 64, x & ((1 << 64) - 1), sc)); want.append(str(_fbits(_scaled(x, sc))))
    half = (M - 1) // 2
    for x in [0, 1, -1, half, -half, half - 1, -(half - 1)] + [rng.randrange(-half, half + 1) >> rng.randint(0, 120)
                                                                for _ in range(3000)]:
        sc = rng.randint(-150, 0)
        res = " ".join(str(sym_residue(x, m)) for m in MS)
        v = _scaled(abs(x), sc)
        cases.append("c %s %d" % (res, sc)); want.append(str(_fbits(-v if x < 0 else v)))
    with tempfile.TemporaryDirectory() as tmp:
        src = os.path.join(tmp, "l8_host.cu")
        with open(src, "w") as f:
            f.write(HOST_PROG)
        exe = os.path.join(tmp, "l8_host")
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-I", os.path.dirname(HDR),
                        "-o", exe, src], check=True, capture_output=True)
        out = subprocess.run([exe], input="\n".join(cases) + "\n", capture_output=True, text=True, check=True).stdout
    got = out.split()
    assert len(got) == len(want)
    bad = [(c, g, w) for c, g, w in zip(cases, got, want) if g != w]
    assert not bad, bad[:5]


def _exact_kinv(U, rows, cols, npad):
    """{(r, c): the exactly rounded (A'_r . A'_c) 2^-(s_r + s_c)} from the engine's U, converted as k_l8_convert does."""
    b = bits(npad)
    idx = sorted(set(rows) | set(cols))
    pos = {r: k for k, r in enumerate(idx)}
    sub = U[idx]
    mx = np.max(np.abs(sub), axis=1)
    e = np.frexp(mx)[1]
    s = np.where(mx > 0, b - 1 - e, 0).astype(np.int64)
    A = np.rint(np.ldexp(sub, s[:, None].astype(np.int32))).astype(np.int64)
    assert np.max(np.abs(A)) <= 2 ** (b - 1)
    sg, mag = np.sign(A), np.abs(A)
    # 19-bit limbs: every product < 2^38 and every partial sum < 2^52, so the float64 products are exact
    limbs = [(sg * ((mag >> (19 * p)) & ((1 << 19) - 1))).astype(np.float64) for p in range(3)]
    P = [[limbs[p] @ limbs[q].T for q in range(3)] for p in range(3)]
    out = {}
    for r in rows:
        for c in cols:
            if c // 128 > r // 128:
                continue
            i, j = pos[r], pos[c]
            x = sum(int(P[p][q][i, j]) << (19 * (p + q)) for p in range(3) for q in range(3))
            out[(r, c)] = _scaled(x, -int(s[i] + s[j])) if x >= 0 else -_scaled(-x, -int(s[i] + s[j]))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("n", [MIN_NPAD, 16384])
def test_kinv_is_exactly_rounded_product(cuda_device, n):
    """kinv() after nlml_grad equals, bit for bit, the exact product of the engine's own U (uinv()) converted to
    integers in Python and rounded once: diagonal blocks, first and last row blocks, the last valid row."""
    from discontinuum_b200 import capi, models, synthetic
    import helpers as H

    X, y, noise = synthetic.loadest_site(n, 1000)
    npad = (n + 127) // 128 * 128
    eng = capi.Engine(max_n=n, max_m=256)
    try:
        eng.set_train(models.loadest_spec(2).to_c(), X, y, noise)
        eng.set_debug_kinv(True)
        _, _, info = eng.nlml_grad(H.loadest_theta1())
        assert info == 0
        U = eng.uinv()
        K = eng.kinv()
    finally:
        eng.close()
    rng = np.random.default_rng(5)
    rows = sorted({0, 1, 127, 128, 255, n // 2, n // 2 + 77, npad - 129, npad - 128, n - 2, n - 1}
                  | set(int(v) for v in rng.integers(0, n, 20)))
    last = (n - 1) // 128 * 128
    cols = sorted(set(rows) | set(range(0, 128, 3)) | set(range(last, n, 3)) | {n - 1})
    want = _exact_kinv(U, rows, cols, npad)
    got = np.array([K[r, c] for r, c in want])
    exp = np.array(list(want.values()))
    bad = np.flatnonzero(got.view(np.uint64) != exp.view(np.uint64))
    assert bad.size == 0, (bad.size, len(want), [(list(want)[k], got[k], exp[k]) for k in bad[:5]])
    assert len(want) > 1500


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["loadest", "rating"])
def test_batch_equals_per_site_across_size_rule(cuda_device, model):
    """Sites above and below L8_MIN_NPAD padded points in one batch handle (loadest sites, or rating gauges with the
    gate, learned noise and power-law mean): NLML, gradient and alpha equal per-site handles bit for bit."""
    from discontinuum_b200 import capi, models, synthetic
    import helpers as H

    if model == "loadest":
        spec = models.loadest_spec(2)
        ns = (MIN_NPAD + 1000, MIN_NPAD - 128, 1500)
        sites = [synthetic.loadest_site(n, 4100 + k) for k, n in enumerate(ns)]
        thetas = np.stack([H.loadest_theta1() * (1.0 + 0.01 * k) for k in range(len(ns))])
    else:
        ns = (MIN_NPAD + 500, 3000)
        sites = [synthetic.rating_gauge(n, 7 + k) for k, n in enumerate(ns)]
        b_lo, b_hi = models.stage_quantile_bounds(sites[0][0][:, 1])
        spec = models.rating_spec(b_lo, b_hi)
        thetas = np.stack([H.rating_theta1(b_lo, b_hi)] * len(ns))
    b = capi.BatchEngine(max_sites=len(ns), max_n=max(ns))
    try:
        b.set_train(spec.to_c(), sites)
        val, grad, info = b.nlml_grad(thetas)
        assert np.all(info == 0)
        alphas = [b.alpha(k) for k in range(len(ns))]
    finally:
        b.close()
    for k, (X, y, noise) in enumerate(sites):
        eng = capi.Engine(max_n=X.shape[0], max_m=256)
        try:
            eng.set_train(spec.to_c(), X, y, noise)
            v, g, i = eng.nlml_grad(thetas[k])
            assert i == 0 and val[k] == v and np.array_equal(grad[k], g), (k, val[k] - v, grad[k] - g)
            assert np.array_equal(alphas[k], eng.alpha())
        finally:
            eng.close()
