"""The top merges of U = L^-T on the INT8 tensor cores (inv_merge_i8 of csrc/dgp_api.cu) and the limb CRT reconstruction
shared by every emulated product (l8_crt of csrc/dgp_lauum8.cuh).

CPU: l8_crt as compiled from the header against exact Python integers (random and extreme residues, x next to +-M/2,
ties, the sticky bit, zero, residue vectors whose CRT sum S = sum_j t_j M/m_j sits next to every multiple of M); the
quotient estimate of the limb CRT on the same sums; the operand width b(K) against exact arithmetic.
GPU: at n = 16 384 and at the ragged 12 289 (97 blocks: 64 | 33), M' = U11 L21' and U12 = -M' T22' equal, bit for bit, the
exactly rounded product of the engine's own operands converted in Python integers; batches with sites on both sides of
the size rule equal per-site handles bit for bit (nlml_grad, factorize + predict).
"""
import os
import random
import re
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from test_lauum_emulated import HDR, M, MODS, MS, _fbits, _scaled, bits, sym_residue

API = os.path.join(os.path.dirname(HDR), "dgp_api.cu")
_src = open(API).read()
INV8_MIN_HB = int(re.search(r"INV8_MIN_HB = (\d+)", _src).group(1))
INV8_MIN_W2 = int(re.search(r"INV8_MIN_W2 = (\d+)", _src).group(1))

HOST_PROG = r"""
#include <cstdio>
#include "dgp_lauum8.cuh"
using namespace dgp;
int main() {
  char op[8];
  while (scanf("%7s", op) == 1) {
    if (op[0] == 'b') { long long k; scanf("%lld", &k); printf("%d\n", l8_bits(k)); }
    else {
      int y[L8_NMOD], sc;
      for (int j = 0; j < L8_NMOD; j++) scanf("%d", &y[j]);
      scanf("%d", &sc);
      const double v = l8_crt(y, sc);
      unsigned long long u;
      memcpy(&u, &v, 8);
      printf("%llu\n", u);
    }
  }
  return 0;
}
"""


def _crt_case(x, sc):
    """the residues of x and the bits of x 2^sc rounded once (sign kept)."""
    v = _scaled(abs(x), sc)
    return "c %s %d" % (" ".join(str(sym_residue(x, m)) for m in MS), sc), str(_fbits(-v if x < 0 else v))


def _from_t(ts):
    """x = (sum_j t_j M/m_j) mod M as a signed integer, |x| <= (M - 1) / 2."""
    x = sum(t * (M // m) for t, m in zip(ts, MS)) % M
    return x - M if x > M // 2 else x


def _limb_quotient(S):
    """q of l8_crt: floor(a3 / (M_top + 1)) from the top bits a3 = S >> 96 of the sum."""
    return (S >> 96) // ((M >> 96) + 1)


def test_limb_crt_quotient_estimate():
    """For every S < 16 M that the limb sum can take, the quotient estimate is floor(S / M) or one less, and one
    correction brings S - q M below M (S next to every multiple of M, the largest S, random S)."""
    rng = random.Random(3)
    smax = sum((m - 1) * (M // m) for m in MS)
    assert smax < 16 * M and smax < 1 << 129
    samples = [0, 1, smax] + [q * M + d for q in range(1, 16) for d in (-2, -1, 0, 1, 2)]
    samples += [rng.randrange(smax + 1) for _ in range(20000)]
    for S in samples:
        if not 0 <= S <= smax:
            continue
        q = _limb_quotient(S)
        assert S // M - 1 <= q <= S // M, S
        x = S - q * M
        assert 0 <= x < 2 * M and (x - M if x >= M else x) == S % M


def test_operand_width_rule():
    """b(K) is the largest b with 2 K 2^(2b-2) < M: K products of two b-bit operands stay below M / 2 (exact), and one
    more bit would not; the merges emulated at 8192-row ranges use b = 56."""
    for K in (128, 4224, 8192, 16384, 1 << 17):
        b = bits(K)
        assert 2 * K * (1 << (2 * b - 2)) < M <= 2 * K * (1 << (2 * b))
        assert K * (1 << (b - 1)) ** 2 < M // 2
    assert bits(64 * 128) == 56


def test_limb_crt_host_exact():
    """l8_crt compiled from the header against exact Python integers: random and extreme residues, +-(M - 1) / 2 and its
    neighbours, ties to even and the sticky bit at several binades, zero, and S next to multiples of M."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not (os.path.exists(nvcc) or shutil.which(nvcc)):
        pytest.skip("nvcc not available")
    rng = random.Random(17)
    half = (M - 1) // 2
    xs = [0, 1, -1, half, -half, half - 1, -(half - 1), half - 2, -(half - 2), 1 << 64, -(1 << 64), (1 << 64) - 1]
    for k in (0, 11, 40, 64, 68):   # ties (53 significant bits + exactly one half) and one past them, both signs
        t = ((((1 << 53) + 1) << 1) | 1) << k
        xs += [t, -t, t + 1, -(t + 1), t - 1]
        t2 = ((((1 << 53) + 2) << 1) | 1) << k
        xs += [t2, -t2]
    xs += [rng.randrange(-half, half + 1) >> rng.randint(0, 124) for _ in range(4000)]
    assert all(abs(x) <= half for x in xs)
    cases, want = [], []
    for x in xs:
        c, w = _crt_case(x, rng.randint(-160, 0))
        cases.append(c); want.append(w)
    # residue vectors with extreme t_j (all m_j - 1, all 0 but one, alternating): S at the top of its range
    for ts in ([m - 1 for m in MS], [0] * 15 + [MS[15] - 1], [m - 1 if j % 2 else 0 for j, m in enumerate(MS)],
               [rng.randrange(m) for m in MS]):
        c, w = _crt_case(_from_t(ts), -100)
        cases.append(c); want.append(w)
    for K in (128, 4224, 8192, 16384):
        cases.append("b %d" % K); want.append(str(bits(K)))
    with tempfile.TemporaryDirectory() as tmp:
        src = os.path.join(tmp, "crt_host.cu")
        with open(src, "w") as f:
            f.write(HOST_PROG)
        exe = os.path.join(tmp, "crt_host")
        subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-I", os.path.dirname(HDR),
                        "-o", exe, src], check=True, capture_output=True)
        out = subprocess.run([exe], input="\n".join(cases) + "\n", capture_output=True, text=True, check=True).stdout
    got = out.split()
    assert len(got) == len(want)
    bad = [(c[:60], g, w) for c, g, w in zip(cases, got, want) if g != w]
    assert not bad, bad[:5]


def _convert(rows, b):
    """k_l8_convert on host rows (entries outside a row's range already zero): scale exponents and integers."""
    mx = np.max(np.abs(rows), axis=1)
    e = np.frexp(mx)[1]
    s = np.where(mx > 0, b - 1 - e, 0).astype(np.int64)
    A = np.rint(np.ldexp(rows, s[:, None].astype(np.int32))).astype(np.int64)
    assert np.max(np.abs(A)) <= 2 ** (b - 1)
    return s, A


def _exact_product(sa, A, sb, B, sign):
    """sign (A B') 2^-(sa + sb), every entry rounded once, from int64 operands (19-bit limbs, exact float64 partials)."""
    def limbs(X):
        sg, mag = np.sign(X), np.abs(X)
        return [(sg * ((mag >> (19 * p)) & ((1 << 19) - 1))).astype(np.float64) for p in range(3)]
    la, lb = limbs(A), limbs(B)
    P = [[la[p] @ lb[q].T for q in range(3)] for p in range(3)]
    out = np.empty((A.shape[0], B.shape[0]))
    for i in range(A.shape[0]):
        for j in range(B.shape[0]):
            x = sum(int(P[p][q][i, j]) << (19 * (p + q)) for p in range(3) for q in range(3))
            sc = -int(sa[i] + sb[j])
            v = _scaled(x, sc) if x >= 0 else -_scaled(-x, sc)
            out[i, j] = sign * v
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("n", [16384, 12289])
def test_top_merge_is_exactly_rounded_product(cuda_device, n):
    """M' (upper triangle of the work matrix after nlml_grad, read through kinv()) and U12 (uinv()) of the top merge equal
    the exactly rounded products of the engine's own operands (U11, L21 from chol(), T22 from linv() of factorize),
    converted in Python integers: first and last row and column blocks, diagonal-block boundaries, the last valid row."""
    from discontinuum_b200 import capi, models, synthetic
    import helpers as H

    X, y, noise = synthetic.loadest_site(n, 1000)
    npad = (n + 127) // 128 * 128
    nb = npad // 128
    hb = 1
    while 2 * hb < nb:
        hb *= 2
    w2 = nb - hb
    assert hb >= INV8_MIN_HB and w2 >= INV8_MIN_W2   # the size rule sends this merge to the INT8 tensor cores
    o1, o2 = 0, hb * 128
    eng = capi.Engine(max_n=n, max_m=256)
    try:
        eng.set_train(models.loadest_spec(2).to_c(), X, y, noise)
        _, info = eng.factorize(H.loadest_theta1())
        assert info == 0
        T = eng.linv()
        Uf = eng.uinv()
        L = eng.chol()
        eng.set_debug_kinv(True)
        _, _, info = eng.nlml_grad(H.loadest_theta1())
        assert info == 0
        W = eng.kinv()
        U = eng.uinv()
    finally:
        eng.close()
    assert np.array_equal(U, Uf)
    rng = np.random.default_rng(7)
    rows = sorted({0, 1, 127, 128, 255, 4095, 4096, o2 - 129, o2 - 128, o2 - 1} | set(int(v) for v in rng.integers(0, o2, 12)))
    cols = sorted({o2, o2 + 1, o2 + 63, o2 + 64, o2 + 127, o2 + 128, n - 129, n - 128, n - 65, n - 64, n - 2, n - 1}
                  | set(int(v) for v in rng.integers(o2, n, 12)))
    # M' = U11 L21': rows of U11 from their diagonal block to the end of range 1, rows of L21 over range 1
    b1 = bits(hb * 128)
    A1 = np.array([np.where(np.arange(o2) >= r // 128 * 128, U[r, :o2], 0.0) for r in rows])
    sa, Ai = _convert(A1, b1)
    sb, Bi = _convert(L[cols, :o2], b1)
    want = _exact_product(sa, Ai, sb, Bi, 1.0)
    got = W[np.ix_(rows, cols)]
    bad = np.argwhere(got.view(np.uint64) != want.view(np.uint64))
    assert bad.size == 0, ("M'", len(bad), [(rows[i], cols[j], got[i, j], want[i, j]) for i, j in bad[:5]])
    # U12 = -M' T22': M' rows over range 2 (dense; the padded columns hold zeros), T22 rows up to their 64-row half
    kw = w2 * 128
    b2 = bits(kw)
    Mp = np.zeros((len(rows), kw))
    Mp[:, :n - o2] = W[rows, o2:n]
    T22 = np.zeros((len(cols), kw))
    for k, c in enumerate(cols):
        hi = min((c - o2) // 64 * 64 + 64, n - o2)
        T22[k, :hi] = T[c, o2:o2 + hi]
    sa, Ai = _convert(Mp, b2)
    sb, Bi = _convert(T22, b2)
    want = _exact_product(sa, Ai, sb, Bi, -1.0)
    got = U[np.ix_(rows, cols)]
    bad = np.argwhere(got.view(np.uint64) != want.view(np.uint64))
    assert bad.size == 0, ("U12", len(bad), [(rows[i], cols[j], got[i, j], want[i, j]) for i, j in bad[:5]])


@pytest.mark.gpu
def test_batch_equals_per_site_across_inverse_rule(cuda_device):
    """Sites above the merge size rule (12 289 points: top merge 64 | 33 blocks emulated) and below it (8 000 and 3 000
    points) in one batch handle: nlml_grad (NLML, gradient, alpha) and factorize + predict (mean, variance) equal per-site
    handles bit for bit."""
    from discontinuum_b200 import capi, models, synthetic
    import helpers as H

    spec = models.loadest_spec(2)
    ns = (12289, 8000, 3000)
    sites = [synthetic.loadest_site(n, 5100 + k) for k, n in enumerate(ns)]
    thetas = np.stack([H.loadest_theta1() * (1.0 + 0.01 * k) for k in range(len(ns))])
    rng = np.random.default_rng(3)
    grids = [X[rng.integers(0, X.shape[0], 300)] + 0.01 for X, _, _ in sites]
    b = capi.BatchEngine(max_sites=len(ns), max_n=max(ns))
    try:
        b.set_train(spec.to_c(), sites)
        val, grad, info = b.nlml_grad(thetas)
        assert np.all(info == 0)
        alphas = [b.alpha(k) for k in range(len(ns))]
        fval, finfo = b.factorize(thetas)
        assert np.all(finfo == 0)
        preds = b.predict(grids)
    finally:
        b.close()
    for k, (X, y, noise) in enumerate(sites):
        eng = capi.Engine(max_n=X.shape[0], max_m=512)
        try:
            eng.set_train(spec.to_c(), X, y, noise)
            v, g, i = eng.nlml_grad(thetas[k])
            assert i == 0 and val[k] == v and np.array_equal(grad[k], g), (k, val[k] - v, grad[k] - g)
            assert np.array_equal(alphas[k], eng.alpha())
            fv, fi = eng.factorize(thetas[k])
            assert fi == 0 and fv == fval[k]
            mu, var = eng.predict(grids[k])
            assert np.array_equal(mu, preds[k][0]) and np.array_equal(var, preds[k][1]), k
        finally:
            eng.close()
