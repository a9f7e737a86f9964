"""Prediction of a group of sites at group close: (a) one capi.Engine per site in turn (set_train + factorize + predict, the
driver's path before dgp_batch_predict) against (b) the group's batch handle (BatchEngine.factorize + predict).

Default group: 16 sites of the BASELINE config-4 size distribution (n = 2000 + 6000 U(0, 1), seed 42, the first 16), each
with its 10 958-point daily grid.  Host clock around synchronised calls, 2 warm-ups, 5 alternating repetitions of each;
prints the median and range of both, the split of (b) into factorize / predict, and the achieved FP64 rate of the variance
GEMMs, sum_s m_s n_s^2 flop over the time.  `small` / `one` add a group of 16 n = 1000 sites and a single n = 8000 site."""
import os
import sys
import time

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, R)
sys.path.insert(0, os.path.join(R, "tests"))
import numpy as np  # noqa: E402

import helpers as H  # noqa: E402
from discontinuum_b200 import capi, models, synthetic  # noqa: E402

M = 10958
spec = models.loadest_spec(2)


def probe(ns, label, warm=2, reps=5):
    sites = [synthetic.loadest_site(int(n), 1000 + k) for k, n in enumerate(ns)]
    grids = [synthetic.daily_grid(s[0], M) for s in sites]
    thetas = np.stack([H.loadest_theta1() * (1.0 + 1e-3 * k) for k in range(len(ns))])
    eng = capi.Engine(max_n=max(ns), max_m=2048)
    b = capi.BatchEngine(max_sites=len(ns), max_n=max(ns))
    b.set_train(spec.to_c(), sites)

    def per_site():
        out = []
        for k, (X, y, nz) in enumerate(sites):
            eng.set_train(spec.to_c(), X, y, nz)
            _, info = eng.factorize(thetas[k])
            assert info == 0
            out.append(eng.predict(grids[k]))
        return out

    def batched():
        t0 = time.perf_counter()
        _, info = b.factorize(thetas)
        t1 = time.perf_counter()
        assert not info.any()
        out = b.predict(grids)
        return out, t1 - t0, time.perf_counter() - t1

    ta, tb, tf, tp = [], [], [], []
    for it in range(warm + reps):
        t0 = time.perf_counter()
        ra = per_site()
        t1 = time.perf_counter()
        rb, f, p = batched()
        t2 = time.perf_counter()
        if it >= warm:
            ta.append(t1 - t0); tb.append(t2 - t1); tf.append(f); tp.append(p)
    same = all(np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1]) for x, y in zip(ra, rb))
    flop = float(sum(M * float(n) ** 2 for n in ns))
    med = lambda v: float(np.median(v))  # noqa: E731
    print(f"{label}: G={len(ns)} n={min(ns)}..{max(ns)} m={M} per site, bit-identical={same}")
    print(f"  (a) per-site Engine set_train+factorize+predict: median {med(ta):.4f} s  [{min(ta):.4f}, {max(ta):.4f}]")
    print(f"  (b) BatchEngine factorize+predict:               median {med(tb):.4f} s  [{min(tb):.4f}, {max(tb):.4f}]"
          f"  = factorize {med(tf):.4f} + predict {med(tp):.4f}")
    print(f"  (a)/(b) = {med(ta) / med(tb):.2f};  variance GEMMs sum m n^2 = {flop / 1e12:.3f} TFLOP: "
          f"{flop / med(tb) / 1e12:.2f} TFLOP/s over (b), {flop / med(tp) / 1e12:.2f} TFLOP/s over its predict", flush=True)
    b.close()
    eng.close()


if __name__ == "__main__":
    which = sys.argv[1:] or ["config4"]
    if "config4" in which:
        rng = np.random.default_rng(42)
        probe([int(v) for v in (2000 + 6000 * rng.uniform(size=128)).astype(int)[:16]], "config-4 first 16")
    if "small" in which:
        probe([1000] * 16, "16 x 1000")
    if "one" in which:
        probe([8000], "1 x 8000")
