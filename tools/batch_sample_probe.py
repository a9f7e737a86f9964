"""Annual-flux sampling of a group of sites: (a) the group's batch handle (BatchEngine.sample, one dgp_batch_sample_ex
launch sequence for all sites, on the factorised group) against (b) a loop of per-site Engine.sample_ex on per-site
handles that are already factorised and (c) what a user does without the batch form: one capi.Engine per site in turn,
set_train + factorize + sample_ex.

Group: 16 sites of the BASELINE config-4 size distribution (n = 2000 + 6000 U(0, 1), seed 42, the first 16, bench.py's
draw), each with its 10 958-point daily grid, S = 1000 Philox draws reduced to 30 "years" on the device.  Host clock
around synchronised calls, 1 warm-up, then 3 alternating repetitions of (a), (b), (c); prints the median and range of
each, whether the three give the same bits, the shape-derived flop count and FP64 rate of (a), the sampling arena of (a),
and the GPU name and power limit read in the same run.  Flop per site (m grid points, n training points, S draws):
m n^2 (V' = Kx T', T triangular) + m^2 n (lower half of Sigma*) + m^3 / 3 (its Cholesky) + S m^2 (draws, Lpost triangular).
`small` runs a group of 16 n = 1000 sites with 2 000-point grids instead."""
import os
import subprocess
import sys
import time

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, R)
sys.path.insert(0, os.path.join(R, "tests"))
import numpy as np  # noqa: E402

import helpers as H  # noqa: E402
from discontinuum_b200 import capi, models, synthetic  # noqa: E402

S = 1000
spec = models.loadest_spec(2)


def gpu_info() -> str:
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def flux_of(m):
    rng = np.random.default_rng(7)
    w = np.exp(rng.standard_normal(m)) * 86.4
    gs = np.linspace(0, m, 31).astype(np.int32)
    return dict(y_mean=0.2, y_scale=0.9, log_transform=1, weight=w, group_start=gs)


def probe(ns, M, label, warm=1, reps=3):
    G = len(ns)
    sites = [synthetic.loadest_site(int(n), 1000 + k) for k, n in enumerate(ns)]
    grids = [synthetic.daily_grid(s[0], M) for s in sites]
    thetas = np.stack([H.loadest_theta1() * (1.0 + 1e-3 * k) for k in range(G)])
    flux = [flux_of(M) for _ in range(G)]
    seeds = list(range(G))
    b = capi.BatchEngine(max_sites=G, max_n=max(ns))
    b.set_train(spec.to_c(), sites)
    _, info = b.factorize(thetas)
    assert not info.any()
    engs = []
    for k, (X, y, nz) in enumerate(sites):   # (b): factorised per-site handles
        e = capi.Engine(max_n=X.shape[0], max_m=2048)
        e.set_train(spec.to_c(), X, y, nz)
        assert e.factorize(thetas[k])[1] == 0
        engs.append(e)
    eng = capi.Engine(max_n=max(ns), max_m=2048)   # (c): one handle, reloaded per site

    def run_a():
        return [o for o, _ in b.sample(grids, S, seeds=seeds, flux=flux)]

    def run_b():
        return [engs[k].sample_ex(grids[k], S, seed=seeds[k], flux=flux[k])[0] for k in range(G)]

    def run_c():
        out = []
        for k, (X, y, nz) in enumerate(sites):
            eng.set_train(spec.to_c(), X, y, nz)
            assert eng.factorize(thetas[k])[1] == 0
            out.append(eng.sample_ex(grids[k], S, seed=seeds[k], flux=flux[k])[0])
        return out

    times = {"a": [], "b": [], "c": []}
    res = {}
    for it in range(warm + reps):
        for key, fn in (("a", run_a), ("b", run_b), ("c", run_c)):
            t0 = time.perf_counter()
            res[key] = fn()   # every call ends in a device synchronise (results copied to the host)
            if it >= warm:
                times[key].append(time.perf_counter() - t0)
    same = all(np.array_equal(x, y) and np.array_equal(x, z) for x, y, z in zip(res["a"], res["b"], res["c"]))
    flop = float(sum(M * float(n) ** 2 + M * M * float(n) + M ** 3 / 3.0 + S * M * M for n in ns))
    arena = b.sample_bytes([M] * G, S, flux)
    med = lambda v: float(np.median(v))  # noqa: E731
    print(f"{label}: G={G} n={min(ns)}..{max(ns)} m={M} S={S}, 30 groups; GPU: {gpu_info()}")
    print(f"  bit-identical (a) = (b) = (c): {same}")
    for key, what in (("a", "batched BatchEngine.sample on the factorised group"),
                      ("b", "per-site Engine.sample_ex on factorised handles"),
                      ("c", "per-site set_train + factorize + sample_ex")):
        v = times[key]
        print(f"  ({key}) {what:52s} median {med(v):.4f} s  [{min(v):.4f}, {max(v):.4f}]")
    print(f"  (b)/(a) = {med(times['b']) / med(times['a']):.2f}, (c)/(a) = {med(times['c']) / med(times['a']):.2f}")
    print(f"  shape-derived flop of (a): {flop / 1e12:.2f} TFLOP -> {flop / med(times['a']) / 1e12:.2f} TFLOP/s FP64; "
          f"sampling arena of (a): {arena / 1e9:.2f} GB ({arena / G / 1e9:.2f} GB per site)", flush=True)
    b.close()
    eng.close()
    for e in engs:
        e.close()


if __name__ == "__main__":
    which = sys.argv[1:] or ["config4"]
    if "config4" in which:
        rng = np.random.default_rng(42)
        probe([int(v) for v in (2000 + 6000 * rng.uniform(size=128)).astype(int)[:16]], 10958, "config-4 first 16")
    if "small" in which:
        probe([1000] * 16, 2000, "16 x 1000")
