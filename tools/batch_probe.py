"""Phase split (factorisation / inverse / LAUUM + gradient) of batched evaluations for a few group compositions."""
import os, sys, time
R = os.path.dirname(os.path.dirname(os.path.abspath(__file__))); sys.path.insert(0, R); sys.path.insert(0, os.path.join(R, "tests"))
import numpy as np
import helpers as H
from discontinuum_b200 import capi, models, synthetic

spec = models.loadest_spec(2)
th = H.loadest_theta1()

def run(ns, label, reps=3):
    sites = [synthetic.loadest_site(n, 2000 + k) for k, n in enumerate(ns)]
    b = capi.BatchEngine(max_sites=len(ns), max_n=max(ns))
    b.set_train(spec.to_c(), sites)
    thetas = np.stack([th] * len(ns))
    b.nlml_grad(thetas)
    b.set_timing(True)
    ph = np.zeros(4); wall = 0.0
    l0 = b.launches
    for _ in range(reps):
        t0 = time.perf_counter(); v, g, info = b.nlml_grad(thetas); wall += time.perf_counter() - t0
        ph += np.array(b.last_timing())
    assert not info.any()
    ph /= reps; wall /= reps
    fl = sum(float(n) ** 3 for n in ns)
    print(f"{label:34s} G={len(ns):2d} launches={(b.launches - l0) // reps:4d} wall {wall * 1e3:8.2f} ms  dev {ph.sum():8.2f} ms = {fl / ph.sum() / 1e9:5.1f} TF | "
          f"potrf {ph[0]:7.2f} ({fl / 3 / ph[0] / 1e9:5.1f}) trtri {ph[1]:7.2f} ({fl / 3 / ph[1] / 1e9:5.1f}) lauum+grad {ph[2]:7.2f} ({fl / 3 / ph[2] / 1e9:5.1f}) rest {ph[3]:.2f}", flush=True)
    b.close()

rng = np.random.default_rng(42)
ns_all = np.sort((2000 + 6000 * rng.uniform(size=128)).astype(int))[::-1]
which = sys.argv[1:] or ["all"]
if "all" in which or "uniform" in which:
    run([7680] * 1, "1 x 7680")
    run([7680] * 4, "4 x 7680")
    run([7680] * 16, "16 x 7680")
    run([4096] * 16, "16 x 4096")
    run([2048] * 16, "16 x 2048")
    run([2048] * 32, "32 x 2048")
    run([1000] * 32, "32 x 1000")
if "all" in which or "config4" in which:
    for g in range(0, 128, 16):
        run([int(v) for v in ns_all[g:g + 16]], f"config-4 group {g // 16} ({ns_all[g]}..{ns_all[g + 15]})")
    run([int(v) for v in ns_all[:32]], "config-4 32 largest")
    run([int(v) for v in ns_all[::8]], "config-4 every 8th (mixed)")
if "rule" in which:   # groups just below (FP64 DMMA LAUUM) and at (INT8 LAUUM, one site at a time) the 8192-point size rule
    for g in (1, 4, 8):
        run([8064] * g, f"{g} x 8064")
        run([8192] * g, f"{g} x 8192")
if "single" in which:
    for n in (2048, 4096, 7680, 8192, 16384):
        run([n], f"1 x {n}")
