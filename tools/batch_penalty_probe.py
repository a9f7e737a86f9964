"""Penalised rating-curve fits of a group of gauges: (a) one RatingGP.fit per gauge in turn (the reference notebook's
per-gauge loop) against (b) multisite.fit_sites on the same model-space data, batched (dgp_batch_* with the batched
posterior-mean adjoint behind the monotonicity penalty).

Default: 16 gauges, n = 200 + 1800 U(0, 1) (seed 42), monotonic_penalty_weight 0.5, grid_size 64, 100 iterations.  Host
clock around work that ends in a device synchronise (every fit returns host results); one warm-up of each path on the first
two gauges.  Prints the card's name and power limit, both wall times, the split of one batched iteration (lanes = 1, one
group of 16) into evaluation / penalty / host step, and, for an early-stopped batched fit, the share of site evaluations
spent on sites that had already stopped or failed (still evaluated with their group)."""
import os
import subprocess
import sys
import time

R = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, R)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from discontinuum_b200 import models, multisite  # noqa: E402

PEN = dict(monotonic_penalty_weight=0.5, grid_size=64)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return name, pl


def raw_gauge(n, seed):
    rng = np.random.default_rng(seed)
    days = np.sort(rng.uniform(0, 3650, n))
    time_ = np.datetime64("2005-01-01") + (days * 86400e9).astype("timedelta64[ns]")
    stage = rng.lognormal(1.0, 0.5, n)
    q = 3.0 * (stage - 0.5 * stage.min()) ** 1.6 * np.exp(0.05 * rng.standard_normal(n))
    gse = rng.choice(np.array([1.02, 1.05, 1.08]), n)
    return {"time": time_, "stage": stage}, q, gse


def per_gauge(gauges, iters, seed0=0):
    out = []
    for i, (cov, q, gse) in enumerate(gauges):
        torch.manual_seed(seed0 + i)
        m = models.RatingGP()
        m.fit(cov, q, target_unc=gse, iterations=iters, **PEN)
        out.append(m)
    return out


def main(G=16, iters=100):
    name, pl = card()
    rng = np.random.default_rng(42)
    ns = (200 + 1800 * rng.uniform(size=G)).astype(int)
    gauges = [raw_gauge(int(n), 100 + k) for k, n in enumerate(ns)]
    print(f"{name}, power limit {pl}; {G} gauges, n = {ns.min()}..{ns.max()}, {iters} iterations, {PEN}", flush=True)
    per_gauge(gauges[:2], 3)                                  # warm-up: module loads, allocations
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fitted = per_gauge(gauges, iters)
    torch.cuda.synchronize()
    ta = time.perf_counter() - t0
    sites = {i: (m.X, m.y, m.fixed_noise) for i, m in enumerate(fitted)}
    multisite.fit_sites({k: sites[k] for k in (0, 1)}, iterations=3, model="rating", **PEN)   # warm-up
    torch.cuda.synchronize()
    torch.manual_seed(0)
    t0 = time.perf_counter()
    res = multisite.fit_sites(sites, iterations=iters, model="rating", **PEN)
    torch.cuda.synchronize()
    tb = time.perf_counter() - t0
    assert all(r["failed"] is None for r in res.values())
    print(f"  (a) per-gauge RatingGP.fit in turn: {ta:.3f} s   ({ta / (G * iters) * 1e3:.3f} ms per gauge-iteration)")
    print(f"  (b) fit_sites batched (lanes 2):    {tb:.3f} s   ({tb / (G * iters) * 1e3:.3f} ms per gauge-iteration)")
    print(f"  (a)/(b) = {ta / tb:.2f}", flush=True)
    st = {}
    torch.manual_seed(0)
    multisite.fit_sites_local(sites, iterations=iters, model="rating", lanes=1, group=G, stats=st, **PEN)
    ev = st["evals"]
    rest = st["fit_wall_s"] - st["penalty_s"] - st["host_step_s"]
    print(f"  one batched iteration of the group (lanes 1, G = {G}, {ev} iterations): evaluation {rest / ev * 1e3:.3f} ms "
          f"(device {st['gpu_eval_ms'] / ev:.3f} ms), penalty {st['penalty_s'] / ev * 1e3:.3f} ms, host step "
          f"{st['host_step_s'] / ev * 1e3:.3f} ms", flush=True)
    st = {}
    torch.manual_seed(0)
    res = multisite.fit_sites_local(sites, iterations=2000, model="rating", early_stopping=True, stats=st, **PEN)
    stops = sorted(r["stopped_at"] for r in res.values() if r["stopped_at"] is not None)
    print(f"  early stopping, 2000 iterations: {len(stops)} of {G} stopped (at {stops[:3]} .. {stops[-3:]}); "
          f"{st['wasted_site_evals']} of {st['site_evals']} site evaluations "
          f"({100.0 * st['wasted_site_evals'] / max(st['site_evals'], 1):.1f} %) spent on stopped or failed sites; "
          f"fit {st['fit_wall_s']:.3f} s", flush=True)


if __name__ == "__main__":
    main(*[int(v) for v in sys.argv[1:3]])
