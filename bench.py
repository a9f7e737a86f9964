"""bench.py -- NLML + hyper-parameter-gradient evaluations per second at n = 16 384 (BASELINE.json metric,
configs[2]: "loadest-gp large single site n=16k, FP64 Cholesky + hyperparameter gradient, 1xB200").

A step = one evaluation of {NLML, dNLML/dtheta} of the loadest-gp model on one synthetic river-like site.
  value   : evaluations/s with the training set already resident in HBM (set_train done before timing),
            timed with CUDA events on the stream the engine launches on.
  e2e     : the same through the C ABI with HOST buffers every step: dgp_set_train(host X, y, noise)
            + dgp_nlml_grad(host theta -> host nlml, grad).
  N > 1   : one process per GPU, every rank evaluates its own site (sites are independent: no data-path
            collective, "weak" scaling); value = total evaluations / max-over-ranks time.
  extra   : the other legs of the BASELINE metric, under the same clock --
            sites   : BASELINE config 4, the FIXED 128-site NWQN-style batch (n = 2000..8000, 100 Adam iterations + daily
                      grid each) sharded over the N ranks (strong scaling), batched multi-site evaluation per rank;
            config5 : BASELINE config 5, ONE site (n = 32 768) replicated on every rank: posterior mean + variance on a
                      100 000-point daily grid sharded by rows (multisite.predict_sharded) and 1 000 joint posterior draws
                      with the posterior-covariance Cholesky distributed panel-cyclically (multisite.sample_sharded).
  --impl reference : the reference's CPU path restated by the oracle (dense covariance build, torch.linalg.cholesky,
            autograd backward -- what discontinuum/engines/gpytorch.py:353,384 executes), float64, every host thread,
            MEASURED at n = 16 384 itself (one timed evaluation) with n = 4096 / 8192 alongside.
  --dump-outputs DIR : after the timed steps, rank 0 writes what the last timed step returned (DIR/nlml.npy, DIR/grad.npy,
            float64).  The inputs depend only on the arguments, so two builds can be compared output for output.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

N_TRAIN = 16384
METRIC = "nlml_grad_evals_per_sec_n16k"
UNIT = "evals/s"
DMMA_PIPE_TFLOPS = 37.2  # FP64 tensor-pipe rate implied by ncu (36.46 Tflop/s at 98.0 % pipe-active, profiles/ncu_lauum_n16384_r01d.txt)


class ClockSampler:
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.QUERY}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            for k, nm in enumerate(names):
                if len(r) > 3 + k and r[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def fp64_peak_live(local: int):
    """FP64 roofline denominator, measured in this run (MEASURED_PEAKS.json has no FP64 entry): cuBLAS DGEMM 8192^3
    through torch.matmul -- best of 8 single launches ("burst") and back to back for ~1.5 s ("sustained"), with the SM
    clock sampled meanwhile.  A library GEMM used as a yardstick only; nothing on the measured path calls it."""
    import torch

    dev = torch.device("cuda", local)
    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device=dev)
    b = torch.randn(n, n, dtype=torch.float64, device=dev)
    c = torch.empty(n, n, dtype=torch.float64, device=dev)
    flop = 2.0 * n ** 3
    for _ in range(2):
        torch.matmul(a, b, out=c)
    torch.cuda.synchronize(dev)
    sampler = ClockSampler(local)
    sampler.start()
    best = 1e30
    for _ in range(8):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b, out=c)
        e1.record()
        torch.cuda.synchronize(dev)
        best = min(best, e0.elapsed_time(e1))
    reps = max(4, int(1500.0 / best))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        torch.matmul(a, b, out=c)
    e1.record()
    torch.cuda.synchronize(dev)
    sus = e0.elapsed_time(e1) / reps
    clocks = sampler.stop()
    del a, b, c
    torch.cuda.empty_cache()
    return {"burst_tflops": flop / best / 1e9, "sustained_tflops": flop / sus / 1e9, "clocks": clocks,
            "how": f"torch.matmul float64 {n}^3 (cuBLAS DGEMM): best of 8 / mean of {reps} back to back, CUDA events"}


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """One float64 DIR/<name>.npy per array."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(a, dtype=np.float64))


def cpu_eval(n: int, mode: str = "autograd"):
    """One oracle NLML+grad evaluation at size n on the host: dense covariance build + torch.linalg.cholesky + backward.
    mode "autograd": autograd straight through the Cholesky factorisation (what the reference's objective.backward()
    does, discontinuum/engines/gpytorch.py:384); "closed_form": the trace identity on an explicit inverse."""
    import torch

    import helpers as H
    from discontinuum_b200 import synthetic
    from oracle import gp_oracle as orc

    X, y, noise = synthetic.loadest_site(n, 1000)
    Xt, yt, nt = torch.tensor(X), torch.tensor(y), torch.tensor(noise)
    nat = H.loadest_nat_from_theta(H.loadest_theta1())
    t0 = time.perf_counter()
    if mode == "autograd":
        v, _ = orc.nlml_grad_autograd(orc.loadest_cov, orc.loadest_mean, nat, Xt, yt, nt)
    else:
        v = orc.nlml_grad_closed_form(orc.loadest_cov, orc.loadest_mean, nat, Xt, yt, nt)[0]
    return time.perf_counter() - t0, float(v)


def cpu_arm(n_full: int, small=(4096, 8192)):
    """Measured points of the CPU arm: the small sizes (also the warm-up of torch's thread pool), then ONE timed
    evaluation at the full size if the host has the memory for it (the autograd graph of the dense covariance holds
    ~70 GB at n = 16 384).  Returns (seconds at n_full or None, {n: seconds}, threads, note)."""
    import psutil
    import torch

    torch.set_num_threads(os.cpu_count() or 1)
    cpu_eval(1024)
    pts = {}
    for ns in small:
        if ns < n_full:
            pts[ns] = cpu_eval(ns)[0]
    need_gb = 5.0 * (n_full / 4096.0) ** 2 * 1.25
    avail = psutil.virtual_memory().available / 1e9
    note = ""
    full = None
    if avail > need_gb + 8:
        full = cpu_eval(n_full)[0]
    else:
        note = f"host has {avail:.0f} GB available, the autograd graph at n={n_full} needs ~{need_gb:.0f} GB: "
    return full, pts, torch.get_num_threads(), note


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.n
    full, pts, threads, note = cpu_arm(n)
    measured = full is not None
    if not measured:   # not enough host memory for the full size: closed-form (no n x n autograd graph), still measured at n
        import torch

        full = cpu_eval(n, "closed_form")[0]
        note += "closed-form gradient (explicit inverse) timed instead of autograd"
    value = 1.0 / full
    pts_s = ", ".join(f"n={k}: {v:.2f} s" for k, v in pts.items())
    sample = (f"oracle NLML+grad (dense K build + torch.linalg.cholesky + autograd backward) MEASURED at n={n}: {full:.1f} s for one "
              f"evaluation on {threads} torch threads (1 timed evaluation whatever --steps says; smaller sizes for the exponent: {pts_s}). {note}")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": full * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "timed_evaluations": 1,
            "config": {"workload": f"loadest-gp single site n={n}, NLML + gradient (10 hyper-parameters)"},
            "measured_points_s": {str(k): v for k, v in list(pts.items()) + [(n, full)]},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--n", type=int, default=N_TRAIN, help="development only; the judged workload is n=16384")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (development)")
    ap.add_argument("--no-extra", action="store_true", help="skip the sites/s and config-5 legs (development)")
    ap.add_argument("--sites", type=int, default=128, help="sites of the NWQN-style batch (BASELINE config 4: 128), sharded over the ranks")
    ap.add_argument("--site-iterations", type=int, default=100)
    ap.add_argument("--site-group", type=int, default=16, help="sites per batched launch sequence")
    ap.add_argument("--site-lanes", type=int, default=2, help="groups in flight per GPU (each on its own batch handle)")
    ap.add_argument("--c5-n", type=int, default=32768)
    ap.add_argument("--c5-m", type=int, default=100000)
    ap.add_argument("--c5-draws", type=int, default=1000)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the NLML and gradient of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path only")
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch

    import helpers as H
    from discontinuum_b200 import capi, models, multisite, synthetic

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a B200; there is no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    # torchrun exports OMP_NUM_THREADS=1; the host steps are numpy / tiny torch ops: a couple of threads per rank is plenty
    torch.set_num_threads(max(1, min(4, (os.cpu_count() or 8) // max(world, 1))))
    dist = None
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # keep NCCL's banner off stdout: rank 0 prints ONE JSON line
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    n = args.n
    warm = max(args.warmup, 3)
    X, y, noise = synthetic.loadest_site(n, 1000 + rank)
    spec = models.loadest_spec(2)
    work_stream = torch.cuda.Stream(device=local)  # the engine launches on this stream; the events below are recorded on it
    torch.cuda.set_stream(work_stream)
    eng = capi.Engine(max_n=n, max_m=2048, device=local, stream=work_stream.cuda_stream)
    eng.set_train(spec.to_c(), X, y, noise)
    base = H.loadest_theta1()
    thetas = [base * (1.0 + 1e-3 * k) for k in range(warm + args.steps)]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: inputs resident in HBM
    for k in range(warm):
        eng.nlml_grad(thetas[k])
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    l0 = eng.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    infos = []
    for k in range(args.steps):
        val, grad, info = eng.nlml_grad(thetas[warm + k])
        infos.append(info)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = eng.launches - l0
    clocks = sampler.stop()
    if any(infos) or not np.isfinite(val):
        raise RuntimeError(f"factorisation failed inside the timed region: info={infos} nlml={val}")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"nlml": np.array([val]), "grad": grad})

    # ---- phase split of one evaluation (CUDA events on the launching stream inside libdgp)
    eng.set_timing(True)
    eng.nlml_grad(base)
    phase = eng.last_timing()
    eng.set_timing(False)

    # ---- e2e: host buffers through the C ABI every step
    Xh, yh, nh = np.ascontiguousarray(X), np.ascontiguousarray(y), np.ascontiguousarray(noise)
    c_spec = spec.to_c()
    for k in range(2):
        eng.set_train(c_spec, Xh, yh, nh)
        eng.nlml_grad(thetas[k])
    barrier()
    t0 = time.perf_counter()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for k in range(args.steps):
        eng.set_train(c_spec, Xh, yh, nh)
        val2, grad2, info2 = eng.nlml_grad(thetas[warm + k])
    e3.record()
    barrier()
    ms_e2e = max(e2.elapsed_time(e3), (time.perf_counter() - t0) * 1e3)
    eng.close()
    eng = None

    extra = None
    if not args.no_extra:
        extra = {}
        # ================= sites/s: BASELINE config 4, the fixed 128-site batch sharded over the ranks (strong scaling)
        rng = np.random.default_rng(42)
        ns_all = (2000 + 6000 * rng.uniform(size=128)).astype(int)   # SURVEY 8d config 4 sizes
        keys = list(range(min(args.sites, 128)))
        costs = [multisite.site_cost(int(ns_all[k]), args.site_iterations, 10958) for k in keys]
        mine = [keys[i] for i in multisite.assign_sites(costs, world)[rank]]   # the driver's own LPT assignment
        sites = {k: synthetic.loadest_site(int(ns_all[k]), 1000 + k) for k in mine}
        grids = {k: synthetic.daily_grid(sites[k][0], 10958) for k in mine}
        multisite.fit_sites_local({999: synthetic.loadest_site(512, 7), 998: synthetic.loadest_site(300, 8)}, iterations=3,
                                  device=local, group=2)   # warm-up: kernels loaded, pinned buffers touched
        multisite.gather_results({-1 - rank: {"warm": True}}, dist)   # ... and the gather's point-to-point channels connected
        barrier()
        stats = {}
        t0 = time.perf_counter()
        res = multisite.fit_sites_local(sites, iterations=args.site_iterations, device=local, group=args.site_group,
                                        predict=grids, stats=stats, lanes=args.site_lanes)
        t_local = time.perf_counter() - t0
        summary = {k: {"theta": r["theta"], "objective": r["objective"], "failed": r["failed"]} for k, r in res.items()}
        merged = multisite.gather_results(summary, dist)   # the only collective: final gather on rank 0
        torch.cuda.synchronize()
        t_sites = time.perf_counter() - t0
        bad = [k for k, r in res.items() if r["failed"] is not None or not np.all(np.isfinite(r["mu"]))]
        if bad or (rank == 0 and sorted(merged) != keys):
            raise RuntimeError(f"site fits failed: {bad}")
        flop_local = float(sum(float(ns_all[k]) ** 3 * args.site_iterations for k in mine))
        per_rank = torch.tensor([t_local, stats["fit_wall_s"], stats["predict_s"], stats["host_step_s"], flop_local, float(len(mine))],
                                dtype=torch.float64, device="cuda")
        all_ranks = [torch.zeros_like(per_rank) for _ in range(world)]
        if dist is not None:
            dist.all_gather(all_ranks, per_rank)
        else:
            all_ranks = [per_rank]
        tt = torch.tensor([t_sites], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        t_sites_max = float(tt[0])
        rows = [[float(v) for v in r.tolist()] for r in all_ranks]
        flop_total = sum(r[4] for r in rows)
        extra["sites"] = {
            "metric": "sites_per_sec", "value": len(keys) / t_sites_max, "unit": "sites/s", "sites": len(keys), "scaling": "strong",
            "iterations": args.site_iterations, "predict_grid": 10958, "group": args.site_group, "lanes": args.site_lanes,
            "fit_tflops": flop_total / t_sites_max / 1e12, "fit_tflops_per_gpu": flop_total / t_sites_max / 1e12 / world,
            "n_range": {"n_min": int(ns_all[keys].min()), "n_max": int(ns_all[keys].max())},
            "per_rank": [{"sites": int(r[5]), "wall_s": r[0], "fit_loop_s": r[1], "other_s": r[0] - r[1] - r[2],
                          "predict_s": r[2], "host_step_s": r[3], "fit_tflops_in_fit_loop": (r[4] / r[1] / 1e12) if r[1] > 0 else None}
                         for r in rows],
            "what": "BASELINE config 4: the fixed 128-site NWQN-style batch (SURVEY 8d sizes, n = 2000 + 6000 u, seed 42), fit (100 Adam "
                    "iterations) + daily-grid prediction per site, host arrays in / host results out, sites assigned to ranks by cost (LPT), "
                    "groups of sites evaluated by one batched launch sequence per iteration (dgp_batch_nlml_grad), one final gather; "
                    "time = max over ranks incl. the gather; gpu_busy_s = device time of the batched evaluations (CUDA events)"}
        del sites, grids, res
        # ================= config 5: one site replicated on every rank, grid sharded, joint draws distributed
        n5, m5, S5 = args.c5_n, args.c5_m, args.c5_draws
        X5, y5, nz5 = synthetic.loadest_site(n5, 1000)   # the SAME site on every rank
        grid5 = synthetic.daily_grid(X5, m5) + np.array([1e-4, 0.0])
        torch.cuda.set_stream(work_stream)
        eng5 = capi.Engine(max_n=n5, max_m=2048, device=local, stream=work_stream.cuda_stream)
        eng5.set_train(spec.to_c(), X5, y5, nz5)
        barrier()
        t0 = time.perf_counter()
        _, info5 = eng5.factorize(base)
        torch.cuda.synchronize()
        t_fact = time.perf_counter() - t0
        if info5 != 0:
            raise RuntimeError(f"config 5 factorisation failed: info={info5}")
        # built-in check: the distributed draws equal the single-GPU dgp_sample_ex draws (same Philox stream)
        mc, Sc = 3000, 48
        want, iw = eng5.sample_ex(grid5[:mc], Sc, Z=None, seed=5, jitter=1e-6)
        got, ig = multisite.sample_sharded(eng5, grid5[:mc], Sc, dist=dist, seed=5, jitter=1e-6)
        check = float(np.max(np.abs(got - want)) / np.max(np.abs(want)))
        if iw != 0 or ig != 0 or not check <= 1e-9:
            raise RuntimeError(f"sharded draws differ from the single-GPU draws: rel {check:g}, info {iw} {ig}")
        del want, got
        barrier()
        t0 = time.perf_counter()
        mu5, var5 = multisite.predict_sharded(eng5, grid5, dist)          # every rank gets the whole mean / variance
        torch.cuda.synchronize()
        tp = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(tp, op=dist.ReduceOp.MAX)
        if not (np.all(np.isfinite(mu5)) and np.all(var5 > -1e-8)):
            raise RuntimeError("config 5 prediction produced invalid output")
        barrier()
        cstats = {}
        t0 = time.perf_counter()
        draws, info_s = multisite.sample_sharded(eng5, grid5, S5, dist=dist, seed=11, jitter=1e-6, stats=cstats)
        torch.cuda.synchronize()
        ts = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(ts, op=dist.ReduceOp.MAX)
        if info_s != 0 or not np.all(np.isfinite(draws)):
            raise RuntimeError(f"config 5 sampling failed: info={info_s}")
        sd = draws.std(axis=0)
        ratio = float(np.median(sd / np.sqrt(np.maximum(var5, 1e-12))))
        del draws
        eng5.close()
        t_pred, t_samp = float(tp[0]), float(ts[0])
        extra["config5"] = {
            "n_train": n5, "m_grid": m5, "draws": S5, "factorize_s": t_fact,
            "predict": {"metric": "predictive_points_per_sec", "value": m5 / t_pred, "unit": "points/s", "seconds": t_pred,
                        "tflops": float(m5) * float(n5) ** 2 / t_pred / 1e12,
                        "what": "posterior mean + latent variance of ONE site on the 100 000-point grid, rows sharded over the ranks "
                                "(multisite.predict_sharded: host grid in, all_gather of 16 m bytes, host mean/variance out on every rank)",
                        "all_gather_bytes": 16 * m5 if world > 1 else 0},
            "sample": {"metric": "joint_posterior_draws", "seconds": t_samp, "draws_per_sec": S5 / t_samp,
                       "tflops": (float(m5) ** 2 * n5 + float(m5) ** 3 / 3 + float(m5) * n5 ** 2 + 2.0 * float(m5) ** 2 * S5) / t_samp / 1e12,
                       "sd_over_sqrt_var_median": ratio, "collectives": cstats,
                       "what": "exact joint draws [S, m]: panel-cyclic Cholesky of the m x m posterior covariance over the ranks "
                               "(multisite.sample_sharded, NCCL all_gather / broadcast per panel / all_reduce), host draws out"},
            "check_sharded_vs_single_gpu_draws_rel": check}

    t = torch.tensor([ms, ms_e2e], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max, ms_e2e_max = float(t[0]), float(t[1])
    value = world * args.steps / (ms_max * 1e-3)
    e2e_value = world * args.steps / (ms_e2e_max * 1e-3)

    if rank == 0:
        peak = fp64_peak_live(local)
        flop = float(n) ** 3  # SURVEY 8d: n^3/3 POTRF + n^3/3 triangular inverse + n^3/3 LAUUM
        dev_ms = sum(phase)
        achieved = flop / (dev_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "achieved": achieved, "peak": peak["burst_tflops"], "unit": "TFLOP/s",
                "frac": achieved / peak["burst_tflops"],
                "peak_sustained": peak["sustained_tflops"], "frac_of_sustained": achieved / peak["sustained_tflops"],
                "dmma_pipe_peak": DMMA_PIPE_TFLOPS, "frac_of_dmma_pipe": achieved / DMMA_PIPE_TFLOPS,
                "peak_source": "measured in this run (MEASURED_PEAKS.json has no FP64 entry, B200_PROFILING.md states no FP64 fallback): "
                               + peak["how"] + "; dmma_pipe_peak = tensor-pipe rate implied by ncu (profiles/ncu_lauum_n16384_r01d.txt)",
                "peak_clocks": peak["clocks"],
                "traffic": 62.7e9 if n == N_TRAIN else None,
                "traffic_note": "dram__bytes_read+write summed over the launches of one evaluation (ncu, profiles/dram_n16384_r02d_summary.txt; working set 3 n^2 x 8 B = 6.4 GB, operand panels re-read through L2)",
                "kernel": "dgp::k_gemm (FP64 DMMA tile engine): every launch of one evaluation",
                "algorithmic_flop_per_eval": flop,
                "phases_ms": {"potrf": phase[0], "trtri": phase[1], "lauum_grad": phase[2], "rest": phase[3]},
                "phases_tflops": {"potrf": flop / 3 / phase[0] / 1e9, "trtri": flop / 3 / phase[1] / 1e9,
                                  "lauum_grad_single_launch": flop / 3 / phase[2] / 1e9}}
        cpu = None
        if not args.no_cpu:
            full, pts, threads, note = cpu_arm(n, small=(4096,))
            if full is not None:
                cpu = {"value": 1.0 / full, "unit": UNIT, "cores": threads, "kind": "port",
                       "sample": f"oracle NLML+grad (dense K build + torch.linalg.cholesky + autograd backward) MEASURED at n={n}: one "
                                 f"evaluation, {full:.1f} s on {threads} torch threads (n=4096: {pts.get(4096, float('nan')):.2f} s)"}
            else:
                s8 = cpu_eval(8192)[0]
                cpu = {"value": 1.0 / (s8 * (n / 8192.0) ** 3), "unit": UNIT, "cores": threads, "kind": "port", "extrapolated": True,
                       "sample": note + f"n=8192 measured ({s8:.1f} s), scaled by (n/8192)^3"}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
                "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": f"loadest-gp single site n={n}, NLML + gradient (10 hyper-parameters), one site per GPU",
                           "l2": "working set 3 x n^2 x 8 B = 6.4 GB per site, far larger than the 126 MB L2 (no flush needed)",
                           "parallelism": f"independent sites x{world}"},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(n * (2 + 2) * 8 + 10 * 8),
                        "d2h_bytes_per_step": int((1 + 10) * 8)},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "cpu_baseline": cpu,
                "nlml": val, "extra": extra}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
