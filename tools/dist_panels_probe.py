"""Memory and time of the distributed posterior sampler with panel-slab storage (multisite.sample_sharded).

    python tools/dist_panels_probe.py table                 # (a) per-rank device bytes, replicated layout vs panel slabs
    python tools/dist_panels_probe.py compare OTHER_ROOT    # (b) config-5 sampling call, OTHER_ROOT's package vs this one
    python tools/dist_panels_probe.py run ROOT              #     one such run with ROOT's package (a JSON line)

(a) needs a GPU only for the handle that dgp_dist_arena_bytes asks: per rank, the workspace (dgp_dist_arena_bytes) plus the
caller's buffers (V', the draws' partial sums, the mean, two broadcast buffers); "replicated" restates the workspace of
the layout before panel slabs (an m x m posterior covariance on every rank).
(b) runs the config-5 sampling call of bench.py (n = 32 768, m = 100 000, S = 1000, seed 11, jitter 1e-6, world 1) once per
subprocess, alternating the two package trees twice, and reports the time of the call, the device-memory low-water mark
during it (torch.cuda.mem_get_info, polled) and the SHA-256 of the draws.  OTHER_ROOT holds a discontinuum_b200/ with its
own libdgp.so (capi.library_path() is the package directory).  Card name and power limit are printed with the numbers."""
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N5, M5, S5, SEED5 = 32768, 100000, 1000, 11
TABLE = [(100000, 32768), (140000, 8192), (200000, 8192), (350640, 8192)]
WORLDS = (1, 2, 4, 8)
MAX_COLS, XS, SC_SIZE = 8, 8, 56   # include/dgp.h, csrc/dgp_cov.cuh, csrc/dgp_panel.cuh


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def _pkg(root):
    sys.path.insert(0, root)
    sys.path.insert(1, os.path.join(ROOT, "tests"))
    import discontinuum_b200  # noqa: F401  (before tests/helpers.py puts this repository on the path)
    from discontinuum_b200 import capi, models, multisite, synthetic
    return capi, models, multisite, synthetic


def _r32(x):
    return (x + 31) // 32 * 32


def replicated_workspace(mpad, Spad, nb):
    """doubles the dist_* workspace took when every rank held the m x m posterior covariance"""
    parts = [mpad * MAX_COLS, mpad * XS, mpad, nb * mpad, mpad * mpad, mpad * 128, mpad * 128, Spad * mpad, mpad, SC_SIZE]
    return sum(_r32(p) for p in parts)


def table():
    capi, models, _, synthetic = _pkg(ROOT)
    print(f"card: {card()}")
    print("GB per rank (1e9 B): workspace + caller buffers (V' [world rpr, npad], Od [Spad, mpad], mu, 2 packs [mpad, 512])")
    print("| m | n | replicated, any world | " + " | ".join(f"panels, G = {g}" for g in WORLDS) + " |")
    for m, n in TABLE:
        X, y, nz = synthetic.loadest_site(n, 1000)
        eng = capi.Engine(max_n=n, max_m=128)
        try:
            eng.set_train(models.loadest_spec(2).to_c(), X, y, nz)
            row = []
            rep = None
            for g in WORLDS:
                d = eng.dist_dims(m, S5, g)
                mpad, Spad, npad, rpr = d["mpad"], d["Spad"], d["npad"], d["rows_per_rank"]
                caller = 8 * (rpr * g * npad + Spad * mpad + mpad + 2 * mpad * d["panel_cols"])
                if rep is None:
                    rep = 8 * replicated_workspace(mpad, Spad, npad // 128) + 8 * (mpad * npad + Spad * mpad + mpad + 2 * mpad * 512)
                row.append(max(eng.dist_arena_bytes(m, S5, g, r) for r in range(g)) + caller)
            print(f"| {m} | {n} | {rep / 1e9:.0f} | " + " | ".join(f"{b / 1e9:.0f}" for b in row) + " |")
        finally:
            eng.close()


def run(root):
    capi, models, multisite, synthetic = _pkg(root)
    import numpy as np
    import torch

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import helpers as H

    X, y, nz = synthetic.loadest_site(N5, 1000)
    grid = synthetic.daily_grid(X, M5) + np.array([1e-4, 0.0])
    st = torch.cuda.Stream(device=0)
    torch.cuda.set_stream(st)
    eng = capi.Engine(max_n=N5, max_m=2048, device=0, stream=st.cuda_stream)
    eng.set_train(models.loadest_spec(2).to_c(), X, y, nz)
    _, info = eng.factorize(H.loadest_theta1())
    assert info == 0
    torch.cuda.synchronize()
    low = [torch.cuda.mem_get_info()[0]]
    stop = threading.Event()

    def poll():
        while not stop.is_set():
            low[0] = min(low[0], torch.cuda.mem_get_info()[0])
            time.sleep(0.01)

    th = threading.Thread(target=poll, daemon=True)
    th.start()
    t0 = time.perf_counter()
    draws, info = multisite.sample_sharded(eng, grid, S5, seed=SEED5, jitter=1e-6)
    torch.cuda.synchronize()
    t = time.perf_counter() - t0
    low[0] = min(low[0], torch.cuda.mem_get_info()[0])
    stop.set()
    th.join()
    free, total = torch.cuda.mem_get_info()
    eng.close()
    print(json.dumps(dict(root=root, library=capi.library_path(), seconds=t, info=int(info), peak_used_gb=(total - low[0]) / 1e9,
                          sha256=hashlib.sha256(np.ascontiguousarray(draws).tobytes()).hexdigest())))


def compare(other):
    print(f"card: {card()}", flush=True)
    res = []
    for root in (other, ROOT, other, ROOT):
        p = subprocess.run([sys.executable, os.path.abspath(__file__), "run", os.path.abspath(root)], capture_output=True, text=True)
        if p.returncode != 0:
            sys.stderr.write(p.stdout + p.stderr)
            raise SystemExit(f"run with {root} failed")
        r = json.loads(p.stdout.strip().splitlines()[-1])
        res.append(r)
        print(f"{r['library']}: {r['seconds']:.2f} s, peak {r['peak_used_gb']:.1f} GB, info {r['info']}, sha256 {r['sha256'][:16]}",
              flush=True)
    print("draws equal:", len({r["sha256"] for r in res}) == 1)


if __name__ == "__main__":
    if len(sys.argv) < 2 or sys.argv[1] not in ("table", "compare", "run"):
        raise SystemExit(__doc__)
    {"table": lambda: table(), "compare": lambda: compare(sys.argv[2]), "run": lambda: run(sys.argv[2])}[sys.argv[1]]()
