"""Multi-site batch timing (development aid): S synthetic loadest sites of SURVEY 8d config 4, fit + predict."""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
from discontinuum_b200 import multisite, synthetic

S = int(sys.argv[1]) if len(sys.argv) > 1 else 8
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 100
conc = int(sys.argv[3]) if len(sys.argv) > 3 else 4
m = int(sys.argv[4]) if len(sys.argv) > 4 else 10958
rng = np.random.default_rng(42)
ns = (2000 + 6000 * rng.uniform(size=128)).astype(int)[:S]
sites, grids = {}, {}
for s, n in enumerate(ns):
    X, y, noise = synthetic.loadest_site(int(n), 1000 + s)
    sites[s] = (X, y, noise)
    grids[s] = synthetic.daily_grid(X, m)
t0 = time.perf_counter()
res = multisite.fit_sites_local(sites, iterations=iters, device=0, concurrency=conc, predict=grids)
dt = time.perf_counter() - t0
flop = sum(float(n) ** 3 * iters for n in ns)
print(f"sites={S} iters={iters} conc={conc} m={m} n=[{ns.min()}..{ns.max()}] wall={dt:.2f}s sites/s={S/dt:.3f} "
      f"fit TF/s={flop/dt/1e12:.2f} failed={[k for k, r in res.items() if r['failed']]}", flush=True)
print("final objectives:", [round(res[k]["objective"], 5) for k in sorted(res)][:8])

if os.environ.get("PHASES"):
    # per-phase device time of every evaluation under contention (events on each site's stream)
    acc = {}
    o0 = multisite._open_site
    def o1(*a, **k):
        st = o0(*a, **k); st.engine.set_timing(True); return st
    multisite._open_site = o1
    f0 = multisite._finish_step
    def f1(st):
        f0(st)
        ms = st.engine.last_timing()
        a = acc.setdefault(st.X.shape[0], [0, 0.0, 0.0, 0.0])
        a[0] += 1; a[1] += ms[0]; a[2] += ms[1]; a[3] += ms[2]
    multisite._finish_step = f1
    t0 = time.perf_counter()
    multisite.fit_sites_local(sites, iterations=iters, device=0, concurrency=conc, predict=grids)
    print("phases run total", round(time.perf_counter() - t0, 2))
    for n in sorted(acc):
        c, a, b, d = acc[n]
        print(f"  n={n}: per evaluation potrf {a/c:.2f} ms  trtri {b/c:.2f} ms  lauum+grad {d/c:.2f} ms  sum {(a+b+d)/c:.2f}  ({n**3/((a+b+d)/c)/1e9:.1f} TF if alone)")

if os.environ.get("BREAKDOWN"):
    import collections
    acc = collections.defaultdict(float)
    def wrap(name):
        f = getattr(multisite, name)
        def g(*a, **k):
            t = time.perf_counter(); r = f(*a, **k); acc[name] += time.perf_counter() - t; return r
        setattr(multisite, name, g)
    for nm in ("_open_site", "_launch_step", "_finish_step", "_close_site"):
        wrap(nm)
    from discontinuum_b200 import capi
    w0 = capi.Engine.nlml_grad_wait
    def w1(self):
        t = time.perf_counter(); r = w0(self); acc["wait"] += time.perf_counter() - t; return r
    capi.Engine.nlml_grad_wait = w1
    t0 = time.perf_counter()
    multisite.fit_sites_local(sites, iterations=iters, device=0, concurrency=conc, predict=grids)
    print("breakdown total", round(time.perf_counter() - t0, 2), {k: round(v, 2) for k, v in acc.items()})
