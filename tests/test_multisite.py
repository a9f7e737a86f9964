"""Site sharding: CPU tests of the assignment and of the final gather with world_size = 2 on gloo, plus a GPU
test that the concurrent multi-site driver reproduces single-site fits."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from discontinuum_b200 import multisite


def test_assign_sites_lpt_balanced_and_complete():
    rng = np.random.default_rng(42)
    ns = (2000 + 6000 * rng.uniform(size=128)).astype(int)  # SURVEY 8d config 4
    costs = [multisite.site_cost(int(n), 100, 10958) for n in ns]
    for world in (1, 2, 4, 8):
        parts = multisite.assign_sites(costs, world)
        flat = sorted(i for p in parts for i in p)
        assert flat == list(range(128))
        loads = [sum(costs[i] for i in p) for p in parts]
        assert max(loads) / (sum(loads) / world) < 1.05
    assert multisite.assign_sites(costs, 4) == multisite.assign_sites(list(costs), 4)  # deterministic


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    costs = [float(c) for c in (9, 7, 5, 4, 3, 1)]
    mine = multisite.assign_sites(costs, world)[rank]
    local = {i: {"theta": np.full(3, float(i)), "rank": rank} for i in mine}
    merged = multisite.gather_results(local, dist)
    if rank == 0:
        assert sorted(merged) == list(range(6))
        assert all(np.array_equal(merged[i]["theta"], np.full(3, float(i))) for i in merged)
        assert {merged[i]["rank"] for i in merged} == {0, 1}
        open(os.path.join(out_dir, "ok"), "w").write("ok")
    else:
        assert merged is None
    dist.barrier()
    dist.destroy_process_group()


def test_gather_results_world2_gloo(tmp_path):
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok").exists()


def test_group_optimizer_matches_torch_adam_clip_and_plateau():
    """GroupOptimizer (vectorised host step of a site group) against the per-site torch objects the reference loop uses:
    clip_grad_norm_(1.0), Adam(lr .05, wd 1e-4) and ReduceLROnPlateau, over enough steps for the scheduler to act."""
    from discontinuum_b200.models import loadest_spec
    from discontinuum_b200.spec import GPModule

    rng = np.random.default_rng(0)
    G, steps = 3, 130
    mods = [GPModule(loadest_spec(2)) for _ in range(G)]
    refs = [GPModule(loadest_spec(2)) for _ in range(G)]
    P = len(mods[0].spec.params)
    opt = multisite.GroupOptimizer(mods, lr=0.05, scheduler=True, patience=60)
    topt = [torch.optim.Adam(m.raw_list(), lr=0.05, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-4, fused=True) for m in refs]
    tsch = [torch.optim.lr_scheduler.ReduceLROnPlateau(o, mode="min", factor=0.7, patience=30, threshold=1e-4,
                                                       threshold_mode="rel", min_lr=1e-6, cooldown=10) for o in topt]
    for t in range(steps):
        g = rng.standard_normal((G, P)) * np.array([0.01, 1.0, 30.0])[:, None]   # below / around / far above the clip norm
        obj = np.array([1.0 / (1 + t), 1.0, 1.0 + 0.5 * np.sin(t)])               # improving / flat (plateau) / noisy
        active = np.array([True, True, t % 7 != 3])                              # site 2 skips some iterations
        nat, dnat, lp, dlp = opt.chain()
        for k in range(G):
            n2, d2, l2, dl2 = refs[k].host_chain()
            assert np.max(np.abs(nat[k] - n2)) <= 1e-13 and np.max(np.abs(dnat[k] - d2)) <= 1e-13
            assert abs(lp[k] - l2) <= 1e-12 * max(1.0, abs(l2)) and np.max(np.abs(dlp[k] - dl2)) <= 1e-12 * max(1.0, np.max(np.abs(dl2)))
        opt.step(g, obj, active)
        for k in range(G):
            if not active[k]:
                continue
            gk = g[k].copy()
            coef = 1.0 / (float(np.sqrt(np.sum(gk * gk))) + 1e-6)
            if not coef >= 1.0:
                gk = gk * coef
            for p, gv in zip(refs[k].raw_list(), gk):
                p.grad = torch.tensor([gv], dtype=torch.float64)
            topt[k].step()
            tsch[k].step(float(obj[k]))
        want = np.array([[float(r.detach()) for r in m.raw_list()] for m in refs])
        assert np.max(np.abs(opt.raw - want)) <= 1e-12, (t, np.max(np.abs(opt.raw - want)))
        assert np.allclose(opt.lr, [o.param_groups[0]["lr"] for o in topt], rtol=0, atol=0)
    assert opt.lr[1] < 0.05 and opt.lr[0] == 0.05  # the flat objective did trigger the plateau scheduler
    opt.push()
    assert all(float(a.detach()) == float(b_) for a, b_ in zip(mods[1].raw_list(), opt.raw[1]))


def test_observed_variance_rule():
    """likelihood(model(x)) in eval mode (SURVEY A.5): + learned noise always, + fixed noise only when m == n, clamp."""
    from discontinuum_b200.models import loadest_spec, rating_spec

    lat = np.array([1e-12, 0.5, 0.2])
    fixed = np.full(3, 0.01)
    th = np.arange(20) * 0.01
    assert np.array_equal(multisite.observed_variance(loadest_spec(2), th, lat, fixed, 3), np.maximum(lat + fixed, 1e-10))
    assert np.array_equal(multisite.observed_variance(loadest_spec(2), th, lat[:2], fixed, 2), np.maximum(lat[:2], 1e-10))
    rs = rating_spec(1.0, 2.0)
    assert np.allclose(multisite.observed_variance(rs, th, lat[:2], fixed, 2), lat[:2] + th[rs.noise_theta])


class _FakeEngine:
    """Stands in for capi.Engine on the CPU: 'predicts' a known function of the inputs."""

    def predict(self, Xs, want_var=True):
        return Xs[:, 0] * 2.0 + Xs[:, 1], (Xs[:, 0] ** 2 if want_var else None)


def _pred_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    Xs = np.stack([np.arange(11.0), np.arange(11.0)[::-1]], axis=1)
    mu, var = multisite.predict_sharded(_FakeEngine(), Xs, dist)
    assert np.array_equal(mu, Xs[:, 0] * 2.0 + Xs[:, 1]) and np.array_equal(var, Xs[:, 0] ** 2)
    mu2, var2 = multisite.predict_sharded(_FakeEngine(), Xs[:1], dist, want_var=False)  # fewer points than ranks
    assert mu2.shape == (1,) and var2 is None
    open(os.path.join(out_dir, f"ok{rank}"), "w").write("ok")
    dist.barrier()
    dist.destroy_process_group()


def test_shard_rows_and_sharded_prediction_world2_gloo(tmp_path):
    assert multisite.shard_rows(10, 4) == [(0, 3), (3, 6), (6, 8), (8, 10)]
    assert multisite.shard_rows(2, 4) == [(0, 1), (1, 2), (2, 2), (2, 2)]
    for m, w in ((100000, 8), (10958, 3), (7, 7)):
        rows = multisite.shard_rows(m, w)
        assert rows[0][0] == 0 and rows[-1][1] == m and all(a[1] == b[0] for a, b in zip(rows, rows[1:]))
    mp.spawn(_pred_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    assert (tmp_path / "ok0").exists() and (tmp_path / "ok1").exists()


@pytest.mark.gpu
def test_concurrent_sites_match_single_site_fits(cuda_device):
    from discontinuum_b200 import synthetic
    import helpers as H
    from helpers import orc

    sites = {i: synthetic.loadest_site(n, 1000 + i)[:2] for i, n in enumerate((300, 450, 700))}
    grid = {i: synthetic.daily_grid(sites[i][0], 200) for i in sites}
    res = multisite.fit_sites(sites, iterations=8, predict=grid, concurrency=3)   # per-handle pipelines (round 1)
    stats = {}
    resb = multisite.fit_sites(sites, iterations=8, predict=grid, group=2, stats=stats)  # batched groups: (700, 450), (300)
    assert sorted(res) == [0, 1, 2] and sorted(resb) == [0, 1, 2]
    assert stats["groups"] == 2 and stats["evals"] == 16 and stats["gpu_eval_ms"] > 0 and stats["lanes"] == 2
    # two groups in flight (default) or one after the other: every site sees the same evaluations
    resb1 = multisite.fit_sites(sites, iterations=8, predict=grid, group=2, lanes=1)
    for i in sites:
        assert resb1[i]["history"] == resb[i]["history"] and np.array_equal(resb1[i]["theta"], resb[i]["theta"])
        assert np.array_equal(resb1[i]["mu"], resb[i]["mu"])
    for i, (X, y) in sites.items():
        raw = orc.loadest_init_raw()
        _, hist = orc.fit_adam("loadest", raw, torch.tensor(X), torch.tensor(y), orc.loadest_noise(X.shape[0]), iterations=8)
        for r in (res, resb):
            assert r[i]["failed"] is None
            assert np.max(np.abs(np.array(r[i]["history"]) - np.array(hist)) / np.abs(hist)) <= 1e-6
            assert r[i]["mu"].shape == (200,) and np.all(r[i]["var"] > 0)
        # the batched groups reproduce the per-handle fits (same evaluations bit for bit, host step equal to rounding)
        assert np.max(np.abs(np.array(resb[i]["history"]) - np.array(res[i]["history"]))) <= 1e-12
        assert np.max(np.abs(resb[i]["theta"] - res[i]["theta"])) <= 1e-11
        assert np.max(np.abs(resb[i]["mu"] - res[i]["mu"])) <= 1e-9


@pytest.mark.gpu
def test_rating_gauges_through_the_batch_driver(cuda_device):
    """Four rating-gp gauges (the per-gauge loop of docs/source/notebooks/rating-gp-demo.ipynb cell 18; model
    rating_gp/models/gpytorch.py:64-79) fitted as one group: objective trajectories equal the oracle's restatement of
    the reference loop with the same random initial draws, per-point noise and per-iteration projection."""
    from discontinuum_b200 import models, synthetic
    from helpers import orc

    ns = (150, 260, 200, 330)
    sites = {i: synthetic.rating_gauge(n, 20 + i) for i, n in enumerate(ns)}
    grids = {i: synthetic.daily_grid(sites[i][0], 120) for i in sites}
    torch.manual_seed(0)
    res = multisite.fit_sites(sites, iterations=8, predict=grids, model="rating", group=4)
    torch.manual_seed(0)
    for i in sorted(sites):
        X, y, noise = sites[i]
        a = float(torch.randn(1)); b = float(torch.randn(1) + 1.3); c = float(torch.rand(1)); u = float(torch.rand(1))
        b_lo, b_hi = models.stage_quantile_bounds(X[:, 1])
        raw = orc.rating_init_raw(b_lo, b_hi, gate_b=b_lo + u * (b_hi - b_lo), pl_a=a, pl_b=b, pl_c=c)
        _, hist = orc.fit_adam("rating", raw, torch.tensor(X), torch.tensor(y), torch.tensor(noise), iterations=8,
                               b_lo=b_lo, b_hi=b_hi, h_min=float(X[:, 1].min()))
        assert res[i]["failed"] is None
        assert np.max(np.abs(np.array(res[i]["history"]) - np.array(hist)) / np.abs(hist)) <= 1e-6
        spec = models.rating_spec(b_lo, b_hi)
        assert np.all(res[i]["var"] >= res[i]["var_latent"] + res[i]["theta"][spec.noise_theta] - 1e-15)
        assert res[i]["mu"].shape == (120,) and np.all(np.isfinite(res[i]["mu"]))


@pytest.mark.gpu
def test_sample_sharded_single_rank_matches_engine_sample(cuda_device):
    """world = 1: the panel-by-panel distributed schedule reproduces dgp_sample (same Philox normals)."""
    import helpers as H
    from discontinuum_b200 import capi, models, synthetic

    n, m, S = 400, 1300, 12
    X, y, noise = synthetic.loadest_site(n, 51)
    Xs = synthetic.daily_grid(X, m) + np.array([0.0009, 0.0])
    eng = capi.Engine(max_n=n, max_m=512)
    eng.set_train(models.loadest_spec(2).to_c(), X, y, noise)
    eng.factorize(H.loadest_theta1())
    want, info = eng.sample_ex(Xs, S, Z=None, seed=99, jitter=1e-7)
    got, info2 = multisite.sample_sharded(eng, Xs, S, dist=None, seed=99, jitter=1e-7)
    assert info == 0 and info2 == 0
    assert np.max(np.abs(got - want)) <= 1e-9 * np.max(np.abs(want))
    eng.close()


def test_panel_owner_cyclic():
    assert [multisite.panel_owner(p, 4) for p in range(6)] == [0, 1, 2, 3, 0, 1]


@pytest.mark.gpu
def test_sample_sharded_two_ranks_match_single_gpu_draws(cuda_device):
    """world = 2 over NCCL (one process per GPU, torchrun): the panel-cyclic distributed draws equal single-GPU dgp_sample_ex
    with the same Philox normals on every rank (tests/dist_sample_check.py).  Needs two visible GPUs; on a one-GPU box the
    same check runs inside `bench.py --gpus N` (extra.config5.check_sharded_vs_single_gpu_draws_rel)."""
    import os
    import subprocess
    import sys

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible GPUs")
    here = os.path.dirname(os.path.abspath(__file__))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29547", os.path.join(here, "dist_sample_check.py"), "900", "2600", "8"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-2000:])
    assert r.stdout.count(" OK") == 2, r.stdout[-2000:]


class _OracleBatch:
    """capi.BatchEngine's surface as fit_sites_local drives it, served by the CPU oracle (loadest sites)."""
    created = 0

    def __init__(self, max_sites, max_n, device=0):
        type(self).created += 1
        self.inflight = None

    def set_train(self, spec_c, sites):
        self.sites = [(torch.tensor(X), torch.tensor(y), torch.tensor(nz)) for X, y, nz in sites]

    def set_timing(self, on):
        pass

    def last_timing(self):
        return [0.0, 0.0, 0.0, 0.0]

    def _eval(self, theta):
        import helpers as H
        from helpers import orc

        G = len(self.sites)
        val, grad, info = np.zeros(G), np.zeros((G, theta.shape[1])), np.zeros(G, dtype=np.int32)
        for k, (X, y, nz) in enumerate(self.sites):
            nat = H.loadest_nat_from_theta(theta[k], X.shape[1])
            with torch.enable_grad():
                v, g, _, _ = orc.nlml_grad_closed_form(orc.loadest_cov, orc.loadest_mean, nat, X, y, nz)
            val[k], grad[k] = float(v), H.loadest_theta_from_nat({n: t.numpy() for n, t in g.items()})
        return val, grad, info

    def nlml_grad_launch(self, theta, jitter=None):
        assert self.inflight is None, "one evaluation in flight per handle"
        self.inflight = np.array(theta)

    def nlml_grad_wait(self):
        theta, self.inflight = self.inflight, None
        return self._eval(theta)

    def nlml_grad(self, theta, jitter=None):
        return self._eval(np.array(theta))

    def close(self):
        pass


@pytest.mark.parametrize("nsites,group", [(5, 2), (4, 16), (1, 16), (7, 3)])
def test_groups_in_flight_schedule_is_result_neutral(monkeypatch, nsites, group):
    """fit_sites_local with 1, 2 or 3 groups in flight (the pairing of large and small groups, a rank whose sites fit one group
    being split, odd group counts, a single site): every site ends with the same history and parameters.  CPU stand-in for the
    batch handle; the same property is checked on the GPU with the real one."""
    from discontinuum_b200 import capi, synthetic

    monkeypatch.setattr(capi, "BatchEngine", _OracleBatch)
    sites = {i: synthetic.loadest_site(24 + 5 * i, 300 + i)[:2] for i in range(nsites)}
    out = {}
    for lanes in (1, 2, 3):
        stats = {}
        _OracleBatch.created = 0
        res = multisite.fit_sites_local(sites, iterations=4, group=group, lanes=lanes, stats=stats)
        assert sorted(res) == list(range(nsites)) and all(r["failed"] is None and len(r["history"]) == 4 for r in res.values())
        assert stats["lanes"] == _OracleBatch.created <= lanes and stats["evals"] == 4 * stats["groups"]
        if nsites >= 2 * lanes:
            assert stats["lanes"] == lanes      # enough sites: no lane stays empty (one group's worth of sites is split)
        out[lanes] = res
    for i in range(nsites):
        for lanes in (2, 3):
            assert out[lanes][i]["history"] == out[1][i]["history"]
            assert np.array_equal(out[lanes][i]["theta"], out[1][i]["theta"])
