"""Joint posterior draws over a grid sharded across 2 ... 8 ranks (multisite.sample_sharded + the dgp_dist_* entry points),
emulated in one process on one GPU.

NCCL cannot put two ranks on one GPU, but sample_sharded takes its collectives from the `dist` object it is passed.
FakeDist below is that object for one rank of an in-process group: one Python thread per rank, each with its own
capi.Engine on device 0, each calling the unchanged sample_sharded.  Every collective
  synchronises the device, deposits this rank's tensor, waits for all ranks, computes the result from all ranks' tensors
  in rank order into a temporary, synchronises, waits again, writes this rank's own tensor and synchronises,
so every rank gets bit-identical results and the order of kernels and collectives is what is tested; stream-event races
under real NCCL are not (tests/dist_sample_check.py on two GPUs and bench.py keep that).  The barrier times out, the first
exception on any rank aborts it, and a rank whose collective differs from the others' (name, shape, dtype, source, op)
fails all of them, so a protocol mismatch fails the test instead of hanging it.

What only the distributed path reaches, and the case that reaches it (PANEL_BLOCKS = 4 block columns of 128 per panel,
panel p owned by rank p mod world, rank r's V' shard rows [r rpr, (r + 1) rpr), rpr = ceil(mb / world) 128):
  * M_ZL tile mode, the per-panel partial draws Z[:, K] L[c, K]' (dgp_dist_draws_partial): every case; the factor check
    (Z = [I; 0], draws = [Lpost'; 0]) sees it read above the diagonal or leave a diagonal block unzeroed
  * M_TRAIL_COL with INIT_COV over one panel's columns (dgp_dist_sigma): every case, ragged last panels at m = 1300, 600, 5200
  * k_pack_panel, pack on the owner and unpack (dir = 1) on the others: every case with world > 1 and more than one panel
  * dgp_dist_trail over the panels a rank owns, and the look-ahead order of sample_sharded (trail(p, p+1, p+1) first, the
    next panel factored and broadcast on a side stream): "shared" mode, where the engine runs on the thread's current stream
  * shards that start past mpad (world 3 / m 100, world 4 / m 600, world 8 / m 5200), ranks that own no panel
  * the MIN all-reduce of info: a duplicated grid point in a panel of rank 1 under a negative jitter
"""
import threading
import time

import numpy as np
import pytest
import torch

import helpers as H
from helpers import orc
from discontinuum_b200 import capi, models, multisite, synthetic
from test_factor_schedule import EPS, _free, _n1

PANEL_BLOCKS = 4             # csrc/dgp_api.cu
N_TRAIN = 800
JITTER = 1e-6                # what bench.py samples with
DRAW_REL = 1e-9              # sharded vs single-GPU draws, relative to max |draw| (bench.py, dist_sample_check.py)
RATIO_MAX = 1.0
SHIFT = np.array([0.0004, 0.01])
DEV = "cuda"
BARRIER_TIMEOUT = 120.0


# ------------------------------------------------------------------------------------------------------------------
# torch.distributed, emulated by threads of one process
# ------------------------------------------------------------------------------------------------------------------
class ReduceOp:
    SUM = "sum"
    MIN = "min"


class _Done:
    """what an async collective returns: the fake has finished by the time it returns"""

    def wait(self):
        return True


class FakeGroup:
    """State shared by the ranks of one emulated process group."""

    def __init__(self, world, timeout=BARRIER_TIMEOUT):
        self.world = world
        self.barrier = threading.Barrier(world, timeout=timeout)
        self.slots = [None] * world
        self.sigs = [None] * world
        self.logs = [[] for _ in range(world)]

    def rank(self, r):
        return FakeDist(self, r)

    def abort(self):
        self.barrier.abort()


class FakeDist:
    """The torch.distributed surface sample_sharded uses, for rank `rank` of `group`."""
    ReduceOp = ReduceOp

    def __init__(self, group, rank):
        self.group, self.r = group, rank

    def is_initialized(self):
        return True

    def get_world_size(self):
        return self.group.world

    def get_rank(self):
        return self.r

    @staticmethod
    def _sync(t):
        if t.is_cuda:
            torch.cuda.synchronize(t.device)

    def _collective(self, name, mine, out, src, op, combine):
        g, r = self.group, self.r
        sig = (name, tuple(mine.shape), str(mine.dtype), src, op)
        g.logs[r].append(sig)
        self._sync(mine)
        g.slots[r], g.sigs[r] = mine, sig
        g.barrier.wait()
        if any(s != g.sigs[0] for s in g.sigs):
            raise RuntimeError(f"rank {r}: ranks issued different collectives: {g.sigs}")
        res = combine(list(g.slots))
        self._sync(res)
        g.barrier.wait()
        out.copy_(res)
        self._sync(out)

    def all_gather_into_tensor(self, output, input):
        if output.numel() != self.group.world * input.numel():
            raise RuntimeError("all_gather_into_tensor: output must hold world x input")
        self._collective("all_gather_into_tensor", input, output, None, None,
                         lambda ts: torch.cat([t.reshape(-1) for t in ts]).reshape(output.shape))

    def all_reduce(self, tensor, op=ReduceOp.SUM):
        if op == ReduceOp.SUM:
            combine = lambda ts: torch.stack(ts).sum(0)     # noqa: E731  (rank order: the same sum on every rank)
        elif op == ReduceOp.MIN:
            combine = lambda ts: torch.stack(ts).amin(0)    # noqa: E731
        else:
            raise ValueError(f"all_reduce: op {op} is not emulated")
        self._collective("all_reduce", tensor, tensor, None, op, combine)

    def broadcast(self, tensor, src, async_op=False):
        self._collective("broadcast", tensor, tensor, int(src), None, lambda ts: ts[src].clone())
        return _Done() if async_op else None


def run_ranks(world, fn, timeout=BARRIER_TIMEOUT):
    """fn(dist) on `world` threads, one per rank -> ([result of rank r], [collective log of rank r]).  The first exception
    on any thread aborts the group's barrier; the first one that is not the resulting BrokenBarrierError is raised."""
    group = FakeGroup(world, timeout)
    results, errors = [None] * world, [None] * world

    def body(r):
        try:
            results[r] = fn(group.rank(r))
        except BaseException as e:  # noqa: BLE001  (re-raised on the calling thread)
            errors[r] = e
            group.abort()

    threads = [threading.Thread(target=body, args=(r,), daemon=True) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout=10 * timeout)
    assert not any(t.is_alive() for t in threads), "a rank did not finish"
    errs = [e for e in errors if e is not None]
    if errs:
        raise next((e for e in errs if not isinstance(e, threading.BrokenBarrierError)), errs[0])
    return results, group.logs


def test_fake_collectives_match_torch_distributed():
    """CPU: with 3 ranks, all_gather_into_tensor concatenates in rank order, all_reduce SUM / MIN reduce elementwise,
    broadcast (blocking and async) copies the source rank's tensor; the logs of all ranks agree."""
    world = 3

    def fn(d):
        r = d.get_rank()
        assert d.is_initialized() and d.get_world_size() == world
        x = torch.arange(4, dtype=torch.float64) + 10.0 * r
        gat = torch.empty(world * 4, dtype=torch.float64)
        d.all_gather_into_tensor(gat, x)
        s = x.clone()
        d.all_reduce(s)
        mn = torch.tensor([5.0 - r, float(r), 7.0], dtype=torch.float64)
        d.all_reduce(mn, op=d.ReduceOp.MIN)
        b = torch.full((2, 3), float(r))
        d.broadcast(b, src=1)
        b2 = torch.full((5,), float(r))
        w = d.broadcast(b2, src=2, async_op=True)
        w.wait()
        return gat, s, mn, b, b2

    out, logs = run_ranks(world, fn, timeout=20.0)
    xs = [torch.arange(4, dtype=torch.float64) + 10.0 * r for r in range(world)]
    for gat, s, mn, b, b2 in out:
        assert torch.equal(gat, torch.cat(xs))
        assert torch.equal(s, xs[0] + xs[1] + xs[2])
        assert torch.equal(mn, torch.tensor([3.0, 0.0, 7.0], dtype=torch.float64))
        assert torch.equal(b, torch.full((2, 3), 1.0))
        assert torch.equal(b2, torch.full((5,), 2.0))
    assert logs[0] == logs[1] == logs[2] and [e[0] for e in logs[0]] == \
        ["all_gather_into_tensor", "all_reduce", "all_reduce", "broadcast", "broadcast"]


@pytest.mark.parametrize("how", ["skip", "mismatch"])
def test_fake_collectives_fail_instead_of_hanging(how):
    """CPU: a rank that skips a collective makes the others raise within the barrier timeout; a rank that issues a
    different collective makes every rank raise at once."""
    world, timeout = 3, 2.0

    def fn(d):
        t = torch.ones(3, dtype=torch.float64)
        d.all_reduce(t)
        if d.get_rank() == 2:
            if how == "skip":
                return None
            d.broadcast(t, src=0)
        else:
            d.all_reduce(t)
        return t

    t0 = time.time()
    with pytest.raises((threading.BrokenBarrierError, RuntimeError)):
        run_ranks(world, fn, timeout=timeout)
    assert time.time() - t0 < timeout + 10.0


# ------------------------------------------------------------------------------------------------------------------
# sites, ranks and the single-GPU reference
# ------------------------------------------------------------------------------------------------------------------
def _site(zero_y=False):
    """the training site, theta1 (with y = 0 and a zero constant mean for the factor check, so that mu* = 0 exactly)"""
    X, y, noise = synthetic.loadest_site(N_TRAIN, 1005)
    theta = H.loadest_theta1()
    if zero_y:
        y = np.zeros_like(y)
        theta[0] = 0.0
    return X, y, noise, theta


def _engine(site, max_m, stream=0):
    X, y, noise, theta = site
    eng = capi.Engine(max_n=X.shape[0], max_m=max_m, device=0, stream=stream)
    try:
        eng.set_train(models.loadest_spec(2).to_c(), X, y, noise)
        _, info = eng.factorize(theta)
        assert info == 0
    except BaseException:
        eng.close()
        raise
    return eng


def _sharded(world, mode, site, Xs, S, Z=None, seed=0, jitter=JITTER, max_m=512):
    """sample_sharded on `world` emulated ranks -> ([draws], [info], [collective log]), one entry per rank.
    mode "private": each engine on its own stream (sample_sharded fences through the host).  "shared": each thread makes a
    stream current (torch's current stream is per thread) and creates its engine on it: the look-ahead branch."""
    def fn(d):
        st = None
        if mode == "shared":
            st = torch.cuda.Stream(device=0)
            torch.cuda.set_stream(st)
        eng = None
        try:
            eng = _engine(site, max_m, st.cuda_stream if st is not None else 0)
            return multisite.sample_sharded(eng, Xs, S, dist=d, seed=seed, jitter=jitter, Z=Z)
        finally:
            if eng is not None:
                eng.close()

    out, logs = run_ranks(world, fn)
    return [o[0] for o in out], [o[1] for o in out], logs


def _check_ranks(draws, infos, logs, want_info=0):
    """(a) info on every rank, (b) bit-identical draws, (d) identical collective sequences"""
    assert all(i == want_info for i in infos), infos
    assert all(np.array_equal(d, draws[0], equal_nan=True) for d in draws[1:]), "ranks returned different draws"
    assert all(lg == logs[0] for lg in logs[1:]), "ranks issued different collective sequences"


def _rel(got, want):
    return float(np.max(np.abs(got - want)) / np.max(np.abs(want)))


def _geometry(site, world, m, S, max_m=512):
    """engine.dist_dims plus what follows from it: panel owners, shards that start past mpad, V' chunks per rank"""
    eng = capi.Engine(max_n=site[0].shape[0], max_m=max_m, device=0)
    try:
        eng.set_train(models.loadest_spec(2).to_c(), *site[:3])
        d = eng.dist_dims(m, S, world)
    finally:
        eng.close()
    mb, rpr, npanels = d["mpad"] // 128, d["rows_per_rank"], d["npanels"]
    owners = [multisite.panel_owner(p, world) for p in range(npanels)]
    shard = [(r * rpr, min((r + 1) * rpr, d["mpad"])) for r in range(world)]
    return dict(dims=d, mb=mb, Spad=d["Spad"], npanels=npanels, last_panel_blocks=mb - (npanels - 1) * PANEL_BLOCKS,
                last_block_rows=m - (mb - 1) * 128, idle=[r for r in range(world) if r not in owners],
                past_mpad=[r for r in range(world) if shard[r][0] > d["mpad"]],
                chunks=[max(0, -(-(hi - lo) // max_m)) for lo, hi in shard])


# ------------------------------------------------------------------------------------------------------------------
# draws against single-GPU dgp_sample_ex
# ------------------------------------------------------------------------------------------------------------------
# world, m, S, normals ("philox" or "host"), stream modes, max_m, the geometry the case is chosen for
CASES = [
    (2, 1300, 48, "philox", ("private", "shared"), 256,
     dict(mb=11, npanels=3, last_panel_blocks=3, last_block_rows=20, idle=[], past_mpad=[], chunks=[3, 3])),
    (3, 100, 1, "host", ("private",), 512,
     dict(mb=1, npanels=1, idle=[1, 2], past_mpad=[2])),
    (4, 600, 130, "philox", ("shared",), 512,
     dict(mb=5, Spad=256, npanels=2, last_panel_blocks=1, idle=[2, 3], past_mpad=[3])),
    (5, 2560, 48, "host", ("private",), 512,
     dict(mb=20, npanels=5, last_panel_blocks=4, last_block_rows=128, idle=[], past_mpad=[])),
    (8, 3000, 48, "philox", ("shared",), 512,
     dict(mb=24, npanels=6, idle=[6, 7], past_mpad=[])),
    (8, 5200, 16, "philox", ("private",), 512,
     dict(mb=41, npanels=11, last_panel_blocks=1, idle=[], past_mpad=[7])),
]
DRAW_CASES = [pytest.param(w, m, S, nz, mode, mm, geo, id=f"w{w}-m{m}-{mode}")
              for (w, m, S, nz, modes, mm, geo) in CASES for mode in modes]


def _assert_geometry(site, world, m, S, max_m, expect):
    geo = _geometry(site, world, m, S, max_m)
    assert geo["dims"]["panel_cols"] == PANEL_BLOCKS * 128, geo["dims"]
    assert {k: geo[k] for k in expect} == expect, (world, m, geo)
    return geo


@pytest.mark.gpu
@pytest.mark.parametrize("world,m,S,normals,mode,max_m,expect", DRAW_CASES)
def test_sharded_draws_match_single_gpu(cuda_device, world, m, S, normals, mode, max_m, expect):
    """(a) info = 0 on every rank, (b) the draws bit-identical across ranks, (c) equal to single-GPU sample_ex with the
    same normals to 1e-9 max|draw|, (d) the same collective sequence on every rank."""
    site = _site()
    geo = _assert_geometry(site, world, m, S, max_m, expect)
    Xs = synthetic.daily_grid(site[0], m) + SHIFT
    Z = np.random.default_rng(m).standard_normal((S, m)) if normals == "host" else None
    seed = 17 + world
    t0 = time.time()
    try:
        draws, infos, logs = _sharded(world, mode, site, Xs, S, Z=Z, seed=seed, max_m=max_m)
        t1 = time.time()
        eng = _engine(site, max_m)
        try:
            want, info1 = eng.sample_ex(Xs, S, Z=Z, seed=seed, jitter=JITTER)
        finally:
            eng.close()
    finally:
        _free()
    _check_ranks(draws, infos, logs)
    assert info1 == 0
    err = _rel(draws[0], want)
    print(f"\nsharded draws world={world} m={m} S={S} {normals} {mode}: mb={geo['mb']} panels={geo['npanels']} "
          f"idle ranks={geo['idle']} shards past mpad={geo['past_mpad']} collectives={len(logs[0])}; "
          f"rel diff vs single GPU {err:.2e} ({t1 - t0:.1f} s sharded)")
    assert err <= DRAW_REL, err


# ------------------------------------------------------------------------------------------------------------------
# the distributed posterior factor against a float64 reference
# ------------------------------------------------------------------------------------------------------------------
FACTOR_CASES = [pytest.param(w, m, mode, mm, id=f"w{w}-m{m}-{mode}")
                for (w, m, mode, mm) in ((2, 1300, "private", 256), (2, 1300, "shared", 256), (4, 600, "shared", 512),
                                         (8, 3000, "shared", 512))]


@pytest.mark.gpu
@pytest.mark.parametrize("world,m,mode,max_m", FACTOR_CASES)
def test_sharded_posterior_factor(cuda_device, world, m, mode, max_m):
    """test_factor_schedule.test_sampler_posterior_factor for the distributed factor: y = 0 and a zero constant mean make
    mu* = 0 exactly, and host normals Z = [I_m; 0] make the draws [Lpost'; 0].  The last row must be exactly zero, Lpost'
    upper triangular (M_ZL reads no entry above the diagonal and every diagonal block is zeroed above it), and
    ||Sigma - Lpost Lpost'||_1 / (m (||K**||_1 + ||V'V||_1) eps) <= 1 with Sigma formed by cuBLAS from the engine's own
    T = L^-1.  The ranks must also agree bit for bit and match single-GPU sample_ex with the same Z."""
    site = _site(zero_y=True)
    X, _, _, theta = site
    n = X.shape[0]
    Xs = synthetic.daily_grid(X, m) + SHIFT
    S = m + 1
    Z = np.zeros((S, m))
    Z[:m] = np.eye(m)
    t0 = time.time()
    eng = T = D = V = VtV = Sg = None
    try:
        draws, infos, logs = _sharded(world, mode, site, Xs, S, Z=Z, max_m=max_m)
        _check_ranks(draws, infos, logs)
        D = draws[0]
        assert not np.any(D[m]), "mu* is not exactly zero: the draws are not Lpost'"
        assert not np.any(np.tril(D[:m], -1)), "Lpost has entries above the diagonal"
        eng = _engine(site, max_m)
        want, info1 = eng.sample_ex(Xs, S, Z=Z, jitter=JITTER)
        assert info1 == 0
        err = _rel(D, want)
        T = eng.linv(out=torch.empty((n, n), dtype=torch.float64, device=DEV))
        with torch.no_grad():
            nat = H.loadest_nat_from_theta(torch.tensor(theta, device=DEV))
            Xt, Xst = torch.tensor(X, device=DEV), torch.tensor(Xs, device=DEV)
            V = T @ orc.loadest_cov(Xst, Xt, nat).T        # [n, m]
            T = None
            VtV = V.T @ V
            V = None
            Sg = orc.loadest_cov(Xst, Xst, nat)
            nK, nV = _n1(Sg), _n1(VtV)
            Sg.diagonal().add_(JITTER)
            Sg -= VtV
            VtV = None
            Lt = torch.tensor(D[:m], device=DEV)            # Lpost'
            Sg -= torch.mm(Lt.T, Lt)
            Lt = None
            ratio = _n1(Sg) / (m * (nK + nV) * EPS)
    finally:
        if eng is not None:
            eng.close()
        eng = T = D = V = VtV = Sg = draws = None
        _free()
    print(f"\nsharded factor world={world} m={m} {mode}: dpot01={ratio:.2e} rel diff vs single GPU {err:.2e} "
          f"({time.time() - t0:.1f} s)")
    assert err <= DRAW_REL, err
    assert ratio <= RATIO_MAX, ratio


# ------------------------------------------------------------------------------------------------------------------
# a failing pivot on one rank, reported on all of them
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_sharded_info_is_min_over_ranks(cuda_device):
    """World 3, m = 3000: 24 block columns, panels 0 ... 5 owned by ranks 0 1 2 0 1 2.  The grid points are far apart in
    time and flow and far from the data, so every posterior pivot is close to the prior variance; point q (in panel 4,
    rank 1) is an exact copy of point 7.  Under the jitter -delta the duplicate's Schur pivot is about -2 delta and every
    other pivot about s_i - delta.  delta is chosen with a margin of 1e3 on both sides, asserted from the float64
    reference: min s_i >= 1e3 delta (s_i = diag(L)^2 of the reference Cholesky of Sigma* on the grid without the
    duplicate) and delta >= 1e3 m eps ||Sigma*||_1.  The sharded info, single-GPU sample_ex info and torch's cholesky_ex
    info must all be q + 1; rank 0 reports 0 for its own panels and rank 2 may report a later pivot, so this is the MIN
    all-reduce at work."""
    world, m, S, delta, src, q = 3, 3000, 4, 1e-6, 7, 2300
    site = _site()
    X, _, noise, theta = site
    geo = _geometry(site, world, m, S)
    assert geo["npanels"] == 6 and geo["mb"] == 24
    pw = PANEL_BLOCKS * 128
    assert q // pw == 4 and multisite.panel_owner(q // pw, world) == 1
    i = np.arange(m, dtype=np.float64)
    Xs = np.ascontiguousarray(np.stack([100.0 + 12.5 * i, 10.0 + 3.0 * i], axis=1))   # 6 l_time and 6 l_flow apart
    Xs[q] = Xs[src]
    t0 = time.time()
    Sg = L = None
    try:
        with torch.no_grad():
            nat = H.loadest_nat_from_theta(torch.tensor(theta, device=DEV))
            Xt, Xst = torch.tensor(X, device=DEV), torch.tensor(Xs, device=DEV)
            Ky = orc.loadest_cov(Xt, Xt, nat)
            Ky.diagonal().add_(torch.tensor(noise, device=DEV))
            L = torch.linalg.cholesky(Ky)
            Ky = None
            V = torch.linalg.solve_triangular(L, orc.loadest_cov(Xst, Xt, nat).T, upper=False)
            L = None
            Sg = orc.loadest_cov(Xst, Xst, nat) - V.T @ V     # Sigma*, jitter 0
            V = None
            keep = torch.tensor([k for k in range(m) if k != q], device=DEV)
            piv = torch.diagonal(torch.linalg.cholesky(Sg[keep][:, keep])) ** 2
            s_min, rounding = float(piv.min()), m * EPS * _n1(Sg)
            Sg.diagonal().sub_(delta)
            ref_info = int(torch.linalg.cholesky_ex(Sg).info)
    finally:
        Sg = L = None
        _free()
    print(f"\nsharded info world={world} m={m} q={q}: min pivot / delta = {s_min / delta:.1e}, "
          f"delta / (m eps ||Sigma*||_1) = {delta / rounding:.1e}")
    assert s_min >= 1e3 * delta and delta >= 1e3 * rounding, (s_min, delta, rounding)
    assert ref_info == q + 1, ref_info
    try:
        draws, infos, logs = _sharded(world, "private", site, Xs, S, seed=3, jitter=-delta)
        eng = _engine(site, 512)
        try:
            _, info1 = eng.sample_ex(Xs, S, seed=3, jitter=-delta)
        finally:
            eng.close()
    finally:
        draws = None
        _free()
    print(f"  sharded info {infos}, single GPU {info1}, cholesky_ex {ref_info} ({time.time() - t0:.1f} s)")
    assert infos == [q + 1] * world and info1 == q + 1
    assert all(lg == logs[0] for lg in logs[1:])


# ------------------------------------------------------------------------------------------------------------------
# the C entry point: shards at or past mpad
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_vt_rows_accepts_empty_shards(cuda_device):
    """dgp_dist_vt_rows clamps both ends to mpad: a range wholly at or past mpad (as sample_sharded passes it for a rank
    whose shard starts past mpad, or unclamped) returns 0 and writes nothing; negative, unaligned and reversed ranges are
    still refused; afterwards the whole range gives the posterior mean of dgp_predict."""
    m = 600
    site = _site()
    Xs = synthetic.daily_grid(site[0], m) + SHIFT
    eng = _engine(site, 512)
    tok = None
    try:
        d = eng.dist_dims(m, 1, 1)
        mpad = d["mpad"]
        assert mpad == 640 and d["rows_per_rank"] == mpad
        f64 = dict(dtype=torch.float64, device=DEV)
        VT = torch.empty((d["rows_per_rank"], d["npad"]), **f64)
        Od = torch.empty((d["Spad"], mpad), **f64)
        mu = torch.empty((mpad,), **f64)
        tok = eng.dist_begin(Xs, 1, None, 0, JITTER, 0, 1, VT, Od, mu)
        torch.cuda.synchronize()
        VT.fill_(3.0)
        mu.fill_(5.0)
        torch.cuda.synchronize()
        for r0, r1 in ((mpad + 128, mpad + 256), (mpad + 128, mpad), (mpad, mpad), (mpad, mpad + 128)):
            assert eng.dist_call("vt_rows", tok, r0, r1) == 0, (r0, r1)
        torch.cuda.synchronize()
        assert bool(torch.all(VT == 3.0)) and bool(torch.all(mu == 5.0))
        for r0, r1 in ((256, 128), (-128, 0), (64, 128), (0, 192)):
            with pytest.raises(capi.DgpError, match="bad row range"):
                eng.dist_call("vt_rows", tok, r0, r1)
        mu.zero_()
        torch.cuda.synchronize()
        assert eng.dist_call("vt_rows", tok, 0, mpad) == 0
        torch.cuda.synchronize()
        got = mu[:m].cpu().numpy()
        assert not bool(torch.any(mu[m:] != 0.0))
        want, _ = eng.predict(Xs, want_var=False)
        assert _rel(got, want) <= 1e-12
    finally:
        if tok is not None:
            eng.dist_call("end", tok)
        eng.close()
        _free()
