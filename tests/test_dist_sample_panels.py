"""The distributed posterior sampler with panel-slab storage: each rank keeps only the lower trapezoids of its own panels
of the m x m posterior covariance (plus two receive slots for broadcast panels), and can reduce its draws to grouped
(annual) flux sums on the device (dgp_dist_finish_ex, sample_sharded(flux=...)).  Ranks are emulated in one process on one
GPU with test_dist_sample.py's FakeGroup.

  * bit identity: the draws' SHA-256 and the info of every case in golden/dist_draws_parent.json, written by
    tools/dist_draws_digest.py from the replicated m x m layout that came before, at worlds 1 ... 8 in both stream modes
  * info: the duplicated grid point under a negative jitter reports the same global 1-based pivot at worlds 1, 2, 3 and
    8 (a pivot index local to the slab would come out 128 pb too small)
  * memory: dgp_dist_arena_bytes is what a fresh handle's dist_begin allocates, for an idle rank, a ragged last panel and
    a full one; the slab parts of all ranks add up to world 1's, 8 sum_p (mb - 4p) 128 w_p 128 bytes, and the rest of the
    workspace is the same on every rank
  * flux: rank-identical sums, equal to a numpy restatement of k_flux_reduce on the draws of the same call without flux,
    and to single-GPU sample_ex(flux=...); a malformed reduction is refused with dgp_sample_ex's messages
"""
import hashlib
import json
import os
import time

import numpy as np
import pytest
import torch

from discontinuum_b200 import capi, models, multisite, synthetic
from test_dist_sample import CASES, JITTER, PANEL_BLOCKS, SHIFT, _engine, _site, run_ranks
from test_factor_schedule import _free

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dist_draws_parent.json")
with open(GOLDEN) as _f:
    PARENT = json.load(_f)["cases"]
DUP_SRC, DUP_Q = 7, 2300          # test_sharded_info_is_min_over_ranks: point q (panel 4) is a copy of point 7
FLUX_REL = 1e-10                  # sums against the numpy reduction of the same draws (test_gpu_parity.py's bound)
SINGLE_REL = 1e-9                 # sums against single-GPU sample_ex (the draws agree to 1e-9, test_dist_sample.py)


def _grid(site, m, kind):
    if kind == "daily":
        return synthetic.daily_grid(site[0], m) + SHIFT
    i = np.arange(m, dtype=np.float64)
    Xs = np.ascontiguousarray(np.stack([100.0 + 12.5 * i, 10.0 + 3.0 * i], axis=1))
    Xs[DUP_Q] = Xs[DUP_SRC]
    return Xs


def _normals(m, S, kind):
    return np.random.default_rng(m).standard_normal((S, m)) if kind == "host" else None


def _run(world, mode, site, Xs, S, max_m, **kw):
    """sample_sharded(**kw) on `world` emulated ranks -> ([(out, info, stats)], [collective log]) per rank (see
    test_dist_sample._sharded for the two stream modes)"""
    def fn(d):
        st = None
        if mode == "shared":
            st = torch.cuda.Stream(device=0)
            torch.cuda.set_stream(st)
        eng = None
        try:
            eng = _engine(site, max_m, st.cuda_stream if st is not None else 0)
            stats = {}
            out, info = multisite.sample_sharded(eng, Xs, S, dist=d, stats=stats, **kw)
            return out, info, stats
        finally:
            if eng is not None:
                eng.close()

    try:
        return run_ranks(world, fn)
    finally:
        _free()


# ------------------------------------------------------------------------------------------------------------------
# the same bits as the replicated layout
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cid", sorted(PARENT))
def test_draws_bit_identical_to_replicated_layout(cuda_device, cid):
    """every rank's draws hash to the parent layout's SHA-256, with its info; the ranks issue the same collectives"""
    c = PARENT[cid]
    site = _site()
    Xs = _grid(site, c["m"], c["grid"])
    t0 = time.time()
    res, logs = _run(c["world"], c["mode"], site, Xs, c["S"], c["max_m"], Z=_normals(c["m"], c["S"], c["normals"]),
                     seed=c["seed"], jitter=c["jitter"])
    digs = [hashlib.sha256(np.ascontiguousarray(r[0]).tobytes()).hexdigest() for r in res]
    infos = [r[1] for r in res]
    print(f"\n{cid}: info {infos[0]} sha256 {digs[0][:16]} ({time.time() - t0:.1f} s)")
    assert all(lg == logs[0] for lg in logs[1:])
    assert infos == [c["info"]] * c["world"], (infos, c["info"])
    if c["grid"] == "dup":
        assert c["info"] == DUP_Q + 1     # the global 1-based pivot, whichever rank owns the panel
    assert digs == [c["sha256"]] * c["world"], "draws differ from the replicated layout's"


# ------------------------------------------------------------------------------------------------------------------
# workspace accounting
# ------------------------------------------------------------------------------------------------------------------
def _slab_bytes(mb, world, rank):
    """8 sum over rank's panels p of (mb - 4p) 128 rows x w_p 128 columns"""
    npanels = -(-mb // PANEL_BLOCKS)
    return sum(8 * (mb - PANEL_BLOCKS * p) * 128 * (min(PANEL_BLOCKS * (p + 1), mb) - PANEL_BLOCKS * p) * 128
               for p in range(rank, npanels, world))


@pytest.mark.gpu
@pytest.mark.parametrize("m", [3000, 5200, 100])
def test_arena_bytes_split_into_slabs(cuda_device, m):
    """over worlds 1 ... 8: the slab parts of the ranks add up to world 1's (about 4 mpad^2 bytes) and the rest is the
    same on every rank"""
    S = 48
    eng = _engine(_site(), 512)
    try:
        mb = -(-m // 128)
        whole = eng.dist_arena_bytes(m, S, 1, 0)
        slabs1 = _slab_bytes(mb, 1, 0)
        assert slabs1 == sum(_slab_bytes(mb, 8, r) for r in range(8))
        assert abs(slabs1 - 4 * (mb * 128) ** 2) <= 8 * 128 * 128 * PANEL_BLOCKS * mb  # the panels' diagonal triangles
        rest = whole - slabs1
        assert rest > 0
        for world in range(1, 9):
            got = [eng.dist_arena_bytes(m, S, world, r) for r in range(world)]
            assert [g - _slab_bytes(mb, world, r) for r, g in enumerate(got)] == [rest] * world, (world, got)
            assert sum(g - rest for g in got) == slabs1
        with pytest.raises(ValueError):
            eng.dist_arena_bytes(m, S, 2, 2)
    finally:
        eng.close()
        _free()


@pytest.mark.gpu
@pytest.mark.parametrize("world,m,rank", [(8, 3000, 7), (8, 3000, 0), (1, 5200, 0), (8, 5200, 2)],
                         ids=["idle-rank", "w8-m3000-r0", "ragged-w1", "ragged-w8-r2"])
def test_arena_bytes_is_what_dist_begin_allocates(cuda_device, world, m, rank):
    """the mem_get_info delta of a fresh handle's first dist_begin is dgp_dist_arena_bytes (cudaMalloc granularity
    aside); world 8, m 3000: rank 7 owns no panel and has no slab"""
    S = 48
    site = _site()
    Xs = synthetic.daily_grid(site[0], m) + SHIFT
    warm = _engine(site, 512)   # every kernel dist_begin launches is loaded before the measurement
    try:
        multisite.sample_sharded(warm, Xs[:300], 4)
    finally:
        warm.close()
    eng = _engine(site, 512)
    tok = None
    try:
        need = eng.dist_arena_bytes(m, S, world, rank)
        mb = -(-m // 128)
        if world == 8 and m == 3000 and rank == 7:
            assert _slab_bytes(mb, world, rank) == 0
        d = eng.dist_dims(m, S, world)
        f64 = dict(dtype=torch.float64, device="cuda")
        VT = torch.zeros((d["rows_per_rank"] * world, d["npad"]), **f64)
        Od = torch.empty((d["Spad"], d["mpad"]), **f64)
        mu = torch.empty((d["mpad"],), **f64)
        torch.cuda.synchronize()
        free0 = torch.cuda.mem_get_info()[0]
        tok = eng.dist_begin(Xs, S, None, 5, JITTER, rank, world, VT, Od, mu)
        torch.cuda.synchronize()
        free1 = torch.cuda.mem_get_info()[0]
        print(f"\nworld {world} m {m} rank {rank}: dgp_dist_arena_bytes {need} B, allocated {free0 - free1} B")
        assert need <= free0 - free1 <= need + (4 << 20)
    finally:
        if tok is not None:
            eng.dist_call("end", tok)
        eng.close()
        _free()


# ------------------------------------------------------------------------------------------------------------------
# annual flux on the device
# ------------------------------------------------------------------------------------------------------------------
def _flux(m, kind=1):
    """weights (flow dt 1e-3 like), "years" of 365 grid points and a log-standard target pipeline"""
    rng = np.random.default_rng(300 + m)
    gs = np.concatenate([np.arange(0, m, 365), [m]]).astype(np.int32)
    return dict(y_mean=0.4, y_scale=0.7, log_transform=kind, weight=np.exp(rng.standard_normal(m)) * 86.4, group_start=gs)


def _flux_ref(draws, f):
    """k_flux_reduce restated: out[s, g] = sum_{i in group g} weight[i] T(draw[s, i])"""
    v = draws * f["y_scale"] + f["y_mean"]
    if f["log_transform"] == 1:
        v = np.maximum(np.exp(v), 1e-6)
    elif f["log_transform"] == 2:
        v = np.maximum(v, 0.0)
    wv = v * f["weight"]
    gs = f["group_start"]
    return np.stack([wv[:, a:b].sum(1) for a, b in zip(gs[:-1], gs[1:])], axis=1)


FLUX_CASES = [pytest.param(w, m, S, nz, modes[0], mm, id=f"w{w}-m{m}-{modes[0]}") for (w, m, S, nz, modes, mm, _) in CASES]
FLUX_CASES.append(pytest.param(1, 5200, 16, "philox", "shared", 512, id="w1-m5200-shared"))


@pytest.mark.gpu
@pytest.mark.parametrize("world,m,S,normals,mode,max_m", FLUX_CASES)
def test_sharded_flux_matches_draws_and_single_gpu(cuda_device, world, m, S, normals, mode, max_m):
    """sample_sharded(flux=FluxSpec): the same sums on every rank, equal to the numpy reduction of the same call's draws
    (1e-10 relative) and to single-GPU sample_ex(flux=...) (1e-9 relative), the same collectives as without flux, and
    stats["arena_bytes"] = dist_arena_bytes"""
    site = _site()
    Xs = synthetic.daily_grid(site[0], m) + SHIFT
    Z = _normals(m, S, normals)
    f = _flux(m)
    spec = models.FluxSpec(Xs, f["weight"], f["group_start"], np.arange(f["group_start"].shape[0] - 1), f["y_mean"],
                           f["y_scale"], f["log_transform"])
    seed = 40 + world
    plain, logs0 = _run(world, mode, site, Xs, S, max_m, Z=Z, seed=seed, jitter=JITTER)
    red, logs1 = _run(world, mode, site, Xs, S, max_m, Z=Z, seed=seed, jitter=JITTER, flux=spec)
    eng = _engine(site, max_m)
    try:
        want, info1 = eng.sample_ex(Xs, S, Z=Z, seed=seed, jitter=JITTER, flux=f)
        for r in range(world):
            assert red[r][2]["arena_bytes"] == eng.dist_arena_bytes(m, S, world, r)
    finally:
        eng.close()
        _free()
    sums = red[0][0]
    assert [r[1] for r in plain] == [0] * world and [r[1] for r in red] == [0] * world and info1 == 0
    assert sums.shape == (S, f["group_start"].shape[0] - 1)
    assert all(np.array_equal(r[0], sums) for r in red[1:]), "ranks returned different sums"
    assert logs1 == logs0 and all(lg == logs1[0] for lg in logs1[1:])
    ref = _flux_ref(plain[0][0], f)
    e_ref = float(np.max(np.abs(sums - ref) / np.abs(ref)))
    e_one = float(np.max(np.abs(sums - want) / np.abs(want)))
    print(f"\nflux world={world} m={m} S={S} {mode}: vs numpy on the draws {e_ref:.1e}, vs single GPU {e_one:.1e}")
    assert e_ref <= FLUX_REL and e_one <= SINGLE_REL


@pytest.mark.gpu
def test_sharded_flux_dict_and_malformed_reduction(cuda_device):
    """world 1 without a process group: the flux dict of sample_ex gives sample_ex's sums; a reduction without groups,
    with a group past the grid or with decreasing group starts is refused with dgp_sample_ex's messages, a weight vector
    of the wrong length before anything runs, and the engine samples the same sums afterwards"""
    m, S = 1300, 8
    site = _site()
    Xs = synthetic.daily_grid(site[0], m) + SHIFT
    f = _flux(m)
    eng = _engine(site, 256)
    try:
        a, ia = multisite.sample_sharded(eng, Xs, S, seed=2, jitter=JITTER, flux=f)
        b, ib = eng.sample_ex(Xs, S, seed=2, jitter=JITTER, flux=f)
        assert ia == ib == 0 and float(np.max(np.abs(a - b) / np.abs(b))) <= SINGLE_REL
        bad = [(np.array([0], dtype=np.int32), "bad reduction spec"),
               (np.array([0, 400, m + 1], dtype=np.int32), "group range outside the grid"),
               (np.array([-1, 400, m], dtype=np.int32), "group range outside the grid"),
               (np.array([0, 700, 400, m], dtype=np.int32), "group_start must be non-decreasing")]
        for gs, msg in bad:
            g = dict(f, group_start=gs)
            with pytest.raises(capi.DgpError, match=msg):
                eng.sample_ex(Xs, S, seed=2, jitter=JITTER, flux=g)
            with pytest.raises(capi.DgpError, match="dgp_dist_finish_ex: " + msg):
                multisite.sample_sharded(eng, Xs, S, seed=2, jitter=JITTER, flux=g)
        with pytest.raises(ValueError, match="weight"):
            multisite.sample_sharded(eng, Xs, S, flux=dict(f, weight=f["weight"][:-1]))
        c, ic = multisite.sample_sharded(eng, Xs, S, seed=2, jitter=JITTER, flux=f)
        assert ic == 0 and np.array_equal(c, a)
    finally:
        eng.close()
        _free()
