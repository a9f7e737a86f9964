"""SHA-256 of the draws and the info of multisite.sample_sharded on emulated ranks (tests/test_dist_sample.py's
FakeGroup), for the geometries of test_dist_sample.CASES (each listed stream mode, and world 1), and for the duplicated
grid point under a negative jitter of test_sharded_info_is_min_over_ranks at worlds 1, 2, 3 and 8.

    python tools/dist_draws_digest.py --out digests.json [--pkg DIR]

--pkg: directory that holds the discontinuum_b200 package to run (default: this repository), so that the digests of
another build of the package, e.g. a copy of an earlier commit with its own libdgp.so, come from the same script.
tests/golden/dist_draws_parent.json holds the digests of the commit before the panel-slab storage of the posterior
covariance; tests/test_dist_sample_panels.py requires the same bits from the current layout."""
import argparse
import hashlib
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def cases(tds):
    """(id, world, mode, m, S, normals, max_m, seed, jitter, grid) for every digest; grid is 'daily' or 'dup'"""
    out = []
    for (w, m, S, nz, modes, mm, _geo) in tds.CASES:
        for world in (w, 1):
            for mode in modes:
                out.append((f"w{world}-m{m}-{mode}", world, mode, m, S, nz, mm, 17 + w, tds.JITTER, "daily"))
    for w in (1, 2, 3, 8):
        out.append((f"dup-w{w}", w, "private", 3000, 4, "philox", 512, 3, -1e-6, "dup"))
    return out


def grid_of(tds, site, m, kind):
    import numpy as np
    from discontinuum_b200 import synthetic

    if kind == "daily":
        return synthetic.daily_grid(site[0], m) + tds.SHIFT
    # test_sharded_info_is_min_over_ranks: far-apart points, point 2300 (panel 4) a copy of point 7
    i = np.arange(m, dtype=np.float64)
    Xs = np.ascontiguousarray(np.stack([100.0 + 12.5 * i, 10.0 + 3.0 * i], axis=1))
    Xs[2300] = Xs[7]
    return Xs


def normals(m, S, kind):
    import numpy as np

    return np.random.default_rng(m).standard_normal((S, m)) if kind == "host" else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--pkg", default=ROOT)
    a = ap.parse_args()
    pkg = os.path.abspath(a.pkg)
    sys.path.insert(0, pkg)
    import discontinuum_b200  # noqa: F401  (first, so that tests/helpers.py's path entry cannot shadow it)
    from discontinuum_b200 import capi

    sys.path.insert(1, os.path.join(ROOT, "tests"))
    import test_dist_sample as tds

    site = tds._site()
    res = {}
    for (cid, w, mode, m, S, nz, mm, seed, jit, kind) in cases(tds):
        Xs = grid_of(tds, site, m, kind)
        t0 = time.time()
        draws, infos, _ = tds._sharded(w, mode, site, Xs, S, Z=normals(m, S, nz), seed=seed, jitter=jit, max_m=mm)
        tds._free()
        digs = {hashlib.sha256(d.tobytes()).hexdigest() for d in draws}
        if len(digs) != 1 or len(set(infos)) != 1:
            raise SystemExit(f"{cid}: ranks disagree ({len(digs)} digests, infos {infos})")
        res[cid] = dict(sha256=digs.pop(), info=int(infos[0]), world=w, mode=mode, m=m, S=S, normals=nz, max_m=mm,
                        seed=seed, jitter=jit, grid=kind)
        print(f"{cid}: info {infos[0]} {res[cid]['sha256'][:16]} ({time.time() - t0:.1f} s)", flush=True)
    doc = dict(library=os.path.relpath(capi.library_path(), pkg), cases=res)
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
