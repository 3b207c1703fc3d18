#!/usr/bin/env python
"""Generate the committed golden fixtures from the UNMODIFIED reference.

Run in the build container (needs /root/reference and oracle/_ref/libwrref.so):

    python tests/golden/make_golden.py

Outputs (all under tests/golden/):
  meshes.npz        triangle lists of the reference's four STL assets as parsed by its own
                    STLReader (read_STL.hpp) — (T,12) float32: normal, v0, v1, v2
  ref_kat.json      voxel-grid KATs (dims, occupied count, SHA-256 of isFree[z][y][x]),
                    single selectNext KATs (incl. a NaN-plane and a boundary case), GTSP runs
  ref_acs.npz       whole searches of the unmodified reference on the C1 weld-point set
                    (SURVEY.md §8d): best path ids + length per pair, SHA-256 of the full
                    pheromone field after 1/2/10 iterations, under the sequential Philox stream
  ref_bspline.npz   BS_Basic<float, 3, D, CI, CF> of the unmodified core/BSplineBasic.h for eight setups: knots, control
                    points, curve points and return values at 261 times each (`python tests/golden/make_golden.py bspline`
                    regenerates only this file; the inputs are a pure function of the case, see bspline_inputs)
  ref_live.json     what tests/test_oracle_vs_reference.py compares with, for exactly its inputs: voxel grid, grid file
                    and its reload, a search on the `test` mesh, the all-pairs driver, GTSP on unrounded distances,
                    36 B-spline setups (`python tests/golden/make_golden.py live` regenerates only this file; its
                    "source" field names the code that produced it, see live_fixtures)
Everything else here is produced by reference code, not by the oracle restatement; the tests then
hold the oracle (and through it the GPU) to these values on machines without the reference sources.
"""
import hashlib
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle import oracle as O  # noqa: E402

REF_FILES = "/root/reference/files"
SEED = 0x5EED

# SURVEY.md §8d, C1: six points on the free plane x = min_x - 2p of the cube, all 15 pairs,
# plus one pair beyond the duplicate-coordinate plane y = max_y (NaN propagation, expected inf).
C1_POINTS = [(1.600931, y, z) for y in (-0.259319, -0.074319, 0.085681) for z in (1.224003, 1.399003)]
C1_NAN_PAIR = ((1.59, -0.27, 1.22), (1.59, 0.12, 1.22))


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


BSPLINE_CASES = [(0, 0, 0, 57, 150.0), (2, 2, 2, 16, 6000.0), (3, 2, 2, 40, 100.0), (3, 0, 0, 9, 10.0), (1, 0, 0, 5, 1.0), (2, 1, 1, 33, 77.7),
                 (5, 2, 2, 64, 1000.0), (3, 2, 1, 12, 3.5)]


def bspline_inputs(case):
    """The inputs of a B-spline fixture, a pure function of the case (tests rebuild them instead of storing them)."""
    d, ci, cf, n, tf = case
    rng = np.random.default_rng(1000 * d + 100 * ci + 10 * cf + n)
    mid = (rng.random((n, 9), dtype=np.float32) * 2 - 1)                      # rows of nine, like main.cpp:325-334
    init = np.concatenate([mid[0, :3], (rng.random(3 * ci) - 0.5)]).astype(np.float32)
    fin = np.concatenate([mid[-1, :3], (rng.random(3 * cf) - 0.5)]).astype(np.float32)
    u = np.concatenate([np.linspace(-0.05 * tf, 1.05 * tf, 257), [0.0, tf, tf * (1 - 1e-7), np.nan]]).astype(np.float32)
    pre = rng.random((u.size, 3), dtype=np.float32)                           # what `ret` holds before the call (kept by a failed call)
    return init, fin, mid, tf, u, pre


def bspline_fixtures():
    """BS_Basic<float, 3, D, CI, CF> of the UNMODIFIED core/BSplineBasic.h: knots, control points, curve points, return values."""
    assert O.have_ref(), "oracle/_ref/libwrref.so missing: run make -C oracle"
    out = {}
    for i, case in enumerate(BSPLINE_CASES):
        init, fin, mid, tf, u, pre = bspline_inputs(case)
        pts, ok, knots, cps = O.bspline(case[0], case[1], case[2], init, fin, mid, tf, u, out=pre, use_ref=True)
        out["pts%d" % i] = pts; out["ok%d" % i] = ok; out["knots%d" % i] = knots; out["cps%d" % i] = cps
        print("bspline", case, "ok", int(ok.sum()), "of", ok.size)
    np.savez_compressed(os.path.join(HERE, "ref_bspline.npz"), **out)


def main():
    assert O.have_ref(), "oracle/_ref/libwrref.so missing: run make -C oracle"
    bspline_fixtures()
    meshes = {n: O.Ref.stl_read("%s/%s.stl" % (REF_FILES, n)) for n in ("cubic", "test", "simplified_piece", "origin_piece")}
    np.savez_compressed(os.path.join(HERE, "meshes.npz"), **meshes)
    kat = {"seed": SEED, "grids": [], "steps": [], "gtsp": []}

    # ---- voxel grids (model_grid_map.hpp:151-273, unmodified) -------------------------------
    for name, precision, wall in (("cubic", 0.005, 10), ("simplified_piece", 0.008, 5), ("test", 0.018692, 10),
                                  ("simplified_piece", 0.02, 3), ("origin_piece", 0.03, 2)):
        R = O.Ref()
        R.voxelize(meshes[name], precision, wall)
        free, xs, ys, zs = R.grid()
        kat["grids"].append(dict(mesh=name, precision=precision, wall=wall, dims=list(R.dims), occupied=int((free == 0).sum()),
                                 sha256_isfree=sha(free), sha256_xs=sha(xs), sha256_ys=sha(ys), sha256_zs=sha(zs)))
        print("grid", kat["grids"][-1])

    # ---- the C1 searches ---------------------------------------------------------------------
    R = O.Ref()
    R.voxelize(meshes["cubic"], 0.005, 10)
    R.acs_init()
    out = {}
    pairs = [(i, j) for i in range(6) for j in range(i + 1, 6)]
    lens = []
    for (i, j) in pairs:
        ok, s, e = R.set_points(C1_POINTS[i], C1_POINTS[j])
        assert ok
        R.compute(0.5, 150, SEED)
        ids, dirs, L = R.best()
        R.reset()
        out["pair_%d_%d_ids" % (i, j)] = ids.astype(np.int32)
        out["pair_%d_%d_dirs" % (i, j)] = dirs.astype(np.int8)
        out["pair_%d_%d_meta" % (i, j)] = np.array([s, e, np.float32(L).view(np.int32)], np.int64)
        lens.append(L)
        print("pair", i, j, "start", s, "goal", e, "L", L, "nodes", len(ids))
    ok, s, e = R.set_points(*C1_NAN_PAIR)
    R.compute(0.5, 20, SEED)
    _, _, L = R.best()
    R.reset()
    out["nan_pair_meta"] = np.array([int(ok), s, e, np.float32(L).view(np.int32)], np.int64)
    print("nan pair", ok, s, e, L)
    snaps = {}
    ok, s, e = R.set_points(C1_POINTS[0], C1_POINTS[5])
    for iters in (1, 2, 10):
        R.compute(0.5, iters, SEED)
        ids, dirs, L = R.best()
        snaps[str(iters)] = dict(sha256_tau=sha(R.pheromone()), L_bits=int(np.float32(L).view(np.int32)), nodes=int(len(ids)), sha256_ids=sha(ids.astype(np.int32)))
        R.reset()
    kat["c1_tau_snapshots_pair_0_5"] = snaps
    np.savez_compressed(os.path.join(HERE, "ref_acs.npz"), **out)

    # ---- single selectNext KATs (ACSRank_3D.hpp:134-193, unmodified) ---------------------------
    free, xs, ys, zs = R.grid()
    rx, ry, rz = R.dims
    nid = lambda x, y, z: (z * ry + y) * rx + x  # noqa: E731
    rng = np.random.default_rng(11)
    cases = []
    # interior, boundary (self-neighbour slots), next to the cube, on the duplicate-y plane (NaN)
    dup_y = int(np.where(np.diff(ys) == 0)[0][0])
    spots = [(5, 5, 5), (0, 0, 0), (rx - 1, ry - 1, rz - 1), (0, 40, 20), (9, 30, 30), (8, dup_y, 8), (8, dup_y + 1, 8), (30, 9, 30), (3, 3, rz - 1)]
    for (x, y, z) in spots:
        cur = nid(x, y, z)
        if not free[cur]:
            continue
        for goal in (nid(2, 2, 2), nid(rx - 3, 5, rz - 4), nid(4, ry - 2, 4)):
            if goal == cur:
                continue
            for r31 in (0, 1 << 30, (1 << 31) - 1, int(rng.integers(0, 1 << 31))):
                tabu = []
                if rng.random() < 0.5:
                    for d in rng.choice(6, 2, replace=False):
                        dx, dy, dz = [(0, 0, -1), (0, -1, 0), (-1, 0, 0), (1, 0, 0), (0, 1, 0), (0, 0, 1)][d]
                        if 0 <= x + dx < rx and 0 <= y + dy < ry and 0 <= z + dz < rz:
                            tabu.append(nid(x + dx, y + dy, z + dz))
                more, infos, d, nxt, L = R.select_step(cur, goal, tabu, r31)
                cases.append(dict(cur=cur, goal=goal, tabu=tabu, r31=r31, more=more, infos_bits=[int(v) for v in infos.view(np.int32)],
                                  dir=d, next=nxt, L_bits=int(np.float32(L).view(np.int32))))
    kat["steps"] = cases
    print("step KATs:", len(cases), "of which dead:", sum(c["dir"] < 0 for c in cases))

    # ---- seam ordering (ACS_GTSP.hpp, unmodified) ---------------------------------------------
    with tempfile.TemporaryDirectory() as td:
        for n, iters, seed in ((8, 20, 77), (16, 40, 78), (48, 12, 79)):
            P = np.random.default_rng(n).random((n, 3))
            D = np.sqrt(((P[:, None] - P[None]) ** 2).sum(-1))
            D = np.array([[float("%.6f" % v) for v in row] for row in D])
            Rg = O.RefGtsp(D, os.path.join(td, "graph.in"))
            ran, calls = Rg.run(iters, seed)
            tour, L = Rg.best()
            kat["gtsp"].append(dict(n=n, iters=iters, seed=seed, ran=ran, rand_calls=calls, points_seed=n, L=L, tour=tour.ravel().tolist(),
                                    tau0=Rg.tau0(), sha256_pheromone=sha(Rg.pheromone())))
            print("gtsp", n, ran, L)
    with open(os.path.join(HERE, "ref_kat.json"), "w") as f:
        json.dump(kat, f, indent=1)
    live_fixtures()
    print("wrote fixtures to", HERE)


# ---- inputs of tests/test_oracle_vs_reference.py (shared, so that the fixture and the tests cannot drift apart) -----------
def search_points(G):
    xs, ys, zs = G.coords()
    return (xs[1], ys[1], zs[1]), (xs[-2], ys[-3], zs[-2])


def all_pairs_points(G):
    xs, ys, zs = G.coords()
    return [(xs[2], ys[2], zs[2]), (xs[2], ys[-4], zs[3]), (xs[3], ys[5], zs[-3])]


def gtsp_distances():
    P = np.random.default_rng(21).random((24, 3))
    return np.sqrt(((P[:, None] - P[None]) ** 2).sum(-1))


def bspline_live_cases():
    """Random valid setups of every (DEGREE, CI, CF) the harness instantiates, three sizes each (one rng, consumed in order)."""
    rng = np.random.default_rng(3)
    for (d, ci, cf) in [(0, 0, 0), (1, 0, 0), (2, 0, 0), (3, 0, 0), (2, 1, 1), (3, 1, 1), (2, 2, 2), (3, 2, 2), (4, 2, 2), (5, 2, 2), (3, 2, 1), (3, 0, 2)]:
        for n, tf in [(max(1, d + 1 - ci - cf), 1.0), (57, 150.0), (1000, 123.456)]:
            mid = rng.random((n, 9), dtype=np.float32) * 2 - 1
            init = np.concatenate([mid[0, :3], rng.random(3 * ci) - 0.5]).astype(np.float32)
            fin = np.concatenate([mid[-1, :3], rng.random(3 * cf) - 0.5]).astype(np.float32)
            u = np.concatenate([np.linspace(-1, tf * 1.01, 301), [0, tf, tf * (1 - 1e-7), np.nan]]).astype(np.float32)
            pre = rng.random((u.size, 3), dtype=np.float32)
            yield (d, ci, cf, n, tf), (init, fin, mid, tf, u, pre)


def live_fixtures():
    """ref_live.json: what tests/test_oracle_vs_reference.py compares with.  Computed by the unmodified reference
    (oracle/_ref/libwrref.so) where it is built.  Without it the values come from the oracle restatement, which that module
    held bit-equal to the reference, live, on these very inputs when the restatement's sources last changed; "source"
    records which of the two produced the file, and a run with the reference built re-records (and so re-checks) it."""
    use_ref = O.have_ref()
    meshes = dict(np.load(os.path.join(HERE, "meshes.npz")))
    out = {"source": "reference (oracle/_ref/libwrref.so)" if use_ref else
           "oracle restatement, as held bit-equal to the reference by tests/test_oracle_vs_reference.py when oracle/ last changed"}
    # voxel grid, the grid file (the reference's dump carries the LAST triangle's box) and the reload of that file
    tris = meshes["simplified_piece"]
    with tempfile.TemporaryDirectory() as td:
        f = os.path.join(td, "grid.in")
        if use_ref:
            R = O.Ref(); R.voxelize(tris, 0.015, 4, file=f)
            dims, (free, xs, ys, zs) = R.dims, R.grid()
            R3 = O.Ref(); R3.read_grid_file(f)
            reload = R3.grid()
        else:
            G = O.Grid.from_triangles(tris, 0.015, 4, O.VOX_AABB); G.write_file(f, compat=True)
            dims, (free, xs, ys, zs) = G.dims, (G.isfree(),) + G.coords()
            H = O.Grid.read_file(f)
            reload = (H.isfree(),) + H.coords()
        out["grid"] = dict(dims=list(dims), sha256_isfree=sha(free), sha256_xyz=[sha(v) for v in (xs, ys, zs)],
                           sha256_file=hashlib.sha256(open(f, "rb").read()).hexdigest(),
                           reload_sha256_isfree=sha(reload[0]), reload_sha256_xyz=[sha(v) for v in reload[1:]])
    # a search on the `test` mesh: best path, length and the whole pheromone field after 1, 3 and 25 iterations
    G = O.Grid.from_triangles(meshes["test"], 0.08, 4, O.VOX_AABB)
    p, q = search_points(G)
    if use_ref:
        R = O.Ref(); R.voxelize(meshes["test"], 0.08, 4); R.acs_init()
    else:
        A = O.Acs(G, rng_mode=O.RNG_SEQUENTIAL, sort_mode=O.SORT_STD, seed=99)
    out["search"] = {"set_points": list(R.set_points(p, q) if use_ref else A.set_points(p, q))}
    for iters in (1, 3, 25):
        if use_ref:
            R.compute(3.0, iters, 99); ids, dirs, L = R.best(); tau = R.pheromone(); R.reset()
        else:
            A.begin(3.0); A.iterate(iters); ids, dirs, L = A.best(); tau = A.pheromone(); A.reset()
        out["search"][str(iters)] = dict(L_bits=int(np.float32(L).view(np.int32)), sha256_ids=sha(ids.astype(np.int64)),
                                         sha256_dirs=sha(dirs.astype(np.int32)), sha256_tau=sha(tau))
    # the all-pairs driver (searchBestPathOfPoints, ACSRank_3D.hpp:427-504): one Philox stream over the pairs, never reseeded
    G = O.Grid.from_triangles(meshes["cubic"], 0.01, 5, O.VOX_AABB)
    pts = all_pairs_points(G)
    pairs = []
    if use_ref:
        R = O.Ref(); R.voxelize(meshes["cubic"], 0.01, 5)
        with tempfile.TemporaryDirectory() as td:
            cnt, lens = R.search_all(pts, 0.4, 4242, td)
            graph = open(os.path.join(td, "graph.in")).read()
        assert cnt == 3 and graph.startswith("3 3")   # "%d %d\r" header rewrite (:500-501)
        for i in range(3):
            for j in range(i + 1, 3):
                ids, L = R.pair_best(i, j)
                assert np.float32(L).tobytes() == np.float32(lens[i, j]).tobytes()
                pairs.append(dict(L_bits=int(np.float32(L).view(np.int32)), sha256_ids=sha(ids.astype(np.int64))))
    else:
        A = O.Acs(G, rng_mode=O.RNG_SEQUENTIAL, sort_mode=O.SORT_STD, seed=4242)
        for k, (i, j) in enumerate([(0, 1), (0, 2), (1, 2)]):
            assert A.set_points(pts[i], pts[j])[0]
            A.begin(0.4, seq_pos=None if k else 0); A.iterate(150)
            ids, _, L = A.best(); A.reset()
            pairs.append(dict(L_bits=int(np.float32(L).view(np.int32)), sha256_ids=sha(ids.astype(np.int64))))
    out["all_pairs"] = pairs
    # seam ordering on unrounded distances, stagnation stop
    D = gtsp_distances()
    if use_ref:
        with tempfile.TemporaryDirectory() as td:
            T = O.RefGtsp(D, os.path.join(td, "g.in")); ran, _ = T.run(30, 5)
    else:
        T = O.Gtsp(D, seed=5, rng_mode=O.RNG_SEQUENTIAL); ran = T.iterate(30, early_stop=True)
    tour, L = T.best()
    out["gtsp"] = dict(ran=int(ran), tour=tour.ravel().tolist(), L_hex=float(L).hex(), sha256_pheromone=sha(T.pheromone()))
    # BS_Basic<float, 3, D, CI, CF>: points, return values, knots, control points
    out["bspline"] = []
    for case, (init, fin, mid, tf, u, pre) in bspline_live_cases():
        pts_, ok, knots, cps = O.bspline(case[0], case[1], case[2], init, fin, mid, tf, u, out=pre, use_ref=use_ref)
        out["bspline"].append(dict(case=list(case), sha256=[sha(pts_), sha(ok), sha(knots), sha(cps)]))
    with open(os.path.join(HERE, "ref_live.json"), "w") as fp:
        json.dump(out, fp, indent=1)
    print("ref_live.json from", out["source"])


if __name__ == "__main__" and sys.argv[1:] == ["bspline"]:
    bspline_fixtures()
elif __name__ == "__main__" and sys.argv[1:] == ["live"]:
    live_fixtures()
elif __name__ == "__main__":
    main()
