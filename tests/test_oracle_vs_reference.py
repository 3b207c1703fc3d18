"""CPU: the oracle restatement against what the UNMODIFIED reference computes for these inputs, stored in
tests/golden/ref_live.json (tests/golden/make_golden.py live: recorded through oracle/_ref/libwrref.so where that is built,
its "source" field says by what), bit for bit."""
import hashlib
import json
import os
import sys
import tempfile

import numpy as np
import pytest

from conftest import GOLDEN

sys.path.insert(0, GOLDEN)
import make_golden as MG  # noqa: E402


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def live():
    with open(os.path.join(GOLDEN, "ref_live.json")) as f:
        return json.load(f)


def test_voxel_grid_and_grid_file_round_trip(oracle, meshes, live):
    want = live["grid"]
    G = oracle.Grid.from_triangles(meshes["simplified_piece"], 0.015, 4, oracle.VOX_AABB)
    xs, ys, zs = G.coords()
    assert list(G.dims) == want["dims"] and sha(G.isfree()) == want["sha256_isfree"]
    assert [sha(v) for v in (xs, ys, zs)] == want["sha256_xyz"]
    with tempfile.TemporaryDirectory() as td:
        # the reference's dump carries the LAST triangle's box (model_grid_map.hpp:279): its own reload
        # rebuilds wrong coordinates; compat=True reproduces that, compat=False writes the global box
        f_compat = os.path.join(td, "compat.in"); f_fixed = os.path.join(td, "fixed.in")
        G.write_file(f_compat, compat=True); G.write_file(f_fixed, compat=False)
        assert hashlib.sha256(open(f_compat, "rb").read()).hexdigest() == want["sha256_file"]
        H = oracle.Grid.read_file(f_compat)
        assert sha(H.isfree()) == want["reload_sha256_isfree"]
        assert [sha(v) for v in H.coords()] == want["reload_sha256_xyz"]
        assert not np.array_equal(H.coords()[0], xs)        # the reference bug, reproduced
        F = oracle.Grid.read_file(f_fixed)
        assert np.allclose(F.coords()[0], xs, atol=1e-6)


def test_search_live_on_second_mesh(oracle, meshes, live):
    """A search on a mesh the other fixtures do not cover: best path, length and the full pheromone field
    after 1, 3 and 25 iterations, bit for bit, under the shared sequential Philox stream."""
    want = live["search"]
    G = oracle.Grid.from_triangles(meshes["test"], 0.08, 4, oracle.VOX_AABB)
    A = oracle.Acs(G, rng_mode=oracle.RNG_SEQUENTIAL, sort_mode=oracle.SORT_STD, seed=99)
    p, q = MG.search_points(G)
    assert list(A.set_points(p, q)) == want["set_points"]
    for iters in (1, 3, 25):
        A.begin(3.0); A.iterate(iters)
        ids, dirs, L = A.best()
        w = want[str(iters)]
        assert int(np.float32(L).view(np.int32)) == w["L_bits"]
        assert sha(ids.astype(np.int64)) == w["sha256_ids"] and sha(dirs.astype(np.int32)) == w["sha256_dirs"]
        assert sha(A.pheromone()) == w["sha256_tau"]
        A.reset()
    assert A.counters()["finite_fallthrough"] == 0


def test_all_pairs_driver_through_files(oracle, meshes, live):
    """The genuine searchBestPathOfPoints (ACSRank_3D.hpp:427-504), which drives the pairs through its file interface:
    every pair's best path and length."""
    G = oracle.Grid.from_triangles(meshes["cubic"], 0.01, 5, oracle.VOX_AABB)
    pts = MG.all_pairs_points(G)
    A = oracle.Acs(G, rng_mode=oracle.RNG_SEQUENTIAL, sort_mode=oracle.SORT_STD, seed=4242)
    pairs = [(i, j) for i in range(3) for j in range(i + 1, 3)]
    assert len(pairs) == len(live["all_pairs"]) == 3
    for k, ((i, j), w) in enumerate(zip(pairs, live["all_pairs"])):
        assert A.set_points(pts[i], pts[j])[0]
        A.begin(0.4, seq_pos=None if k else 0); A.iterate(150)   # the driver never reseeds between pairs
        ids, dirs, L = A.best()
        A.reset()
        assert int(np.float32(L).view(np.int32)) == w["L_bits"] and sha(ids.astype(np.int64)) == w["sha256_ids"]


def test_gtsp_live(oracle, live):
    want = live["gtsp"]
    T = oracle.Gtsp(MG.gtsp_distances(), seed=5, rng_mode=oracle.RNG_SEQUENTIAL)
    assert T.iterate(30, early_stop=True) == want["ran"]
    tour, L = T.best()
    assert tour.ravel().tolist() == want["tour"] and float(L).hex() == want["L_hex"]
    assert sha(T.pheromone()) == want["sha256_pheromone"]


def test_bspline_restatement_equals_reference_header(oracle, live):
    """Random valid setups of every (DEGREE, CI, CF) the harness instantiates, restatement == unmodified BSplineBasic.h."""
    cases = list(MG.bspline_live_cases())
    assert len(cases) == len(live["bspline"]) == 36
    for (case, (init, fin, mid, tf, u, pre)), w in zip(cases, live["bspline"]):
        assert list(case) == w["case"]
        pts, ok, knots, cps = oracle.bspline(case[0], case[1], case[2], init, fin, mid, tf, u, out=pre)
        assert [sha(pts), sha(ok), sha(knots), sha(cps)] == w["sha256"], case
