"""Path verification of converged iterations (path_verify.cuh): ants that follow the best path are checked against
per-position roulette thresholds instead of walking it, and k_walk3 resumes each warp where its first ant leaves the path.
The walk must produce the same bits as walking every step: against the same search with WR_WALK_VERIFY=0 on the bench
workload, and against the CPU oracle where the predicted walk runs from the first iteration (WR_RANKSET_POLICY=1)."""
import contextlib
import io
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import C1_NAN_PAIR, GOLDEN
from test_gpu_parity import compare_iteration, make_pair

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def wr():
    import welding_robot_b200 as wr
    return wr

# The C2 workload exactly as bench.py builds it (256^3 grid, 4096 ants, step cap 8192, seed 1), 60 iterations; a digest of
# every ant's trail, step count and order, the best path and the whole pheromone field after iterations 30, 45 and 60.
CHILD = r"""
import contextlib, hashlib, io, json, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import bench
import welding_robot_b200 as wr
wl = bench.build_workload_gpu()
acs = wr.ACS_Rank(seed=bench.SEED, fixed_colony=bench.ANTS_PER_GPU, step_cap=bench.STEP_CAP, update_mode=4)
acs.creatFromOccupancy(wl["isfree"], wl["xs"], wl["ys"], wl["zs"], bench.PRECISION)
with contextlib.redirect_stdout(io.StringIO()):
    acs.initFromGridMap()
acs.setEndpoints(wl["start"], wl["goal"])
acs.begin(bench.PREDICT)
out = {"digests": []}
done = 0
for upto in (30, 45, 60):
    acs.iterate(upto - done); done = upto
    h = hashlib.sha256()
    colony = acs.lastColony()[0]
    for k in range(colony):
        ids, dirs, L, order = acs.lastAnt(k)
        h.update(ids.tobytes()); h.update(dirs.tobytes()); h.update(np.float32(L).tobytes()); h.update(np.int64(order).tobytes())
    b = acs.bestPath()
    h.update(b[0].tobytes()); h.update(b[1].tobytes()); h.update(np.float32(b[2]).tobytes())
    h.update(acs.pheromone().view(np.uint32).tobytes())
    out["digests"].append(h.hexdigest())
out["counters"] = acs.counters()
out["walk"] = acs.walkStats()
out["rankset_iterations"] = acs.updateStats()["rankset_iterations"]
print("RESULT " + json.dumps(out))
"""


def _child(verify):
    env = dict(os.environ, WR_WALK_VERIFY=verify)
    r = subprocess.run([sys.executable, "-c", CHILD, ROOT], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stderr[-4000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1]
    return json.loads(line[len("RESULT "):])


@pytest.mark.timeout(1500)
def test_bench_workload_verify_on_equals_off():
    on, off = _child("1"), _child("0")
    assert on["digests"] == off["digests"]
    assert on["counters"] == off["counters"]
    assert off["walk"] == {"verified_ants": 0, "verified_steps": 0}
    # iterations 37-60 of this search are rank-set iterations in which a shrinking minority of ants still leaves the path
    # (profiles/r3_walk_deviation.json): the check decides most of their steps, and completes every ant of the warps without one
    rs = on["rankset_iterations"]
    assert rs > 0
    assert on["walk"]["verified_steps"] > 0.4 * 735 * 4096 * rs, on
    assert on["walk"]["verified_ants"] > 0.2 * 4096 * rs, on
    print("C2 60 iterations:", on["walk"], "rank-set iterations", on["rankset_iterations"])


def _endpoints(A):
    ids = np.flatnonzero(A.grid.isfree())
    return int(ids[10]), int(ids[-10])


def tile_of(node, rx, ry):
    """k_walk3's visited-table key of a node: its 4 x 4 x 2 tile."""
    x, y, z = node % rx, (node // rx) % ry, node // (rx * ry)
    return (x >> 2, y >> 2, z >> 1)


def expected_walk_stats(best, trails, start, goal, cap, dims, table_log2=0, colony=None, world=1, nonfinite=()):
    """walkStats() increments of one converged iteration, from the CPU oracle alone.

    best: the best path's node ids before the iteration; trails: every ant's node ids from the iteration (the oracle keeps
    them for dead ants too); nonfinite: best-path positions whose roulette total or suffix sums are not finite.  The
    verifiable prefix D is the first position the check cannot decide (step cap, visited table full, non-finite sums); an
    ant's dev is the first step it leaves the best path.  Warps of four consecutive ants of a shard either book their ants
    complete (every ant followed the whole path) or resume at the lowest floor8(dev) of their ants.
    Returns ([{verified_ants, verified_steps} per shard], {D, n, dev, warps: [(shard, first ant, present, T, done)]})."""
    rx, ry, _ = dims
    n = len(best)
    D = n - 1 if 2 <= n <= cap + 1 else 0
    limit = ((1 << table_log2 if table_log2 > 0 else 768) >> 2) * 3
    if D > 0:
        assert int(best[0]) == start and int(best[-1]) == goal
        tiles = set()
        for t in range(D):
            tiles.add(tile_of(int(best[t]), rx, ry))
            if t + 1 >= cap or len(tiles) > limit or t in nonfinite:
                D = t
                break
    colony = len(trails) if colony is None else colony
    dev = np.empty(colony, np.int64)
    for k in range(colony):
        tr = trails[k]
        m = min(D, len(tr) - 1)
        diff = np.flatnonzero(np.asarray(tr[1:m + 1]) != np.asarray(best[1:m + 1]))
        dev[k] = diff[0] if len(diff) else m
    complete = (D == n - 1) & (dev == D)
    chunk = (max(colony, 1) + world - 1) // world
    counts, warps = [], []
    for r in range(world):
        first, last = min(r * chunk, colony), min((r + 1) * chunk, colony)
        ants = steps = 0
        for w0 in range(first, last, 4):
            present = list(range(w0, min(w0 + 4, last)))
            done = bool(all(complete[present]))
            T = min(int(dev[k]) & ~7 for k in present)
            if done:
                ants += len(present); steps += len(present) * (n - 1)
            else:
                steps += len(present) * T
            warps.append((r, w0, len(present), T, done))
        counts.append({"verified_ants": ants, "verified_steps": steps})
    return counts, {"D": D, "n": n, "dev": dev, "warps": warps}


def oracle_step(A, start, goal, cap, dims, table_log2=0, world=1, nonfinite=()):
    """One oracle iteration and its expected walkStats() increments per shard (expected_walk_stats)."""
    best = A.best()[0]
    A.iterate(1)
    colony = A.last_colony()[0]
    trails = [A.last_ant(k)[0] for k in range(colony)]
    return expected_walk_stats(best, trails, start, goal, cap, dims, table_log2, colony, world, nonfinite)


def add_stats(total, counts):
    return [{k: t[k] + c[k] for k in t} for t, c in zip(total, counts)]


def _run_vs_oracle(A, g, iters=(1, 1, 1, 1, 12, 14), table_log2=0):
    s, e = _endpoints(A)
    A.set_endpoints(s, e); g.setEndpoints(s, e)
    A.begin(1.0); g.begin(1.0)
    dims = (g.rangeX, g.rangeY, g.rangeZ)
    want = [{"verified_ants": 0, "verified_steps": 0}]
    for n in iters:
        for _ in range(n):
            want = add_stats(want, oracle_step(A, s, e, g.stepCap(), dims, table_log2)[0])
        g.iterate(n)
        compare_iteration(A, g)
        assert g.walkStats() == want[0]
    oc, gc = A.counters(), g.counters()
    for key in ("ant_steps", "ants", "arrived", "dead_no_candidate", "dead_fallthrough", "dead_step_cap"):
        assert oc[key] == gc[key], key
    assert g.updateStats()["rankset_iterations"] == sum(iters)
    return gc


@pytest.mark.parametrize("alpha", [1, 2, 0])
def test_piece_alpha_bit_exact(wr, oracle, meshes, alpha, monkeypatch):
    monkeypatch.setenv("WR_RANKSET_POLICY", "1")
    A, g = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, seed=51, fixed_colony=640, step_cap=300, update_mode=4, alpha=alpha)
    _run_vs_oracle(A, g)
    st = g.walkStats()
    print("alpha", alpha, st)
    if alpha == 1:
        assert st["verified_steps"] > 0, st


def test_small_tables_fill_inside_the_verified_prefix(wr, oracle, meshes, monkeypatch):
    """16-entry visited tables (12 tiles): the verifiable prefix ends where a table would fill; the rest parks and resumes in HBM."""
    monkeypatch.setenv("WR_RANKSET_POLICY", "1")
    A, g = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, seed=52, fixed_colony=512, step_cap=300, update_mode=4, walk_table_log2=4)
    gc = _run_vs_oracle(A, g, table_log2=4)
    assert gc["table_overflows"] > 0


def test_step_cap_around_the_best_length(wr, oracle, meshes, monkeypatch):
    monkeypatch.setenv("WR_RANKSET_POLICY", "1")
    A, g = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, seed=53, fixed_colony=512, step_cap=300, update_mode=4)
    _run_vs_oracle(A, g)
    best_steps = len(g.bestPath()[0]) - 1
    assert best_steps > 2
    for cap in (best_steps + 1, best_steps - 1):
        A, g = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, seed=53, fixed_colony=512, step_cap=cap, update_mode=4)
        _run_vs_oracle(A, g)


def test_nan_pair_has_no_path_to_verify(wr, oracle, meshes, monkeypatch):
    monkeypatch.setenv("WR_RANKSET_POLICY", "1")
    A, g = make_pair(wr, oracle, meshes["cubic"], 0.005, 10, seed=0x5EED, update_mode=4)
    ok, s, e = A.set_points(*C1_NAN_PAIR)
    assert g.setPoints(*C1_NAN_PAIR) and ok
    A.begin(0.5); g.begin(0.5)
    for _ in range(3):
        A.iterate(1); g.iterate(1)
        compare_iteration(A, g)
    assert np.isinf(g.bestPath()[2]) and g.walkStats()["verified_steps"] == 0


@pytest.mark.timeout(600)
@pytest.mark.parametrize("world", [2, 3])
def test_in_process_shards_equal_one_handle(world, monkeypatch):
    import welding_robot_b200 as wr
    from welding_robot_b200.dist import LocalShards
    monkeypatch.setenv("WR_PEER_TIMEOUT_MS", "8000")
    monkeypatch.setenv("WR_RANKSET_POLICY", "1")
    tris = np.load(os.path.join(GOLDEN, "meshes.npz"))["simplified_piece"]

    def make():
        a = wr.ACS_Rank(seed=23, fixed_colony=700, step_cap=600)
        with contextlib.redirect_stdout(io.StringIO()):
            a.creatGridMap(tris, 0.012, 4)
            a.initFromGridMap()
        free = np.flatnonzero(a.isfree())
        a.setEndpoints(int(free[11]), int(free[-11]))
        return a

    single = make(); single.begin(1.0)
    shards = [make() for _ in range(world)]
    S = LocalShards(shards); S.begin(1.0)
    for its in (1, 1, 6, 12):
        single.iterate(its); S.iterate(its)
        S.sync()
        t1, b1 = single.pheromone(), single.bestPath()
        for a in shards:
            assert np.array_equal(t1.view(np.uint32), a.pheromone().view(np.uint32))
            b2 = a.bestPath()
            assert np.array_equal(b1[0], b2[0]) and np.array_equal(b1[1], b2[1]) and np.float32(b1[2]) == np.float32(b2[2])
    assert sum(a.counters()["ant_steps"] for a in shards) == single.counters()["ant_steps"]
    assert all(a.walkStats()["verified_steps"] > 0 for a in shards)
