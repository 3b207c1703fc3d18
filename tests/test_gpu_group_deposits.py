"""GPU: group deposits of converged rank-set iterations (rankset.cuh, rank_small.cuh).  An eligible rank whose local ant
k_path_verify saw follow the whole best path does not walk its trail in k_rankset_gen: the ranking marks it in a 1024-bit
mask per rank group, and extra CTAs of the same launch walk one such ant's trail once and OR each group's mask into the block
of every step.  The table must end up with the same (key, rank bits) as when every rank sets its own bits, so the field is
the same bit for bit.  Every case compares the ants, the best path and the whole field with the CPU oracle (or a sharded
colony with one handle) and checks updateStats()["group_ranks"] against the count the oracle's trails imply:

  * a converging colony whose eligible ranks are a mix of complete ants and ants that leave the path;
  * iterations in which a deviating ant finds a shorter best path, so k_best_copy replaces the path that the group's trail
    was verified against;
  * a colony above 5120 ants (two rank groups, complete ants in both);
  * a 64-block table that overflows into k_deposit_serial;
  * two and three in-process shards against one handle on a small mesh, and two on C2;
  * C2 as bench.py builds it, against the same search with WR_WALK_VERIFY=0 (no group).
"""
import contextlib
import io
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import GOLDEN
from test_gpu_parity import compare_iteration, make_pair
from test_gpu_path_verify import expected_walk_stats

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def wr():
    import welding_robot_b200 as wr
    return wr


def group_expected(best, last_colony, last_ant, start, goal, cap, dims, world=1):
    """Eligible ranks whose ant walked exactly the best path of the start of the iteration (verified as a whole), per shard,
    and a row of what else the iteration reached: eligible ranks, group ranks >= 1024 (the second rank group), and eligible
    ranks with the best path's step count that took another route (not complete).  last_colony / last_ant: the oracle's or
    a handle's accessors of the iteration that just ran."""
    colony, lam, _ = last_colony()
    trails, eligible, orders, keys = [], np.zeros(colony, bool), np.zeros(colony, np.int64), np.zeros(colony, np.int64)
    for k in range(colony):
        ids, _, L, order = last_ant(k)
        trails.append(ids)
        orders[k] = order
        keys[k] = len(ids) - 1 if np.isfinite(L) else cap + 1
        eligible[k] = np.isfinite(L) and not (np.float32(order) > np.float32(np.float32(lam) - np.float32(1.0)))
    _, info = expected_walk_stats(best, trails, start, goal, cap, dims, 0, colony, world)
    complete = (info["D"] == info["n"] - 1) & (info["dev"] == info["D"])
    grp = eligible & complete
    chunk = (max(colony, 1) + world - 1) // world
    per_shard = [int(grp[r * chunk:(r + 1) * chunk].sum()) for r in range(world)]
    row = {"group": int(grp.sum()), "eligible": int(eligible.sum()), "second": int((grp & (orders > 1024)).sum()),
           "same_steps_other_route": int((eligible & (keys == len(best) - 1) & ~complete).sum())}
    return per_shard, row


def _endpoints(A):
    ids = np.flatnonzero(A.grid.isfree())
    return int(ids[10]), int(ids[-10])


def run_vs_oracle(A, g, iters):
    """One iteration at a time: oracle parity and the group counter.  Returns per-iteration rows."""
    s, e = _endpoints(A)
    A.set_endpoints(s, e); g.setEndpoints(s, e)
    A.begin(1.0); g.begin(1.0)
    dims = (g.rangeX, g.rangeY, g.rangeZ)
    rows, total = [], 0
    for it in range(1, iters + 1):
        best = A.best()[0]
        A.iterate(1); g.iterate(1)
        compare_iteration(A, g)
        (want,), row = group_expected(best, A.last_colony, A.last_ant, s, e, g.stepCap(), dims)
        st = g.updateStats()
        assert st["group_ranks"] == want, (it, st, want)
        total += want
        assert st["group_ranks_total"] == total
        rows.append(dict(row, it=it, best_before=len(best) - 1, best_after=len(A.best()[0]) - 1))
    return rows


def test_mixed_group_and_deviating_ranks(wr, oracle, meshes, monkeypatch):
    monkeypatch.setenv("WR_RANKSET_POLICY", "1")
    A, g = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, seed=51, fixed_colony=640, step_cap=300, update_mode=4)
    rows = run_vs_oracle(A, g, 30)
    mixed = [r for r in rows if 0 < r["group"] < r["eligible"]]
    assert len(mixed) >= 10, rows
    assert any(r["group"] > 0 and r["same_steps_other_route"] > 0 for r in rows), rows
    assert rows[-1]["group"] > 0.8 * rows[-1]["eligible"], rows[-1]


def test_shorter_best_path_found_in_a_group_iteration(wr, oracle, meshes, monkeypatch):
    """A small, fast-evaporating colony converges on a detour and keeps shortening it: in those iterations the group's trail is
    the best path of the iteration's start while k_best_copy installs the new, shorter one before the rank sets are built."""
    monkeypatch.setenv("WR_RANKSET_POLICY", "1")
    A, g = make_pair(wr, oracle, meshes["simplified_piece"], 0.012, 4, seed=9, fixed_colony=64, step_cap=600, update_mode=4, rho=0.5)
    rows = run_vs_oracle(A, g, 20)
    events = [r for r in rows if r["group"] > 0 and 0 < r["best_after"] < r["best_before"]]
    assert len(events) >= 2, rows


def test_two_rank_groups(wr, oracle, meshes, monkeypatch):
    """6000 ants: 1199 eligible ranks, so ranks 1024.. live in the second group's mask and blocks."""
    monkeypatch.setenv("WR_RANKSET_POLICY", "1")
    A, g = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, seed=54, fixed_colony=6000, step_cap=300, update_mode=4)
    rows = run_vs_oracle(A, g, 16)
    assert rows[-1]["eligible"] > 1024
    assert sum(r["second"] for r in rows) > 100, rows


def test_table_overflow_into_the_serial_pass(wr, oracle, meshes, monkeypatch):
    """A 64-block table: the group CTAs claim through the same claim limit, the overflow flag is raised and k_deposit_serial
    applies every eligible trail."""
    monkeypatch.setenv("WR_RANKSET_POLICY", "1")
    monkeypatch.setenv("WR_RANKSET_LOG2", "6")
    A, g = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, seed=51, fixed_colony=640, step_cap=300, update_mode=4)
    rows = run_vs_oracle(A, g, 20)
    assert rows[-1]["group"] > 0 and rows[-2]["group"] > 0
    assert g.updateStats()["distinct_slots"] == 0xFFFFFFFF   # iteration 19 overflowed


def _shards(world, monkeypatch):
    """Each shard masks only its own complete ants.  Ties of the ranking go to the lower ant index, so on this mesh the
    eligible complete ants all live in the first shard; the counts per shard are checked exactly, from the single handle's
    trails."""
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
    free = np.flatnonzero(single.isfree())
    s, e = int(free[11]), int(free[-11])
    dims = (single.rangeX, single.rangeY, single.rangeZ)
    totals = np.zeros(world, np.int64)
    for it in range(1, 23):
        best = single.bestPath()[0] if it > 1 else np.zeros(0, np.uint32)
        single.iterate(1); S.iterate(1)
        S.sync()
        want, _ = group_expected(best, single.lastColony, single.lastAnt, s, e, single.stepCap(), dims, world)
        totals += want
        got = [a.updateStats() for a in shards]
        assert [x["group_ranks"] for x in got] == want, (it, got, want)
        assert [x["group_ranks_total"] for x in got] == totals.tolist()
        assert single.updateStats()["group_ranks"] == sum(want)
        if it in (1, 2, 8, 20, 21, 22):
            t1, b1 = single.pheromone(), single.bestPath()
            for a in shards:
                assert np.array_equal(t1.view(np.uint32), a.pheromone().view(np.uint32))
                b2 = a.bestPath()
                assert np.array_equal(b1[0], b2[0]) and np.array_equal(b1[1], b2[1]) and np.float32(b1[2]) == np.float32(b2[2])
    assert totals[0] > 0, totals


@pytest.mark.timeout(900)
@pytest.mark.parametrize("world", [2, 3])
def test_in_process_shards_equal_one_handle(world, monkeypatch):
    import welding_robot_b200 as wr
    for attempt in range(3):   # a barrier timeout between shards of one process is retried on fresh handles (test_gpu_shards_local.py)
        try:
            return _shards(world, monkeypatch)
        except wr.WrError as e:
            if "did not reach a barrier" not in str(e) or attempt == 2:
                raise
            print("barrier timeout between in-process shards, retrying (%d)" % (attempt + 1))


def _c2_shards(monkeypatch):
    import bench
    import welding_robot_b200 as wr
    from welding_robot_b200.dist import LocalShards
    monkeypatch.setenv("WR_PEER_TIMEOUT_MS", "8000")
    wl = bench.build_workload_gpu()

    def make():
        a = wr.ACS_Rank(seed=bench.SEED, fixed_colony=bench.ANTS_PER_GPU, step_cap=bench.STEP_CAP, update_mode=4)
        a.creatFromOccupancy(wl["isfree"], wl["xs"], wl["ys"], wl["zs"], bench.PRECISION)
        with contextlib.redirect_stdout(io.StringIO()):
            a.initFromGridMap()
        a.setEndpoints(wl["start"], wl["goal"])
        return a

    single = make(); single.begin(bench.PREDICT)
    shards = [make() for _ in range(2)]
    S = LocalShards(shards); S.begin(bench.PREDICT)
    per_shard = np.zeros(2, np.int64)
    for it in range(1, 61):
        single.iterate(1); S.iterate(1)
        S.sync()
        got = [a.updateStats()["group_ranks"] for a in shards]
        assert sum(got) == single.updateStats()["group_ranks"], (it, got)
        per_shard += got
        if it in (38, 45, 60):
            t1, b1 = single.pheromone(), single.bestPath()
            for a in shards:
                assert np.array_equal(t1.view(np.uint32), a.pheromone().view(np.uint32)), it
                b2 = a.bestPath()
                assert np.array_equal(b1[0], b2[0]) and np.float32(b1[2]) == np.float32(b2[2])
    print("C2, two shards: group ranks per shard over 60 iterations", per_shard.tolist())
    assert per_shard[0] > 0, per_shard


@pytest.mark.timeout(900)
def test_c2_two_shards_equal_one_handle(monkeypatch):
    """C2 through its switch to rank sets and its convergence, on two shards: the shard that holds the group's ants and the
    one that holds none build one table between them (k_rankset_merge), and the field equals the single handle's."""
    import welding_robot_b200 as wr
    for attempt in range(3):
        try:
            return _c2_shards(monkeypatch)
        except wr.WrError as e:
            if "did not reach a barrier" not in str(e) or attempt == 2:
                raise
            print("barrier timeout between in-process shards, retrying (%d)" % (attempt + 1))


# C2 exactly as bench.py builds it: field, best path and counters after iterations 60 and 125, and the group counters
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
out = {"digests": [], "group": []}
done = 0
for upto in (60, 125):
    acs.iterate(upto - done); done = upto
    h = hashlib.sha256()
    b = acs.bestPath()
    h.update(b[0].tobytes()); h.update(b[1].tobytes()); h.update(np.float32(b[2]).tobytes())
    h.update(acs.pheromone().view(np.uint32).tobytes())
    out["digests"].append(h.hexdigest())
    out["group"].append(acs.updateStats())
out["counters"] = acs.counters()
print("RESULT " + json.dumps(out))
"""


def _child(verify):
    env = dict(os.environ, WR_WALK_VERIFY=verify)
    r = subprocess.run([sys.executable, "-c", CHILD, ROOT], cwd=ROOT, env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stderr[-4000:]
    line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")][-1]
    return json.loads(line[len("RESULT "):])


@pytest.mark.timeout(1500)
def test_bench_workload_group_equals_no_group():
    on, off = _child("1"), _child("0")
    assert on["digests"] == off["digests"]
    assert on["counters"] == off["counters"]
    assert all(s["group_ranks_total"] == 0 for s in off["group"])
    last = on["group"][-1]
    # iteration 125 is a converged rank-set iteration: nearly all of its 820 eligible ranks walked the best path
    assert last["rankset_last"] == 1 and last["group_ranks"] > 700, last
    assert last["group_ranks_total"] > 50 * 700, last
    print("C2 group deposits:", on["group"])
