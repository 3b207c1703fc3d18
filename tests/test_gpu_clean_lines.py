"""GPU: the line flags of the clean-tile pheromone field.  The evaporation passes read and write only the 128-byte lines
(32 slots) that ever received a deposit, so a writer that forgets to mark a line leaves a real value un-evaporated from
the next iteration on.  Every case counts, from the CPU oracle's field alone, the lines that hold a value other than the
clean-field scalar (tau0 * rho per iteration) and other than the exact zeros of out-of-bounds slots, and checks
fieldLines() / fieldStats() against that count and the whole field bit for bit:

  * C2 exactly as bench.py builds it, iterations 1 and 2 (record path, k_update_fused);
  * a small mesh through each deposit path: sorted records (k_update_fused), rank sets (k_evaporate_lines +
    k_rankset_apply), a rank-set table too small for the iteration (k_deposit_serial), and two in-process shards on the
    record path (k_pull_finals) and on rank sets;
  * reset() (no dirty line), an upload (every line), and a clean line of an already-dirty tile that takes its first deposit
    several iterations later.
"""
import contextlib
import io
import os
import sys

import numpy as np
import pytest

from conftest import GOLDEN, ROOT
from test_gpu_parity import compare_iteration, make_pair

pytestmark = pytest.mark.gpu

LINE, TILE = 32, 4096   # slots per 128-byte line / per 16 KB tile


@pytest.fixture(scope="module")
def wr():
    import welding_robot_b200 as wr
    return wr


def dirty_mask(tau, base):
    """slots of an oracle field that hold a real value: not the clean-field scalar, not an exact +0 (out of bounds)"""
    bits = tau.view(np.uint32)
    m = (bits != np.float32(base).view(np.uint32)) & (bits != 0)
    return np.concatenate([m, np.zeros((-m.size) % TILE, bool)])


def lines_of(mask):
    return mask.reshape(-1, LINE).any(1)


class Tracker:
    """Follows the oracle: the clean-field scalar, and per iteration the dirty lines and tiles it implies."""

    def __init__(self, A, g, tau0=1.0, rho=0.8):
        self.A, self.g, self.rho = A, g, np.float32(rho)
        self.base = np.float32(tau0)
        self.lines = None
        self.late = 0             # lines first dirtied at iteration >= 3 inside a tile dirty since an earlier iteration
        self.it = 0

    def step(self, n=1, compare=True):
        for _ in range(n):
            self.A.iterate(1); self.g.iterate(1)
            self.base = np.float32(self.base * self.rho)
            self.it += 1
            if compare:
                compare_iteration(self.A, self.g)
            self.check()

    def check(self):
        lines = lines_of(dirty_mask(self.A.pheromone(), self.base))
        tiles = lines.reshape(-1, TILE // LINE).any(1)
        if self.lines is not None:
            prev_tiles = self.lines.reshape(-1, TILE // LINE).any(1)
            new = np.flatnonzero(lines & ~self.lines)
            if self.it >= 3:
                self.late += int(prev_tiles[new // (TILE // LINE)].sum())
        self.lines = lines
        assert self.g.fieldLines() == (int(lines.sum()), lines.size)
        assert self.g.fieldStats() == (int(tiles.sum()), tiles.size)

    def reset(self, tau0=1.0):
        self.A.reset(); self.g.reset()
        self.base = np.float32(tau0)
        self.lines = None
        assert self.g.fieldLines()[0] == 0 and self.g.fieldStats()[0] == 0
        assert np.array_equal(self.A.pheromone().view(np.uint32), self.g.pheromone().view(np.uint32))


def deposited_slots(prev, cur, rho=0.8):
    """slots that received a deposit in the iteration between two oracle fields"""
    return int(((np.float32(rho) * prev).view(np.uint32) != cur.view(np.uint32)).sum())


@pytest.mark.timeout(900)
def test_c2_bench_workload_lines(wr, oracle):
    """The bench workload: iteration 1 leaves 211 732 dirty lines (10 404 tiles), iteration 2 adds more."""
    sys.path.insert(0, ROOT)
    import bench
    bench.select_workload("C2")
    wl = bench.build_workload_gpu()
    G = oracle.Grid.from_occupancy(wl["isfree"], wl["xs"], wl["ys"], wl["zs"], bench.PRECISION)
    A = oracle.Acs(G, seed=bench.SEED, fixed_colony=bench.ANTS_PER_GPU, step_cap=bench.STEP_CAP)
    g = wr.ACS_Rank(seed=bench.SEED, fixed_colony=bench.ANTS_PER_GPU, step_cap=bench.STEP_CAP, update_mode=4)
    g.creatFromOccupancy(wl["isfree"], wl["xs"], wl["ys"], wl["zs"], bench.PRECISION)
    g.initFromGridMap()
    A.set_endpoints(wl["start"], wl["goal"]); g.setEndpoints(wl["start"], wl["goal"])
    A.begin(bench.PREDICT); g.begin(bench.PREDICT)
    assert g.fieldLines() == (0, 3145728)
    T = Tracker(A, g)
    T.step(1, compare=False)
    assert g.fieldLines()[0] == 211732 and g.fieldStats()[0] == 10404
    T.step(1, compare=False)
    assert g.fieldLines()[0] > 211732
    assert np.array_equal(A.pheromone().view(np.uint32), g.pheromone().view(np.uint32))


PATHS = {   # deposit path -> (update_mode, environment)
    "records": (0, {}),
    "ranksets": (4, {"WR_RANKSET_POLICY": "1"}),
    "serial": (4, {"WR_RANKSET_POLICY": "1", "WR_RANKSET_LOG2": "6"}),   # 64-block table: every iteration overflows
}


@pytest.mark.parametrize("path", sorted(PATHS))
def test_small_mesh_lines_per_deposit_path(wr, oracle, meshes, path, monkeypatch):
    mode, env = PATHS[path]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    A, g = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, seed=13, fixed_colony=256, step_cap=400, update_mode=mode)
    ids = np.flatnonzero(A.grid.isfree())
    s, e = int(ids[60]), int(ids[-60])
    A.set_endpoints(s, e); g.setEndpoints(s, e)
    A.begin(1.0); g.begin(1.0)
    T = Tracker(A, g)
    T.check()
    prev = A.pheromone()
    for _ in range(8):
        T.step()
        cur = A.pheromone()
        if path == "serial":   # more slots than the 32 blocks the table lists: the chains are skipped for the serial pass
            assert deposited_slots(prev, cur) > 32
        prev = cur
    assert T.late > 0, "no line of an already-dirty tile took its first deposit late"
    st = g.updateStats()
    assert (st["rankset_iterations"] == 8) == (mode == 4), st
    # reset(): no dirty line; the first reset also turns the out-of-bounds zeros into clean slots
    T.reset()
    A.begin(1.0); g.begin(1.0)
    T.step(3)
    # upload: explicit values everywhere, every line dirty
    rng = np.random.default_rng(4)
    tau = (0.25 + rng.random(A.pheromone().size)).astype(np.float32)
    A.set_pheromone(tau); g.setPheromone(tau)
    total = g.fieldLines()[1]
    assert g.fieldLines() == (total, total) and g.fieldStats()[0] == g.fieldStats()[1]
    A.begin(1.0); g.begin(1.0)
    for _ in range(2):
        A.iterate(1); g.iterate(1)
        compare_iteration(A, g)
    assert g.fieldLines() == (total, total)
    T.reset()


@pytest.mark.timeout(600)
def test_late_first_deposit_in_a_dirty_tile(wr, oracle, meshes, monkeypatch):
    """A converging colony on rank sets: lines whose tile has been dirty for several iterations take their first deposit
    late (the best path shifts); the whole field is compared at every iteration, so an evaporation that skipped such a
    line — or streamed a line it should not — shows up within one iteration."""
    monkeypatch.setenv("WR_RANKSET_POLICY", "1")
    A, g = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, seed=13, fixed_colony=256, step_cap=400, update_mode=4)
    ids = np.flatnonzero(A.grid.isfree())
    s, e = int(ids[60]), int(ids[-60])
    A.set_endpoints(s, e); g.setEndpoints(s, e)
    A.begin(1.0); g.begin(1.0)
    T = Tracker(A, g)
    tiles_at = {}
    late_gap = 0
    for it in range(1, 16):
        before = None if T.lines is None else T.lines.copy()
        T.step()
        tiles = T.lines.reshape(-1, TILE // LINE).any(1)
        for t in np.flatnonzero(tiles):
            tiles_at.setdefault(int(t), it)
        if before is not None:
            for ln in np.flatnonzero(T.lines & ~before):
                late_gap = max(late_gap, it - tiles_at[int(ln) // (TILE // LINE)])
    assert late_gap >= 3, late_gap   # a tile dirty since iteration k had a clean line that took its first deposit at k + 3 or later
    assert g.updateStats()["rankset_iterations"] == 15


def _shard_run(wr, oracle, meshes, policy, world, monkeypatch):
    from welding_robot_b200.dist import LocalShards
    monkeypatch.setenv("WR_PEER_TIMEOUT_MS", "8000")
    tris = np.load(os.path.join(GOLDEN, "meshes.npz"))["simplified_piece"]
    G = oracle.Grid.from_triangles(tris, 0.012, 4, oracle.VOX_AABB)
    A = oracle.Acs(G, seed=21, fixed_colony=501, step_cap=600)
    monkeypatch.setenv("WR_RANKSET_POLICY", policy)
    shards = []
    for _ in range(world):
        a = wr.ACS_Rank(seed=21, fixed_colony=501, step_cap=600)
        with contextlib.redirect_stdout(io.StringIO()):
            a.creatGridMap(tris, 0.012, 4)
            a.initFromGridMap()
        shards.append(a)
    monkeypatch.delenv("WR_RANKSET_POLICY")
    free = np.flatnonzero(A.grid.isfree())
    A.set_endpoints(int(free[11]), int(free[-11]))
    for a in shards:
        a.setEndpoints(int(free[11]), int(free[-11]))
    S = LocalShards(shards)
    A.begin(1.0); S.begin(1.0)
    base = np.float32(1.0)
    for _ in range(5):
        A.iterate(1); S.iterate(1); S.sync()
        base = np.float32(base * np.float32(0.8))
        to = A.pheromone()
        lines = lines_of(dirty_mask(to, base))
        for a in shards:
            assert np.array_equal(to.view(np.uint32), a.pheromone().view(np.uint32)), "shard field differs from the oracle"
            assert a.fieldLines() == (int(lines.sum()), lines.size)
    for a in shards:
        assert (a.updateStats()["rankset_iterations"] > 0) == (policy == "1")


@pytest.mark.timeout(600)
@pytest.mark.parametrize("policy", ["2", "1"])   # 2: sorted records + final-value lists (k_pull_finals), 1: rank sets
def test_two_in_process_shards_lines(wr, oracle, meshes, policy, monkeypatch):
    for attempt in range(3):   # a barrier timeout between shards of one process is retried (see test_gpu_shards_local.py)
        try:
            return _shard_run(wr, oracle, meshes, policy, 2, monkeypatch)
        except wr.WrError as e:
            if "did not reach a barrier" not in str(e) or attempt == 2:
                raise
