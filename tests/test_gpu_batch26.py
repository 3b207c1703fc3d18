"""GPU: concurrent searches (wr_acs_search_batch) with the K = 26 neighbourhood against the same searches run one after the
other (wr_acs_search_pairs) and against the oracle's K = 26 mode — best path, its slots and its float32 length of every
query, bit for bit.  Covers the reference's all-pairs workload (C1), non-default parameters, ants that park on a full
visited table and resume from HBM, a chunk that falls back, several chunks, a step cap, the C5 shape, an axis beyond the
1024 nodes of packed coordinates, the colony bounds of the batch, and a used handle (sequential loop)."""
import numpy as np
import pytest

from conftest import C1_NAN_PAIR, C1_POINTS
from test_gpu_batch import same
from test_gpu_dispatch_edges import occupancy_pair
from test_gpu_parity import make_pair, synthetic_boxes

pytestmark = pytest.mark.gpu

COUNTERS = ("ant_steps", "ants", "arrived", "dead_no_candidate", "dead_fallthrough", "dead_step_cap", "deposit_records", "table_overflows")


@pytest.fixture(scope="module")
def wr():
    import welding_robot_b200 as wr
    return wr


def check_oracle(A, s, e, predict, iters, bat, queries):
    """Query q of a batch is search index q: the oracle runs it alone with that index."""
    for q in queries:
        A.set_endpoints(s[q], e[q]); A.set_next_search(q)
        A.begin(predict); A.iterate(iters)
        ids, dirs, L = A.best()
        assert (np.isinf(L) and np.isinf(bat[q][2])) or (np.float32(L) == np.float32(bat[q][2]) and np.array_equal(ids, bat[q][0])
                                                         and np.array_equal(dirs, bat[q][1])), q
        A.reset()


def ran_batched(g):
    st = g.batchStats()
    assert st["queries_per_chunk"] > 0 and st["fallbacks"] == 0, st


def test_c1_all_pairs_k26(wr, oracle, meshes):
    """cubic.stl @ (0.005, 10), K = 26: the 15 pairs + the NaN-plane pair, 150 iterations, adaptive colonies."""
    A, g = make_pair(wr, oracle, meshes["cubic"], 0.005, 10, seed=0x5EED, K=26)
    _, g2 = make_pair(wr, oracle, meshes["cubic"], 0.005, 10, seed=0x5EED, K=26)
    pts = list(C1_POINTS) + list(C1_NAN_PAIR)
    node = g.snapPoints(pts)
    assert (node >= 0).all()
    pairs = [(i, j) for i in range(6) for j in range(i + 1, 6)] + [(6, 7)]
    s = [int(node[i]) for i, _ in pairs]; e = [int(node[j]) for _, j in pairs]
    seq = g.searchPairs(s, e, 0.5, iterations=150)
    bat = g2.searchBatch(s, e, 0.5, iterations=150)
    same(seq, bat)
    ran_batched(g2)
    assert g2.batchStats()["entries_used"] > 0
    assert all(np.isfinite(r[2]) for r in bat[:15])
    for key in COUNTERS:
        assert g.counters()[key] == g2.counters()[key], key
    tau, tau2 = g.pheromone(), g2.pheromone()
    assert tau.size == 26 * g.rangeX * g.rangeY * g.rangeZ
    assert np.array_equal(tau.view(np.uint32), tau2.view(np.uint32))   # both end in the reset() state
    check_oracle(A, s, e, 0.5, 150, bat, (0, 7, 14, 15))
    # a second batch on the same handle continues the search indices, like a second sequential call
    seq2 = g.searchPairs(s[:4], e[:4], 0.5, iterations=40)
    bat2 = g2.searchBatch(s[:4], e[:4], 0.5, iterations=40)
    same(seq2, bat2)
    ran_batched(g2)


@pytest.mark.parametrize("params,env", [
    (dict(fixed_colony=200, step_cap=300), {}),
    (dict(fixed_colony=96, step_cap=300, alpha=2, beta=0.9, rho=0.7, tau0=0.5), {}),
    (dict(fixed_colony=150, step_cap=400, walk_table_log2=4), {}),                     # 16-entry visited tables: ants park and resume
    (dict(fixed_colony=150, step_cap=300), {"WR_BATCH_LOG2": "10"}),                  # 1024-entry pheromone table: the chunk falls back
    (dict(fixed_colony=64, step_cap=300), {"WR_BATCH_MEM_MB": "4", "WR_BATCH_LOG2": "18"}),   # memory for a few queries per chunk only
    (dict(fixed_colony=128, step_cap=24), {}),                                        # a step cap that some ants hit
], ids=["defaults", "alpha2", "parked", "fallback", "chunks", "step_cap"])
def test_fixed_colony_queries_k26(wr, oracle, meshes, params, env, monkeypatch):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    A, g = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, seed=17, K=26, **params)
    _, g2 = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, seed=17, K=26, **params)
    free = np.flatnonzero(A.grid.isfree())
    rng = np.random.default_rng(2)
    s = [int(v) for v in free[rng.integers(0, len(free), 24)]]
    e = [int(v) for v in free[rng.integers(0, len(free), 24)]]
    s[5] = e[5] = int(free[100])            # a query whose start is its goal
    seq = g.searchPairs(s, e, 1.0, iterations=12)
    bat = g2.searchBatch(s, e, 1.0, iterations=12)
    same(seq, bat)
    st = g2.batchStats()
    assert st["queries_per_chunk"] > 0, st
    assert (st["fallbacks"] > 0) == (env.get("WR_BATCH_LOG2") == "10"), st
    if "walk_table_log2" in params:
        assert g2.counters()["table_overflows"] > 0
    if "WR_BATCH_MEM_MB" in env:
        assert st["queries_per_chunk"] < 24, st
    if params["step_cap"] < 100:
        assert g2.counters()["dead_step_cap"] > 0 and g2.counters()["arrived"] > 0
    for key in COUNTERS:
        assert g.counters()[key] == g2.counters()[key], key
    check_oracle(A, s, e, 1.0, 12, bat, (0, 11, 23))


def test_queries_on_an_obstacle_grid_k26(wr):
    """C5 shape at 1/64 of the volume, K = 26: 128^3 boxes grid, coordinates = indices, 96 queries x 256 ants."""
    n = 128
    free = synthetic_boxes(n, 60, 4)
    axis = np.arange(n, dtype=np.float32)
    ids = np.flatnonzero(free)
    rng = np.random.default_rng(5)
    s = [int(v) for v in ids[rng.integers(0, len(ids), 96)]]
    e = [int(v) for v in ids[rng.integers(0, len(ids), 96)]]
    res = []
    for batch in (False, True):
        g = wr.ACS_Rank(seed=5, fixed_colony=256, step_cap=1024, K=26)
        g.creatFromOccupancy(free, axis, axis, axis, 1.0)
        g.initFromGridMap()
        res.append(g.searchPairs(s, e, 100.0, iterations=10, batch=batch))
        if batch:
            ran_batched(g)
        del g
    same(res[0], res[1])
    assert sum(np.isfinite(r[2]) for r in res[1]) > 48


def test_axis_beyond_1024_k26(wr, oracle):
    """A 1100 x 6 x 5 corridor with scattered obstacles: k_walk_batch26 uses unpacked coordinates, so an axis beyond 1024
    nodes batches like any other grid."""
    dims = (1100, 6, 5)
    rx, ry, rz = dims
    free = np.ones((rz, ry, rx), np.uint8)
    rng = np.random.default_rng(3)
    for _ in range(40):
        free[int(rng.integers(0, rz)), int(rng.integers(0, ry)), int(rng.integers(5, rx - 5))] = 0
    params = dict(seed=5, fixed_colony=128, step_cap=8000, K=26)
    A, g = occupancy_pair(wr, oracle, free.ravel(), dims, **params)
    _, g2 = occupancy_pair(wr, oracle, free.ravel(), dims, **params)
    assert max(g.rangeX, g.rangeY, g.rangeZ) > 1024
    nid = lambda x, y, z: (z * ry + y) * rx + x  # noqa: E731
    s = [nid(0, 2, 2), nid(rx - 1, 0, 0), nid(300, 5, 4)]
    e = [nid(rx - 1, 3, 2), nid(2, 5, 4), nid(800, 0, 1)]
    assert all(free.ravel()[v] for v in s + e)
    seq = g.searchPairs(s, e, 100.0, iterations=3)
    bat = g2.searchBatch(s, e, 100.0, iterations=3)
    same(seq, bat)
    ran_batched(g2)
    assert all(np.isfinite(r[2]) for r in bat)
    for key in COUNTERS:
        assert g.counters()[key] == g2.counters()[key], key
    check_oracle(A, s, e, 100.0, 3, bat, (0, 2))


@pytest.mark.parametrize("colony,batched", [(4096, True), (4097, False)])
def test_colony_bounds_k26(wr, oracle, meshes, colony, batched):
    """4096 ants (the largest batch colony) run concurrently; 4097 run as the sequential loop.  Same answers either way."""
    params = dict(seed=17, fixed_colony=colony, step_cap=300, K=26)
    A, g = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, **params)
    _, g2 = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, **params)
    free = np.flatnonzero(A.grid.isfree())
    rng = np.random.default_rng(2)
    s = [int(v) for v in free[rng.integers(0, len(free), 4)]]
    e = [int(v) for v in free[rng.integers(0, len(free), 4)]]
    seq = g.searchPairs(s, e, 1.0, iterations=4)
    bat = g2.searchBatch(s, e, 1.0, iterations=4)
    same(seq, bat)
    if batched:
        ran_batched(g2)
    else:
        assert g2.batchStats()["queries_per_chunk"] == 0
    assert g.counters()["ant_steps"] == g2.counters()["ant_steps"]
    assert sum(np.isfinite(r[2]) for r in bat) > 0
    check_oracle(A, s, e, 1.0, 4, bat, (3,))


def test_used_handle_runs_sequentially_k26(wr, oracle, meshes):
    """A K = 26 handle whose field carries deposits (iterated without reset()): the batch call takes the sequential loop."""
    _, g = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, seed=4, fixed_colony=128, step_cap=300, K=26)
    _, g2 = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, seed=4, fixed_colony=128, step_cap=300, K=26)
    free = np.flatnonzero(g.isfree())
    s = [int(free[10]), int(free[500])]; e = [int(free[-10]), int(free[-700])]
    for h in (g, g2):
        h.setEndpoints(s[0], e[1]); h.begin(1.0); h.iterate(3)
    same(g.searchPairs(s, e, 1.0, iterations=8), g2.searchBatch(s, e, 1.0, iterations=8))
    assert g2.batchStats()["queries_per_chunk"] == 0
