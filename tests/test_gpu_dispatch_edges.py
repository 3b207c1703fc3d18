"""GPU parity at the dispatch edges: the host code picks kernel variants on alpha, K, axis length, colony size, step cap,
visited-table size and batch colony size, and the seam ordering sizes its shared memory from the city count.  Every case
here runs a variant (or a size limit) the default configurations never reach, compares it with the CPU oracle, and asserts
the counter or the condition that shows the intended variant ran — so a later change of a threshold cannot silently turn
the case into a duplicate of another one.

  * colony ranking: the last single-CTA colony and the first chunked one, the second staging round of k_rank_merge, and
    step caps whose dead-ant key (cap + 1) no longer fits the 16-bit staged keys;
  * walk kernels with alpha != 1 (resume pass, predicted gathers), the K = 26 variants with non-default parameters, the
    K = 26 walk for axes beyond 1024 nodes, the 10-bit packed coordinates at their limit, K = 26 atomic deposits;
  * concurrent searches: alpha != 1 with parked ants, the largest batch colony and the first colony beyond it;
  * seam ordering at 2, 3, 257 and 464 cities, and the rejection of 465;
  * the debug switches that must not change a single bit.
"""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from conftest import C1_POINTS, ROOT
from test_gpu_batch import same
from test_gpu_gtsp import matrix
from test_gpu_parity import compare_iteration, make_pair

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def wr():
    import welding_robot_b200 as wr
    return wr


def piece_pair(wr, oracle, meshes, **params):
    A, g = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, **params)
    ids = np.flatnonzero(A.grid.isfree())
    s, e = int(ids[40]), int(ids[len(ids) // 3])
    A.set_endpoints(s, e); g.setEndpoints(s, e)
    A.begin(1.0); g.begin(1.0)
    return A, g


def occupancy_pair(wr, oracle, free, dims, **params):
    axes = [np.arange(n, dtype=np.float32) for n in dims]
    G = oracle.Grid.from_occupancy(free, *axes, 1.0)
    A = oracle.Acs(G, **params)
    g = wr.ACS_Rank(**params)
    g.creatFromOccupancy(free, *axes, 1.0)
    g.initFromGridMap()
    return A, g


# ---------------------------------------------------------------------------------------------
# 1. colony ranking (launch_rank, rank_small.cuh)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [6, 26])
@pytest.mark.parametrize("colony", [8192, 8193])
def test_ranking_at_the_single_cta_limit(wr, oracle, meshes, colony, K):
    """8192 ants: the last colony k_rank_small ranks alone; 8193: the chunked path (k_rank_chunks + k_rank_merge +
    k_rank_finish_prefix) with a one-ant last chunk.  Every ant's order, lambda, Q, the best path and the field."""
    A, g = piece_pair(wr, oracle, meshes, seed=31, fixed_colony=colony, step_cap=160, K=K)
    for _ in range(2):
        A.iterate(1); g.iterate(1)
        compare_iteration(A, g)
    c = g.counters()
    assert g.lastColony()[0] == colony and c["ants"] == 2 * colony
    assert c["arrived"] > 0 and c["arrived"] < c["ants"]


def test_ranking_second_staging_round(wr, oracle, meshes):
    """100 000 ants = 25 chunks of 4096: k_rank_merge stages 24 chunks per round, so the last chunk is searched in a second
    staging round.  A step cap of 64 leaves a few dozen distinct keys: long runs of ties across every chunk."""
    A, g = piece_pair(wr, oracle, meshes, seed=53, fixed_colony=100000, step_cap=64)
    A.iterate(1); g.iterate(1)
    compare_iteration(A, g)
    c = g.counters()
    assert g.lastColony()[0] == 100000 and (100000 + 4095) // 4096 > 24
    assert c["ants"] == 100000 and c["arrived"] > 0 and c["dead_step_cap"] > 0


@pytest.mark.timeout(900)
@pytest.mark.parametrize("update_mode", [0, 4])
@pytest.mark.parametrize("step_cap", [65534, 65535, 70000])
def test_ranking_step_caps_beyond_16_bit_keys(wr, oracle, meshes, step_cap, update_mode):
    """A dead ant ranks with the key cap + 1.  The chunked ranking stages keys 16 bits wide only while cap + 1 fits them;
    at cap 65535 the key would wrap to 0 and dead ants would rank ahead of the arrived ones.  9000 ants (chunked path),
    about a fifth of them dead."""
    A, g = piece_pair(wr, oracle, meshes, seed=77, fixed_colony=9000, step_cap=step_cap, update_mode=update_mode)
    assert g.stepCap() == step_cap
    for _ in range(2):
        A.iterate(1); g.iterate(1)
        compare_iteration(A, g)
    oc, gc = A.counters(), g.counters()
    for key in ("ant_steps", "ants", "arrived", "dead_no_candidate", "dead_fallthrough", "dead_step_cap"):
        assert oc[key] == gc[key], key
    assert gc["ants"] == 2 * 9000 and gc["dead_no_candidate"] > 1000 and gc["arrived"] > 0


# ---------------------------------------------------------------------------------------------
# 2. walk kernels
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("alpha", [2, 0])
def test_k6_resume_pass_with_alpha(wr, oracle, meshes, alpha):
    """16-slot visited tables: ants park in k_walk3 and finish in k_walk2<Dense6, false> (the alpha != 1 resume pass)."""
    A, g = piece_pair(wr, oracle, meshes, seed=7, fixed_colony=512, step_cap=300, walk_table_log2=4, alpha=alpha)
    for _ in range(4):
        A.iterate(1); g.iterate(1)
        compare_iteration(A, g)
    c = g.counters()
    assert c["table_overflows"] > 0 and c["arrived"] > 0
    assert c["dead_step_cap"] == A.counters()["dead_step_cap"]


def test_k6_predicted_gathers_with_alpha(wr, oracle, meshes, monkeypatch):
    """Rank-set iterations walk with k_walk3<false, 0>: gathers predicted a trip ahead, power<T> for alpha = 2."""
    monkeypatch.setenv("WR_RANKSET_POLICY", "1")
    A, g = piece_pair(wr, oracle, meshes, seed=19, fixed_colony=640, step_cap=300, update_mode=4, alpha=2, beta=0.9, rho=0.7, tau0=0.5)
    for _ in range(3):
        A.iterate(1); g.iterate(1)
        compare_iteration(A, g)
    A.iterate(8); g.iterate(8)
    compare_iteration(A, g)
    assert g.updateStats()["rankset_iterations"] == 11
    assert g.counters()["arrived"] > 0


@pytest.mark.parametrize("table_log2", [9, 4])
@pytest.mark.parametrize("update_mode", [0, 4])
@pytest.mark.parametrize("alpha,beta,rho,tau0", [(2, 0.9, 0.7, 0.5), (3, 0.3, 0.93, 2.5), (0, 0.6, 0.8, 1.0)])
def test_k26_non_default_parameters(wr, oracle, meshes, alpha, beta, rho, tau0, update_mode, table_log2):
    """K = 26 away from the defaults: k_walk26p's alpha branch, k_heuristic26 with beta != 0.6, evaporation and initial
    pheromone away from 0.8 / 1; with 16-slot tables the ants park and finish in k_walk26<Dense26, true> with alpha != 1."""
    A, g = piece_pair(wr, oracle, meshes, seed=11, fixed_colony=384, step_cap=200, K=26, walk_table_log2=table_log2,
                      alpha=alpha, beta=beta, rho=rho, tau0=tau0, update_mode=update_mode)
    for it in range(3):
        A.iterate(1); g.iterate(1)
        compare_iteration(A, g, check_tau=it in (0, 2))
    A.iterate(6); g.iterate(6)
    compare_iteration(A, g)
    c = g.counters()
    assert c["arrived"] > 0
    assert (c["table_overflows"] > 0) == (table_log2 == 4)
    A.reset(); g.reset()
    assert np.array_equal(A.pheromone().view(np.uint32), g.pheromone().view(np.uint32))


def test_k26_axis_beyond_1024(wr, oracle):
    """A 1100 x 6 x 5 corridor with scattered obstacles, endpoints at both ends: an axis beyond the 10-bit packed
    coordinates, so K = 26 walks with k_walk26<Dense26, false> instead of k_walk26p."""
    dims = (1100, 6, 5)
    rx, ry, rz = dims
    free = np.ones((rz, ry, rx), np.uint8)
    rng = np.random.default_rng(3)
    for _ in range(40):
        free[int(rng.integers(0, rz)), int(rng.integers(0, ry)), int(rng.integers(5, rx - 5))] = 0
    A, g = occupancy_pair(wr, oracle, free.ravel(), dims, seed=5, fixed_colony=128, step_cap=8000, K=26)
    assert max(g.rangeX, g.rangeY, g.rangeZ) > 1024
    nid = lambda x, y, z: (z * ry + y) * rx + x  # noqa: E731
    A.set_endpoints(nid(0, 2, 2), nid(rx - 1, 3, 2)); g.setEndpoints(nid(0, 2, 2), nid(rx - 1, 3, 2))
    A.begin(100.0); g.begin(100.0)
    for _ in range(3):
        A.iterate(1); g.iterate(1)
        compare_iteration(A, g)
    assert g.counters()["arrived"] > 0
    assert g.counters()["ant_steps"] == A.counters()["ant_steps"]


@pytest.mark.parametrize("dims", [(1024, 4, 4), (4, 4, 1024)])
def test_k6_packed_coordinates_at_their_limit(wr, oracle, dims):
    """k_walk3 packs node coordinates into 10 bits per axis: a 1024-node axis walked end to end, from coordinate 0 to
    1023, bit for bit with the oracle."""
    rx, ry, rz = dims
    A, g = occupancy_pair(wr, oracle, np.ones(rx * ry * rz, np.uint8), dims, seed=7, fixed_colony=1024, step_cap=8000)
    assert max(g.rangeX, g.rangeY, g.rangeZ) == 1024
    s, e = 0, rx * ry * rz - 1          # (0, 0, 0) and (rx-1, ry-1, rz-1)
    A.set_endpoints(s, e); g.setEndpoints(s, e)
    A.begin(100.0); g.begin(100.0)
    for _ in range(3):
        A.iterate(1); g.iterate(1)
        compare_iteration(A, g)
    c = g.counters()
    assert c["arrived"] > 0 and c["ant_steps"] == A.counters()["ant_steps"]
    ids = g.bestPath()[0]
    assert ids[0] == s and ids[-1] == e


def test_k26_atomic_update_within_tolerance(wr, oracle, meshes):
    """update_mode 2 with K = 26: k_deposit_gen<true> adds in arbitrary order, hence 1e-5 relative like the K = 6 atomic test;
    the walks of the following iterations read that field and still match the oracle step for step."""
    A, g = piece_pair(wr, oracle, meshes, seed=9, fixed_colony=256, step_cap=400, K=26, update_mode=2)
    A.iterate(1); g.iterate(1)
    compare_iteration(A, g, exact_tau=False)
    assert g.counters()["arrived"] > 0


# ---------------------------------------------------------------------------------------------
# 3. concurrent searches (wr_acs_search_batch)
# ---------------------------------------------------------------------------------------------
def batch_vs_sequential(wr, oracle, meshes, nq, iters, oracle_queries, **params):
    A, g = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, seed=17, **params)
    _, g2 = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, seed=17, **params)
    free = np.flatnonzero(A.grid.isfree())
    rng = np.random.default_rng(2)
    s = [int(v) for v in free[rng.integers(0, len(free), nq)]]
    e = [int(v) for v in free[rng.integers(0, len(free), nq)]]
    seq = g.searchPairs(s, e, 1.0, iterations=iters)
    bat = g2.searchBatch(s, e, 1.0, iterations=iters)
    same(seq, bat)
    assert g.counters()["ant_steps"] == g2.counters()["ant_steps"]
    for q in oracle_queries:
        A.set_endpoints(s[q], e[q]); A.set_next_search(q)
        A.begin(1.0); A.iterate(iters)
        ids, dirs, L = A.best()
        assert (np.isinf(L) and np.isinf(bat[q][2])) or (np.float32(L) == np.float32(bat[q][2]) and np.array_equal(ids, bat[q][0])
                                                         and np.array_equal(dirs, bat[q][1])), q
        A.reset()
    assert sum(np.isfinite(r[2]) for r in bat) > 0
    return g2


def test_batch_alpha2_parked_ants(wr, oracle, meshes, monkeypatch):
    """16-entry batch visited tables with alpha = 2: the parked ants finish in k_walk2<Batch6, false>."""
    monkeypatch.setenv("WR_BATCH_TABLE", "16")
    g2 = batch_vs_sequential(wr, oracle, meshes, 16, 10, (0, 15), fixed_colony=150, step_cap=400, alpha=2, beta=0.9, rho=0.7, tau0=0.5)
    st = g2.batchStats()
    assert st["queries_per_chunk"] > 0 and st["fallbacks"] == 0, st
    assert g2.counters()["table_overflows"] > 0


def test_batch_largest_colony(wr, oracle, meshes):
    """4096 ants (kBatchMaxColony): the batch path with k_batch_rank at its largest shared memory."""
    g2 = batch_vs_sequential(wr, oracle, meshes, 6, 6, (0, 5), fixed_colony=4096, step_cap=300)
    st = g2.batchStats()
    assert st["queries_per_chunk"] > 0 and st["fallbacks"] == 0, st


def test_batch_colony_beyond_batch_limit(wr, oracle, meshes):
    """4097 ants: the batch call runs the sequential loop (no batch buffers), with the same answers."""
    g2 = batch_vs_sequential(wr, oracle, meshes, 4, 4, (3,), fixed_colony=4097, step_cap=300)
    assert g2.batchStats()["queries_per_chunk"] == 0


# ---------------------------------------------------------------------------------------------
# 4. seam ordering sizes (gtsp.cu)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,iters,batch", [(2, 4, 2), (3, 4, 2), (257, 3, 2), (464, 2, 2)])
def test_gtsp_sizes(wr, oracle, n, iters, batch):
    """The smallest tours, the first city count past a warp multiple of 256, and the largest count whose check-points,
    visited bits and TMA ring fit 227 KB of shared memory."""
    D = matrix(n, n)
    g = wr.ACS_GTSP(seed=77)
    g.dis, g.city_num, g.cnt = D, n, n * (n - 1) // 2
    res = g.computeBatch(batch, iters, colony_first=5)
    for b in range(batch):
        T = oracle.Gtsp(D, seed=77, colony_id=5 + b)
        assert T.iterate(iters) == iters
        tour, L = T.best()
        assert g.tau0() == T.tau0()
        assert len(res[b][0]) == len(tour) > 0
        assert np.array_equal(res[b][0], tour), (n, b)
        assert res[b][1] == L
        assert np.array_equal(g.pheromone(b).view(np.uint64), T.pheromone().view(np.uint64))


def test_gtsp_city_limit(wr):
    from welding_robot_b200._lib import WrError
    g = wr.ACS_GTSP(seed=1)
    assert g.setDistanceMatrix(matrix(464, 1))
    with pytest.raises(WrError, match="at most 464 cities"):
        g.setDistanceMatrix(matrix(465, 1))


# ---------------------------------------------------------------------------------------------
# 5. debug switches that must give identical bits (DESIGN.md §6)
# ---------------------------------------------------------------------------------------------
# WR_WALK_PREFETCH, WR_STREAM_CS and WR_GRAPH are read once per process: each setting runs in a child process
# of its own.  The child runs the C1 adaptive scenario, records which kernels ran (torch.profiler) and saves the best path,
# the counters and the final field.
_CHILD = r"""
import sys
import numpy as np
root, out = sys.argv[1], sys.argv[2]
sys.path[:0] = [root, root + "/tests"]
import welding_robot_b200 as wr
from conftest import C1_POINTS
from torch.profiler import ProfilerActivity, profile
g = wr.ACS_Rank(seed=0x5EED, update_mode=4)
g.creatGridMap(np.load(root + "/tests/golden/meshes.npz")["cubic"], 0.005, 10)
g.initFromGridMap()
assert g.setPoints(C1_POINTS[0], C1_POINTS[5])
g.begin(0.5)
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    g.iterate(30)
    g.sync()
kernels = sorted({e.key for e in prof.key_averages()})
ids, dirs, L = g.bestPath()
c = g.counters()
np.savez(out, ids=ids, dirs=dirs, L=np.float32(L), tau=g.pheromone(), kernels=np.array(kernels),
         counter_keys=np.array(list(c)), counter_vals=np.array(list(c.values()), np.uint64))
"""


@pytest.fixture(scope="module")
def c1_oracle_30(oracle, meshes):
    G = oracle.Grid.from_triangles(meshes["cubic"], 0.005, 10, oracle.VOX_AABB)
    A = oracle.Acs(G, seed=0x5EED)
    assert A.set_points(C1_POINTS[0], C1_POINTS[5])[0]
    A.begin(0.5); A.iterate(30)
    return A.best(), A.counters(), A.pheromone()


def _has(kernels, pattern):
    return any(re.search(pattern, k) for k in kernels)


@pytest.mark.parametrize("var,value", [("WR_WALK_PREFETCH", "0"), ("WR_WALK_PREFETCH", "1"), ("WR_STREAM_CS", "0"), ("WR_GRAPH", "0")])
def test_debug_switch_gives_identical_bits(c1_oracle_30, tmp_path, var, value):
    out = tmp_path / "run.npz"
    env = dict(os.environ)
    env[var] = value
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", _CHILD, ROOT, str(out)]
    r = subprocess.run(cmd, env=env, cwd=str(tmp_path), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    res = np.load(out)
    (oids, odirs, oL), oc, otau = c1_oracle_30
    assert np.float32(oL).tobytes() == res["L"].tobytes() and np.isfinite(oL)
    assert np.array_equal(oids, res["ids"]) and np.array_equal(odirs, res["dirs"])
    gc = dict(zip(res["counter_keys"].tolist(), res["counter_vals"].tolist()))
    for key in ("ant_steps", "ants", "arrived", "dead_no_candidate", "dead_fallthrough", "dead_step_cap", "iterations"):
        assert gc[key] == oc[key], key
    assert np.array_equal(otau.view(np.uint32), res["tau"].view(np.uint32)), "pheromone field differs: max |d| = %g" % np.abs(otau - res["tau"]).max()
    # what the setting selects
    kernels = res["kernels"].tolist()
    assert _has(kernels, r"k_walk3<true, ?[01]>"), kernels
    if var == "WR_WALK_PREFETCH":
        assert not _has(kernels, r"k_walk3<true, ?%d>" % (1 - int(value))), kernels
        assert _has(kernels, r"k_walk3<true, ?%s>" % value), kernels
    else:   # the defaults: prefetching walks on record iterations, plain ones on rank-set iterations
        assert _has(kernels, r"k_walk3<true, ?1>"), kernels
        assert _has(kernels, r"k_walk3<true, ?0>") == _has(kernels, r"k_rankset_apply"), kernels


@pytest.mark.parametrize("update_mode", [0, 4])
def test_materialised_field_without_clean_tiles(wr, oracle, meshes, update_mode, monkeypatch):
    """WR_LAZY_TAU=0 (read per handle): the field is explicit from the start — every tile counts as touched — and the
    uploaded-field / reset scenario gives the oracle's bits."""
    monkeypatch.setenv("WR_LAZY_TAU", "0")
    A, g = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, seed=5, fixed_colony=300, step_cap=250, update_mode=update_mode)
    ids = np.flatnonzero(A.grid.isfree())
    s, e = int(ids[30]), int(ids[len(ids) // 3])
    A.set_endpoints(s, e); g.setEndpoints(s, e)
    A.begin(1.0); g.begin(1.0)
    dirty, tiles = g.fieldStats()
    assert dirty == tiles > 0
    assert np.array_equal(A.pheromone().view(np.uint32), g.pheromone().view(np.uint32))
    A.iterate(3); g.iterate(3)
    compare_iteration(A, g)
    A.reset(); g.reset()
    assert g.fieldStats()[0] == tiles
    assert np.array_equal(A.pheromone().view(np.uint32), g.pheromone().view(np.uint32))
    A.begin(1.0); g.begin(1.0)
    A.iterate(2); g.iterate(2)
    compare_iteration(A, g)
    rng = np.random.default_rng(3)
    tau = (0.25 + rng.random(A.pheromone().size)).astype(np.float32)
    A.set_pheromone(tau); g.setPheromone(tau)
    A.begin(1.0); g.begin(1.0)
    for _ in range(3):
        A.iterate(1); g.iterate(1)
        compare_iteration(A, g)
    assert g.fieldStats()[0] == tiles
