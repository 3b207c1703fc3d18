"""GPU parity of concurrent searches (wr_acs_search_batch) at the edges where the batch path branches.  Every case runs
on a synthetic occupancy grid whose path lengths and pheromone-table claims are known in advance, and checks EVERY query
three ways: against the CPU oracle run query by query with the same search index, against the sequential loop
(searchPairs) on a twin handle, and through the counter sums.  The batch's pheromone table cannot be downloaded, so the
counters (ant steps, ants, arrivals, deaths) are the fingerprint of every ant's walk: a pheromone difference that changes
one choice shows up there.  Each case also asserts the condition that shows it reached its edge.

  1. the pheromone-table claim limit (T/2) hit exactly, and a probe cluster that wraps past slot T - 1;
  2. the pool of HBM visited tables for parked ants, exactly full and one short (WR_BATCH_POOL);
  3. chunks with mixed outcomes: one middle chunk falls back to the sequential loop, the last chunk holds one query, and
     later calls on the same handle reuse or re-size the buffers;
  4. k_batch_deposit's 256-step trips: eligible ants of exactly 256 and 512 steps and longer, every iteration count;
  5. adaptive colonies that shrink to 0-3 ants;
  6. search indices that cross 2^16 and wrap at 2^32 inside one batch.
"""
import numpy as np
import pytest

from test_gpu_dispatch_edges import occupancy_pair

pytestmark = pytest.mark.gpu

KEYS = ("ant_steps", "ants", "arrived", "dead_no_candidate", "dead_fallthrough", "dead_step_cap")
U32 = 0xFFFFFFFF


@pytest.fixture(scope="module")
def wr():
    import welding_robot_b200 as wr
    return wr


def nid(dims, x, y, z=0):
    rx, ry, _ = dims
    return (z * ry + y) * rx + x


def handles(wr, oracle, free, dims, **params):
    """(oracle, batch handle, sequential twin) on the same occupancy grid with the same parameters."""
    A, g = occupancy_pair(wr, oracle, free, dims, **params)
    _, twin = occupancy_pair(wr, oracle, free, dims, **params)
    return A, g, twin


def oracle_queries(A, s, e, predict, iters, first):
    """The oracle, query by query with search index first + q: best (ids, dirs, L) per query, the colony size of each of
    its iterations and the sum of the per-query counters."""
    res, colonies, tot = [], [], dict.fromkeys(KEYS, 0)
    for q in range(len(s)):
        c0 = A.counters()
        A.set_endpoints(s[q], e[q]); A.set_next_search((first + q) & U32)
        A.begin(predict)
        col = []
        for _ in range(iters):
            A.iterate(1)
            col.append(A.last_colony()[0])
        res.append(A.best()); colonies.append(col)
        c1 = A.counters()
        for k in KEYS:
            tot[k] += c1[k] - c0[k]
        A.reset()
    return res, colonies, tot


def counted(g, fn):
    c0 = g.counters()
    out = fn()
    c1 = g.counters()
    return out, {k: c1[k] - c0[k] for k in KEYS}


def run_batch(g, s, e, predict, iters, first):
    g.setNextSearch(first)
    return counted(g, lambda: g.searchBatch(s, e, predict, iterations=iters))


def run_sequential(g, s, e, predict, iters, first):
    g.setNextSearch(first)
    return counted(g, lambda: g.searchPairs(s, e, predict, iterations=iters))


def same_as_oracle(ores, gres, what):
    assert len(ores) == len(gres)
    for q, ((oi, od, oL), (gi, gd, gL)) in enumerate(zip(ores, gres)):
        if np.isinf(oL):   # no path: the oracle keeps the ids of an earlier search, the handle reports none
            assert np.isinf(gL) and len(gi) == 0, (what, q, gL)
            continue
        assert np.float32(oL).tobytes() == np.float32(gL).tobytes(), (what, q, oL, gL)
        assert np.array_equal(oi, gi) and np.array_equal(od, gd), (what, q)


def check_all(A, g, twin, s, e, predict, iters, first):
    """Every query of one batch call against the oracle and the sequential loop; returns the oracle's colony sizes per
    query and iteration, and its counter sums."""
    ores, colonies, otot = oracle_queries(A, s, e, predict, iters, first)
    bres, bcnt = run_batch(g, s, e, predict, iters, first)
    sres, scnt = run_sequential(twin, s, e, predict, iters, first)
    same_as_oracle(ores, bres, "batch")
    same_as_oracle(ores, sres, "sequential")
    assert bcnt == otot, (bcnt, otot)
    assert scnt == otot, (scnt, otot)
    return colonies, otot


# ---------------------------------------------------------------------------------------------
# 1. pheromone-table claim limit (batch_find_or_insert: claim `at < limit`, limit = T/2)
# ---------------------------------------------------------------------------------------------
CORRIDOR_DIMS = (64, 3, 1)   # only row y = 2 is free: a 1 x 64 corridor whose node ids make a probe cluster wrap (below)
CORRIDOR_ROW = 2


def corridor():
    free = np.zeros(CORRIDOR_DIMS[::-1], np.uint8)
    free[0, CORRIDOR_ROW, :] = 1
    return free.ravel()


def batch_hash(node, q):
    """batch.cuh batch_hash in u32 arithmetic."""
    node = np.asarray(node, np.uint64); q = np.asarray(q, np.uint64); m = np.uint64(U32)
    return ((node * np.uint64(2654435761)) & m) ^ ((q * np.uint64(0x85EBCA6B) + (q << np.uint64(13))) & m)


def wrapping_keys(keys, log2):
    """Keys (node, query-in-chunk) of a linear-probing table of 2^log2 entries: the number of keys that MUST be placed past
    slot T - 1 (0 when no probe chain wraps).  The occupied slots do not depend on the insertion order; slots [a, T - 1] of
    the cluster that ends at T - 1 can only hold keys homed in [a, T - 1], so any excess wraps whatever the order."""
    T = 1 << log2
    homes = (batch_hash([k[0] for k in keys], [k[1] for k in keys]) >> np.uint64(32 - log2)).astype(np.int64)
    occ = np.zeros(T, bool)
    for h in homes:
        while occ[h]:
            h = (h + 1) % T
        occ[h] = True
    if not (occ[T - 1] and occ[0]):
        return 0
    a = T - 1
    while occ[a - 1]:
        a -= 1
    return max(0, int((homes >= a).sum()) - (T - a))


@pytest.mark.parametrize("K", [6, 26])
def test_claim_limit_exact(wr, oracle, K, monkeypatch):
    """T = 1024, limit 512.  Each full-corridor query claims exactly 64 entries: deposits on nodes 0-62 of its path and the
    best-path flag on the goal.  8 queries claim 512 (no fallback), a start == goal query adds none, and a one-step query
    adds two more (exactly one fallback, same results)."""
    monkeypatch.setenv("WR_BATCH_LOG2", "10")
    dims = CORRIDOR_DIMS
    A, g, twin = handles(wr, oracle, corridor(), dims, seed=41, fixed_colony=10, step_cap=200, K=K)
    ends = (nid(dims, 0, CORRIDOR_ROW), nid(dims, 63, CORRIDOR_ROW))
    s = [ends[q % 2] for q in range(8)]
    e = [ends[1 - q % 2] for q in range(8)]
    nodes = range(nid(dims, 0, CORRIDOR_ROW), nid(dims, 64, CORRIDOR_ROW))
    assert wrapping_keys([(n, q) for q in range(8) for n in nodes], 10) > 0   # batch_find follows a chain past slot T - 1

    _, tot = check_all(A, g, twin, s, e, 64.0, 3, 100)
    st = g.batchStats()
    assert st["table_entries"] == 1024 and st["entries_used"] == 512 and st["fallbacks"] == 0, st
    assert tot["arrived"] == tot["ants"] == 8 * 3 * 10 and tot["ant_steps"] == 63 * tot["ants"]

    mid = nid(dims, 30, CORRIDOR_ROW)
    _, tot = check_all(A, g, twin, s + [mid], e + [mid], 64.0, 3, 200)   # start == goal: no ant arrives, nothing is claimed
    st = g.batchStats()
    assert st["entries_used"] == 512 and st["fallbacks"] == 0, st
    assert tot["dead_fallthrough"] == 3 * 10

    check_all(A, g, twin, s + [mid], e + [mid + 1], 64.0, 3, 300)         # one step: two claims past the limit
    st = g.batchStats()
    assert st["entries_used"] > 512 and st["fallbacks"] == 1, st


# ---------------------------------------------------------------------------------------------
# 2. pool of HBM visited tables for parked ants (k_walk_batch3 `fits = o < pool`, Batch26::park)
# ---------------------------------------------------------------------------------------------
def ladder(n):
    """An n x 2 x 1 grid, every node free: two lanes side by side."""
    return np.ones(n * 2, np.uint8), (n, 2, 1)


@pytest.mark.parametrize("K", [6, 26])
def test_overflow_pool_exhaustion(wr, oracle, K, monkeypatch):
    """Visited tables of 16 entries (12 tiles of 4 x 4 x 2 nodes): an ant that gets 48 nodes along a 100-node ladder parks.
    One iteration: P parked ants need P pool tables.  A pool of P gives no fallback, a pool of P - 1 exactly one.  The ant
    that found no table must not be resumed: K = 6's resume pass once walked overflow_n ants, one past the pool, from a
    table and a resume record that were never written; it now stops at the pool, as the K = 26 pass does."""
    free, dims = ladder(100)
    params = dict(seed=23, fixed_colony=24, step_cap=300, beta=1.0, K=K)
    if K == 26:
        params["walk_table_log2"] = 4
    else:
        monkeypatch.setenv("WR_BATCH_TABLE", "16")
    A, g, twin = handles(wr, oracle, free, dims, **params)
    s = [nid(dims, 0, 0), nid(dims, 99, 1), nid(dims, 0, 1)]
    e = [nid(dims, 99, 0), nid(dims, 0, 0), nid(dims, 99, 1)]
    c0 = g.counters()["table_overflows"]
    check_all(A, g, twin, s, e, 100.0, 1, 7)
    P = g.counters()["table_overflows"] - c0
    assert P >= 2 and g.batchStats()["fallbacks"] == 0
    for pool, fallbacks in ((P, 0), (P - 1, 1)):
        monkeypatch.setenv("WR_BATCH_POOL", str(pool))
        _, h = occupancy_pair(wr, oracle, free, dims, **params)
        check_all(A, h, twin, s, e, 100.0, 1, 7)
        assert h.batchStats()["fallbacks"] == fallbacks, (pool, P)


# ---------------------------------------------------------------------------------------------
# 3. chunks with mixed outcomes (per-chunk restore after a fallback; buffers reused or re-sized)
# ---------------------------------------------------------------------------------------------
# rows 0-1: a 2 x 100 ladder (long queries, at least 101 claims each); row 2 blocked; rows 3-4: a 2 x 4 patch (short
# queries, at most 8 claims each)
MIXED_DIMS = (100, 5, 1)


def mixed_grid():
    free = np.zeros(MIXED_DIMS[::-1], np.uint8)
    free[0, 0:2, :] = 1
    free[0, 3:5, 0:4] = 1
    return free.ravel()


def test_mixed_fallback_chunks(wr, oracle, monkeypatch):
    """Adaptive colonies of at most 64 ants with a 420-step cap need 137 265 bytes per query: a 1 MB budget gives chunks of
    3 queries, so 10 queries run as chunks of 3, 3, 3 and 1.  A 256-entry table (limit 128) holds any chunk of patch queries
    (<= 24 claims) and no chunk with a ladder query: only the middle chunk of three ladder queries falls back."""
    monkeypatch.setenv("WR_BATCH_MEM_MB", "1")
    monkeypatch.setenv("WR_BATCH_LOG2", "8")
    dims = MIXED_DIMS
    A, g, twin = handles(wr, oracle, mixed_grid(), dims, seed=61, step_cap=420, beta=1.0)
    P = lambda x, y: nid(dims, x, y)  # noqa: E731
    short = [(P(0, 3), P(3, 4)), (P(3, 3), P(0, 3)), (P(1, 4), P(2, 3)), (P(0, 4), P(3, 3)), (P(2, 4), P(2, 3)),
             (P(3, 4), P(0, 4)), (P(1, 3), P(3, 3))]
    long = [(P(0, 0), P(99, 0)), (P(99, 1), P(0, 1)), (P(0, 1), P(99, 0))]
    pairs = short[:3] + long + short[3:6] + short[6:]
    s, e = [p[0] for p in pairs], [p[1] for p in pairs]
    predict, iters, first = 183.0, 4, 1000                  # colony 0.35 * 183 = 64
    f0 = g.batchStats()["fallbacks"]
    check_all(A, g, twin, s, e, predict, iters, first)
    st = g.batchStats()
    assert st["queries_per_chunk"] == 3 and st["table_entries"] == 256, st
    assert st["fallbacks"] - f0 == 1, st
    assert st["entries_used"] <= 8, st                      # the one-query last chunk ran on the batch path

    # the handle's next search index continues after the batch: first + 10.  The end of every call sets it whatever its
    # chunks did, so this does not cover the restore after a fallback (next_search = first + c0): the fallback chunk's own
    # queries, equal to the oracle at first + 3 .. first + 5 above, do.
    ores, _, otot = oracle_queries(A, [long[0][0]], [long[0][1]], predict, iters, first + 10)
    g.setEndpoints(long[0][0], long[0][1])
    _, gcnt = counted(g, lambda: (g.begin(predict), g.iterate(iters)))
    same_as_oracle(ores, [g.bestPath()], "single search after the batch")
    assert gcnt == otot
    g.reset()

    # more queries than before, same colony: the memory-limited buffers are reused
    pairs2 = (short * 2)[:14]
    s2, e2 = [p[0] for p in pairs2], [p[1] for p in pairs2]
    check_all(A, g, twin, s2, e2, predict, iters, 2000)
    st = g.batchStats()
    assert st["queries_per_chunk"] == 3 and st["fallbacks"] - f0 == 1, st
    # another colony size (0.35 * 100 = 35 ants, 76 075 bytes per query): new buffers, chunks of 6
    check_all(A, g, twin, s2, e2, 100.0, iters, 3000)
    st = g.batchStats()
    assert st["queries_per_chunk"] == 6 and st["fallbacks"] - f0 == 1, st


# ---------------------------------------------------------------------------------------------
# 4. k_batch_deposit's trips of 256 steps
# ---------------------------------------------------------------------------------------------
def oracle_per_iteration(A, s, e, predict, iters, first):
    """Per query and iteration count 1..iters: best, cumulative counters, and the step counts of the eligible ants
    (arrived and rank <= lambda - 1, ACSRank_3D.hpp:200)."""
    best, cnt, elig = [], [], []
    for q in range(len(s)):
        A.set_endpoints(s[q], e[q]); A.set_next_search((first + q) & U32)
        A.begin(predict)
        c0 = A.counters()
        b, c, el = [], [], []
        for _ in range(iters):
            A.iterate(1)
            b.append(A.best())
            c1 = A.counters()
            c.append({k: c1[k] - c0[k] for k in KEYS})
            colony, lam, _ = A.last_colony()
            for k in range(colony):
                ids, _, L, order = A.last_ant(k)
                if np.isfinite(L) and not np.float32(order) > np.float32(lam) - np.float32(1):
                    el.append(len(ids) - 1)
        best.append(b); cnt.append(c); elig.append(el)
        A.reset()
    return best, cnt, elig


@pytest.mark.parametrize("n,K,iters,straight", [(257, 6, 18, 256), (513, 6, 25, 512), (300, 26, 8, None)])
def test_deposit_trips(wr, oracle, n, K, iters, straight):
    """A two-lane ladder from (0, 0, 0) to (n - 1, 0, 0) and back along the other lane.  beta = 1: stepping backwards is
    worth nothing, a lane change half a step forward, so the first ants arrive with dozens of lane changes and the colony
    converges onto a straight lane over the iterations.  Every iteration count 1..iters is a call of its own with the same
    search indices, so a wrong deposit shows in the first iteration after it."""
    free, dims = ladder(n)
    A, g, twin = handles(wr, oracle, free, dims, seed=11, fixed_colony=128, step_cap=2 * n, beta=1.0, K=K)
    s = [nid(dims, 0, 0), nid(dims, n - 1, 1)]
    e = [nid(dims, n - 1, 0), nid(dims, 0, 1)]
    first = 500
    best, cnt, elig = oracle_per_iteration(A, s, e, float(n), iters, first)
    steps = np.concatenate([np.asarray(x) for x in elig])
    if straight is not None:   # the straight lane, exactly two trips of 256 steps or one, and longer ants
        assert (steps == straight).sum() > 0 and (steps > straight).sum() > 0
    assert (steps > 256).sum() > 0
    for it in range(1, iters + 1):
        want = dict.fromkeys(KEYS, 0)
        for q in range(len(s)):
            for k in KEYS:
                want[k] += cnt[q][it - 1][k]
        bres, bcnt = run_batch(g, s, e, float(n), it, first)
        sres, scnt = run_sequential(twin, s, e, float(n), it, first)
        same_as_oracle([b[it - 1] for b in best], bres, ("batch", it))
        same_as_oracle([b[it - 1] for b in best], sres, ("sequential", it))
        assert bcnt == want and scnt == want, (it, bcnt, scnt, want)
    assert g.batchStats()["fallbacks"] == 0


# ---------------------------------------------------------------------------------------------
# 5. adaptive colonies that shrink to 0-3 ants (k_batch_iter_begin: 0.35 * best_L / precision)
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [6, 26])
def test_tiny_adaptive_colonies(wr, oracle, K):
    """precision 1: once a query's best is L long its colony has int(0.35 L) ants — 0 for L <= 2, 1 for 3 to 5, 2 up to 8,
    3 up to 11 — so the near queries run partial groups of four and iterations without ants or eligible ants, next to a
    start == goal query (no best: 14 ants that all die) and a far query (14, then 10 ants)."""
    dims = (16, 16, 1)
    A, g, twin = handles(wr, oracle, np.ones(16 * 16, np.uint8), dims, seed=5, K=K)
    P = lambda x, y: nid(dims, x, y)  # noqa: E731
    ds = (0, 1, 2, 3, 5, 6, 8, 9, 11)
    s = [P(4, 4)] * len(ds) + [P(0, 0)]
    e = [P(4 + d, 4) for d in ds] + [P(15, 15)]
    colonies, tot = check_all(A, g, twin, s, e, 40.0, 6, 70)
    assert {0, 1, 2, 3} <= {c for col in colonies[1:-1] for c in col[1:]}, colonies
    assert g.batchStats()["queries_per_chunk"] == len(s) and g.batchStats()["fallbacks"] == 0
    assert tot["arrived"] > 0 and tot["dead_fallthrough"] > 0   # the start == goal query's ants


# ---------------------------------------------------------------------------------------------
# 6. search indices inside one batch: block_hi changes at 2^16, the index wraps at 2^32
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("first", [0xFFFE, 0xFFFFFFFE])
def test_search_indices_in_a_batch(wr, oracle, first):
    dims = (12, 12, 2)
    A, g, twin = handles(wr, oracle, np.ones(12 * 12 * 2, np.uint8), dims, seed=13, fixed_colony=32, step_cap=200)
    P = lambda x, y, z: nid(dims, x, y, z)  # noqa: E731
    s = [P(0, 0, 0), P(11, 0, 1), P(0, 11, 0), P(5, 5, 1)]
    e = [P(11, 11, 1), P(0, 11, 0), P(11, 0, 1), P(10, 1, 0)]
    check_all(A, g, twin, s, e, 30.0, 5, first)
    assert g.batchStats()["fallbacks"] == 0
    # the next search of the handle takes index first + 4 (mod 2^32)
    nxt = (first + 4) & U32
    ores, _, otot = oracle_queries(A, [s[0]], [e[0]], 30.0, 5, nxt)
    g.setEndpoints(s[0], e[0])
    _, gcnt = counted(g, lambda: (g.begin(30.0), g.iterate(5)))
    same_as_oracle(ores, [g.bestPath()], "next search")
    assert gcnt == otot
