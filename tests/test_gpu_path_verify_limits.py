"""Path verification (path_verify.cuh) where its arithmetic and bookkeeping have edges the short oracle cases of
test_gpu_path_verify.py never reach, each against the CPU oracle bit for bit and with walkStats() checked exactly:

  * best paths of more than 2048 steps: k_path_thresholds counts the visited tiles across three 1024-position chunks, a
    visited table fills in the second chunk, and warps resume at T >= 1024;
  * step caps at the best path's length;
  * colonies whose warps are not full (1, 2, 3, 5, 4099 ants; 1001 ants over three shards);
  * search indices around 2^16, where the Philox counter takes the index's high half (block_hi);
  * pheromone values at the arithmetic edges (inf, NaN, 0, subnormal, underflow, overflow) on a best-path node.

Every iteration takes the predicted walk (WR_RANKSET_POLICY=1), so every iteration after the first verifies the best path.
The expected walkStats() increments come from expected_walk_stats, which reads only the oracle: the best path before the
iteration and every ant's trail."""
import numpy as np
import pytest

from test_gpu_dispatch_edges import occupancy_pair
from test_gpu_parity import compare_iteration, make_pair
from test_gpu_path_verify import _run_vs_oracle, add_stats, expected_walk_stats

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def wr():
    import welding_robot_b200 as wr
    return wr


@pytest.fixture(autouse=True)
def rank_sets_always(monkeypatch):
    monkeypatch.setenv("WR_RANKSET_POLICY", "1")


# ---------------------------------------------------------------------------------------------
# the serpentine corridor: one 2079-node shortest path with side features
# ---------------------------------------------------------------------------------------------
RX, RY, RZ = 64, 63, 2
DIMS = (RX, RY, RZ)
UP = 5                                                     # slot k: dz = +1 (slots 0..5: -z, -y, -x, +x, +y, +z)


def nid(x, y, z):
    return (z * RY + y) * RX + x


def slot_of(a, b):
    d = b - a
    return {-RX * RY: 0, -RX: 1, -1: 2, 1: 3, RX: 4, RX * RY: 5}[d]


def corridor():
    """Rows of 64 nodes on even y at z = 0, joined by one-node connectors at alternating ends: the only path from (0, 0, 0)
    to (0, 62, 0), 2079 nodes.  Above every row, at z = 1: a two-node detour (up at one row node, down at the next, so a
    deviating ant rejoins the corridor) and a one-node pocket (an ant that enters it dies), at positions that vary by row.
    Returns (isfree, path node ids, path positions of detour entries, path positions of pockets)."""
    free = np.zeros((RZ, RY, RX), np.uint8)
    path, detours, pockets = [], [], []
    for r in range(RY // 2 + 1):
        y = 2 * r
        xs = list(range(RX)) if r % 2 == 0 else list(range(RX - 1, -1, -1))
        free[0, y, :] = 1
        a = 8 + (r * 7) % 20
        b = a + 20 + (r * 5) % 16
        for i in (a, a + 1, b):
            free[1, y, xs[i]] = 1
        detours.append(len(path) + a)
        pockets.append(len(path) + b)
        path += [nid(x, y, 0) for x in xs]
        if y + 1 < RY:
            free[0, y + 1, xs[-1]] = 1
            path.append(nid(xs[-1], y + 1, 0))
    return free.ravel(), np.array(path, np.int64), detours, pockets


FREE, PATH, DETOURS, POCKETS = corridor()
START, GOAL = int(PATH[0]), int(PATH[-1])


def corridor_field(tau_path, tau_side):
    """tau_side everywhere, tau_path on the slot each corridor node takes to the next one."""
    tau = np.full(RX * RY * RZ * 6, tau_side, np.float32)
    for p in range(len(PATH) - 1):
        tau[PATH[p] * 6 + slot_of(PATH[p], PATH[p + 1])] = tau_path
    return tau


# The corridor's slots start at about the pheromone the colony's own deposits keep them at; the side slots are low enough
# that a few ants per iteration leave the corridor, at any of its 64 side features, and evaporate from there.
TAU_PATH = 300.0
TAU_SIDE = {1: 0.05, 2: 3.0}                               # per alpha: about the same chance to leave at a feature


class Search:
    """One search on the oracle and the GPU (one handle, or in-process shards) stepped an iteration at a time: every
    iteration is compared bit for bit, and walkStats() is checked against expected_walk_stats on every shard."""

    def __init__(self, A, gs, start, goal, table_log2=0, shards=None):
        self.A, self.gs, self.start, self.goal, self.table_log2, self.S = A, gs, start, goal, table_log2, shards
        g = gs[0]
        self.dims, self.cap = (g.rangeX, g.rangeY, g.rangeZ), g.stepCap()
        self.want = [g.walkStats() for g in gs]
        self.iters = 0
        self.infos = []

    def step(self, nonfinite=()):
        A = self.A
        best = A.best()[0]
        A.iterate(1)
        if self.S:
            self.S.iterate(1); self.S.sync()
        else:
            self.gs[0].iterate(1)
        self.iters += 1
        colony = A.last_colony()[0]
        trails = [A.last_ant(k)[0] for k in range(colony)]
        counts, info = expected_walk_stats(best, trails, self.start, self.goal, self.cap, self.dims, self.table_log2, colony,
                                           len(self.gs), nonfinite)
        info["trails"] = trails
        self.infos.append(info)
        self.want = add_stats(self.want, counts)
        if self.S:
            compare_shards(A, self.gs)
        else:
            compare_iteration(A, self.gs[0])
        for g, w in zip(self.gs, self.want):
            assert g.walkStats() == w, (self.iters, info["D"], info["n"])
            assert g.updateStats()["rankset_iterations"] == self.iters
        return info


def compare_shards(A, shards):
    """compare_iteration for a colony split over in-process shards: each ant is read from the shard that walked it."""
    world = len(shards)
    oc, olam, oq = A.last_colony()
    chunk = (max(oc, 1) + world - 1) // world
    for g in shards:
        gc, glam, gq = g.lastColony()
        assert (oc, np.float32(olam).tobytes(), np.float32(oq).tobytes()) == (gc, np.float32(glam).tobytes(), np.float32(gq).tobytes())
    for k in range(oc):
        oid, odir, oL, oorder = A.last_ant(k)
        gid, gdir, gL, gorder = shards[k // chunk].lastAnt(k)
        assert gorder == oorder, (k, gorder, oorder)
        if np.isinf(oL):
            assert np.isinf(gL), k
        else:
            assert np.float32(oL).tobytes() == np.float32(gL).tobytes(), (k, oL, gL)
            assert np.array_equal(oid, gid) and np.array_equal(odir, gdir), k
    ob, to = A.best(), A.pheromone()
    for g in shards:
        gb = g.bestPath()
        assert np.float32(ob[2]).tobytes() == np.float32(gb[2]).tobytes()
        assert np.array_equal(ob[0], gb[0]) and np.array_equal(ob[1], gb[1])
        assert np.array_equal(to.view(np.uint32), g.pheromone().view(np.uint32))


def corridor_search(wr, oracle, colony, alpha=1, seed=3, step_cap=4096, walk_table_log2=0, search=None):
    params = dict(seed=seed, fixed_colony=colony, step_cap=step_cap, alpha=alpha, update_mode=4)
    if walk_table_log2:
        params["walk_table_log2"] = walk_table_log2
    A, g = occupancy_pair(wr, oracle, FREE, DIMS, **params)
    tau = corridor_field(TAU_PATH, TAU_SIDE[alpha])
    A.set_pheromone(tau); g.setPheromone(tau)
    A.set_endpoints(START, GOAL); g.setEndpoints(START, GOAL)
    if search is not None:
        A.set_next_search(search); g.setNextSearch(search)
    A.begin(2100.0); g.begin(2100.0)
    return Search(A, [g], START, GOAL, walk_table_log2)


def converge(run, iters):
    """Iteration 1 finds the corridor (no best path yet: nothing to verify); the following ones verify it."""
    first = run.step()
    assert first["D"] == 0 and np.array_equal(run.A.best()[0], PATH)
    return [run.step() for _ in range(iters - 1)]


def warps_resumed(infos):
    return [w for i in infos for w in i["warps"] if not w[4]]


# ---------------------------------------------------------------------------------------------
# 1. long best paths
# ---------------------------------------------------------------------------------------------
def test_corridor_three_threshold_chunks(wr, oracle):
    """D = 2078 > 2048: the thresholds of three 1024-position chunks, the tile count carried across them; ants that leave the
    path beyond position 1024 and warps that resume there."""
    run = corridor_search(wr, oracle, colony=256)
    infos = converge(run, 8)
    assert all(i["D"] == len(PATH) - 1 > 2048 for i in infos)
    assert sum(w[4] for i in infos for w in i["warps"]) > 0                      # warps completed by the check
    assert max(int(d) for i in infos for d in i["dev"] if d < i["D"]) >= 1024     # an ant leaves the path beyond 1024
    assert max(w[3] for w in warps_resumed(infos)) >= 1024                        # a warp resumes at T >= 1024
    assert run.gs[0].counters()["arrived"] > 0


def test_corridor_table_fills_in_the_second_chunk(wr, oracle):
    """256-entry visited tables (192 tiles): the corridor's 193rd tile is at position 1560, so the tile count that ends the
    verifiable prefix is found in the second chunk; the ants walk on from there, park on the full table and finish in pass 2."""
    run = corridor_search(wr, oracle, colony=256, walk_table_log2=8)
    infos = converge(run, 5)
    assert all(1024 <= i["D"] < 2048 for i in infos), [i["D"] for i in infos]
    assert run.gs[0].counters()["table_overflows"] > 0
    assert run.gs[0].walkStats()["verified_ants"] == 0


@pytest.mark.parametrize("extra", [0, 1])
def test_corridor_step_cap_at_the_path_length(wr, oracle, extra):
    """step_cap = n - 1 (the best path's steps): the ant deciding step n - 2 is at the cap, so D = n - 2 and no ant is
    complete — every warp walks the tail.  step_cap = n: the whole path verifies."""
    n = len(PATH)
    run = corridor_search(wr, oracle, colony=128, step_cap=n - 1 + extra)
    infos = converge(run, 4)
    assert all(i["D"] == n - 2 + extra for i in infos)
    if extra:
        assert run.gs[0].walkStats()["verified_ants"] > 0
    else:
        assert run.gs[0].walkStats()["verified_ants"] == 0
        assert max(w[3] for i in infos for w in i["warps"]) == (n - 2) & ~7   # warps without a deviating ant re-walk the last steps


# ---------------------------------------------------------------------------------------------
# 2. partial warps
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("colony", [1, 2, 3, 5, 4099])
def test_piece_partial_warps(wr, oracle, meshes, colony):
    """Colonies that leave lanes of the last warp without an ant (k_path_verify's grid rounds up; k_walk3's min and all-complete
    votes skip them).  The small colonies barely converge here: their ants leave the best path within its first steps."""
    A, g = make_pair(wr, oracle, meshes["simplified_piece"], 0.02, 3, seed=54, fixed_colony=colony, step_cap=300, update_mode=4)
    _run_vs_oracle(A, g, iters=(1,) * 16)
    assert colony % 4 != 0 and len(A.best()[0]) > 1
    if colony == 4099:
        assert g.walkStats()["verified_ants"] > 0


@pytest.mark.parametrize("colony", [1, 2, 3, 5])
def test_corridor_partial_warps(wr, oracle, colony):
    """The same colonies on the corridor, where they follow the best path: a warp with idle lanes is booked complete."""
    run = corridor_search(wr, oracle, colony=colony, seed=10 + colony)
    infos = converge(run, 5)
    partial = [w for i in infos for w in i["warps"] if w[2] < 4]
    assert partial and any(w[4] for w in partial)


@pytest.mark.timeout(900)
def test_corridor_three_shards_partial_warps(wr, oracle, monkeypatch):
    """1001 ants over three in-process shards: chunks of 334, 334 and 333 ants, each shard with a partial last warp."""
    from welding_robot_b200.dist import LocalShards
    monkeypatch.setenv("WR_PEER_TIMEOUT_MS", "8000")
    params = dict(seed=8, fixed_colony=1001, step_cap=4096, update_mode=4)
    A, _ = occupancy_pair(wr, oracle, FREE, DIMS, **params)
    shards = []
    tau = corridor_field(TAU_PATH, TAU_SIDE[1])
    for _ in range(3):
        g = wr.ACS_Rank(**params)
        g.creatFromOccupancy(FREE, *[np.arange(n, dtype=np.float32) for n in DIMS], 1.0)
        g.initFromGridMap()
        g.setPheromone(tau)
        g.setEndpoints(START, GOAL)
        shards.append(g)
    A.set_pheromone(tau); A.set_endpoints(START, GOAL)
    S = LocalShards(shards)
    A.begin(2100.0); S.begin(2100.0)
    run = Search(A, shards, START, GOAL, shards=S)
    infos = converge(run, 5)
    last = {r: max(w[1] for w in infos[0]["warps"] if w[0] == r) for r in range(3)}
    assert [w[2] for w in infos[0]["warps"] if w[1] == last[w[0]]] == [2, 2, 1]
    assert any(w[4] for i in infos for w in i["warps"] if w[1] == last[w[0]])    # a partial warp completed by the check
    assert all(s["verified_ants"] > 0 for s in run.want)


# ---------------------------------------------------------------------------------------------
# 3. search indices at the 16-bit boundary
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("search", [0xFFFF, 0x10000, 0x12345, 0xFFFFFFFF])
def test_corridor_search_index(wr, oracle, search):
    """The draws of search i use the Philox counter words (i & 0xFFFF) and (block | (i >> 16) << 16): k_path_verify builds
    the second one itself.  Ants that leave the corridor are found by their draws; the others complete."""
    run = corridor_search(wr, oracle, colony=256, seed=4, search=search)
    infos = converge(run, 5)
    assert sum(int((i["dev"] < i["D"]).sum()) for i in infos) > 0
    assert any(w[4] for i in infos for w in i["warps"]) and len(warps_resumed(infos)) > 0


# ---------------------------------------------------------------------------------------------
# 4. pheromone at the arithmetic edges on a best-path node, uploaded mid-search
# ---------------------------------------------------------------------------------------------
def thresholds_finite(A, best, t, goal):
    """Whether the roulette total and every suffix sum at best[t] are finite for an ant that followed best[0..t]: the oracle's
    scores of that step (select_step), summed in the walk's order."""
    _, infos, _, _, _ = A.select_step(int(best[t]), goal, best[:t + 1], 0)
    v = np.where(infos == np.float32(-12345.0), np.float32(0), infos).astype(np.float32)
    total, suffix, ok = np.float32(0), np.float32(0), True
    with np.errstate(all="ignore"):
        for k in range(6):
            total = np.float32(total + v[k])
        for k in range(5, -1, -1):
            suffix = np.float32(suffix + v[k])
            ok = ok and bool(np.isfinite(suffix))
    return ok and bool(np.isfinite(total))


SUBNORMAL = np.float32(1e-39)
QNAN = np.array([0x7FFFFFFF], np.uint32).view(np.float32)[0]   # the NaN the GPU's arithmetic produces: the field compares bitwise


def _edit(tau, t, case):
    node = int(PATH[t])
    d = slot_of(PATH[t], PATH[t + 1])
    row = tau[node * 6:node * 6 + 6]
    if case == "inf_side":
        row[UP] = np.inf
    elif case == "nan_side":
        row[UP] = QNAN
    elif case in ("zero_path",):
        row[d] = 0.0
    elif case == "subnormal_all":
        row[:] = SUBNORMAL
    elif case == "tiny_path_alpha2":
        row[d] = np.float32(1e-30)
    elif case == "huge_two":
        row[d] = row[UP] = np.float32(3e38)


@pytest.mark.parametrize("case,alpha", [("inf_side", 1), ("nan_side", 1), ("zero_path", 1), ("subnormal_all", 1), ("tiny_path_alpha2", 2),
                                        ("huge_two", 1)])
def test_corridor_pheromone_edges(wr, oracle, case, alpha):
    """Once the corridor is the best path, the field is downloaded, one best-path node t (with a side feature, beyond the
    first threshold chunk) is edited, and the field uploaded to both sides:
      inf / NaN on the side slot, 3e38 on two candidate slots: the roulette at t is not finite, so D = t (NaN: ants reaching
      t die by fall-through);  0 on the path slot, 1e-30 on it with alpha = 2 (tau^2 underflows): every ant reaching t
      leaves there, D unchanged;  all six slots subnormal: no flush to zero anywhere in the roulette or the thresholds."""
    run = corridor_search(wr, oracle, colony=128, alpha=alpha, seed=9)
    converge(run, 3)
    A, g = run.A, run.gs[0]
    n = len(PATH)
    t = next(p for p in (POCKETS if case == "nan_side" else DETOURS) if p >= 1100)
    tau = g.pheromone()
    assert np.array_equal(tau.view(np.uint32), A.pheromone().view(np.uint32))
    _edit(tau, t, case)
    A.set_pheromone(tau); g.setPheromone(tau)
    for _ in range(4):
        best = A.best()[0]
        assert np.array_equal(best, PATH)
        fin = thresholds_finite(A, best, t, GOAL)
        info = run.step(nonfinite=() if fin else (t,))
        reached = [k for k in range(len(info["dev"])) if info["dev"][k] >= t]
        if case in ("inf_side", "nan_side", "huge_two") and run.iters == 4:
            assert not fin and info["D"] == t
        if case in ("zero_path", "subnormal_all", "tiny_path_alpha2"):
            assert fin and info["D"] == n - 1
        if run.iters == 4:
            assert reached, "no ant reached the edited node"
            trails = info["trails"]
            if case in ("zero_path", "tiny_path_alpha2"):
                assert all(info["dev"][k] == t for k in reached)
            if case == "nan_side":
                assert all(len(trails[k]) == t + 1 for k in reached)                # died at t: the roulette fell through
            if case == "subnormal_all":
                assert 0 < sum(info["dev"][k] == t for k in reached) < len(reached)   # both subnormal candidates are taken
