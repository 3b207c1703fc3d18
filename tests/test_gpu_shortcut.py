"""Line-of-sight shortcutting of node rows (wr_grid_shortcut_paths, GridMap.shortcutPaths, ACS_Rank.shortcutBestMatrix).

The reference below restates the definition of include/wr_gpu.h in exact int64 arithmetic: the cover of a segment between two
index points is every cube [c - 1/2, c + 1/2]^3 that meets the closed segment, decided per candidate cube by a slab test whose
rational bounds are compared by cross-multiplication.  Candidates: along the axis of largest |d|, every integer c_m between the
endpoints; on the other axes, round(centre) + {-1, 0, 1} (the segment moves by at most 1/2 on either side of the slab's centre).
Greedy waypoints, fallback counts and lengths (summed in order in a Python loop) are compared for exact equality.
The reference's own checks run without a GPU; everything else is marked gpu."""
import contextlib
import ctypes as C
import io
import math
import os
import subprocess
from fractions import Fraction

import numpy as np
import pytest

from conftest import C1_POINTS, ROOT

FAR = 0xFFFFFFFF
PAIRS = [(i, j) for i in range(6) for j in range(i + 1, 6)]
# per axis m of largest |d|: the 9 offsets on the two other axes
OFFS9 = np.array([[o for o in np.ndindex(3, 3, 3) if o[m] == 1] for m in range(3)], np.int64) - 1


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


# ---- the reference ----------------------------------------------------------------------------------------------------
def covers(a, B):
    """Covers of the segments a -> B[q] (int index points).  -> (segment index, cube xyz) of every covered cube, exact."""
    a = np.asarray(a, np.int64)
    B = np.asarray(B, np.int64).reshape(-1, 3)
    q = len(B)
    D = B - a
    m = np.abs(D).argmax(1)
    dm = D[np.arange(q), m]
    cnt = np.abs(dm) + 1
    seg = np.repeat(np.arange(q), cnt)
    step = np.arange(cnt.sum()) - np.repeat(np.cumsum(cnt) - cnt, cnt)
    u = a[m][seg] + np.sign(dm)[seg] * step                 # the slab's coordinate along m
    d, dms, ms = D[seg], dm[seg], m[seg]
    den = np.where(dms == 0, 1, dms)
    base = np.empty((len(seg), 3), np.int64)
    for k in range(3):
        num = a[k] * den + (u - a[m][seg]) * d[:, k]          # centre = num / den
        sgn = np.sign(den)
        base[:, k] = np.where(ms == k, u, np.floor_divide(sgn * (2 * num + den), 2 * np.abs(den)))   # round half up
    cand = (base[:, None, :] + OFFS9[ms]).reshape(-1, 3)
    cseg = np.repeat(seg, 9)
    d = D[cseg]
    lo_n, lo_d = np.zeros(len(cand), np.int64), np.ones(len(cand), np.int64)
    hi_n, hi_d = np.ones(len(cand), np.int64), np.ones(len(cand), np.int64)
    ok = np.ones(len(cand), bool)
    for k in range(3):
        dk = d[:, k]
        e = np.sign(dk) * (cand[:, k] - a[k])
        den2 = 2 * np.abs(dk)
        ok &= (dk != 0) | (cand[:, k] == a[k])
        act = dk != 0
        n1, n2 = 2 * e - 1, 2 * e + 1
        up = act & (n1 * lo_d > lo_n * den2)
        lo_n, lo_d = np.where(up, n1, lo_n), np.where(up, den2, lo_d)
        dn = act & (n2 * hi_d < hi_n * den2)
        hi_n, hi_d = np.where(dn, n2, hi_n), np.where(dn, den2, hi_d)
    ok &= lo_n * hi_d <= hi_n * lo_d
    return cseg[ok], cand[ok]                              # a cube may appear more than once


def cover(a, b):
    return {tuple(int(v) for v in c) for c in covers(a, [b])[1]}


def cover_fraction(a, b):
    """The definition with Fractions over the whole bounding box (slow; for small segments only)."""
    d = [b[k] - a[k] for k in range(3)]
    out = set()
    rng = [range(min(a[k], b[k]) - 1, max(a[k], b[k]) + 2) for k in range(3)]
    for c in ((x, y, z) for x in rng[0] for y in rng[1] for z in rng[2]):
        lo, hi, ok = Fraction(0), Fraction(1), True
        for k in range(3):
            if d[k] == 0:
                ok &= abs(2 * (c[k] - a[k])) <= 1
                continue
            t1, t2 = sorted((Fraction(2 * (c[k] - a[k]) - 1, 2 * d[k]), Fraction(2 * (c[k] - a[k]) + 1, 2 * d[k])))
            lo, hi = max(lo, t1), min(hi, t2)
        if ok and lo <= hi:
            out.add(c)
    return out


def xyz_of(ids, dims):
    rx, ry, _ = dims
    ids = np.asarray(ids, np.int64)
    z, r = np.divmod(ids, rx * ry)
    y, x = np.divmod(r, rx)
    return np.stack([x, y, z], 1)


def clear_many(P, i, js, block):
    """clear(P[i], P[j]) for every j in js; block is bool [z, y, x]."""
    seg, c = covers(P[i], P[js])
    bad = np.zeros(len(js), bool)
    np.logical_or.at(bad, seg, block[c[:, 2], c[:, 1], c[:, 0]])
    return ~bad


def shortcut_ref(row, dims, block, max_span=0, chunk=64):
    """Greedy waypoints of one row -> (keep indices, blocked)."""
    n = len(row)
    if n == 0:
        return np.zeros(0, np.int32), 0
    P = xyz_of(row, dims)
    span = max_span if max_span > 0 else n
    w, nb = [0], 0
    while w[-1] < n - 1:
        i = w[-1]
        nxt = None
        for hi in range(min(n - 1, i + span), i, -chunk):
            js = np.arange(hi, max(i, hi - chunk), -1)
            ok = clear_many(P, i, js, block)
            if ok.any():
                nxt = int(js[np.argmax(ok)])
                break
        if nxt is None:
            nxt, nb = i + 1, nb + 1
        w.append(nxt)
    return np.array(w, np.int32), nb


def world_length(row, keep, dims, coords):
    """Sum in order, in double, of sqrt(dx*dx + dy*dy + dz*dz) with dx = (double)c[a] - (double)c[b]."""
    P = xyz_of(np.asarray(row)[keep], dims)
    xs, ys, zs = (np.asarray(c, np.float32) for c in coords)
    L = 0.0
    for k in range(len(P) - 1):
        a, b = P[k], P[k + 1]
        dx = float(xs[a[0]]) - float(xs[b[0]]); dy = float(ys[a[1]]) - float(ys[b[1]]); dz = float(zs[a[2]]) - float(zs[b[2]])
        L += math.sqrt(dx * dx + dy * dy + dz * dz)
    return L


def grid_dims(g):
    return (g.rangeX, g.rangeY, g.rangeZ)


def blocks(g, r2):
    if r2 == 0:
        b = g.isfree() == 0
    else:
        b = g.clearanceMap() <= r2
    return b.reshape(g.rangeZ, g.rangeY, g.rangeX)


def assert_matches_reference(g, rows, r2, max_span=0, radius=None):
    """GPU result == reference for every row: keep, nkeep, blocked, and length to the bit."""
    if radius is None:
        got = raw_shortcut(g, rows, r2, max_span)
    else:
        got = [(k, b, L) for _, k, b, L in g.shortcutPaths(rows, radius, max_span)]
    blk = blocks(g, r2)
    dims, coords = grid_dims(g), g.coords()
    for q, row in enumerate(rows):
        keep, nb = shortcut_ref(row, dims, blk, max_span)
        assert np.array_equal(got[q][0], keep), (q, got[q][0][:20], keep[:20])
        assert got[q][1] == nb, q
        L = world_length(row, keep, dims, coords)
        assert got[q][2] == L, (q, got[q][2], L)
        check_waypoints(row, keep, nb, dims, blk)
    return got


def check_waypoints(row, keep, nb, dims, blk):
    n = len(row)
    if n == 0:
        assert len(keep) == 0
        return
    assert keep[0] == 0 and keep[-1] == n - 1 and (np.diff(keep) > 0).all()
    P = xyz_of(row, dims)
    fallbacks = 0
    for a, b in zip(keep[:-1], keep[1:]):
        if not clear_many(P, a, np.array([b]), blk)[0]:
            assert b == a + 1
            fallbacks += 1
    assert fallbacks == nb


def raw_shortcut(g, rows, r2, max_span=0):
    """wr_grid_shortcut_paths on an explicit r2 -> per row (keep, blocked, length)."""
    from welding_robot_b200._lib import check, lib, ptr
    rows = [np.asarray(r, np.int64) for r in rows]
    off = np.zeros(len(rows) + 1, np.int64)
    off[1:] = np.cumsum([len(r) for r in rows])
    ids = np.concatenate(rows) if rows else np.zeros(0, np.int64)
    ids = np.ascontiguousarray(ids if len(ids) else np.zeros(1, np.int64))
    keep = np.full(max(int(off[-1]), 1), -7, np.int32)
    nkeep = np.full(max(len(rows), 1), -7, np.int32); nb = nkeep.copy(); L = np.full(len(nkeep), -7.0)
    check(lib().wr_grid_shortcut_paths(g._g, ptr(ids), ptr(off), len(rows), r2, max_span, ptr(keep), ptr(nkeep), ptr(nb), ptr(L)))
    return [(keep[off[p]:off[p] + nkeep[p]].copy(), int(nb[p]), float(L[p])) for p in range(len(rows))]


def occupancy_grid(free_zyx, precision=1.0):
    import welding_robot_b200 as wr
    rz, ry, rx = free_zyx.shape
    return wr.GridMap().creatFromOccupancy(np.ascontiguousarray(free_zyx, np.uint8).ravel(), np.arange(rx, dtype=np.float32),
                                           np.arange(ry, dtype=np.float32), np.arange(rz, dtype=np.float32), precision)


def node_id(dims, p):
    return (int(p[2]) * dims[1] + int(p[1])) * dims[0] + int(p[0])


# ---- 0. the reference itself (no GPU) ---------------------------------------------------------------------------------
def test_reference_cover_sizes():
    assert cover((0, 0, 0), (1, 0, 0)) == {(0, 0, 0), (1, 0, 0)}
    assert len(cover((0, 0, 0), (1, 1, 0))) == 4 and len(cover((0, 0, 0), (1, 1, 1))) == 8
    assert len(cover((5, 5, 5), (4, 6, 4))) == 8 and cover((2, 3, 4), (2, 3, 4)) == {(2, 3, 4)}
    # |dx| = 3, |dy| = 1 crosses the x = 1.5 / y = 0.5 edge at t = 1/2: all four cubes around it
    assert cover((0, 0, 0), (3, 1, 0)) == {(0, 0, 0), (1, 0, 0), (1, 1, 0), (2, 0, 0), (2, 1, 0), (3, 1, 0)}


def test_reference_equals_fraction_definition():
    a = (1, -2, 3)
    for d in np.ndindex(9, 9, 9):
        b = tuple(a[k] + d[k] - 4 for k in range(3))
        assert cover(a, b) == cover_fraction(a, b), b
    rng = np.random.default_rng(1)
    for _ in range(200):
        a, b = rng.integers(-9, 9, 3), rng.integers(-9, 9, 3)
        assert cover(a, b) == cover_fraction(tuple(a), tuple(b)), (a, b)


def test_reference_greedy_on_a_wall():
    free = np.ones((1, 5, 7), np.uint8)
    free[0, 1:, 3] = 0                                     # a wall at x = 3 with a gap at y = 0
    row = [node_id((7, 5, 1), (x, 4, 0)) for x in (0,)] + [node_id((7, 5, 1), (0, y, 0)) for y in (3, 2, 1, 0)] + \
          [node_id((7, 5, 1), (x, 0, 0)) for x in range(1, 7)] + [node_id((7, 5, 1), (6, y, 0)) for y in range(1, 5)]
    keep, nb = shortcut_ref(np.array(row), (7, 5, 1), free == 0)
    # (0,4) -> (2,0) stays left of the wall; (2,0) -> (6,1) passes the gap below y = 1/2; (2,0) -> (6,2) would meet cube (3,1)
    assert nb == 0 and list(keep) == [0, 6, 11, 14]


# ---- 1. the predicate, exhaustively -----------------------------------------------------------------------------------
DELTAS = np.array([d for d in np.ndindex(13, 13, 13)], np.int64) - 6


def two_node_rows(dims, anchor):
    a = np.asarray(anchor, np.int64)
    return [[node_id(dims, a), node_id(dims, a + d)] for d in DELTAS]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["random0.1", "random0.3", "single"])
def test_predicate_on_every_delta(kind):
    n = 24
    rng = np.random.default_rng(7)
    if kind == "single":
        free = np.ones((n, n, n), np.uint8)
        free[12, 12, 12] = 0
        anchors = [(12 + dx, 12 + dy, 12 + dz) for dx, dy, dz in
                   [(-3, -1, 0), (-2, -2, -2), (-3, 0, -1), (1, -3, -3), (-1, -1, 0), (0, -2, 1), (2, 2, -3), (-4, 1, 1)]]
        radii = [0, 1, 2, 3]
    else:
        free = (rng.random((n, n, n)) >= float(kind[6:])).astype(np.uint8)
        cand = np.argwhere(free[6:18, 6:18, 6:18])[::-1] + 6
        anchors = [tuple(int(v) for v in cand[k][::-1]) for k in rng.choice(len(cand), 4, replace=False)]
        radii = [0, 1]
    g = occupancy_grid(free)
    dims = grid_dims(g)
    for r2 in radii:
        blk = blocks(g, r2)
        for a in anchors:
            rows = two_node_rows(dims, a)
            got = raw_shortcut(g, rows, r2)
            seg, c = covers(a, np.asarray(a) + DELTAS)
            bad = np.zeros(len(DELTAS), bool)
            np.logical_or.at(bad, seg, blk[c[:, 2], c[:, 1], c[:, 0]])
            assert np.array_equal(np.array([b for _, b, _ in got]), bad.astype(int)), (kind, r2, a)
            assert all(list(k) == [0, 1] for k, _, _ in got)


@pytest.mark.gpu
@pytest.mark.parametrize("step", [(1, 0, 0), (0, -1, 0), (1, 1, 0), (-1, 0, 1), (1, 1, 1), (-1, 1, -1)])
def test_unit_step_cover_sizes(step):
    """One blocker at every cube of a 4 x 4 x 4 block around the step on an otherwise empty grid: the step is blocked exactly
    when the blocker is in its cover, 2 / 4 / 8 cubes."""
    n = 8
    a = np.array([3, 3, 3]); b = a + np.array(step)
    want = cover(a, b)
    assert len(want) == {1: 2, 2: 4, 3: 8}[int(np.abs(step).sum())]
    hit = set()
    for o in np.ndindex(4, 4, 4):
        o = tuple(int(v) + 2 for v in o)
        free = np.ones((n, n, n), np.uint8)
        free[o[2], o[1], o[0]] = 0
        g = occupancy_grid(free)
        (_, nb, _), = raw_shortcut(g, [[node_id((n, n, n), a), node_id((n, n, n), b)]], 0)
        if nb:
            hit.add(o)
    assert hit == want


# ---- 2. greedy on synthetic grids ---------------------------------------------------------------------------------------
def synthetic(kind):
    n = 32 if kind != "random64" else 64
    free = np.ones((n, n, n), np.uint8)
    if kind == "wall":
        free[:, :, 16] = 0
        free[20:23, 9:12, 16] = 1                        # one hole
    elif kind == "u":
        free[6:26, 8:24, 20:23] = 0                      # the U's bottom
        free[6:26, 8:11, 8:23] = 0                       # its arms
        free[6:26, 21:24, 8:23] = 0
    else:
        rng = np.random.default_rng(64)
        free = (rng.random((n, n, n)) >= 0.08).astype(np.uint8)
    return free


def random_walk(free, n, seed):
    rng = np.random.default_rng(seed)
    rz, ry, rx = free.shape
    p = np.array([rx // 4, ry // 4, rz // 4])
    while not free[p[2], p[1], p[0]]:
        p = rng.integers(0, [rx, ry, rz])
    steps = np.array([(1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1)])
    out = [p.copy()]
    while len(out) < n:
        q = p + steps[rng.integers(6)]
        if (q >= 0).all() and (q < [rx, ry, rz]).all() and free[q[2], q[1], q[0]]:
            p = q
            out.append(p.copy())
    return np.array([node_id((rx, ry, rz), v) for v in out], np.int64)


def oracle_rows(oracle, free, pairs):
    rz, ry, rx = free.shape
    ax = [np.arange(v, dtype=np.float32) for v in (rx, ry, rz)]
    G = oracle.Grid.from_occupancy(free.ravel(), *ax, 1.0)
    A = oracle.Acs(G, seed=0)
    rows = []
    for s, e in pairs:
        A.set_endpoints(node_id((rx, ry, rz), s), node_id((rx, ry, rz), e))
        A.begin(float(np.abs(np.subtract(e, s)).sum()))
        A.iterate(40)
        rows.append(np.asarray(A.best()[0], np.int64))
        A.reset()
    assert all(len(r) for r in rows)
    return rows


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["wall", "u", "random64"])
def test_greedy_on_synthetic_grids(kind, oracle):
    free = synthetic(kind)
    g = occupancy_grid(free)
    n = free.shape[0]
    pairs = [((3, 3, 3), (n - 4, n - 5, n - 4)), ((n - 3, 4, n // 2), (2, n - 3, n // 2)), ((n // 2, 2, 2), (n // 2, n - 3, n - 3))]
    pairs = [(s, e) for s, e in pairs if free[s[2], s[1], s[0]] and free[e[2], e[1], e[0]]]
    rows = oracle_rows(oracle, free, pairs)
    long_walk = 5000 if kind != "random64" else 3000
    rows += [random_walk(free, 400, 1), random_walk(free, long_walk, 2)]
    for r2 in (0, 1):
        assert_matches_reference(g, rows[:-1], r2)
        assert_matches_reference(g, rows, r2, max_span=48)
        assert_matches_reference(g, [rows[-1][:800]], r2, max_span=1)


@pytest.mark.gpu
def test_long_walk_without_span():
    """A 5000-node random walk around the wall's hole, window = the whole row."""
    free = synthetic("wall")
    g = occupancy_grid(free)
    row = random_walk(free, 5000, 3)
    got = assert_matches_reference(g, [row], 0)
    assert got[0][0].size < 5000


# ---- 3. r2 against inflation --------------------------------------------------------------------------------------------
def inflated(g, r2):
    import welding_robot_b200 as wr
    from welding_robot_b200._lib import check, lib
    h = C.c_void_p()
    check(lib().wr_grid_inflate(g._g, r2, C.byref(h)))
    out = wr.GridMap()
    out._adopt(h)
    return out


def weld_points_file(path):
    with open(path, "w") as fp:
        fp.write("%d\n" % len(C1_POINTS))
        for p in C1_POINTS:
            fp.write("%f %f %f\n" % p)


@pytest.fixture(scope="module")
def c1(meshes, tmp_path_factory):
    """C1: all 15 best paths of searchBestPathOfPoints (seed 0, defaults) and its graph file."""
    import welding_robot_b200 as wr
    d = tmp_path_factory.mktemp("c1")
    weld_points_file(d / "pts.in")
    g = wr.ACS_Rank(seed=0)
    quiet(g.creatGridMap, meshes["cubic"], 0.005, 10)
    quiet(g.searchBestPathOfPoints, 0.5, str(d / "pts.in"), str(d / "graph.in"))
    rows = [g.best_matrix[i][j].ids for i, j in PAIRS]
    assert all(len(r) for r in rows)
    return g, rows, d


@pytest.mark.gpu
@pytest.mark.parametrize("r2", [1, 2, 4])
def test_r2_equals_inflated_grid_at_zero(c1, r2):
    g, rows, _ = c1
    a = raw_shortcut(g, rows, r2)
    b = raw_shortcut(inflated(g, r2), rows, 0)
    assert all(np.array_equal(x[0], y[0]) and x[1] == y[1] and x[2] == y[2] for x, y in zip(a, b))
    free = synthetic("u")
    s = occupancy_grid(free)
    srows = [random_walk(free, 600, 4), random_walk(free, 2000, 5)]
    a = raw_shortcut(s, srows, r2, 64)
    b = raw_shortcut(inflated(s, r2), srows, 0, 64)
    assert all(np.array_equal(x[0], y[0]) and x[1] == y[1] and x[2] == y[2] for x, y in zip(a, b))


@pytest.mark.gpu
def test_r2_zero_builds_no_field_and_max_r2_keeps_the_row(meshes, c1):
    import welding_robot_b200 as wr
    from welding_robot_b200._lib import lib
    _, rows, _ = c1
    g = wr.GridMap()
    quiet(g.creatGridMap, meshes["cubic"], 0.005, 10)
    raw_shortcut(g, rows, 0)
    ms = C.c_float()
    assert lib().wr_grid_clearance_ms(g._g, C.byref(ms)) == 0 and ms.value == 0.0
    for (keep, nb, L), row in zip(raw_shortcut(g, rows, FAR), rows):
        assert np.array_equal(keep, np.arange(len(row))) and nb == len(row) - 1
        assert L == world_length(row, keep, grid_dims(g), g.coords())
    assert lib().wr_grid_clearance_ms(g._g, C.byref(ms)) == 0 and ms.value > 0.0


# ---- 4. C1 end to end through the Python facade -------------------------------------------------------------------------
def smoothed(path_xyz, m):
    """The demo's two curves (main.cpp:299-352): degree 0 through the path, then degree 2 through its samples."""
    import welding_robot_b200 as wr
    c0 = wr.BS_Basic(len(path_xyz), 0, 0, 0)
    c0.SetParam(path_xyz[0], path_xyz[-1], path_xyz, 150.0)
    first = c0.getCurvePoints(np.arange(10, 161, 10, dtype=np.float32))[0]
    c2 = wr.BS_Basic(len(first), 2, 2, 2)
    z6 = np.zeros(6, np.float32)
    c2.SetParam(np.concatenate([path_xyz[0], z6]), np.concatenate([path_xyz[-1], z6]), first, 6000.0)
    pts, ok = c2.getCurvePoints(np.linspace(0, 6000, m).astype(np.float32))
    assert ok.all()
    return pts


def table_row(g, m, rows):
    """(input nodes, waypoints, fallbacks, input length, shortcut length) over the 15 pairs of a shortcut matrix."""
    dims, coords = grid_dims(g), g.coords()
    nodes = sum(len(r) for r in rows)
    Lin = sum(world_length(r, np.arange(len(r)), dims, coords) for r in rows)
    way = sum(len(m[i][j].ids) for i, j in PAIRS)
    return nodes, way, Lin


@pytest.mark.gpu
def test_c1_table(c1, capsys):
    import welding_robot_b200 as wr
    g, rows, d = c1
    full = g.shortcutPaths(rows, 0.0)
    assert sum(len(w) for w, _, _, _ in full) == 30 and sum(b for _, _, b, _ in full) == 0
    assert round(sum(L for _, _, _, L in full), 4) == 3.6622
    one = g.shortcutPaths(rows, 0.005)                     # r2 = floor((0.005 / 0.005f)^2) = 1
    assert sum(len(w) for w, _, _, _ in one) == 485 and sum(b for _, _, b, _ in one) == 456
    assert round(sum(L for _, _, _, L in one), 4) == 4.2710
    nodes, _, Lin = table_row(g, g.best_matrix, rows)
    assert nodes == 1020 and round(Lin, 4) == 5.0250
    for r2, res in ((0, full), (1, one)):
        for (w, k, b, L), row in zip(res, rows):
            assert np.array_equal(w, row[k])
        got = raw_shortcut(g, rows, r2)
        assert all(np.array_equal(x[0], y[1]) and x[1] == y[2] and x[2] == y[3] for x, y in zip(got, res))
    assert_matches_reference(g, rows, 1, radius=0.005)
    # the matrix: [i][j] and [j][i] share one Agent, L is float32 of the length, dirs are empty
    m = g.shortcutBestMatrix()
    for q, (i, j) in enumerate(PAIRS):
        assert m[i][j] is m[j][i]
        assert np.array_equal(m[i][j].ids, full[q][0]) and m[i][j].dirs.size == 0 and m[i][j].L == float(np.float32(full[q][3]))
    assert all(m[i][i].L == g.best_matrix[i][i].L and m[i][i].ids.size == 0 for i in range(6))
    # seam ordering on the search lengths, then the shortcut paths stitched and smoothed
    route = wr.ACS_GTSP()
    assert route.readFromGraphFile(str(d / "graph.in"))
    quiet(route.computeSolution)
    route.read_all_segments(m)
    pts = np.stack([route.g_path_x, route.g_path_y, route.g_path_z], 1).astype(np.float32)
    assert len(pts) == sum(len(m[r][s].ids) for r, s in route.best_path[:-1])
    curve = smoothed(pts, 20000)
    with capsys.disabled():
        print("\nC1 shortcut (r2 = 0) stitched %d points; smoothed points' min d2 %d" % (len(pts), int(g.clearanceAt(curve)[1].min())))


@pytest.mark.gpu
def test_c1_inflate_search_shortcut(meshes, c1, tmp_path):
    import welding_robot_b200 as wr
    g0, _, _ = c1
    d2 = g0.clearanceMap()
    weld_points_file(tmp_path / "pts.in")
    g = wr.ACS_Rank(seed=0)
    quiet(g.creatGridMap, meshes["cubic"], 0.005, 10)
    g.inflateGridMap(0.005)
    quiet(g.searchBestPathOfPoints, 0.5, str(tmp_path / "pts.in"))
    rows = [g.best_matrix[i][j].ids for i, j in PAIRS]
    assert sum(len(r) for r in rows) == 1032
    # the inflated grid at 0 == the original grid at r2 = 1
    res = g.shortcutPaths(rows, 0.0)
    res1 = g0.shortcutPaths(rows, 0.005)
    assert all(np.array_equal(a[1], b[1]) and a[2] == b[2] and a[3] == b[3] for a, b in zip(res, res1))
    assert sum(len(w) for w, _, _, _ in res1) == 30 and sum(b for _, _, b, _ in res1) == 0
    assert all(d2[w].min() >= 4 for w, _, _, _ in res1)
    assert round(sum(L for _, _, _, L in res1), 4) == 3.6622
    assert_matches_reference(g0, rows, 1)


# ---- 5. K = 26 rows and C2 ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_k26_rows_on_c1(meshes, c1):
    import welding_robot_b200 as wr
    g0, _, _ = c1
    g = wr.ACS_Rank(seed=0, K=26)
    quiet(g.creatGridMap, meshes["cubic"], 0.005, 10)
    node = g.snapPoints(C1_POINTS)
    res = quiet(g.searchBatch, [int(node[i]) for i, _ in PAIRS], [int(node[j]) for _, j in PAIRS], 0.5, iterations=150)
    rows = [ids for ids, _, _ in res if len(ids)]
    assert len(rows) == len(PAIRS)
    for r2 in (0, 1):
        got = assert_matches_reference(g, rows, r2)
        if r2 == 1:
            assert sum(b for _, b, _ in got) > 0           # diagonals that cut a corner near the part are kept by the fallback


@pytest.mark.gpu
def test_c2_best_path():
    import sys
    sys.path.insert(0, ROOT)
    import bench
    import welding_robot_b200 as wr
    wl = bench.build_workload_gpu()
    g = wr.ACS_Rank(seed=bench.SEED, fixed_colony=4096, step_cap=bench.STEP_CAP)
    g.creatFromOccupancy(wl["isfree"], wl["xs"], wl["ys"], wl["zs"], bench.PRECISION)
    g.setEndpoints(wl["start"], wl["goal"])
    g.begin(bench.PREDICT)
    g.iterate(60)
    row = g.bestPath()[0]
    assert len(row) > 100
    for r2 in (0, 1):
        assert_matches_reference(g, [row], r2)
    assert_matches_reference(g, [row], 0, max_span=100)


# ---- 6. edge rows and arguments -----------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_edge_rows():
    free = synthetic("wall")
    g = occupancy_grid(free)
    dims = grid_dims(g)
    a, b = node_id(dims, (3, 3, 3)), node_id(dims, (9, 5, 4))
    rows = [[], [a], [a, a], [a, a, b, b, a], [], [b, a, a, b], [a]]
    got = assert_matches_reference(g, rows, 0)
    assert [len(k) for k, _, _ in got] == [0, 1, 2, 2, 0, 2, 1]
    assert got[0][2] == 0.0 and got[1][2] == 0.0 and got[2][2] == 0.0
    assert raw_shortcut(g, [], 0) == []
    assert [len(r[0]) for r in g.shortcutPaths([[], [a]])] == [0, 1]


@pytest.mark.gpu
def test_invalid_arguments_write_nothing():
    from welding_robot_b200._lib import lib, ptr
    free = synthetic("wall")
    g = occupancy_grid(free)
    N = g.size_of_map()
    L = lib()

    def call(ids, off, nrows, r2=0, span=0):
        ids = np.ascontiguousarray(ids, np.int64); off = np.ascontiguousarray(off, np.int64)
        keep = np.full(8, -7, np.int32); nk = np.full(4, -7, np.int32); nb = nk.copy(); ln = np.full(4, -7.0)
        st = L.wr_grid_shortcut_paths(g._g, ptr(ids), ptr(off), nrows, r2, span, ptr(keep), ptr(nk), ptr(nb), ptr(ln))
        return st, (keep == -7).all() and (nk == -7).all() and (nb == -7).all() and (ln == -7.0).all()

    assert call([0, 1, 2], [0, 3], 1) == (0, False)
    for args in [([0, N, 2], [0, 3], 1), ([0, -1, 2], [0, 3], 1), ([0, 1, 2], [0, 2, 1], 2), ([0, 1, 2], [1, 3], 1),
                 ([0, 1, 2], [0, 3], -1), ([0, 1, 2], [0, 3], 1, 0, -1), ([0, 1, 2], [0, 3], 1, 5, -3)]:
        assert call(*args) == (-1, True), args
    ids = np.zeros(2, np.int64); off = np.array([0, 2], np.int64)
    assert L.wr_grid_shortcut_paths(g._g, ptr(ids), ptr(off), 1, 0, 0, None, None, None, None) == -1
    assert L.wr_grid_shortcut_paths(None, ptr(ids), ptr(off), 1, 0, 0, None, None, None, None) == -1
    assert L.wr_grid_shortcut_paths(g._g, None, None, 0, 0, 0, None, None, None, None) == 0
    keep = np.zeros(2, np.int32); nk = np.zeros(1, np.int32)
    assert L.wr_grid_shortcut_paths(g._g, ptr(ids), ptr(off), 1, 0, 0, ptr(keep), ptr(nk), None, None) == 0 and nk[0] == 2
    big = occupancy_grid(np.ones((1, 1, 40000), np.uint8))
    ids = np.array([0, 39999], np.int64)
    assert L.wr_grid_shortcut_paths(big._g, ptr(ids), ptr(off), 1, 1, 0, ptr(keep), ptr(nk), None, None) == -1
    assert L.wr_grid_shortcut_paths(big._g, ptr(ids), ptr(off), 1, 0, 0, ptr(keep), ptr(nk), None, None) == 0
    assert list(keep) == [0, 1] and nk[0] == 2
    with pytest.raises(ValueError):
        g.shortcutPaths([[0, 1]], radius=-1.0)


# ---- 7. the C++ facade --------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_cpp_facade_prints_what_python_computes(meshes, c1, tmp_path):
    import welding_robot_b200 as wr
    from test_oracle_golden import stl_bytes
    from welding_robot_b200 import _lib
    g, rows, d = c1
    exe = str(tmp_path / "shortcut_test")
    libdir = os.path.dirname(_lib.LIB_PATH)
    subprocess.run(["g++", "-std=c++14", "-O1", "-Wall", "-I" + os.path.join(ROOT, "include", "welding_robot_b200"),
                    os.path.join(ROOT, "tests", "cpp", "shortcut_test.cpp"), "-o", exe, "-L" + libdir, "-lwrgpu",
                    "-Wl,-rpath," + libdir, "-ldl", "-lpthread", "-lrt"], check=True)
    stl = tmp_path / "cubic.stl"
    stl.write_bytes(stl_bytes(meshes["cubic"]))
    weld_points_file(tmp_path / "pts.in")
    r = subprocess.run([exe, str(stl), str(tmp_path / "pts.in"), str(tmp_path / "graph.in")], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    got = [line for line in r.stdout.splitlines() if line.startswith("shortcut ")]
    want = []
    for radius in (0.0, 0.005):
        for (i, j), (_, k, b, L) in zip(PAIRS, g.shortcutPaths(rows, radius)):
            want.append("shortcut pair %d %d radius %s nkeep %d blocked %d length %s" % (i, j, "%g" % radius, len(k), b, "%.17g" % L))
    route = wr.ACS_GTSP()
    assert route.readFromGraphFile(str(d / "graph.in"))
    quiet(route.computeSolution)
    route.read_all_segments(g.best_matrix)
    full = len(route.g_path_x)
    route.g_path_x, route.g_path_y, route.g_path_z = [], [], []
    m = g.shortcutBestMatrix()
    route.read_all_segments(m)
    want.append("shortcut stitched %d of %d" % (len(route.g_path_x), full))
    want.append("shortcut agent 0 1 nodes %d dirs 0 L %.9g" % (len(m[0][1].ids), m[1][0].L))
    assert got == want
