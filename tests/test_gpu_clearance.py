"""GPU: the clearance field (wr_grid_clearance), point queries (wr_grid_clearance_at) and obstacle inflation (wr_grid_inflate).

The field is exact: it equals scipy's Euclidean distance transform squared and rounded, and a numpy brute force on small grids.
Searches on an inflated grid equal the CPU oracle on the thresholded occupancy bit for bit."""
import contextlib
import ctypes as C
import io
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import C1_POINTS, ROOT

pytestmark = pytest.mark.gpu

FAR = np.uint32(0xFFFFFFFF)
PAIRS = [(i, j) for i in range(6) for j in range(i + 1, 6)]


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def occupancy_grid(isfree_zyx, xs=None, ys=None, zs=None, precision=1.0):
    import welding_robot_b200 as wr
    rz, ry, rx = isfree_zyx.shape
    xs = np.arange(rx, dtype=np.float32) if xs is None else xs
    ys = np.arange(ry, dtype=np.float32) if ys is None else ys
    zs = np.arange(rz, dtype=np.float32) if zs is None else zs
    return wr.GridMap().creatFromOccupancy(isfree_zyx.ravel(), xs, ys, zs, precision)


def mesh_grid(tris, precision, wall):
    import welding_robot_b200 as wr
    return quiet(wr.GridMap().creatGridMap, tris, precision, wall)


def field(g):
    return g.clearanceMap().reshape(g.rangeZ, g.rangeY, g.rangeX)


def scipy_d2(isfree_zyx):
    from scipy import ndimage
    return np.rint(ndimage.distance_transform_edt(isfree_zyx) ** 2).astype(np.uint32)


def brute_d2(isfree_zyx):
    occ = np.argwhere(isfree_zyx == 0)
    if len(occ) == 0:
        return np.full(isfree_zyx.shape, FAR)
    nodes = np.indices(isfree_zyx.shape).reshape(3, -1).T
    d2 = np.full(len(nodes), np.iinfo(np.int64).max)
    for chunk in np.array_split(occ, max(1, len(occ) // 256)):
        d2 = np.minimum(d2, ((nodes[:, None, :] - chunk[None]) ** 2).sum(-1).min(1))
    return d2.reshape(isfree_zyx.shape).astype(np.uint32)


def nearest_ref(g, pts):
    """float64 |p - c|.argmin() per axis, then the downloaded field; non-finite coordinates give -1 / UINT32_MAX."""
    pts = np.asarray(pts, np.float32).reshape(-1, 3)
    ok = np.isfinite(pts).all(1)
    p = pts[ok].astype(np.float64)
    ix, iy, iz = (np.abs(p[:, k, None] - c.astype(np.float64)[None]).argmin(1) for k, c in enumerate(g.coords()))
    ids = np.full(len(pts), -1, np.int64); d2 = np.full(len(pts), FAR, np.uint32)
    ids[ok] = (iz * g.rangeY + iy) * g.rangeX + ix
    d2[ok] = g.clearanceMap()[ids[ok]]
    return ids, d2


def inflated(g, r2):
    """wr_grid_inflate's new handle in a GridMap of its own."""
    import welding_robot_b200 as wr
    from welding_robot_b200._lib import check, lib
    h = C.c_void_p()
    check(lib().wr_grid_inflate(g._g, r2, C.byref(h)))
    out = wr.GridMap()
    out._adopt(h)
    return out


@pytest.fixture(scope="module")
def c1(meshes):
    return mesh_grid(meshes["cubic"], 0.005, 10)


# ---- 1. the exact field ---------------------------------------------------------------------------------------------
def test_field_on_mesh_grids(meshes, c1):
    """C1 cubic.stl (57 x 91 x 57, one duplicate y plane) and simplified_piece @ (0.008, 5) against scipy."""
    assert (c1.rangeX, c1.rangeY, c1.rangeZ) == (57, 91, 57)
    ys = c1.coords()[1]
    assert (np.diff(ys) == 0).sum() == 1
    free = c1.isfree().reshape(c1.rangeZ, c1.rangeY, c1.rangeX)
    assert np.array_equal(field(c1), scipy_d2(free))
    g = mesh_grid(meshes["simplified_piece"], 0.008, 5)
    free = g.isfree().reshape(g.rangeZ, g.rangeY, g.rangeX)
    assert np.array_equal(field(g), scipy_d2(free))


def test_field_on_bench_grids():
    """bench.py's C2 256^3 cube and C5 512^3 obstacle grid."""
    sys.path.insert(0, ROOT)
    import bench
    wl = bench.build_workload_gpu()
    n = len(wl["xs"])
    free = wl["isfree"].reshape(n, n, n)
    g = occupancy_grid(free, wl["xs"], wl["ys"], wl["zs"], bench.PRECISION)
    assert np.array_equal(field(g), scipy_d2(free))
    n = 512
    free = bench.synthetic_boxes(n, 4096, 4).reshape(n, n, n)
    g = occupancy_grid(free)
    assert np.array_equal(field(g), scipy_d2(free))


@pytest.mark.parametrize("shape", [(5, 7, 1), (6, 5, 31), (4, 9, 33), (3, 4, 1025), (4000, 3, 33), (2, 2000, 40),
                                   (20000, 1, 1), (1, 1, 30000), (1, 1, 1), (3, 1, 2)])
@pytest.mark.parametrize("p_occ", [0.0005, 0.05, 0.5])
def test_field_on_odd_shapes(shape, p_occ):
    """Line lengths around the 32-lane tiles, long y / z columns (fewer lanes per CTA), 1 x 1 x N and N x 1 x 1."""
    rng = np.random.default_rng(hash((shape, p_occ)) & 0xFFFF)
    free = (rng.random(shape) >= p_occ).astype(np.uint8)
    free.ravel()[rng.integers(free.size)] = 0          # at least one occupied node
    assert np.array_equal(field(occupancy_grid(free)), scipy_d2(free))


def test_field_single_all_and_none_occupied():
    free = np.ones((9, 10, 11), np.uint8)
    free[4, 7, 2] = 0
    assert np.array_equal(field(occupancy_grid(free)), brute_d2(free))
    assert (field(occupancy_grid(np.zeros((9, 10, 11), np.uint8))) == 0).all()
    assert (field(occupancy_grid(np.ones((9, 10, 11), np.uint8))) == FAR).all()
    assert (field(occupancy_grid(np.ones((1, 1, 70), np.uint8))) == FAR).all()


@pytest.mark.parametrize("seed", range(6))
def test_field_equals_brute_force(seed):
    rng = np.random.default_rng(seed)
    shape = tuple(int(v) for v in rng.integers(1, 25, 3))
    free = (rng.random(shape) >= [0.002, 0.01, 0.05, 0.2, 0.6, 0.95][seed]).astype(np.uint8)
    assert np.array_equal(field(occupancy_grid(free)), brute_d2(free)), shape


def test_axis_longer_than_32768_is_rejected():
    import welding_robot_b200 as wr
    g = occupancy_grid(np.ones((1, 1, 40000), np.uint8))
    with pytest.raises(wr.WrError) as e:
        g.clearanceMap()
    assert e.value.status == -1
    with pytest.raises(wr.WrError):
        g.clearanceAt([(1.0, 0.0, 0.0)])


def test_capacity_and_arguments(c1):
    from welding_robot_b200._lib import lib, ptr
    L = lib()
    c1.clearanceMap()
    small = np.zeros(c1.size_of_map() - 1, np.uint32)
    assert L.wr_grid_clearance(c1._g, ptr(small), small.size) == -6
    assert L.wr_grid_clearance(c1._g, None, c1.size_of_map()) == -1
    pts = np.zeros(3, np.float32)
    assert L.wr_grid_clearance_at(c1._g, ptr(pts), -1, None, None) == -1
    assert L.wr_grid_clearance_at(c1._g, None, 1, None, None) == -1
    assert L.wr_grid_clearance_at(c1._g, ptr(pts), 0, None, None) == 0
    assert L.wr_grid_inflate(c1._g, 1, None) == -1
    ms = C.c_float()
    assert L.wr_grid_clearance_ms(c1._g, C.byref(ms)) == 0 and ms.value > 0


# ---- 2. point queries -----------------------------------------------------------------------------------------------
def test_points_on_c1(c1):
    """Random points, exact midpoints between nodes, points on and beside the duplicate y plane, points beyond the grid, NaN / inf."""
    xs, ys, zs = c1.coords()
    rng = np.random.default_rng(3)
    lo = np.array([xs[0], ys[0], zs[0]]) - 0.05; hi = np.array([xs[-1], ys[-1], zs[-1]]) + 0.05
    pts = [rng.uniform(lo, hi, (20000, 3)).astype(np.float32)]
    mid = lambda c, i: np.float32((np.float64(c[i]) + np.float64(c[i + 1])) / 2)   # noqa: E731
    m = np.array([(mid(xs, rng.integers(len(xs) - 1)), mid(ys, rng.integers(len(ys) - 1)), mid(zs, rng.integers(len(zs) - 1)))
                  for _ in range(2000)], np.float32)
    pts.append(m)
    dup = int(np.flatnonzero(np.diff(ys) == 0)[0])
    for y in (ys[dup], np.nextafter(ys[dup], np.float32(-1)), np.nextafter(ys[dup], np.float32(9)), mid(ys, dup - 1), mid(ys, dup + 1)):
        pts.append(np.array([(xs[i], y, zs[j]) for i in range(0, len(xs), 7) for j in range(0, len(zs), 7)], np.float32))
    pts.append(np.array([(-1e30, 0, 0), (1e30, 1e30, -1e30), (xs[0] - 1, ys[-1] + 1, zs[3])], np.float32))
    bad = np.array([(np.nan, 0, 0), (0, np.inf, 0), (0, 0, -np.inf), (np.nan, np.nan, np.nan)], np.float32)
    pts.append(bad)
    pts = np.concatenate(pts)
    ids, d2 = c1.clearanceAt(pts)
    rid, rd2 = nearest_ref(c1, pts)
    assert np.array_equal(ids, rid) and np.array_equal(d2, rd2)
    assert (ids[-4:] == -1).all() and (d2[-4:] == FAR).all()
    on_dup = ids[(pts[:, 1] == ys[dup]) & np.isfinite(pts).all(1)]
    assert len(on_dup) and ((on_dup // c1.rangeX) % c1.rangeY == dup).all()     # the tie goes to the lower plane


def test_points_on_a_shuffled_table():
    """A non-monotone x table (allowed by wr_grid_create_from_occupancy) is scanned, not bisected."""
    rng = np.random.default_rng(8)
    free = (rng.random((6, 7, 40)) >= 0.1).astype(np.uint8)
    xs = rng.permutation(40).astype(np.float32) * np.float32(0.25)
    xs[5] = xs[9]                                        # a duplicate value too
    g = occupancy_grid(free, xs=xs)
    pts = np.concatenate([rng.uniform(-2, 12, (5000, 3)), np.stack([xs, np.full(40, 3.0), np.full(40, 2.5)], 1)]).astype(np.float32)
    ids, d2 = g.clearanceAt(pts)
    rid, rd2 = nearest_ref(g, pts)
    assert np.array_equal(ids, rid) and np.array_equal(d2, rd2)


def test_points_with_null_outputs(c1):
    from welding_robot_b200._lib import check, lib, ptr
    pts = np.random.default_rng(4).uniform(1.5, 1.7, (1000, 3)).astype(np.float32)
    rid, rd2 = nearest_ref(c1, pts)
    ids = np.zeros(1000, np.int64); d2 = np.zeros(1000, np.uint32)
    check(lib().wr_grid_clearance_at(c1._g, ptr(pts), 1000, ptr(ids), None))
    check(lib().wr_grid_clearance_at(c1._g, ptr(pts), 1000, None, ptr(d2)))
    check(lib().wr_grid_clearance_at(c1._g, ptr(pts), 1000, None, None))
    assert np.array_equal(ids, rid) and np.array_equal(d2, rd2)


def surface_samples(tris, n, seed):
    rng = np.random.default_rng(seed)
    v = tris[:, 3:].reshape(-1, 3, 3).astype(np.float64)
    area = 0.5 * np.linalg.norm(np.cross(v[:, 1] - v[:, 0], v[:, 2] - v[:, 0]), axis=1)
    t = rng.choice(len(v), n, p=area / area.sum())
    a, b = rng.random(n), rng.random(n)
    flip = a + b > 1
    a[flip], b[flip] = 1 - a[flip], 1 - b[flip]
    return (v[t, 0] + a[:, None] * (v[t, 1] - v[t, 0]) + b[:, None] * (v[t, 2] - v[t, 0])).astype(np.float32)


@pytest.mark.parametrize("mesh,precision,wall", [("cubic", 0.005, 10), ("simplified_piece", 0.008, 5)])
def test_surface_points_map_to_occupied_nodes(meshes, mesh, precision, wall):
    g = mesh_grid(meshes[mesh], precision, wall)
    ids, d2 = g.clearanceAt(surface_samples(meshes[mesh], 20000, 11))
    assert (ids >= 0).all() and (d2 == 0).all(), int((d2 != 0).sum())


# ---- 3. inflation ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("r2", [0, 1, 2, 3, 1000])
def test_inflate_thresholds_the_field(c1, r2):
    h = inflated(c1, r2)
    d = c1.clearanceMap()
    assert np.array_equal(h.isfree() == 0, d <= r2)
    if r2 == 0:
        assert np.array_equal(h.bits(), c1.bits())
    assert (h.rangeX, h.rangeY, h.rangeZ, h.precision, h.wall) == (c1.rangeX, c1.rangeY, c1.rangeZ, c1.precision, c1.wall)
    assert h.bbox() == c1.bbox()
    assert all(np.array_equal(a.view(np.uint32), b.view(np.uint32)) for a, b in zip(h.coords(), c1.coords()))
    assert h.stats() == dict(occupied=int((d <= r2).sum()), tests=0, kernel_ms=0.0)


# ---- 4. searches on an inflated grid --------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def c1_r1(meshes, c1, oracle):
    """C1 at r2 = 1: all 15 pairs through searchBatch (seed 0, 150 iterations) and through the oracle on the thresholded occupancy."""
    d = c1.clearanceMap()
    g = inflated_search_handle(meshes, 0.005)             # r2 = floor((0.005 / 0.005f)^2) = 1
    assert np.array_equal(g.isfree() == 0, d <= 1)
    node = g.snapPoints(C1_POINTS)
    s = [int(node[i]) for i, _ in PAIRS]; e = [int(node[j]) for _, j in PAIRS]
    bat = quiet(g.searchBatch, s, e, 0.5, iterations=150)
    G = oracle.Grid.from_occupancy((d > 1).astype(np.uint8), *c1.coords(), c1.precision)
    A = oracle.Acs(G, seed=0)
    ref = []
    for q in range(len(PAIRS)):
        A.set_endpoints(s[q], e[q]); A.set_next_search(q)
        A.begin(0.5); A.iterate(150)
        ref.append(A.best())
        A.reset()
    return d, node, bat, ref


def inflated_search_handle(meshes, radius):
    import welding_robot_b200 as wr
    g = wr.ACS_Rank(seed=0)
    quiet(g.creatGridMap, meshes["cubic"], 0.005, 10)
    g.inflateGridMap(radius)
    return g


def test_search_on_inflated_grid_equals_oracle(c1_r1):
    d, node, bat, ref = c1_r1
    assert (node >= 0).all()
    for q, ((ids, dirs, L), (rids, rdirs, rL)) in enumerate(zip(bat, ref)):
        assert np.isfinite(L) and np.float32(L) == np.float32(rL), q
        assert np.array_equal(ids, rids) and np.array_equal(dirs, rdirs), q
        assert d[ids].min() == 4, q            # one node further from the part than on the plain grid


def test_paths_on_plain_grid_touch_the_shell(meshes, c1):
    import welding_robot_b200 as wr
    d = c1.clearanceMap()
    g = wr.ACS_Rank(seed=0)
    quiet(g.creatGridMap, meshes["cubic"], 0.005, 10)
    node = g.snapPoints(C1_POINTS)
    res = quiet(g.searchBatch, [int(node[i]) for i, _ in PAIRS], [int(node[j]) for _, j in PAIRS], 0.5, iterations=150)
    assert [int(d[ids].min()) for ids, _, _ in res] == [1] * len(PAIRS)


def test_inflated_endpoints_that_do_not_snap(meshes, c1):
    """At r2 = 4 the 1.2 * precision box of some weld points holds no free node any more: 9 of the 15 pairs lose an endpoint."""
    g = inflated_search_handle(meshes, 0.01)              # r2 = floor((0.01 / 0.005f)^2) = 4
    assert np.array_equal(g.isfree() == 0, c1.clearanceMap() <= 4)
    node = g.snapPoints(C1_POINTS)
    assert sum(1 for i, j in PAIRS if node[i] < 0 or node[j] < 0) == 9
    assert not g.setPoints(C1_POINTS[int(np.flatnonzero(node < 0)[0])], C1_POINTS[0])


# ---- 5. facades -----------------------------------------------------------------------------------------------------
def weld_points_file(path):
    with open(path, "w") as fp:
        fp.write("%d\n" % len(C1_POINTS))
        for p in C1_POINTS:
            fp.write("%f %f %f\n" % p)


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


def test_python_facade_inflate_then_search(meshes, c1, c1_r1, tmp_path):
    import welding_robot_b200 as wr
    d, _, bat, _ = c1_r1
    g = wr.ACS_Rank(seed=0)
    quiet(g.creatGridMap, meshes["cubic"], 0.005, 10)
    quiet(g.initFromGridMap)
    assert g._a is not None
    g.inflateGridMap(0.005)                               # r2 = floor((0.005 / 0.005f)^2) = 1
    assert g._a is None and g.precision == c1.precision and g.wall == 10
    assert g.stats()["occupied"] == int((d <= 1).sum())
    f = tmp_path / "weld_points.in"
    weld_points_file(f)
    quiet(g.searchBestPathOfPoints, 0.5, str(f))
    assert g._a is not None
    for q, (i, j) in enumerate(PAIRS):
        best = g.best_matrix[i][j]
        assert np.array_equal(best.ids, bat[q][0]) and np.float32(best.L) == np.float32(bat[q][2])
    xs, ys, zs = g.coords()
    for q, (i, j) in enumerate(PAIRS):
        ids = g.best_matrix[i][j].ids
        z, r = np.divmod(ids, g.rangeX * g.rangeY); y, x = np.divmod(r, g.rangeX)
        pts = smoothed(np.stack([xs[x], ys[y], zs[z]], 1).astype(np.float32), 20000)
        got = g.clearanceAt(pts)
        want = nearest_ref(g, pts)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), q


def test_cpp_facade_prints_what_python_computes(meshes, c1, c1_r1, tmp_path):
    from test_oracle_golden import stl_bytes
    from welding_robot_b200 import _lib
    d, _, bat, _ = c1_r1
    exe = str(tmp_path / "clearance_test")
    libdir = os.path.dirname(_lib.LIB_PATH)
    subprocess.run(["g++", "-std=c++14", "-O1", "-Wall", "-I" + os.path.join(ROOT, "include", "welding_robot_b200"),
                    os.path.join(ROOT, "tests", "cpp", "clearance_test.cpp"), "-o", exe, "-L" + libdir, "-lwrgpu",
                    "-Wl,-rpath," + libdir, "-ldl", "-lpthread", "-lrt"], check=True)
    stl = tmp_path / "cubic.stl"
    stl.write_bytes(stl_bytes(meshes["cubic"]))
    pts = tmp_path / "weld_points.in"
    weld_points_file(pts)
    r = subprocess.run([exe, str(stl), str(pts)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    got = [l for l in r.stdout.splitlines() if l.startswith("clearance ")]
    want = ["clearance occupied %d inflated %d" % (int((d == 0).sum()), int((d <= 1).sum()))]
    h = inflated(c1, 1)
    xs, ys, zs = c1.coords()
    for q, (i, j) in enumerate(PAIRS):
        ids = bat[q][0]
        z, r = np.divmod(ids, c1.rangeX * c1.rangeY); y, x = np.divmod(r, c1.rangeX)
        at = h.clearanceAt(np.stack([xs[x], ys[y], zs[z]], 1))[1]
        want.append("clearance pair %d %d min_d2 %d inflated_at %d" % (i, j, int(d[ids].min()), int(at.min())))
    want += ["clearance path 0 1 L %.6f" % bat[0][2]]
    assert got == want
