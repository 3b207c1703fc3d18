"""Host-side mirror of the reference's class surface for the ACS hot path, over libwrgpu.so.

Same names, argument meaning and error behaviour as the reference's headers so that parity
tests read like its demo (main.cpp:273-283):

    model = STLReader(); model.readFile("cubic.stl")
    search = ACS_Rank()
    search.creatGridMap(model.TriangleList(), 0.005, 10)
    search.searchBestPathOfPoints(0.5, "weld_points.in", "graph.in")
    route = ACS_GTSP(); route.readFromGraphFile("graph.in"); route.computeSolution()
    route.read_all_segments(search.best_matrix)

All compute runs in hand-written sm_100a CUDA kernels behind the C ABI (include/wr_gpu.h).
The C++ twin of this file is include/welding_robot_b200/*.hpp.
"""
import ctypes as C
import math
import os

import numpy as np

from . import _lib
from ._lib import AcsParams, check, lib, ptr

INF_FLOAT = float("inf")


class Point3f:
    """Point3<float> (core/model_grid_map.hpp:34-70)."""
    __slots__ = ("x", "y", "z")

    def __init__(self, x=0.0, y=0.0, z=0.0):
        self.x, self.y, self.z = float(x), float(y), float(z)

    def __iter__(self):
        return iter((self.x, self.y, self.z))

    def __repr__(self):
        return "Point3f(%g, %g, %g)" % (self.x, self.y, self.z)


class STLReader:
    """STLReader (core/read_STL.hpp:23-175): binary STL -> triangle list."""

    def __init__(self):
        self._tris = np.zeros((0, 12), np.float32)

    def readFile(self, file_name):
        # read_STL.hpp:33-38 exits the process on I/O error; the library never exits: raise instead
        with open(file_name, "rb") as f:
            return self.readBuffer(f.read())

    def readBuffer(self, data: bytes):
        buf = np.frombuffer(data, np.uint8)
        n = C.c_int()
        check(lib().wr_stl_parse(ptr(buf), len(data), None, 0, C.byref(n)))
        t = np.zeros((n.value, 12), np.float32)
        check(lib().wr_stl_parse(ptr(buf), len(data), ptr(t), n.value, C.byref(n)))
        self._tris = t
        return True

    def NumTri(self):
        return len(self._tris)

    def TriangleList(self):
        """(T, 12) float32: normal, v0, v1, v2 — Triangles<float> without the unused `trait`."""
        return self._tris

    def PointList(self):
        return []  # never filled by the reference either (read_STL.hpp:119-120 is commented out)


class Vertex3:
    """Vertex3<float> / ACS_Node<float> as returned by paths (model_grid_map.hpp:81-88)."""
    __slots__ = ("pt", "isFree", "id")

    def __init__(self, pt, is_free, node_id):
        self.pt, self.isFree, self.id = pt, is_free, node_id


class GridMap:
    """GridMap<float> (core/model_grid_map.hpp:140-421) with the grid resident in HBM."""

    def __init__(self):
        self._g = None
        self.precision = 0.0
        self.wall = 0
        self.rangeX = self.rangeY = self.rangeZ = 0
        self._coords = None

    # -- construction ----------------------------------------------------------------------
    def creatGridMap(self, mesh, _precision, _wall, file_name=""):
        """model_grid_map.hpp:151-298.  mesh: (T,12) float32 triangle list."""
        mesh = np.ascontiguousarray(mesh, np.float32).reshape(-1, 12)
        self._destroy_grid()
        h = C.c_void_p()
        check(lib().wr_grid_create_from_triangles(ptr(mesh), len(mesh), _precision, _wall, C.byref(h)))
        self._adopt(h)
        mn, mx = self.bbox()
        print("[Grid Map]max(%.2f, %.2f, %.2f), min(%.2f, %.2f, %.2f) " % (mx[0], mx[1], mx[2], mn[0], mn[1], mn[2]))
        print("[Grid Map] %d triangles is scanned... " % len(mesh))
        print("[Grid Map] %d nodes is created... " % self.size_of_map())
        if file_name:
            self.writeGridMap(file_name)
        print("[Grid Map] Done! \r")
        return self

    def creatFromOccupancy(self, isfree, xs, ys, zs, precision):
        """Synthetic-grid entry point (an addition: the reference can only voxelise a mesh)."""
        isfree = np.ascontiguousarray(isfree, np.uint8).ravel()
        xs, ys, zs = (np.ascontiguousarray(v, np.float32) for v in (xs, ys, zs))
        if isfree.size != len(xs) * len(ys) * len(zs):
            raise ValueError("isfree must hold rx*ry*rz bytes in z,y,x order")
        self._destroy_grid()
        h = C.c_void_p()
        check(lib().wr_grid_create_from_occupancy(ptr(isfree), len(xs), len(ys), len(zs), ptr(xs), ptr(ys), ptr(zs), precision, C.byref(h)))
        self._adopt(h)
        return self

    def _adopt(self, h):
        self._g = h
        d = (C.c_int * 3)()
        check(lib().wr_grid_dims(h, d))
        self.rangeX, self.rangeY, self.rangeZ = d[0], d[1], d[2]
        p = C.c_float(); w = C.c_int()
        check(lib().wr_grid_precision(h, C.byref(p), C.byref(w)))
        self.precision, self.wall = p.value, w.value
        self._coords = None

    def _destroy_grid(self):
        if self._g is not None:
            lib().wr_grid_destroy(self._g)
            self._g = None

    # -- text dump / reload (model_grid_map.hpp:275-356) -----------------------------------
    def writeGridMap(self, file_name):
        """Same layout as :278-290, but the header carries the GLOBAL mesh box: the reference
        writes the last triangle's box there (:279), which makes its own reload wrong."""
        free = self.isfree().reshape(self.rangeZ, self.rangeY, self.rangeX)
        mn, mx = self.bbox()
        with open(file_name, "w") as fp:
            fp.write("%d %d %d %d %f %d\n" % (self.size_of_map(), self.rangeX, self.rangeY, self.rangeZ, self.precision, self.wall))
            fp.write("%f %f %f %f %f %f\n" % (mn[0], mn[1], mn[2], mx[0], mx[1], mx[2]))
            for z in range(self.rangeZ):
                for y in range(self.rangeY):
                    fp.write(" ".join("1" if v else "0" for v in free[z, y]) + " \n")
        print("\n[Grid Map] Successfully write to %s \r" % file_name)

    def readGridMap(self, file_name):
        """model_grid_map.hpp:300-356: coordinates are rebuilt from the header's box."""
        try:
            fp = open(file_name, "r")
        except OSError:
            print("[Grid Map] Failed to read file, skipping...")
            return
        with fp:
            tok = fp.read().split()
        n, rx, ry, rz = (int(t) for t in tok[:4])
        precision = np.float32(float(tok[4])); wall = int(tok[5])
        mn = [np.float32(float(t)) for t in tok[6:9]]; mx = [np.float32(float(t)) for t in tok[9:12]]
        free = np.array(tok[12:12 + rx * ry * rz], dtype=np.int64).astype(np.uint8)
        if free.size != rx * ry * rz:
            raise ValueError("grid file is truncated")
        axes = [_axis_coords(r, wall, a, b, precision) for r, a, b in ((rx, mn[0], mx[0]), (ry, mn[1], mx[1]), (rz, mn[2], mx[2]))]
        self.creatFromOccupancy(free != 0, axes[0], axes[1], axes[2], float(precision))
        self.wall = wall
        print("\n[Grid Map] Successfully read grid map from %s \r" % file_name)

    # -- accessors -------------------------------------------------------------------------
    def size_of_map(self):
        return self.rangeX * self.rangeY * self.rangeZ

    def bbox(self):
        mn = (C.c_float * 3)(); mx = (C.c_float * 3)()
        check(lib().wr_grid_bbox(self._g, mn, mx))
        return list(mn), list(mx)

    def coords(self):
        if self._coords is None:
            xs, ys, zs = (np.zeros(n, np.float32) for n in (self.rangeX, self.rangeY, self.rangeZ))
            check(lib().wr_grid_coords(self._g, ptr(xs), ptr(ys), ptr(zs)))
            self._coords = (xs, ys, zs)
        return self._coords

    def isfree(self):
        """uint8[N] in z,y,x order: Vertex3::isFree of every node."""
        out = np.zeros(self.size_of_map(), np.uint8)
        check(lib().wr_grid_download_isfree(self._g, ptr(out), out.size))
        return out

    def bits(self):
        out = np.zeros((self.size_of_map() + 31) // 32, np.uint32)
        check(lib().wr_grid_download_bits(self._g, ptr(out), out.size))
        return out

    def stats(self):
        occ = C.c_uint64(); tests = C.c_uint64(); ms = C.c_float()
        check(lib().wr_grid_stats(self._g, C.byref(occ), C.byref(tests), C.byref(ms)))
        return dict(occupied=occ.value, tests=tests.value, kernel_ms=ms.value)

    # -- clearance (an addition: the reference never measures how close a path comes to the part) --------------------
    def clearanceMap(self):
        """uint32[N] in z,y,x order: squared INDEX distance of every node to the nearest occupied node (0 on occupied nodes,
        UINT32_MAX everywhere when none is occupied).  World distance ~= sqrt(d2) * precision away from the max-side wall
        planes.  Built on the device on first use and kept with the grid."""
        out = np.zeros(self.size_of_map(), np.uint32)
        check(lib().wr_grid_clearance(self._g, ptr(out), out.size))
        return out

    def clearanceAt(self, points):
        """Per point: the nearest node (per axis argmin |p - c[i]| in double, lowest index on ties; beyond the grid: the
        boundary node) and its d2.  -> (int64 ids, uint32 d2); a non-finite coordinate gives -1 / UINT32_MAX."""
        pts = np.ascontiguousarray(np.asarray(points, np.float32).reshape(-1, 3))
        ids = np.zeros(len(pts), np.int64); d2 = np.zeros(len(pts), np.uint32)
        check(lib().wr_grid_clearance_at(self._g, ptr(pts), len(pts), ptr(ids), ptr(d2)))
        return ids, d2

    def _radius_r2(self, radius, who):
        """A world radius as a squared index radius: floor((radius / precision)^2), saturating at UINT32_MAX."""
        if self._g is None:
            raise _lib.WrError(-4, "%s: no grid map" % who)
        if not radius >= 0:
            raise ValueError("%s: radius must be >= 0" % who)
        return min(math.floor((float(radius) / float(self.precision)) ** 2), 0xFFFFFFFF)

    def inflateGridMap(self, radius):
        """Replace the grid by its obstacles inflated by `radius` (world units): a node becomes occupied iff its squared index
        distance to the part is <= floor((radius / precision)^2).  Dims, coordinates, precision and wall stay; an ACS_Rank
        drops its search handle and creates a new one on next use."""
        r2 = self._radius_r2(radius, "inflateGridMap")
        h = C.c_void_p()
        check(lib().wr_grid_inflate(self._g, r2, C.byref(h)))
        precision, wall = self.precision, self.wall
        self._destroy_grid()
        self._adopt(h)
        self.precision, self.wall = precision, wall
        return self

    def shortcutPaths(self, paths, radius=0.0, max_span=0):
        """Greedy line-of-sight shortcutting of node rows (include/wr_gpu.h, wr_grid_shortcut_paths), all rows in one launch.
        A segment between two nodes is kept clear of every node whose squared index distance to the part is <=
        floor((radius / precision)^2) (radius 0: of occupied nodes); from each waypoint the next one is the furthest row
        node, at most `max_span` ahead (0: no bound), whose segment is clear, else the next node.  -> per row
        (waypoint ids, keep indices into the row, blocked = segments kept by that fallback, world length in double)."""
        r2 = self._radius_r2(radius, "shortcutPaths")
        rows = [np.asarray(p, np.int64).ravel() for p in paths]
        off = np.zeros(len(rows) + 1, np.int64)
        off[1:] = np.cumsum([len(r) for r in rows])
        ids = np.ascontiguousarray(np.concatenate(rows) if rows else np.zeros(0, np.int64))
        keep = np.zeros(max(len(ids), 1), np.int32)
        nkeep = np.zeros(max(len(rows), 1), np.int32); blocked = np.zeros_like(nkeep); length = np.zeros(len(nkeep), np.float64)
        check(lib().wr_grid_shortcut_paths(self._g, ptr(ids), ptr(off), len(rows), r2, int(max_span), ptr(keep), ptr(nkeep),
                                           ptr(blocked), ptr(length)))
        out = []
        for p, r in enumerate(rows):
            k = keep[off[p]:off[p] + nkeep[p]].copy()
            out.append((r[k], k, int(blocked[p]), float(length[p])))
        return out

    def node(self, node_id):
        """The Vertex3 of a node id (materialised on demand; ptr_grid_map()'s cuboid is never built)."""
        xs, ys, zs = self.coords()
        rxy = self.rangeX * self.rangeY
        z, r = divmod(int(node_id), rxy)
        y, x = divmod(r, self.rangeX)
        return Vertex3(Point3f(xs[x], ys[y], zs[z]), True, int(node_id))

    def plot_grid_map(self, figureNumber=1):  # plotting is out of scope (model_grid_map.hpp:368-379)
        pass

    def show_plot(self):
        pass

    def __del__(self):
        try:
            self._destroy_grid()
        except Exception:
            pass


def _axis_coords(rng, wall, mn, mx, precision):
    """model_grid_map.hpp:204-205 in float32."""
    f = np.float32
    out = np.zeros(rng, np.float32)
    for i in range(rng):
        if i < wall:
            out[i] = f(mn) - f(f(wall - i) * f(precision))
        elif i >= rng - wall:
            out[i] = f(mx) + f(f(i - rng + wall) * f(precision))
        else:
            out[i] = f(mn) + f(f(i - wall) * f(precision))
    return out


class Agent:
    """Agent<float> (core/ACSRank_3D.hpp:62-109): a path, its chosen slots and its length."""

    def __init__(self, grid=None, ids=None, dirs=None, L=INF_FLOAT):
        self._grid = grid
        self.ids = np.zeros(0, np.int64) if ids is None else np.asarray(ids, np.int64)
        self.dirs = np.zeros(0, np.int32) if dirs is None else np.asarray(dirs, np.int32)
        self.L = L

    @property
    def tabu_list(self):
        return set(int(i) for i in self.ids)

    def getPath(self):
        return [self._grid.node(i) for i in self.ids]

    def nodeIndex(self):
        return [int(d) for d in self.dirs]

    def findPathNode(self, target):
        tid = target.id if isinstance(target, Vertex3) else int(target)
        return bool((self.ids == tid).any())


class ACS_Rank(GridMap):
    """ACS_Rank (core/ACSRank_3D.hpp:111-599) with the colony on the GPU.

    Additions the reference lacks (SURVEY.md §8b): a parameter struct (`params`), explicit
    `begin` / `iterate` / `bestPath` stepping, counters and per-kernel timings.
    """

    def __init__(self, **params):
        super().__init__()
        self.params = AcsParams()
        check(lib().wr_acs_default_params(C.byref(self.params)))
        self.max_iteration = 150  # ACSRank_3D.hpp:322
        known = {f[0] for f in AcsParams._fields_}
        for k, v in params.items():
            if k == "max_iteration":
                self.max_iteration = v
            elif k in known:
                setattr(self.params, k, v)
            else:   # a typo must not silently run the search with defaults
                raise TypeError("ACS_Rank: unknown parameter %r (known: max_iteration, %s)" % (k, ", ".join(sorted(known))))
        self._a = None
        self.best_matrix = None
        self.route_points = []
        self._start_id = self._goal_id = -1

    # -- lifetime --------------------------------------------------------------------------
    def _destroy_grid(self):
        self._destroy_acs()
        super()._destroy_grid()

    def _destroy_acs(self):
        if getattr(self, "_a", None) is not None:
            lib().wr_acs_destroy(self._a)
            self._a = None

    def initFromGridMap(self):
        """ACSRank_3D.hpp:317-410."""
        if self._g is None:
            raise _lib.WrError(-4, "initFromGridMap: no grid map")
        self._destroy_acs()
        h = C.c_void_p()
        check(lib().wr_acs_create(self._g, C.byref(self.params), C.byref(h)))
        self._a = h
        print("[ACS 3D] Created %d nodes, node cubiod [x: %d, y: %d, z: %d]\r" % (self.size_of_map(), self.rangeX, self.rangeY, self.rangeZ))

    def _need(self):
        if self._a is None:
            self.initFromGridMap()
        return self._a

    # -- reference methods -----------------------------------------------------------------
    def setPoints(self, start, end):
        """ACSRank_3D.hpp:537-565 -> bool."""
        s = np.array(list(start), np.float32); e = np.array(list(end), np.float32)
        ids = np.zeros(2, np.int64)
        st = lib().wr_acs_set_points(self._need(), ptr(s), ptr(e), ptr(ids))
        self._start_id, self._goal_id = int(ids[0]), int(ids[1])
        if st == _lib.WR_ERR_NOTFOUND:
            return False
        check(st)
        return True

    def setEndpoints(self, start_id, goal_id):
        check(lib().wr_acs_set_endpoints(self._need(), start_id, goal_id))
        self._start_id, self._goal_id = int(start_id), int(goal_id)

    def snapPoints(self, points):
        """setPoints' scan (ACSRank_3D.hpp:545-562) for many points in one kernel -> int64 node ids (-1: no free node)."""
        pts = np.ascontiguousarray(np.array([list(p) for p in points], np.float32).reshape(-1, 3))
        ids = np.full(len(pts), -1, np.int64)
        check(lib().wr_acs_snap_points(self._need(), ptr(pts), len(pts), ptr(ids)))
        return ids

    def stepCap(self):
        return self.params.step_cap if self.params.step_cap > 0 else min(self.size_of_map() - 1, 65532)

    def searchPairs(self, start_ids, goal_ids, predict_path_len, iterations=None, with_paths=True, batch=False):
        """The all-pairs loop (ACSRank_3D.hpp:472-499) on the device: per pair computeSolution + reset(), no host
        synchronisation between pairs.  -> list of (ids, dirs, L) per pair (ids/dirs empty when no path).
        batch=True: the same searches advanced concurrently (wr_acs_search_batch) — same results, bit for bit."""
        s = np.ascontiguousarray(start_ids, np.int64); g = np.ascontiguousarray(goal_ids, np.int64)
        n = len(s)
        it = self.max_iteration if iterations is None else iterations
        L = np.zeros(max(n, 1), np.float32); cnt = np.zeros(max(n, 1), np.int32)
        fn = lib().wr_acs_search_batch if batch else lib().wr_acs_search_pairs
        check(fn(self._need(), ptr(s), ptr(g), n, predict_path_len, it, ptr(L), ptr(cnt), None, None, 0))
        out = []
        for p in range(n):
            k = int(cnt[p])
            if not with_paths or k == 0:
                out.append((np.zeros(0, np.int64), np.zeros(0, np.int32), float(L[p])))
                continue
            ids = np.zeros(k, np.int64); dirs = np.zeros(k, np.int32); m = C.c_int(); Lp = C.c_float()
            check(lib().wr_acs_result_path(self._a, p, ptr(ids), ptr(dirs), k, C.byref(m), C.byref(Lp)))
            out.append((ids, dirs[:k - 1].copy(), float(L[p])))
        return out

    def searchBatch(self, start_ids, goal_ids, predict_path_len, iterations=None, with_paths=True):
        return self.searchPairs(start_ids, goal_ids, predict_path_len, iterations, with_paths, batch=True)

    def batchStats(self):
        out = np.zeros(4, np.uint64)
        check(lib().wr_acs_batch_stats(self._need(), ptr(out)))
        return dict(queries_per_chunk=int(out[0]), table_entries=int(out[1]), entries_used=int(out[2]), fallbacks=int(out[3]))

    def checkRoutePoints(self):
        """ACSRank_3D.hpp:511-535."""
        for p in self.route_points:
            q = Point3f(*p)
            if not self.setPoints(q, q):
                print("[ACS 3D] Invalid route point, please reset point(%.3f, %.3f, %.3f) " % (q.x, q.y, q.z))
        print("[ACS 3D] %d route points have been checked. " % len(self.route_points))

    def begin(self, predict_path_len):
        check(lib().wr_acs_begin(self._need(), predict_path_len))

    def setNextSearch(self, index):
        """Philox: the search index the next begin() takes (default: the number of begin() calls so far)."""
        check(lib().wr_acs_set_next_search(self._need(), index))

    def iterate(self, n=1):
        check(lib().wr_acs_iterate(self._need(), n))

    def sync(self):
        check(lib().wr_acs_sync(self._need()))

    def computeSolution(self, predict_path_len):
        """ACSRank_3D.hpp:220-305."""
        self.begin(predict_path_len)
        self.iterate(self.max_iteration)

    def reset(self):
        """ACSRank_3D.hpp:307-315."""
        check(lib().wr_acs_reset(self._need()))

    def bestPath(self):
        n = C.c_int(); L = C.c_float()
        check(lib().wr_acs_best(self._need(), None, None, 0, C.byref(n), C.byref(L)))
        ids = np.zeros(max(n.value, 1), np.int64); dirs = np.zeros(max(n.value, 1), np.int32)
        check(lib().wr_acs_best(self._a, ptr(ids), ptr(dirs), n.value, C.byref(n), C.byref(L)))
        return ids[:n.value].copy(), dirs[:max(n.value - 1, 0)].copy(), L.value

    def getSolution(self):
        """ACSRank_3D.hpp:506-509."""
        ids, dirs, L = self.bestPath()
        return Agent(self, ids, dirs, L)

    def searchBestPathOfPoints(self, predict_path_len=10, read_file="", output_file=""):
        """ACSRank_3D.hpp:427-504: all-pairs searches, best_matrix, graph file."""
        if read_file == "":
            print("[ACS 3D] Please enter passing point number: ", end="")
            point_num = int(input())
            print("[ACS 3D] Please enter passing point in order: ")
            self.route_points = [Point3f(*(float(v) for v in input().split())) for _ in range(point_num)]
        else:
            try:
                with open(read_file, "r") as fp:
                    tok = fp.read().split()
            except OSError:
                print("[ACS 3D] Failed to read file, reject to init.")
                return
            point_num = int(tok[0])
            self.route_points = [Point3f(*(float(v) for v in tok[1 + 3 * i:4 + 3 * i])) for i in range(point_num)]
        self.best_matrix = [[Agent(self) for _ in range(point_num)] for _ in range(point_num)]
        self.initFromGridMap()
        self.checkRoutePoints()
        # the pair loop of :472-499 runs on the device (wr_acs_search_pairs): snap every point once, search all pairs up
        # to the first one the reference would reject, read everything back once
        node = self.snapPoints(self.route_points) if point_num else np.zeros(0, np.int64)
        pairs = [(i, j) for i in range(point_num) for j in range(i + 1, point_num)]
        bad = next((q for q, (i, j) in enumerate(pairs) if node[i] < 0 or node[j] < 0), len(pairs))
        res = self.searchPairs([node[i] for i, _ in pairs[:bad]], [node[j] for _, j in pairs[:bad]], predict_path_len, batch=True) if bad else []
        lengths = []
        for (i, j), (ids, dirs, L) in zip(pairs[:bad], res):
            pi, pj = self.route_points[i], self.route_points[j]
            best = Agent(self, ids, dirs, L)
            self.best_matrix[i][j] = best
            self.best_matrix[j][i] = best
            print("[ACS 3D] <Point (%.3f, %.3f, %.3f) : Point (%.3f, %.3f, %.3f)> Path length: %.3f\r" %
                  (pi.x, pi.y, pi.z, pj.x, pj.y, pj.z, best.L))
            lengths.append(best.L)
        if bad < len(pairs):
            pi, pj = self.route_points[pairs[bad][0]], self.route_points[pairs[bad][1]]
            print("[ACS 3D] Wrong point : (%.3f, %.3f, %.3f) or (%.3f, %.3f, %.3f), program will exit immediately \r" %
                  (pi.x, pi.y, pi.z, pj.x, pj.y, pj.z))
            return
        if output_file:
            # the reference rewrites the header in place with "%d %d\r" (:500-501), which clobbers the
            # first distance once point_num >= 10; the header is written whole here.
            with open(output_file, "w") as fp:
                fp.write("%d %d\n" % (point_num, len(lengths)))
                for L in lengths:
                    fp.write("%.3f\n" % L)
            print("[ACS 3D] %d Result has been written to \"%s\" \r" % (len(lengths), output_file))

    def shortcutBestMatrix(self, radius=0.0, max_span=0):
        """best_matrix with every best path shortcut (GridMap.shortcutPaths, one launch for all pairs): a new matrix of Agents
        whose ids are the waypoint ids, with empty dirs and L = float32 of the waypoint polyline's world length; [i][j] and
        [j][i] share one object as in best_matrix.  ACS_GTSP.read_all_segments stitches it like best_matrix.  Entries
        without a path are copied as they are."""
        if self.best_matrix is None:
            raise _lib.WrError(-4, "shortcutBestMatrix: no best_matrix (run searchBestPathOfPoints first)")
        n = len(self.best_matrix)
        pairs = [(i, j) for i in range(n) for j in range(i + 1, n) if len(self.best_matrix[i][j].ids)]
        res = self.shortcutPaths([self.best_matrix[i][j].ids for i, j in pairs], radius, max_span)
        out = [[Agent(self, L=self.best_matrix[i][j].L) for j in range(n)] for i in range(n)]
        for (i, j), (ids, _, _, L) in zip(pairs, res):
            out[i][j] = out[j][i] = Agent(self, ids, None, float(np.float32(L)))
        return out

    # -- introspection (parity tests, bench) -----------------------------------------------
    def pheromone(self):
        out = np.zeros(self.size_of_map() * int(self.params.K), np.float32)
        check(lib().wr_acs_download_pheromone(self._need(), ptr(out), out.size))
        return out

    def setPheromone(self, tau):
        tau = np.ascontiguousarray(tau, np.float32)
        check(lib().wr_acs_upload_pheromone(self._need(), ptr(tau), tau.size))

    def lastColony(self):
        c = C.c_int(); lam = C.c_float(); q = C.c_float()
        check(lib().wr_acs_last_colony(self._need(), C.byref(c), C.byref(lam), C.byref(q)))
        return c.value, lam.value, q.value

    def lastAnt(self, k):
        n = C.c_int(); L = C.c_float(); order = C.c_int()
        check(lib().wr_acs_last_ant(self._need(), k, None, None, 0, C.byref(n), C.byref(L), C.byref(order)))
        ids = np.zeros(max(n.value, 1), np.int64); dirs = np.zeros(max(n.value, 1), np.int32)
        check(lib().wr_acs_last_ant(self._a, k, ptr(ids), ptr(dirs), n.value, C.byref(n), C.byref(L), C.byref(order)))
        return ids[:n.value].copy(), dirs[:max(n.value - 1, 0)].copy(), L.value, order.value

    def counters(self):
        out = np.zeros(9, np.uint64)
        check(lib().wr_acs_counters(self._need(), ptr(out)))
        keys = ["ant_steps", "ants", "arrived", "dead_no_candidate", "dead_fallthrough", "dead_step_cap", "iterations",
                "deposit_records", "table_overflows"]
        return dict(zip(keys, (int(v) for v in out)))

    def setTiming(self, enabled=True):
        check(lib().wr_acs_set_timing(self._need(), int(enabled)))

    def kernelMs(self):
        out = np.zeros(5, np.float32)
        check(lib().wr_acs_kernel_ms(self._need(), ptr(out)))
        return dict(walk=float(out[0]), rank=float(out[1]), deposit_build=float(out[2]), update=float(out[3]), total=float(out[4]))

    def updateStats(self):
        """WR_UPDATE_RANKSET: which deposit path the last iteration took and how concentrated the deposits were; group_ranks:
        eligible ranks of the last iteration whose bits were set once per best-path slot (ants verified on the whole best path),
        group_ranks_total: the same summed since begin."""
        out = np.zeros(4, np.uint32)
        check(lib().wr_acs_update_stats(self._need(), ptr(out)))
        grp = np.zeros(2, np.uint64)
        check(lib().wr_acs_group_stats(self._need(), ptr(grp)))
        return dict(rankset_last=int(out[0]), deposit_tiles=int(out[1]), distinct_slots=int(out[2]), rankset_iterations=int(out[3]),
                    group_ranks=int(grp[0]), group_ranks_total=int(grp[1]))

    def walkStats(self):
        """Converged iterations: ants completed by checking the best path against roulette thresholds, and the ant-steps that
        check decided (cumulative since the handle was created)."""
        out = np.zeros(2, np.uint64)
        check(lib().wr_acs_walk_stats(self._need(), ptr(out)))
        return dict(verified_ants=int(out[0]), verified_steps=int(out[1]))

    def streamKernelMs(self):
        """(cumulative device ms, launches) of the kernel that streams the pheromone field, timed inside the loop."""
        ms = C.c_float(); n = C.c_int()
        check(lib().wr_acs_stream_kernel_ms(self._need(), C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def fieldStats(self):
        """Clean-tile field: (16 KB tiles with at least one dirty line, tiles of the field)."""
        out = np.zeros(2, np.uint64)
        check(lib().wr_acs_field_stats(self._need(), ptr(out)))
        return int(out[0]), int(out[1])

    def fieldLines(self):
        """Clean-tile field: (128-byte lines the evaporation pass touches, lines of the field)."""
        out = np.zeros(2, np.uint64)
        check(lib().wr_acs_field_lines(self._need(), ptr(out)))
        return int(out[0]), int(out[1])

    def benchKernel(self, which, reps=20):
        """Average device ms of one update-path kernel run alone (0 fused update, 1 float4 evaporation, 2 D2D copy, 3 all-TMA ring variant)."""
        ms = C.c_float()
        check(lib().wr_acs_bench_kernel(self._need(), which, reps, C.byref(ms)))
        return ms.value

    def plot_path(self, agentK=None, figureNumber=1):  # ACSRank_3D.hpp:567-583 — plotting out of scope
        pass

    def plot_route_point(self, figureNumber=1):
        pass

    def __del__(self):
        try:
            self._destroy_acs()
        except Exception:
            pass
        super().__del__()


class ACS_GTSP:
    """ACS_GTSP (core/ACS_GTSP.hpp:82-328): ant-colony ordering of the weld seams (a symmetric TSP
    over the pair-length matrix), on the GPU.  `computeBatch` is the batched entry point the
    reference lacks: B independent colonies on the same matrix, one CTA each.  `colonies` (an
    addition) is the batch setDistanceMatrix creates: computeSolution then runs them all, each to
    the reference's stopping rule, and keeps the best colony's tour (multi-start)."""

    def __init__(self, seed=0, colonies=1):
        self.seed = seed
        self.colonies = colonies
        self.city_num = 0
        self.dis = None
        self.cnt = 0
        self._g = None
        self._batch = 0
        self.best_path = np.zeros((0, 2), np.int32)   # best.path: (r, s) per edge
        self.best_L = float(0x3f3f3f3f)
        self.g_path_x, self.g_path_y, self.g_path_z = [], [], []
        self.init_flag = False

    def readFromGraphFile(self, filename):
        """ACS_GTSP.hpp:224-253: "<city_num> <cnt>" then the upper triangle, row by row."""
        with open(filename, "r") as fp:
            tok = fp.read().split()
        n, cnt = int(tok[0]), int(tok[1])
        vals = [float(t) for t in tok[2:2 + n * (n - 1) // 2]]
        if len(vals) != n * (n - 1) // 2:
            raise _lib.WrError(-7, "graph file holds %d of %d distances" % (len(vals), n * (n - 1) // 2))
        dis = np.zeros((n, n), np.float64)
        it = iter(vals)
        for i in range(n):
            for j in range(i + 1, n):
                dis[i, j] = dis[j, i] = next(it)
                print("distance: %f \r" % dis[i, j])
        return self.setDistanceMatrix(dis, cnt)

    def setDistanceMatrix(self, dis, cnt=None):
        """In-memory variant of readFromGraphFile (the hand-off SURVEY.md §8f asks for)."""
        dis = np.ascontiguousarray(dis, np.float64)
        self.city_num = dis.shape[0]
        self.dis = dis
        self.cnt = self.city_num * (self.city_num - 1) // 2 if cnt is None else cnt
        self._create(self.colonies)
        self.init_flag = True
        return True

    def _create(self, batch, colony_first=0):
        if self._g is not None:
            lib().wr_gtsp_destroy(self._g)
            self._g = None
        h = C.c_void_p()
        check(lib().wr_gtsp_create(ptr(self.dis), self.city_num, self.cnt, batch, colony_first, self.seed, C.byref(h)))
        self._g, self._batch = h, batch
        self.best_L = float(0x3f3f3f3f)

    def tau0(self):
        t = C.c_double()
        check(lib().wr_gtsp_tau0(self._g, C.byref(t)))
        return t.value

    def iterate(self, n=1):
        check(lib().wr_gtsp_iterate(self._g, n))

    def best(self, colony=0):
        n = C.c_int(); L = C.c_double()
        tour = np.zeros(2 * self.city_num, np.int32)
        check(lib().wr_gtsp_best(self._g, colony, ptr(tour), C.byref(n), C.byref(L)))
        return tour[:2 * n.value].reshape(n.value, 2).copy(), L.value

    def pheromone(self, colony=0):
        out = np.zeros((self.city_num, self.city_num), np.float64)
        check(lib().wr_gtsp_download_pheromone(self._g, colony, ptr(out)))
        return out

    def kernelMs(self):
        out = np.zeros(3, np.float32)
        check(lib().wr_gtsp_kernel_ms(self._g, ptr(out)))
        return dict(info=float(out[0]), construct=float(out[1]), update=float(out[2]))

    def solve(self, max_iterations=0):
        """wr_gtsp_solve: every colony iterates until max_iterations (0: N^2) or more than N
        iterations without improvement.  Returns (iterations per colony, [B][cap] best L after each
        iteration (valid up to that colony's count), the colony with the lowest best L)."""
        cap = max_iterations if max_iterations > 0 else self.city_num * self.city_num
        ran = np.zeros(self._batch, np.int32)
        # np.empty: only the pages up to each colony's iteration count are ever touched
        hist = np.empty((self._batch, cap), np.float64)
        bc = C.c_int()
        check(lib().wr_gtsp_solve(self._g, max_iterations, ptr(ran), ptr(hist), C.byref(bc)))
        return ran, hist, bc.value

    def computeSolution(self, max_iterations=None):
        """ACS_GTSP.hpp:255-284: iterate until MAX_itera = N^2 or more than N iterations without
        improvement, on the device for every colony; report the best colony."""
        if not self.init_flag:
            return False
        max_it = self.city_num * self.city_num if max_iterations is None else max_iterations
        if max_it > 0:
            ran, hist, b = self.solve(max_it)
            for index_itera in range(ran[b]):
                print("iteration %d:Best so far = %.2f" % (index_itera, hist[b, index_itera]))
            self.best_path, self.best_L = self.best(b)
        print("Best in all = %.2f" % self.best_L)
        if len(self.best_path):
            print("->".join(str(r + 1) for r, _ in self.best_path) + "->%d" % (self.best_path[-1][1] + 1))
        return True

    def computeBatch(self, batch, iterations, colony_first=0):
        """B independent colonies (Philox streams colony_first .. colony_first+B-1), fixed iterations."""
        self._create(batch, colony_first)
        self.iterate(iterations)
        return [self.best(b) for b in range(batch)]

    def path_segment_nums(self):
        return len(self.best_path) - 1

    def read_segment(self, best_matrix, i):
        """ACS_GTSP.hpp:303-312 (i starts from 1)."""
        r, s = self.best_path[i - 1]
        for node in best_matrix[r][s].getPath():
            self.g_path_x.append(node.pt.x); self.g_path_y.append(node.pt.y); self.g_path_z.append(node.pt.z)

    def read_all_segments(self, best_matrix):
        """ACS_GTSP.hpp:286-298: the first N-1 edges of the best tour."""
        for i in range(1, len(self.best_path)):
            self.read_segment(best_matrix, i)

    def plot_route_path(self, figureNumber=1):
        pass

    def __del__(self):
        try:
            if self._g is not None:
                lib().wr_gtsp_destroy(self._g)
        except Exception:
            pass


class BS_Basic:
    """Mirror of BS_Basic<float, 3, DEGREE, CONST_LEVEL_INI, CONST_LEVEL_FIN> (core/BSplineBasic.h:33-120), the trajectory
    smoothing of main.cpp:287-352: SetParam on the host, curve points for a whole array of times in one kernel launch
    (wr_bspline_eval).  The demo samples at wall-clock times (main.cpp:309-320); here the caller names the times."""

    def __init__(self, num_middle, degree=0, const_level_ini=0, const_level_fin=0):
        self.NUM_MIDDLE = int(num_middle)
        self.DEGREE, self.CI, self.CF = int(degree), int(const_level_ini), int(const_level_fin)
        self.NumKnots_ = self.DEGREE + self.NUM_MIDDLE + 2 + self.CI + self.CF + 1       # :39-40
        self.NumCPs_ = self.NUM_MIDDLE + 2 + self.CI + self.CF                           # :41
        self._set = False

    def SetParam(self, init, fin, middle_pt, fin_time):
        """:70-76.  init / fin: 3 * (level + 1) floats; middle_pt: [NUM_MIDDLE][>= 3] (the first three columns are used)."""
        self._init = np.ascontiguousarray(init, dtype=np.float32).ravel()
        self._fin = np.ascontiguousarray(fin, dtype=np.float32).ravel()
        if self._init.size < 3 * (self.CI + 1) or self._fin.size < 3 * (self.CF + 1):
            raise ValueError("init / fin need 3 * (constraint level + 1) floats")
        self._mid = np.ascontiguousarray(middle_pt, dtype=np.float32).reshape(self.NUM_MIDDLE, -1) if self.NUM_MIDDLE else np.zeros((0, 3), np.float32)
        self._tf = float(fin_time)
        self.Knots_ = np.zeros(self.NumKnots_, np.float32)
        self.CPoints_ = np.zeros((self.NumCPs_, 3), np.float32)
        self._call(np.zeros(0, np.float32))
        self._set = True
        return True

    def _call(self, u, out=None):
        u = np.ascontiguousarray(u, dtype=np.float32).ravel()
        if out is None:
            out = np.zeros((u.size, 3), np.float32)
        ok = np.zeros(u.size, np.uint8)
        check(lib().wr_bspline_eval(self.DEGREE, self.CI, self.CF, ptr(self._init), ptr(self._fin), ptr(self._mid), self.NUM_MIDDLE,
                                    self._mid.shape[1] if self.NUM_MIDDLE else 3, self._tf, ptr(u), u.size, ptr(out), ptr(ok),
                                    ptr(self.Knots_), ptr(self.CPoints_)))
        return out, ok.astype(bool)

    def getCurvePoints(self, times, out=None):
        """getCurvePoint (:85-111) at every time of `times`: ([m][3] points, [m] success flags).  A failed sample keeps the row of
        `out` it was given (zeros without `out`), as the reference leaves `ret` untouched."""
        if not self._set:
            raise RuntimeError("SetParam first")
        return self._call(times, out)

    def getCurvePoint(self, u):
        pts, ok = self.getCurvePoints([u])
        return bool(ok[0]), pts[0]
