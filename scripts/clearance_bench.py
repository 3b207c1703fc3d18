"""Clearance field (wr_grid_clearance), point queries (wr_grid_clearance_at) and inflation (wr_grid_inflate) on one GPU; prints
one JSON line.

  C1  cubic.stl @ (0.005, wall 10): 57 x 91 x 57 (for scale)
  C2  bench.py's 256^3 cube (bench.build_workload_gpu), field 67 MB: fits the 126 MB L2
  C5  bench.py's 512^3 obstacle grid (bench.synthetic_boxes(512, 4096, 4)), field 537 MB: does not

Field build: device ms of the three passes (CUDA events inside the library, wr_grid_clearance_ms) on fresh handles, one untimed
build first, then --builds builds.  A fresh handle is wr_grid_inflate(g, 0): same occupancy, no field yet.  Bytes are what the
passes move at the least: the occupancy bits once, 4 B written per node by pass 1, 4 B read + 4 B written per node by each of
passes 2 and 3 (the re-reads of envelope apexes are L2 hits and not counted), against the data sheet's 7.7 TB/s.
Queries: host clock around wr_grid_clearance_at for --points points uniform in the grid's box (one launch; the call copies the
points in and the results out, and synchronises).  Inflation: host clock around wr_grid_inflate (r2 = 1) on a grid whose field
exists (allocation, one launch, the occupied count read back).  The card's name and power limit are read in the same run.

    python scripts/clearance_bench.py [--builds 20] [--points 1000000] [--out FILE]
"""
import argparse
import contextlib
import ctypes as C
import io
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import welding_robot_b200 as wr  # noqa: E402
from welding_robot_b200._lib import check, lib, ptr  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return q


def grids():
    tris = np.load(os.path.join(ROOT, "tests", "golden", "meshes.npz"))["cubic"]
    with contextlib.redirect_stdout(io.StringIO()):
        c1 = wr.GridMap().creatGridMap(tris, 0.005, 10)
    yield "C1", c1
    wl = bench.build_workload_gpu()
    yield "C2", wr.GridMap().creatFromOccupancy(wl["isfree"], wl["xs"], wl["ys"], wl["zs"], bench.PRECISION)
    axis = np.arange(512, dtype=np.float32)
    yield "C5", wr.GridMap().creatFromOccupancy(bench.synthetic_boxes(512, 4096, 4), axis, axis, axis, 1.0)


def fresh(g):
    h = C.c_void_p()
    check(lib().wr_grid_inflate(g._g, 0, C.byref(h)))
    return h


def build_ms(g, builds):
    one = np.zeros(3, np.float32)
    out = []
    for k in range(builds + 1):
        h = fresh(g)
        check(lib().wr_grid_clearance_at(h, ptr(one), 1, None, None))
        ms = C.c_float()
        check(lib().wr_grid_clearance_ms(h, C.byref(ms)))
        check(lib().wr_grid_destroy(h))
        if k:
            out.append(ms.value)
    return np.array(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--builds", type=int, default=20)
    ap.add_argument("--points", type=int, default=1000000)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    rec = {"gpu_name_power_limit": gpu_info(), "builds": args.builds, "points": args.points, "grids": {}}
    rng = np.random.default_rng(0)
    for name, g in grids():
        n = g.size_of_map()
        g.clearanceAt(np.zeros((1, 3), np.float32))                       # the source's own field (fresh() thresholds it)
        ms = build_ms(g, args.builds)
        nbytes = n * (4 + 8 + 8) + (n + 7) // 8
        med = float(np.median(ms))
        xs, ys, zs = g.coords()
        lo = np.array([xs.min(), ys.min(), zs.min()]); hi = np.array([xs.max(), ys.max(), zs.max()])
        pts = rng.uniform(lo, hi, (args.points, 3)).astype(np.float32)
        g.clearanceAt(pts[:1000])
        q = []
        for _ in range(5):
            t0 = time.perf_counter(); g.clearanceAt(pts); q.append(time.perf_counter() - t0)
        inf = []
        for _ in range(10):
            h = C.c_void_p()
            t0 = time.perf_counter()
            check(lib().wr_grid_inflate(g._g, 1, C.byref(h)))
            inf.append(time.perf_counter() - t0)
            check(lib().wr_grid_destroy(h))
        rec["grids"][name] = {
            "dims": [g.rangeX, g.rangeY, g.rangeZ], "nodes": n, "field_MB": 4 * n / 1e6, "field_fits_126MB_L2": 4 * n < 126e6,
            "build_ms_median": med, "build_ms_min": float(ms.min()), "build_ms_max": float(ms.max()),
            "bytes_moved": nbytes, "bytes_formula": "N*(4 + 8 + 8) + N/8 (pass 1 write, passes 2-3 read+write, occupancy bits)",
            "GB_per_s": nbytes / med / 1e6, "fraction_of_7.7TB_per_s": nbytes / (med * 1e-3) / HBM_BYTES_PER_S,
            "bound": "memory (the passes do a few integer operations per byte)",
            "query_s_median": float(np.median(q)), "query_points_per_s": args.points / float(np.median(q)),
            "inflate_ms_median": 1e3 * float(np.median(inf)), "inflate_ms_min": 1e3 * float(min(inf)),
        }
        del g
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
