"""Line-of-sight shortcutting (wr_grid_shortcut_paths) on one GPU; prints one JSON line.

  C1   the 15 best paths of cubic.stl @ (0.005, wall 10), the six weld points, seed 0, 150 iterations, at r2 = 0 and r2 = 1
  C2   the 4096 ant trails of one early (wandering) and one late iteration of bench.py's 256^3 search (wr_acs_last_ant),
       max_span 0 and 256, r2 = 0
  C5   the best paths of bench.py's 1024 queries on the 512^3 obstacle grid (256 ants x 50 iterations each), r2 = 0

Time: host clock around the whole call (copies in, one launch, copies out, synchronise), median / min / max of --reps calls
after one untimed call.  At r2 > 0 the clearance field is built by the untimed call and cached in the grid, so the timed calls
do not include it; its build time (wr_grid_clearance_ms, device ms) is reported beside them.  The card's name and power limit
are read in the same run.

    python scripts/shortcut_bench.py [--reps 20] [--out FILE]
"""
import argparse
import contextlib
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

C1_POINTS = [(1.600931, y, z) for y in (-0.259319, -0.074319, 0.085681) for z in (1.224003, 1.399003)]


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return q


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def measure(g, rows, r2, max_span, reps):
    rows = [np.asarray(r, np.int64) for r in rows]
    off = np.zeros(len(rows) + 1, np.int64)
    off[1:] = np.cumsum([len(r) for r in rows])
    ids = np.ascontiguousarray(np.concatenate(rows))
    keep = np.zeros(len(ids), np.int32)
    nkeep = np.zeros(len(rows), np.int32); nb = np.zeros(len(rows), np.int32); L = np.zeros(len(rows))

    def call():
        check(lib().wr_grid_shortcut_paths(g._g, ptr(ids), ptr(off), len(rows), r2, max_span, ptr(keep), ptr(nkeep), ptr(nb), ptr(L)))

    t0 = time.perf_counter(); call(); first = time.perf_counter() - t0
    reps = reps if first < 2.0 else 3            # long workloads: fewer calls, reported in the record
    t = []
    for _ in range(reps):
        t0 = time.perf_counter(); call(); t.append(time.perf_counter() - t0)
    t = np.array(t)
    med = float(np.median(t))
    xs, ys, zs = g.coords()
    rx, ry = g.rangeX, g.rangeY
    z, r = np.divmod(ids, rx * ry); y, x = np.divmod(r, rx)
    P = np.stack([xs[x], ys[y], zs[z]], 1).astype(np.float64)
    seg = np.sqrt((np.diff(P, axis=0) ** 2).sum(1))
    inner = np.ones(len(seg), bool); inner[off[1:-1] - 1] = False          # no segment across two rows
    Lin = float(seg[inner].sum())
    ms = np.zeros(1, np.float32)
    check(lib().wr_grid_clearance_ms(g._g, ptr(ms)))
    return {"rows": len(rows), "input_nodes": int(len(ids)), "r2": r2, "max_span": max_span, "reps": reps,
            "s_median": med, "s_min": float(t.min()), "s_max": float(t.max()),
            "rows_per_s": len(rows) / med, "input_nodes_per_s": len(ids) / med,
            "waypoints": int(nkeep.sum()), "waypoint_ratio": float(nkeep.sum()) / len(ids), "blocked": int(nb.sum()),
            "length_in": Lin, "length_out": float(L.sum()), "length_reduction": 1.0 - float(L.sum()) / Lin if Lin else 0.0,
            "field_build_ms": float(ms[0]) if r2 else None,
            "field_build_in_timed_calls": False}


def c1(reps):
    tris = np.load(os.path.join(ROOT, "tests", "golden", "meshes.npz"))["cubic"]
    g = wr.ACS_Rank(seed=0)
    quiet(g.creatGridMap, tris, 0.005, 10)
    node = g.snapPoints(C1_POINTS)
    pairs = [(i, j) for i in range(6) for j in range(i + 1, 6)]
    res = quiet(g.searchBatch, [int(node[i]) for i, _ in pairs], [int(node[j]) for _, j in pairs], 0.5, iterations=150)
    rows = [ids for ids, _, _ in res]
    return {"C1_r2_0": measure(g, rows, 0, 0, reps), "C1_r2_1": measure(g, rows, 1, 0, reps)}


def c2(reps):
    wl = bench.build_workload_gpu()
    g = wr.ACS_Rank(seed=bench.SEED, fixed_colony=bench.ANTS_PER_GPU, step_cap=bench.STEP_CAP)
    g.creatFromOccupancy(wl["isfree"], wl["xs"], wl["ys"], wl["zs"], bench.PRECISION)
    g.setEndpoints(wl["start"], wl["goal"])
    g.begin(bench.PREDICT)
    out = {}
    done = 0
    for name, it in (("early", 5), ("late", 120)):
        g.iterate(it - done); done = it
        rows = [t for t in (g.lastAnt(k)[0] for k in range(bench.ANTS_PER_GPU)) if len(t)]
        for span in (0, 256):
            out["C2_%s_iter%d_span%d" % (name, it, span)] = measure(g, rows, 0, span, reps)
    return out


def c5(reps):
    n = 512
    free = bench.synthetic_boxes(n, 4096, 4)
    axis = np.arange(n, dtype=np.float32)
    starts, goals = bench.c5_queries(free, n, 1024)
    g = wr.ACS_Rank(seed=5, fixed_colony=256, step_cap=4096)
    g.creatFromOccupancy(free, axis, axis, axis, 1.0)
    quiet(g.initFromGridMap)
    g.searchBatch(starts[:8], goals[:8], 300.0, 3, with_paths=False)
    g.setNextSearch(0)
    g.sync()
    t0 = time.perf_counter()
    res = g.searchBatch(starts, goals, 300.0, 50, with_paths=True)
    search_s = time.perf_counter() - t0
    rows = [ids for ids, _, _ in res if len(ids)]
    rec = measure(g, rows, 0, 0, reps)
    rec["search_s"] = search_s
    rec["shortcut_over_search"] = rec["s_median"] / search_s
    return {"C5": rec}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    rec = {"gpu_name_power_limit": gpu_info(), "reps": args.reps,
           "timed": "host clock around wr_grid_shortcut_paths (copies in and out, one launch, synchronise); median of reps"}
    for fn in (c1, c2, c5):
        rec.update(fn(args.reps))
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
