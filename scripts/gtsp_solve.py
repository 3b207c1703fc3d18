"""Seam ordering run to convergence on the device (wr_gtsp_solve) on one GPU; prints one JSON line.

  (a) N = 256, one colony: computeSolution's former host loop (one wr_gtsp_iterate launch, a synchronise and a best-tour
      read-back per iteration, the stopping rule on the host; written out below) against one wr_gtsp_solve call.  Wall time of
      each; the tours, lengths, iteration counts and per-iteration best lengths must be bit-equal.
  (b) N = 256, B colonies (default 1, 148, 296), each to its own stopping rule: wall time of the solve, iterations per colony
      (min / median / max), the best colony's L against colony 0's.
  (c) --c4-against DIR: bench.py's C4 sub-record (1024 colonies x 64 fixed iterations, bench.sub_c4) from this tree and from
      the tree DIR (built), alternated --rounds times, each in its own process.

Wall clock around work that ends in a device synchronise; a warm-up solve on a separate handle first.  The distance matrix is
C4's (bench.sub_c4: 256 random points, seed 3, rounded to 6 decimals).  The card's name and power limit are read in the same run.

    python scripts/gtsp_solve.py [--colonies 1,148,296] [--c4-against DIR] [--rounds 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import welding_robot_b200 as wr  # noqa: E402

N, SEED = 256, 3


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return {"gpu": name, "power_limit_and_max_sm_clock": q}


def c4_matrix(n=N):
    P = np.random.default_rng(3).random((n, 3))
    return np.round(np.sqrt(((P[:, None] - P[None]) ** 2).sum(-1)), 6)


def handle(D, batch):
    n = D.shape[0]
    g = wr.ACS_GTSP(seed=SEED)
    g.dis, g.city_num, g.cnt = D, n, n * (n - 1) // 2
    g._create(batch, 0)
    return g


def host_loop(g):
    """computeSolution as the facades ran it before wr_gtsp_solve: colony 0, one iteration per launch."""
    n = g.city_num
    last, bad_times, hist = float(0x3f3f3f3f), 0, []
    for _ in range(n * n):
        if bad_times > n:
            break
        g.iterate(1)
        _, L = g.best(0)           # wr_gtsp_best synchronises
        hist.append(L)
        if last > L:
            last, bad_times = L, 0
        else:
            bad_times += 1
    return np.array(hist)


def part_a(D):
    g = handle(D, 1)
    t0 = time.perf_counter()
    hist = host_loop(g)
    t_loop = time.perf_counter() - t0
    tour_loop, L_loop = g.best(0)
    g = handle(D, 1)
    t0 = time.perf_counter()
    ran, h, _ = g.solve()          # returns after its last launch has finished
    t_solve = time.perf_counter() - t0
    tour, L = g.best(0)
    same = bool(ran[0] == len(hist) and np.array_equal(h[0, :ran[0]].view(np.uint64), hist.view(np.uint64)) and
                np.array_equal(tour, tour_loop) and L == L_loop)
    return {"n": N, "iterations": int(ran[0]), "host_loop_s": t_loop, "solve_s": t_solve, "speedup": t_loop / t_solve,
            "host_loop_ms_per_iteration": 1e3 * t_loop / len(hist), "solve_ms_per_iteration": 1e3 * t_solve / ran[0],
            "best_L": L, "bit_equal": same}


def part_b(D, batch):
    g = handle(D, batch)
    t0 = time.perf_counter()
    ran, _, bc = g.solve()
    dt = time.perf_counter() - t0
    L0, Lb = g.best(0)[1], g.best(bc)[1]
    return {"n": N, "colonies": batch, "solve_s": dt, "iterations_min": int(ran.min()), "iterations_median": float(np.median(ran)),
            "iterations_max": int(ran.max()), "colony_iterations": int(ran.sum()), "colony_iterations_per_s": float(ran.sum()) / dt,
            "kernel_ms": g.kernelMs(), "best_colony": bc, "best_L": Lb, "colony0_L": L0}


def c4_once(tree):
    code = "import json, sys; sys.path.insert(0, %r); import bench; print(json.dumps(bench.sub_c4(0, 1, None)))" % tree
    r = subprocess.run([sys.executable, "-c", code], cwd=tree, capture_output=True, text=True, timeout=900)
    if r.returncode != 0:
        raise RuntimeError("C4 in %s failed:\n%s" % (tree, r.stderr[-3000:]))
    return json.loads(r.stdout.strip().splitlines()[-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--colonies", default="1,148,296")
    ap.add_argument("--c4-against", metavar="DIR", help="a built tree to alternate bench.py's C4 with")
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    out = gpu_info()
    D = c4_matrix()
    handle(D, 1).solve(1)          # warm-up: module load, first launch
    out["a_host_loop_vs_solve"] = part_a(D)
    out["b_colonies"] = [part_b(D, int(b)) for b in args.colonies.split(",")]
    if args.c4_against:
        rows = []
        for _ in range(args.rounds):
            for name, tree in (("this", ROOT), ("other", os.path.abspath(args.c4_against))):
                r = c4_once(tree)
                rows.append({"tree": name, "colony_iterations_per_s": r["colony_iterations_per_s"], "seconds": r["seconds"],
                             "sample_best_L": r["sample_best_L"]})
        out["c4_alternated"] = rows
        for name in ("this", "other"):
            v = [r["colony_iterations_per_s"] for r in rows if r["tree"] == name]
            out["c4_%s_colony_iterations_per_s" % name] = {"min": min(v), "median": float(np.median(v)), "max": max(v)}
        out["c4_same_sample_best_L"] = len({json.dumps(r["sample_best_L"]) for r in rows}) == 1
    print(json.dumps(out))


if __name__ == "__main__":
    main()
