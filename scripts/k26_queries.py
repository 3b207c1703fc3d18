"""Concurrent (wr_acs_search_batch) against one-after-the-other (wr_acs_search_pairs) searches with the K = 26 neighbourhood,
on one GPU; prints one JSON line.

  C5-K26  1024 queries on bench.py's synthetic 512^3 obstacle grid (bench.synthetic_boxes(512, 4096, 4), bench.c5_queries),
          256 ants x 50 iterations, step cap 4096: all of them through the batch, a sample of 16 through the sequential loop
          (checked bit-equal to the batch's answers for the same queries)
  C1-K26  cubic.stl @ (0.005, wall 10), the 15 pairs of the six weld points, 150 iterations, adaptive colony: both ways

Wall clock with a device synchronise before every host-clock reading; warm-up calls first.  The card's name and power limit
are read in the same run.

    python scripts/k26_queries.py [--queries N] [--sample K] [--profile DIR]

--profile DIR: instead of the timings, one torch.profiler capture of a 256-query C5-K26 batch and of 4 sequential queries
(CUDA activity only), its per-kernel table written to DIR/k26_kernels.txt and summarised on the JSON line.
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
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import welding_robot_b200 as wr  # noqa: E402

C1_POINTS = [(1.600931, y, z) for y in (-0.259319, -0.074319, 0.085681) for z in (1.224003, 1.399003)]


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return {"gpu": name, "power_limit_and_max_sm_clock": q}


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return r, time.perf_counter() - t0


def equal(a, b):
    return len(a) == len(b) and all(np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1]) and
                                    ((np.isinf(x[2]) and np.isinf(y[2])) or np.float32(x[2]) == np.float32(y[2])) for x, y in zip(a, b))


def c5_handle():
    n = 512
    free = bench.synthetic_boxes(n, 4096, 4)
    axis = np.arange(n, dtype=np.float32)
    g = wr.ACS_Rank(seed=5, fixed_colony=256, step_cap=4096, K=26)
    g.creatFromOccupancy(free, axis, axis, axis, 1.0)
    with contextlib.redirect_stdout(io.StringIO()):
        g.initFromGridMap()
    return g, free, n


def c5(nq, sample, iters=50):
    g, free, n = c5_handle()
    s, e = bench.c5_queries(free, n, nq)
    g.searchBatch(s[:8], e[:8], 300.0, 3)              # warm-up: buffers, kernels
    g.searchPairs(s[:1], e[:1], 300.0, 3)
    g.setNextSearch(0)
    bat, dt = timed(lambda: g.searchBatch(s, e, 300.0, iters))
    st = g.batchStats()
    g.setNextSearch(0)
    seq, dt_seq = timed(lambda: g.searchPairs(s[:sample], e[:sample], 300.0, iters))
    del g
    seq_ms = 1e3 * dt_seq / sample
    return {"workload": "C5-K26: %d queries on bench.synthetic_boxes(512, 4096, 4), 256 ants x %d iterations, step cap 4096, K = 26" % (nq, iters),
            "batch_seconds": dt, "batch_queries_per_s": nq / dt, "batch_ms_per_query": 1e3 * dt / nq,
            "sequential_sample": sample, "sequential_ms_per_query": seq_ms, "sequential_queries_per_s": 1e3 / seq_ms,
            "speedup_batch_over_sequential": seq_ms / (1e3 * dt / nq),
            "found": int(sum(np.isfinite(r[2]) for r in bat)), "batch": st, "sample_bit_equal": equal(seq, bat[:sample])}


def c1_handle():
    tris = np.load(os.path.join(ROOT, "tests", "golden", "meshes.npz"))["cubic"]
    g = wr.ACS_Rank(seed=0x5EED, K=26)
    with contextlib.redirect_stdout(io.StringIO()):
        g.creatGridMap(tris, 0.005, 10)
        g.initFromGridMap()
    node = g.snapPoints(C1_POINTS)
    pairs = [(i, j) for i in range(6) for j in range(i + 1, 6)]
    return g, [int(node[i]) for i, _ in pairs], [int(node[j]) for _, j in pairs]


def c1(iters=150):
    g, s, e = c1_handle()
    g.searchBatch(s, e, 0.5, 5)                        # warm-up
    g.searchPairs(s, e, 0.5, 5)
    out = {"workload": "C1-K26: cubic.stl @ (0.005, wall 10), 15 pairs x %d iterations, adaptive colony, K = 26" % iters}
    runs = {}
    for rep in range(2):                               # alternated, twice: the spread is part of the figure
        for mode in ("batch", "sequential"):
            g.setNextSearch(0)
            fn = (lambda: g.searchBatch(s, e, 0.5, iters)) if mode == "batch" else (lambda: g.searchPairs(s, e, 0.5, iters))
            res, dt = timed(fn)
            runs.setdefault(mode, []).append(dt)
            runs[mode + "_res"] = res
    out.update({"batch_seconds": runs["batch"], "sequential_seconds": runs["sequential"],
                "speedup_batch_over_sequential": min(runs["sequential"]) / min(runs["batch"]),
                "bit_equal": equal(runs["batch_res"], runs["sequential_res"]), "batch": g.batchStats()})
    del g
    return out


def profile(outdir, nq=256, iters=50):
    from torch.profiler import ProfilerActivity, profile as tprof
    g, free, n = c5_handle()
    s, e = bench.c5_queries(free, n, nq)
    g.searchBatch(s[:8], e[:8], 300.0, 3)
    g.searchPairs(s[:1], e[:1], 300.0, 3)
    torch.cuda.synchronize()
    tables = {}
    for mode in ("batch", "sequential"):
        g.setNextSearch(0)
        with tprof(activities=[ProfilerActivity.CUDA]) as p:
            if mode == "batch":
                g.searchBatch(s, e, 300.0, iters)
            else:
                g.searchPairs(s[:4], e[:4], 300.0, iters)
            torch.cuda.synchronize()
        ka = p.key_averages()
        tables[mode] = ka.table(sort_by="device_time_total", row_limit=25)
        tables[mode + "_top"] = [{"kernel": k.key[:80], "calls": k.count, "total_ms": k.device_time_total / 1e3}
                                 for k in sorted(ka, key=lambda k: -k.device_time_total)[:8]]
    os.makedirs(outdir, exist_ok=True)
    with open(os.path.join(outdir, "k26_kernels.txt"), "w") as f:
        f.write("C5-K26 batch, %d queries x 256 ants x %d iterations\n%s\n\nC5-K26 sequential, 4 queries\n%s\n" % (nq, iters, tables["batch"], tables["sequential"]))
    return {"workload": "torch.profiler, C5-K26: %d queries through the batch, 4 through the sequential loop, %d iterations" % (nq, iters),
            "batch_top_kernels": tables["batch_top"], "sequential_top_kernels": tables["sequential_top"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--queries", type=int, default=1024)
    ap.add_argument("--sample", type=int, default=16)
    ap.add_argument("--profile", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("k26_queries.py: no CUDA device")
    torch.cuda.set_device(0)
    out = gpu_info()
    if args.profile:
        out["profile"] = profile(args.profile)
    else:
        out["c5_k26"] = c5(args.queries, args.sample)
        out["c1_k26"] = c1()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
