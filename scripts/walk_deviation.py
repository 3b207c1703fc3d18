"""Deviation profile of the C2 search (bench.py's workload): for every iteration, how many ants leave the best path they
start the iteration with, where the earliest one leaves, and how many steps a walk that resumes each warp at the lowest
floor8(first deviating step) of its four ants (path_verify.cuh) still runs step by step.

    python scripts/walk_deviation.py [--iters 150] [--out profiles/r3_walk_deviation.json]

Ants are grouped as k_walk3 takes them off its queue: four consecutive ants per warp."""
import argparse
import contextlib
import io
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=150)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import bench
    import welding_robot_b200 as wr
    wl = bench.build_workload_gpu()
    acs = wr.ACS_Rank(seed=bench.SEED, fixed_colony=bench.ANTS_PER_GPU, step_cap=bench.STEP_CAP, update_mode=4)
    acs.creatFromOccupancy(wl["isfree"], wl["xs"], wl["ys"], wl["zs"], bench.PRECISION)
    with contextlib.redirect_stdout(io.StringIO()):
        acs.initFromGridMap()
    acs.setEndpoints(wl["start"], wl["goal"])
    acs.begin(bench.PREDICT)
    rows = []
    for it in range(1, args.iters + 1):
        bids, _, bL = acs.bestPath()
        n = 0 if np.isinf(bL) else len(bids)
        acs.iterate(1)
        rs = acs.updateStats()["rankset_last"]
        colony = acs.lastColony()[0]
        devs, steps = np.zeros(colony, np.int64), np.zeros(colony, np.int64)
        complete = np.zeros(colony, bool)
        dead = 0
        for k in range(colony):
            ids, _, L, _ = acs.lastAnt(k)
            if np.isinf(L):        # a dead ant's trail is not kept: counted as leaving at step 0
                dead += 1
                continue
            steps[k] = len(ids) - 1
            if n == 0:
                continue
            m = min(len(ids), n)
            diff = np.flatnonzero(ids[:m] != bids[:m])
            if len(diff) == 0 and len(ids) == n:
                complete[k] = True
                devs[k] = n - 1
            else:
                devs[k] = (diff[0] if len(diff) else m) - 1
        left = int((~complete).sum())
        t0 = np.where(complete, (max(n - 1, 0) // 8) * 8, (np.maximum(devs, 0) // 8) * 8)
        rest = 0
        for w in range(0, colony, 4):
            if complete[w:w + 4].all():
                continue
            rest = max(rest, int(steps[w:w + 4].max() - t0[w:w + 4].min()))
        rows.append({"iteration": it, "best_n": n, "rankset": rs, "ants": colony, "left_path": left, "dead": dead,
                     "earliest_leave": int(devs[~complete].min()) if left else None,
                     "warps_all_complete": int(sum(complete[w:w + 4].all() for w in range(0, colony, 4))),
                     "steps_still_walked": rest, "max_steps": int(steps.max()) if colony else 0})
        print(json.dumps(rows[-1]), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"workload": bench.LABEL, "ants": bench.ANTS_PER_GPU, "iterations": rows}, f, indent=1)


if __name__ == "__main__":
    main()
