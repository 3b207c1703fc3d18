"""Ranking and rank-set build of the C2 search (bench.py's workload), iteration by iteration: the device time of the rank
phase (k_rank_small + k_best_copy) and of the deposit build (k_rankset_gen, or k_deposit_gen + record sort on record
iterations), each from the handle's per-phase events, next to the eligible ranks whose bits the group path set
(updateStats()["group_ranks"]: ants verified on the whole best path).

    python scripts/group_deposits.py [--iters 125] [--out profiles/r6_group_deposits.json]

A build without group deposits reports group_ranks as null."""
import argparse
import contextlib
import io
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=125)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import bench
    import welding_robot_b200 as wr
    import torch
    wl = bench.build_workload_gpu()
    acs = wr.ACS_Rank(seed=bench.SEED, fixed_colony=bench.ANTS_PER_GPU, step_cap=bench.STEP_CAP, update_mode=4)
    acs.creatFromOccupancy(wl["isfree"], wl["xs"], wl["ys"], wl["zs"], bench.PRECISION)
    with contextlib.redirect_stdout(io.StringIO()):
        acs.initFromGridMap()
    acs.setEndpoints(wl["start"], wl["goal"])
    acs.begin(bench.PREDICT)
    acs.setTiming(True)
    rows = []
    k0 = acs.kernelMs()
    for it in range(1, args.iters + 1):
        acs.iterate(1)
        acs.sync()
        k1 = acs.kernelMs()
        st = acs.updateStats()
        rows.append({"iteration": it, "rankset": st["rankset_last"], "group_ranks": st.get("group_ranks"),
                     "rank_ms": round(k1["rank"] - k0["rank"], 5), "deposit_build_ms": round(k1["deposit_build"] - k0["deposit_build"], 5),
                     "walk_ms": round(k1["walk"] - k0["walk"], 5), "update_ms": round(k1["update"] - k0["update"], 5)})
        print(json.dumps(rows[-1]), flush=True)
        k0 = k1
    conv = [r for r in rows if r["rankset"] and r["iteration"] > 36]
    summary = {k: round(sum(r[k] for r in conv) / max(1, len(conv)), 5) for k in ("rank_ms", "deposit_build_ms")}
    summary["iterations"] = len(conv)
    print("rank-set iterations after 36:", json.dumps(summary))
    gpu = torch.cuda.get_device_name(0)
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"workload": bench.LABEL, "ants": bench.ANTS_PER_GPU, "gpu": gpu, "rankset_after_36": summary, "iterations": rows}, f, indent=1)


if __name__ == "__main__":
    main()
