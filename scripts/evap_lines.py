"""Evaporation pass of the C2 search (bench.py's workload), iteration by iteration: the device time of the kernel that
streams the pheromone field (k_update_fused on record iterations, k_evaporate_lines on rank-set iterations, timed by its
own event pair), the dirty 16 KB tiles and 128-byte lines it had to move, and the rate that gives.

    python scripts/evap_lines.py [--iters 125] [--out profiles/r5_evap_lines.json]

bytes = dirty lines before the iteration x 256 B (each line read once and written once).  On record iterations
k_update_fused also streams the deposit tiles whole, so there the figure is a lower bound.  A build without line flags
(wr_acs_field_lines) reports lines as null and bytes from its 16 KB tiles."""
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
    has_lines = hasattr(acs, "fieldLines")

    def lines():
        return acs.fieldLines()[0] if has_lines else None

    acs.setTiming(True)
    rows = []
    sk0, _ = acs.streamKernelMs()
    tiles0, lines0 = acs.fieldStats()[0], lines()
    for it in range(1, args.iters + 1):
        acs.iterate(1)
        acs.sync()
        sk1, _ = acs.streamKernelMs()
        ms = sk1 - sk0
        nbytes = lines0 * 256 if has_lines else tiles0 * 4096 * 8
        rows.append({"iteration": it, "rankset": acs.updateStats()["rankset_last"], "stream_kernel_ms": round(ms, 5),
                     "dirty_tiles": tiles0, "dirty_lines": lines0, "bytes": nbytes, "GBps": round(nbytes / (ms * 1e-3) / 1e9, 1) if ms > 0 else None})
        print(json.dumps(rows[-1]), flush=True)
        sk0 = sk1
        tiles0, lines0 = acs.fieldStats()[0], lines()
    gpu = torch.cuda.get_device_name(0)
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"workload": bench.LABEL, "ants": bench.ANTS_PER_GPU, "gpu": gpu, "line_flags": has_lines, "iterations": rows}, f, indent=1)


if __name__ == "__main__":
    main()
