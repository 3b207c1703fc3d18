#!/usr/bin/env python
"""bench.py — ant-steps/s of the rank-based 3-D ACS search on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU code (oracle/_ref)
    python bench.py ... --dump-outputs DIR                   # + what the timed search computed, as DIR/<name>.npy

Workload "C2" (BASELINE.json configs[1], SURVEY.md §8d): the simplified_piece mesh voxelised at a
256-long grid (precision 0.823812/235.5, wall 10) and embedded in a 256^3 lattice whose node
coordinates follow the reference's formula (model_grid_map.hpp:204-211) for a cubic bounding box;
4096 ants per GPU, K = 6, Philox seed 1, start/goal at opposite corners inset by 5 cells, step cap
8192.  One "step" = `--iters` ACS iterations (ant construction + ranking + pheromone update) of one
search.  With N GPUs the colony is 4096*N ants sharded by ant index (weak scaling) with one exchange
per iteration.  The pheromone field (403 MB) is larger than L2 (126 MB): every iteration streams it
from HBM, so no L2 flush is needed between timed iterations.

Prints ONE JSON line.  `value` = whole-job ant-steps/s with the grid already in HBM (CUDA events on
the launching stream, max over ranks); `e2e` = the same metric through the public API from HOST
buffers, every step: occupancy upload, handle creation, search, best-path download.
"""
import argparse
import contextlib
import io
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # no .pyc files in the tree the benchmark runs from (which may be read-only)

ANTS_PER_GPU = 4096
STEP_CAP = 8192
SEED = 1
PRECISION = 0.823812 / 235.5
WALL = 10
CUBE = 256
MESH = "simplified_piece"
LABEL = "C2: ACSRank_3D, simplified_piece @256-long grid in 256^3"


def select_workload(name):
    """C2 (BASELINE.json configs[1]) is the bench workload; C3 (configs[2]: origin_piece at a 512-long grid in 512^3, 8192 ants per
    GPU, the pheromone field 3.2 GB per GPU) is the multi-GPU scaling case north_star names — an exploration run, never the default."""
    global CUBE, PRECISION, MESH, LABEL, ANTS_PER_GPU, STEP_CAP
    if name == "C3":
        CUBE, PRECISION, MESH = 512, 0.823812 / 491.5, "origin_piece"
        ANTS_PER_GPU, STEP_CAP = 8192, 16384
        LABEL = "C3: ACSRank_3D, origin_piece @512-long grid in 512^3"
PREDICT = 1.0                # with a fixed colony only Q of the pre-arrival iterations depends on it (ACSRank_3D.hpp:249)
WALK_BYTES_PER_STEP = 30     # SURVEY.md §8d: 4*K tau + K/8 occupancy + 4 id + 1 dir, K = 6
UPDATE_BYTES_PER_SLOT = 8    # 4 read + 4 write per directed slot per iteration


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """SM clock and clock-event reasons sampled DURING the timed region (B200_PROFILING.md recipe).  NVML is polled in
    process every few ms (a 4 ms step leaves no room for `nvidia-smi -lms`' start-up); where pynvml cannot initialise the
    recipe's `nvidia-smi --query-gpu` loop is the fallback.  Only samples taken between mark_begin() and mark_end() count."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self.proc = index, [], None     # rows: (t, sm_mhz, sm_max_mhz, [reasons])
        self.t0 = self.t1 = None
        self.quit = threading.Event()
        self.ready = threading.Event()
        self.source = None

    def _nvml(self):
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        names = (("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap),
                 ("hw_power_brake_slowdown", nv.nvmlClocksEventReasonHwPowerBrakeSlowdown))
        self.source = "nvml"
        while not self.quit.is_set():
            sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
            bits = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
            self.rows.append((time.perf_counter(), sm, mx, [n for n, b in names if bits & b]))
            self.ready.set()
            time.sleep(0.003)

    def _smi(self):
        self.source = "nvidia-smi"
        self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                                     stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        for line in self.proc.stdout:
            c = [v.strip() for v in line.split(",")]
            try:
                sm, mx = float(c[0]), float(c[1])
            except (ValueError, IndexError):
                continue
            rs = [n for n, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[3:7]) if v.lower().startswith("active")]
            self.rows.append((time.perf_counter(), sm, mx, rs))
            self.ready.set()
            if self.quit.is_set():
                break

    def run(self):
        try:
            self._nvml()
        except Exception:
            try:
                self._smi()
            except OSError:
                pass
        self.ready.set()

    def mark_begin(self):
        self.ready.wait(10.0)       # first sample is in before the timed region starts
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        self.quit.set()
        if self.proc is not None:
            self.proc.terminate()

    def summary(self):
        rows = [r for r in self.rows if self.t0 is not None and self.t0 <= r[0] <= (self.t1 or float("inf"))]
        window = "timed region"
        if not rows:                # never silently empty: say that the window is wider
            rows, window = list(self.rows), "whole run (no sample fell inside the timed region)"
        sm = [r[1] for r in rows]
        mx = [r[2] for r in rows]
        reasons = sorted({n for r in rows for n in r[3]})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "source": self.source, "window": window}


# ---------------------------------------------------------------------------------------------------
# workload
# ---------------------------------------------------------------------------------------------------
def axis_coords(rng, wall, mn, mx, precision):
    """model_grid_map.hpp:204-205 in float32 (bit-identical to the C expression, see tests)."""
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


def embed(free_zyx, gmin, gmax):
    """Natural voxelisation -> CUBE^3 workload: cubic bounding box (the long axis' extent on all axes),
    the reference's coordinate formula, the piece's occupancy centred, everything else free."""
    rz, ry, rx = free_zyx.shape
    assert max(rx, ry, rz) == CUBE, (rx, ry, rz)
    f = np.float32
    ext = max(f(gmax[k]) - f(gmin[k]) for k in range(3))
    cmin = [f(gmin[k]) for k in range(3)]
    cmax = [f(f(gmin[k]) + f(ext)) for k in range(3)]
    axes = [axis_coords(CUBE, WALL, cmin[k], cmax[k], f(PRECISION)) for k in range(3)]
    cube = np.ones((CUBE, CUBE, CUBE), np.uint8)
    oz, oy, ox = (CUBE - rz) // 2, (CUBE - ry) // 2, (CUBE - rx) // 2
    cube[oz:oz + rz, oy:oy + ry, ox:ox + rx] = free_zyx
    nid = lambda x, y, z: (z * CUBE + y) * CUBE + x  # noqa: E731
    start, goal = nid(5, 5, 5), nid(CUBE - 6, CUBE - 6, CUBE - 6)
    flat = np.ascontiguousarray(cube.ravel())
    assert flat[start] and flat[goal]
    return dict(isfree=flat, xs=axes[0], ys=axes[1], zs=axes[2], start=start, goal=goal, natural=(rx, ry, rz),
                cmin=[float(v) for v in cmin], cmax=[float(v) for v in cmax])


def build_workload_gpu():
    """Natural grid from the product's GPU voxeliser (K1)."""
    import welding_robot_b200 as wr
    tris = np.load(os.path.join(ROOT, "tests", "golden", "meshes.npz"))[MESH]
    g = wr.GridMap()
    with contextlib.redirect_stdout(io.StringIO()):
        g.creatGridMap(tris, PRECISION, WALL)
    free = g.isfree().reshape(g.rangeZ, g.rangeY, g.rangeX)
    mn, mx = g.bbox()
    wl = embed(free, mn, mx)
    wl["vox"] = g.stats(); wl["ntri"] = len(tris)
    return wl


def build_workload_cpu():
    """The same workload built on the CPU (reference arm): the oracle's box-restricted voxeliser gives
    the natural grid (the reference's own O(T*N) loop would need ~140 s for it)."""
    from oracle import oracle as O
    tris = np.load(os.path.join(ROOT, "tests", "golden", "meshes.npz"))[MESH]
    G = O.Grid.from_triangles(tris, PRECISION, WALL, O.VOX_AABB)
    rx, ry, rz = G.dims
    v = tris[:, 3:].reshape(-1, 3)
    wl = embed(G.isfree().reshape(rz, ry, rx), v.min(0), v.max(0))
    wl["ntri"] = len(tris)
    return wl


# ---------------------------------------------------------------------------------------------------
# the other BASELINE.json configurations, as sub-records of the same line (short, bounded runs)
# ---------------------------------------------------------------------------------------------------
def synthetic_boxes(n, nboxes, seed):
    """C5 grid (SURVEY.md 8d): union of axis-aligned boxes (edges 4-48 cells), 10-cell free wall, coordinates = indices."""
    rng = np.random.default_rng(seed)
    occ = np.zeros((n, n, n), bool)
    for _ in range(nboxes):
        e = rng.integers(4, 49, 3)
        c = [int(rng.integers(10, n - 10 - int(e[k]))) for k in range(3)]
        occ[c[2]:c[2] + e[2], c[1]:c[1] + e[1], c[0]:c[0] + e[0]] = True
    return (~occ).astype(np.uint8).ravel()


def c5_queries(free, n, nq, seed=5):
    ids = np.flatnonzero(free)
    rng = np.random.default_rng(seed)
    starts, goals = [], []
    while len(starts) < nq:
        s = int(ids[rng.integers(0, len(ids))])
        sz, sy, sx = s // (n * n), (s // n) % n, s % n
        d = int(rng.integers(64, 257))
        for _ in range(64):      # a free cell at Manhattan distance d: random split of d over the axes
            a = rng.multinomial(d, [1 / 3] * 3) * rng.choice([-1, 1], 3)
            gz, gy, gx = sz + a[0], sy + a[1], sx + a[2]
            if 0 <= gz < n and 0 <= gy < n and 0 <= gx < n and free[(gz * n + gy) * n + gx]:
                starts.append(s); goals.append(int((gz * n + gy) * n + gx))
                break
    return starts, goals


def sub_c5(rank, world, dist, nq=1024, iters=50, ants=256):
    """BASELINE configs[4]: independent queries on a synthetic 512^3 obstacle grid, query q -> rank q mod world, no communication;
    every rank advances its queries concurrently (wr_acs_search_batch)."""
    import torch
    import welding_robot_b200 as wr
    from welding_robot_b200.dist import shard_queries
    n = 512
    free = synthetic_boxes(n, 4096, 4)
    axis = np.arange(n, dtype=np.float32)
    starts, goals = c5_queries(free, n, nq)
    mine = shard_queries(nq, rank, world)
    g = wr.ACS_Rank(seed=5, fixed_colony=ants, step_cap=4096)
    g.creatFromOccupancy(free, axis, axis, axis, 1.0)
    with contextlib.redirect_stdout(io.StringIO()):
        g.initFromGridMap()
    s = [starts[q] for q in mine]; e = [goals[q] for q in mine]
    g.searchBatch(s[:8], e[:8], 300.0, 3, with_paths=False)       # warm-up: buffers, kernels
    g.setNextSearch(0)
    g.sync()
    c0 = g.counters()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = g.searchBatch(s, e, 300.0, iters, with_paths=True)     # paths read back: this is the e2e figure (queries in, paths out)
    g.sync()
    dt = time.perf_counter() - t0
    steps = g.counters()["ant_steps"] - c0["ant_steps"]
    found = int(sum(np.isfinite(r[2]) for r in res))
    st = g.batchStats()
    # the same queries one after the other (round 1's path), on a sample, and a sample against... nothing here: parity lives in tests/
    k = min(8, len(s))
    g.setNextSearch(0)
    t1 = time.perf_counter()
    seq = g.searchPairs(s[:k], e[:k], 300.0, iters, with_paths=True)
    g.sync()
    dt_seq = (time.perf_counter() - t1) / max(k, 1)
    same = all(np.array_equal(a[0], b[0]) and (a[2] == b[2] or (np.isinf(a[2]) and np.isinf(b[2]))) for a, b in zip(seq, res[:k]))
    if dist is not None:
        t = torch.tensor([dt], device="cuda", dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX); dt = float(t.item())
        v = torch.tensor([steps, found, int(same)], device="cuda", dtype=torch.int64); dist.all_reduce(v, op=dist.ReduceOp.SUM)
        steps, found, same = int(v[0]), int(v[1]), int(v[2]) == world
    del g
    return {"workload": "C5: %d start/goal queries on a synthetic 512^3 obstacle grid (%.1f %% occupied), %d ants x %d iterations each, Manhattan separation 64-256, "
                        "query q -> rank q mod %d" % (nq, 100.0 * (1 - free.mean()), ants, iters, world),
            "queries_per_s": nq / dt, "seconds": dt, "ant_steps_per_s": steps / dt, "acs_iterations_per_s": nq * iters / dt, "found": found,
            "timed": "wall clock from host query lists to host paths (wr_acs_search_batch), max over ranks",
            "batch": st, "sequential_ms_per_query_sample": 1e3 * dt_seq, "batch_equals_sequential_on_sample": bool(same)}


def sub_c4(rank, world, dist, n=256, colonies=1024, iters=64):
    """BASELINE configs[3]: ACS_GTSP seam ordering, 256 seams, 1024 colonies (colony b -> rank b mod world), 64 iterations (SURVEY 8d)."""
    import torch
    import welding_robot_b200 as wr
    P = np.random.default_rng(3).random((n, 3))
    D = np.sqrt(((P[:, None] - P[None]) ** 2).sum(-1))
    D = np.round(D, 6)                                   # "%.6f", as a graph file would carry it
    per = (colonies + world - 1) // world
    first = rank * per
    mine = max(0, min(per, colonies - first))
    g = wr.ACS_GTSP(seed=3)
    g.dis, g.city_num, g.cnt = D, n, n * (n - 1) // 2
    g._create(max(mine, 1), first)
    g.iterate(1)
    check_sync = lambda: g.best(0)  # noqa: E731  (wr_gtsp_best synchronises)
    check_sync()
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    g.iterate(iters)
    check_sync()
    dt = time.perf_counter() - t0
    ms = g.kernelMs()
    Ls = [g.best(b)[1] for b in range(0, max(mine, 1), max(1, mine // 4))]
    if dist is not None:
        t = torch.tensor([dt], device="cuda", dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX); dt = float(t.item())
    return {"workload": "C4: ACS_GTSP, %d seams, %d colonies x %d iterations, colonies split over %d rank(s)" % (n, colonies, iters, world),
            "colony_iterations_per_s": colonies * iters / dt, "ant_steps_per_s": colonies * iters * n * n / dt, "seconds": dt,
            "phase_ms_rank0": ms, "algorithmic_GBps_at_40N2_B": colonies * iters * 40 * n * n / dt / 1e9, "sample_best_L": Ls}


def sub_c3(rank, world, dist, stream, iters=10, ants_per_gpu=8192):
    """BASELINE configs[2]: origin_piece at a 512-long grid in 512^3, 8192 ants per GPU (65 536 at 8), ant-sharded."""
    import torch
    import welding_robot_b200 as wr
    from welding_robot_b200 import _lib
    from welding_robot_b200.dist import ShardedSearch
    global CUBE, PRECISION, MESH
    keep = (CUBE, PRECISION, MESH)
    CUBE, PRECISION, MESH = 512, 0.823812 / 491.5, "origin_piece"
    try:
        wl = build_workload_gpu()
        a = wr.ACS_Rank(seed=2, fixed_colony=ants_per_gpu * world, step_cap=16384, update_mode=4)
        a.creatFromOccupancy(wl["isfree"], wl["xs"], wl["ys"], wl["zs"], PRECISION)
        with contextlib.redirect_stdout(io.StringIO()):
            a.initFromGridMap()
        _lib.check(_lib.lib().wr_acs_set_stream(a._a, stream.cuda_stream))
        a.setEndpoints(wl["start"], wl["goal"])
        if world > 1:
            S = ShardedSearch(a, rank, world); S.begin(PREDICT); step = S.iterate
        else:
            a.begin(PREDICT); step = a.iterate
        step(3)
        a.sync()
        a.setTiming(True)
        c0 = a.counters()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        step(iters)
        e1.record(stream)
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        steps = a.counters()["ant_steps"] - c0["ant_steps"]
        kms = a.kernelMs()
        dirty, tiles = a.fieldStats()
        if dist is not None:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
            v = torch.tensor([steps], device="cuda", dtype=torch.int64); dist.all_reduce(v, op=dist.ReduceOp.SUM); steps = int(v.item())
        del a
        return {"workload": "C3: ACSRank_3D, origin_piece @512-long grid in 512^3, %d ants (%d per GPU), iterations 4-%d of one search" % (ants_per_gpu * world, ants_per_gpu, 3 + iters),
                "ant_steps_per_s": steps / (ms * 1e-3), "acs_iterations_per_s": iters / (ms * 1e-3), "ms_per_iteration": ms / iters,
                "kernel_ms_per_iteration_rank0": {k: v / iters for k, v in kms.items()}, "dirty_tiles": dirty, "tiles": tiles,
                "pheromone_field_bytes": 512 ** 3 * 6 * 4, "natural_grid": list(wl["natural"])}
    finally:
        CUBE, PRECISION, MESH = keep


def field_digest(acs):
    """order-sensitive 64-bit digest of the downloaded pheromone field"""
    t = acs.pheromone().view(np.uint32).astype(np.uint64)
    w = (np.arange(t.size, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)) | np.uint64(1)
    return int((t * w).sum(dtype=np.uint64))


DUMP_TAU_SLOTS = 1 << 22     # pheromone slots in --dump-outputs: 16 MB of the 403 MB field


def dump_outputs(acs, out_dir):
    """--dump-outputs: what a caller of the timed search receives after its last step, as out_dir/<name>.npy — the best path
    (node ids, directions, length), the search counters (in the order of ACS_Rank.counters(); in a sharded run those of rank 0's
    shard, while the best path and the field are the same on every rank) and the pheromone field at a fixed
    sample of slots (drawn with seed 0, ascending).  The workload and the search are seeded: with the same arguments every run
    searches the same inputs, so two builds of the project can be compared file by file."""
    os.makedirs(out_dir, exist_ok=True)
    ids, dirs, L = acs.bestPath()
    tau = acs.pheromone()
    slots = np.unique(np.random.default_rng(0).integers(0, tau.size, DUMP_TAU_SLOTS))
    arrays = {"best_path_ids": ids.astype(np.float64), "best_path_dirs": dirs.astype(np.float64), "best_length": np.array([L], np.float32),
              "counters": np.array(list(acs.counters().values()), np.float64), "pheromone_sample": tau[slots]}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------------
# this repo's arm
# ---------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import welding_robot_b200 as wr
    from welding_robot_b200 import _lib
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1 and args.gpus > 1:
        raise SystemExit("launch with `python -m torch.distributed.run --nproc-per-node %d bench.py --gpus %d ...`" % (args.gpus, args.gpus))
    torch.cuda.set_device(local)
    _lib.check(_lib.lib().wr_set_device(local))
    torch.cuda.set_stream(torch.cuda.Stream())   # a stream of our own (the default stream cannot be captured into CUDA graphs); events, NCCL and the handles all use it
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    wl = build_workload_gpu()
    n_nodes = CUBE ** 3
    colony = args.ants * world

    def make_search(host_free):
        acs = wr.ACS_Rank(seed=SEED, fixed_colony=colony, step_cap=STEP_CAP, update_mode=args.update_mode)
        acs.creatFromOccupancy(host_free, wl["xs"], wl["ys"], wl["zs"], PRECISION)     # H2D: occupancy + coordinates
        with contextlib.redirect_stdout(io.StringIO()):
            acs.initFromGridMap()
        return acs

    acs = make_search(wl["isfree"])
    stream = torch.cuda.current_stream()
    _lib.check(_lib.lib().wr_acs_set_stream(acs._a, stream.cuda_stream))
    acs.setEndpoints(wl["start"], wl["goal"])
    from welding_robot_b200.dist import ShardedSearch
    if world > 1:
        driver = ShardedSearch(acs, rank, world)
        driver.begin(PREDICT)
        step = lambda: driver.iterate(args.iters)  # noqa: E731
    else:
        acs.begin(PREDICT)
        step = lambda: acs.iterate(args.iters)  # noqa: E731

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    # ---- timed region, device resident -------------------------------------------------------------
    # The timed region runs as a user would run it (no per-phase events, so the steady-state iterations go out as one CUDA graph
    # each); the per-phase / per-kernel times are taken afterwards on a REPLAY of the same iterations (a fresh handle — on every
    # rank, for a sharded search — same seed: the search is deterministic) with the event pairs enabled.
    phase_in_timed = False
    c0 = acs.counters()
    rs0 = acs.updateStats()["rankset_iterations"]
    dirty0, tiles_total = acs.fieldStats()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        sampler.mark_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    sampler.mark_end()
    sampler.stop()
    c1 = acs.counters()
    if args.dump_outputs and rank == 0:
        dump_outputs(acs, args.dump_outputs)     # before the kernels-alone leg below runs more updates on this handle
    if phase_in_timed:
        kms = acs.kernelMs()
        sk_ms, sk_n = acs.streamKernelMs()                  # the streaming kernel alone, by its own events inside the loop
    else:
        rep = make_search(wl["isfree"])
        _lib.check(_lib.lib().wr_acs_set_stream(rep._a, stream.cuda_stream))
        rep.setEndpoints(wl["start"], wl["goal"])
        if world > 1:
            rep_driver = ShardedSearch(rep, rank, world)
            rep_driver.begin(PREDICT)
            rep_step = rep_driver.iterate
        else:
            rep.begin(PREDICT)
            rep_step = rep.iterate
        for _ in range(args.warmup):
            rep_step(args.iters)
        rep.sync()
        rep.setTiming(True)
        for _ in range(args.steps):
            rep_step(args.iters)
        kms = rep.kernelMs()
        sk_ms, sk_n = rep.streamKernelMs()
        assert rep.counters()["ant_steps"] == c1["ant_steps"], "replay diverged from the timed search"
        del rep
    upd_stats = acs.updateStats()
    rs_iters = upd_stats["rankset_iterations"] - rs0        # timed iterations whose deposits went through rank sets (mode 4)
    dirty1, _ = acs.fieldStats()
    dirty_tiles = 0.5 * (dirty0 + dirty1)                    # tiles the evaporation pass streams (clean-tile field), mean over the timed region
    acs.setTiming(False)
    local_steps = c1["ant_steps"] - c0["ant_steps"]
    steps_done = local_steps
    if dist is not None:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        s = torch.tensor([local_steps], device="cuda", dtype=torch.int64)
        dist.all_reduce(s, op=dist.ReduceOp.SUM)
        steps_done = int(s.item())
    iters_done = args.steps * args.iters
    value = steps_done / (ms * 1e-3)

    # ---- kernels timed alone (burst roofline of K3): the single-pass fused kernel over the WHOLE field, i.e. on a handle whose
    #      field is materialised (every tile dirty, WR_LAZY_TAU=0) and that carries the deposit records of a real iteration -------
    alone = {}
    if world == 1 and args.workload == "C2":
        os.environ["WR_LAZY_TAU"] = "0"
        dense = wr.ACS_Rank(seed=SEED, fixed_colony=colony, step_cap=STEP_CAP, update_mode=0)
        dense.creatFromOccupancy(wl["isfree"], wl["xs"], wl["ys"], wl["zs"], PRECISION)
        with contextlib.redirect_stdout(io.StringIO()):
            dense.initFromGridMap()
        del os.environ["WR_LAZY_TAU"]
        _lib.check(_lib.lib().wr_acs_set_stream(dense._a, stream.cuda_stream))
        dense.setEndpoints(wl["start"], wl["goal"])
        dense.begin(PREDICT)
        dense.iterate(3 * args.iters)
        for name, which in (("update_fused", 0), ("evaporate_float4", 1), ("d2d_copy", 2)):
            t_ms = dense.benchKernel(which, 20)
            alone[name] = {"ms": t_ms, "GBps": UPDATE_BYTES_PER_SLOT * n_nodes * 6 / (t_ms * 1e-3) / 1e9}
        alone["what"] = "dense field (every tile streamed), records of iteration %d of the same search; 805 MB per launch" % (3 * args.iters)
        del dense
        # the same kernel on the bench handle itself: its clean-tile field after the timed region, no records (rank-set phase)
        t_ms = acs.benchKernel(0, 20)
        dt, _ = acs.fieldStats()
        alone["update_fused_dirty_tiles_only"] = {"ms": t_ms, "GBps": dt * 4096 * UPDATE_BYTES_PER_SLOT / (t_ms * 1e-3) / 1e9, "tiles_streamed": dt,
                                                  "bytes": dt * 4096 * UPDATE_BYTES_PER_SLOT}

    # ---- the K = 26 neighbourhood (north_star's "26-neighbour" scores; the reference disables it, so it is reported next to
    #      the K = 6 parity workload, never instead of it): same grid, colony and endpoints, 112 B per ant-step --------------
    k26 = None
    if world == 1 and not args.no_k26:
        a26 = wr.ACS_Rank(seed=SEED, fixed_colony=args.ants, step_cap=STEP_CAP, update_mode=args.update_mode, K=26)
        a26.creatFromOccupancy(wl["isfree"], wl["xs"], wl["ys"], wl["zs"], PRECISION)
        with contextlib.redirect_stdout(io.StringIO()):
            a26.initFromGridMap()
        _lib.check(_lib.lib().wr_acs_set_stream(a26._a, stream.cuda_stream))
        a26.setEndpoints(wl["start"], wl["goal"])
        a26.begin(PREDICT)
        a26.iterate(3 * args.iters)
        a26.sync()
        a26.setTiming(True)
        d0 = a26.counters()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n26 = 6 * args.iters
        f0.record(stream)
        a26.iterate(n26)
        f1.record(stream)
        torch.cuda.synchronize()
        ms26 = f0.elapsed_time(f1)
        d1 = a26.counters()
        k26ms = a26.kernelMs()
        st26 = d1["ant_steps"] - d0["ant_steps"]
        hbm26, _ = peaks()
        w26 = 112 * st26 / (k26ms["walk"] * 1e-3) / 1e9
        dt26, tt26 = a26.fieldStats()
        u26 = UPDATE_BYTES_PER_SLOT * dt26 * 4096 * n26 / (k26ms["update"] * 1e-3) / 1e9
        k26 = {"ant_steps_per_s": st26 / (ms26 * 1e-3), "acs_iterations_per_s": n26 / (ms26 * 1e-3), "iterations": n26,
               "mean_steps_per_ant": st26 / max(1, d1["ants"] - d0["ants"]), "arrived": d1["arrived"] - d0["arrived"],
               "kernel_ms_per_iteration": {k: v / n26 for k, v in k26ms.items()},
               "walk_GBps_at_112B_per_step": w26, "walk_frac_of_hbm": w26 / hbm26,
               "update_GBps": u26, "update_frac_of_hbm": u26 / hbm26, "pheromone_field_bytes": n_nodes * 26 * 4, "dirty_tiles": dt26, "tiles": tt26}
        del a26

    # ---- sharded runs carry their own parity evidence: 3 iterations of a fresh sharded search against the same colony on
    #      ONE GPU (rank 0), whole pheromone field + best path -------------------------------------------------------------
    parity = None
    if world > 1 and not args.no_parity_check:
        psh = make_search(wl["isfree"])
        _lib.check(_lib.lib().wr_acs_set_stream(psh._a, stream.cuda_stream))
        psh.setEndpoints(wl["start"], wl["goal"])
        pd = ShardedSearch(psh, rank, world)
        pd.begin(PREDICT); pd.iterate(3); psh.sync()
        mine = (field_digest(psh), float(psh.bestPath()[2]), int(psh.bestPath()[0].sum()))
        del pd, psh
        ref = None
        if rank == 0:
            one = make_search(wl["isfree"])
            one.setEndpoints(wl["start"], wl["goal"])
            one.begin(PREDICT); one.iterate(3); one.sync()
            ref = (field_digest(one), float(one.bestPath()[2]), int(one.bestPath()[0].sum()))
            del one
        allv = [None] * world
        dist.all_gather_object(allv, mine)
        box = [ref]
        dist.broadcast_object_list(box, src=0)
        parity = {"parity_check": "ok" if all(v == box[0] for v in allv) else "FAILED",
                  "what": "3 iterations of a fresh %d-ant sharded search on every rank vs the same colony on one GPU (rank 0): digest of the whole "
                          "pheromone field, best length, best path" % colony, "digests": [hex(v[0]) for v in allv], "single_gpu_digest": hex(box[0][0])}

    # ---- what a user runs: begin + 150 iterations (the reference's max_iteration, ACSRank_3D.hpp:322), from host buffers --------
    full = None
    if world == 1 and args.workload == "C2" and not args.no_sub:
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fs = make_search(wl["isfree"])
        fs.setEndpoints(wl["start"], wl["goal"])
        fs.begin(PREDICT)
        fs.iterate(150)
        ids, dirs, L = fs.bestPath()
        dt_full = time.perf_counter() - t0
        cf = fs.counters()
        full = {"iterations": 150, "seconds_from_host_buffers": dt_full, "ant_steps": cf["ant_steps"], "ant_steps_per_s": cf["ant_steps"] / dt_full,
                "acs_iterations_per_s": 150 / dt_full, "best_L": float(L), "best_path_nodes": int(len(ids)), "rank_set_iterations": fs.updateStats()["rankset_iterations"],
                "what": "occupancy upload + wr_acs_create + wr_acs_begin + 150 x iterate + wr_acs_best, wall clock"}
        del fs

    subs = {}
    if not args.no_sub and args.workload == "C2":
        subs["C3"] = sub_c3(rank, world, dist, stream)
        subs["C4"] = sub_c4(rank, world, dist)
        subs["C5"] = sub_c5(rank, world, dist)

    # ---- end to end through the public API from HOST buffers -------------------------------------------
    e2e = None
    if True:
        pinned = torch.from_numpy(wl["isfree"]).pin_memory()
        host_free = pinned.numpy()
        e2e_steps = max(1, min(args.steps, 5))

        def e2e_step():
            a2 = make_search(host_free)
            a2.setEndpoints(wl["start"], wl["goal"])
            if world > 1:
                _lib.check(_lib.lib().wr_acs_set_stream(a2._a, stream.cuda_stream))
                d2 = ShardedSearch(a2, rank, world)
                d2.begin(PREDICT)                                                       # + exchange of the peer-slab IPC handles
                d2.iterate(args.iters)
            else:
                a2.begin(PREDICT)
                a2.iterate(args.iters)
            ids, dirs, L = a2.bestPath()                                                # D2H: the result
            n = a2.counters()["ant_steps"]
            del a2
            return n, len(ids) * 4 + len(dirs) + 4 + 9 * 8

        for _ in range(2):          # untimed: the first searches grow the stream-ordered memory pool by a second handle's worth
            e2e_step()
        tot_steps, d2h = 0, 0
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            n, d2h = e2e_step()
            tot_steps += n
        barrier()
        dt = time.perf_counter() - t0
        if dist is not None:
            t = torch.tensor([dt], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
            sN = torch.tensor([tot_steps], device="cuda", dtype=torch.int64)
            dist.all_reduce(sN, op=dist.ReduceOp.SUM)
            tot_steps = int(sN.item())
        e2e = {"value": tot_steps / dt, "unit": "ant-steps/s", "h2d_bytes_per_step": int(host_free.nbytes + 3 * CUBE * 4 + 16),
               "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
               "what": "per step and per rank, from host buffers: wr_grid_create_from_occupancy (16.8 MB H2D) -> wr_acs_create -> wr_acs_begin -> "
                       "%d x iterate%s -> wr_acs_best (D2H); wall clock between barriers, max over ranks"
                       % (args.iters, " (sharded: + peer-slab handle exchange)" if world > 1 else "")}
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    hbm, hbm_src = peaks()
    traffic = {}
    tp = os.path.join(ROOT, "profiles", "r2_traffic.json")   # dram__bytes_read+write per launch from the committed ncu --set full captures
    if os.path.exists(tp):
        with open(tp) as f:
            tj = json.load(f)
        traffic = {k: v["dram_bytes_read"] + v["dram_bytes_write"] for k, v in tj.items() if isinstance(v, dict)}
    walk_ms = kms["walk"] / iters_done
    upd_ms = kms["update"] / iters_done
    walk_gbs = WALK_BYTES_PER_STEP * (local_steps / iters_done) / (walk_ms * 1e-3) / 1e9
    upd_bytes = dirty_tiles * 4096 * UPDATE_BYTES_PER_SLOT     # what the pass reads + writes: 4096-float tiles, 8 B per slot
    upd_phase_gbs = upd_bytes / (upd_ms * 1e-3) / 1e9
    upd_kernel_ms = sk_ms / max(1, sk_n)
    upd_gbs = upd_bytes / (upd_kernel_ms * 1e-3) / 1e9
    upd_dense_gbs = UPDATE_BYTES_PER_SLOT * n_nodes * 6 / (upd_ms * 1e-3) / 1e9
    ants_done = max(1, c1["ants"] - c0["ants"])
    out = {
        "metric": "ant-steps/s", "value": value, "unit": "ant-steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic: reference mesh fixture voxelised on the GPU, embedded in 256^3 free space; synthetic start/goal",
        "config": {"workload": "%s, %d ants/GPU, K=6" % (LABEL, args.ants),
                   "grid": [CUBE, CUBE, CUBE], "natural_grid": list(wl["natural"]), "ants": colony, "iters_per_step": args.iters,
                   "step_cap": STEP_CAP, "seed": SEED, "update_mode": ["fused", "split", "atomic", "fused_tma", "rankset"][args.update_mode],
                   "parallelism": "ants sharded x%d" % world,
                   "exchange": ("none (1 GPU)" if world == 1 else
                                "NVLink peer memory inside the library's kernels (barrier flags, step counts, trails, rank-set blocks | final slot values); "
                                "no collective in the iteration loop"),
                   "l2_rule": "inputs larger than L2: the %d MB pheromone field is streamed from HBM every iteration" % (n_nodes * 6 * 4 // 1000000)},
        "acs_iterations_per_s": iters_done / (ms * 1e-3),
        "ant_steps": steps_done, "arrived_local": c1["arrived"] - c0["arrived"], "ants_local": c1["ants"] - c0["ants"],
        "mean_steps_per_ant": local_steps / ants_done,
        "gpu_launches": int(round(launches_per_iteration(0 if args.update_mode == 4 else args.update_mode, colony, args.iters, world > 1) * (iters_done - rs_iters)
                                  + launches_per_iteration(4, colony, args.iters, world > 1) * rs_iters)),
        "deposit_path": {"rank_set_iterations": rs_iters, "record_iterations": iters_done - rs_iters, "last": upd_stats} if args.update_mode == 4 else None,
        "kernel_ms_per_iteration": {k: v / iters_done for k, v in kms.items()},
        "kernel_ms_source": "replay of the timed iterations on a fresh handle with per-phase events (the timed region itself runs without them)",
        "roofline": {"kernel": "k_walk3 (K2 ant construction; dominant by time)", "bound": "hbm", "achieved": walk_gbs, "peak": hbm, "unit": "GB/s",
                     "frac": walk_gbs / hbm, "traffic": traffic.get("k_walk3"),
                     "traffic_source": "static: dram__bytes_read+write per launch from the committed `ncu --set full` capture (profiles/), not measured in this run",
                     "peak_source": hbm_src,
                     "limiter": "(longest ant's steps) x (latency of one warp's dependent instruction chain: 132 warp-instructions per step at 3.9 cycles, "
                                "28 % of the issue slots, 10 % of the warp slots in the round-2 ncu capture) - not HBM (1.5 MB of DRAM traffic per converged launch), "
                                "not issue; see DESIGN.md section 4",
                     "algorithmic_bytes_per_launch": WALK_BYTES_PER_STEP * (local_steps / iters_done),
                     "note": "30 B algorithmic per ant-step; a walk is a chain of dependent gathers, so with 4096 ants the kernel is "
                             "latency-bound, not bandwidth-bound (see DESIGN.md)"},
        "roofline_update": {"kernel": ["k_update_fused (K3: evaporation + rank-ordered deposits, one HBM pass)", "k_evaporate + k_deposit_apply (K3 split)",
                                       "k_evaporate + atomic deposits (K3 atomic)", "(removed)",
                                       "k_update_fused on record-path iterations | k_evaporate_tiles (+ k_rankset_apply) on rank-set iterations (K3 adaptive)"][args.update_mode],
                            "bound": "hbm", "achieved": upd_gbs, "peak": hbm, "unit": "GB/s", "frac": upd_gbs / hbm,
                            "traffic": traffic.get("k_update_fused") if args.update_mode == 0 else (traffic.get("k_evaporate_tiles") if args.update_mode == 4 else None),
                            "traffic_source": "static: committed ncu capture (profiles/), not measured in this run",
                            "algorithmic_bytes_per_launch": upd_bytes,
                            "reference_sweep_bytes": UPDATE_BYTES_PER_SLOT * n_nodes * 6, "reference_sweep_equivalent_GBps": upd_dense_gbs,
                            "dirty_tiles": dirty_tiles, "tiles": tiles_total, "kernel_ms": upd_kernel_ms, "launches_timed": sk_n,
                            "phase_ms": upd_ms, "phase_GBps": upd_phase_gbs,
                            "note": "clean-tile field: the pass streams only the 16 KB tiles that ever received a deposit (8 B per slot of those); "
                                    "`achieved` counts those bytes, `reference_sweep_equivalent_GBps` the reference's sweep of every slot (SURVEY 8d) over the same time",
                            "peak_source": hbm_src,
                            "timed": "the streaming kernel by its own CUDA-event pair inside the iteration loop (`kernel_ms`); `phase_ms` is the whole update "
                                     "phase (k_tile_offsets / k_rankset_apply and launch gaps included)"},
        "kernels_alone": alone,
        "voxelise": {"triangles": wl["ntri"], "grid": list(wl["natural"]), "kernel_ms": wl["vox"]["kernel_ms"], "tests": wl["vox"]["tests"]},
        "clocks": sampler.summary(),
    }
    if e2e:
        out["e2e"] = e2e
    if parity:
        out.update(parity)
    if full:
        out["full_search"] = full
    if subs:
        out["other_configs"] = subs
    if k26:
        out["k26_extension"] = k26
    if not args.no_cpu_baseline and world == 1:
        out["cpu_baseline"] = cpu_baseline(args)
    print(json.dumps(out))


def launches_per_iteration(update_mode, colony=ANTS_PER_GPU, iters=5, sharded=False):
    """Kernels of OURS launched per ACS iteration (welding_robot_b200/csrc/acs.cu: wr_acs_iterate; a steady-state iteration that goes
    out as one CUDA graph launch still runs the same kernels)."""
    slot_bits = int(np.ceil(np.log2(CUBE ** 3 * 6)))
    sort = lambda bits: 3 * ((bits + 9) // 10)  # noqa: E731  hist + scan + scatter per pass of <= 10-bit digits (radix_sort.cu)
    rank = 1 if colony <= 8192 else 3                            # k_rank_small | chunk sorts + merge + prefix finish
    groups = 1 if int(0.2 * colony) + 1 <= 1024 else 2           # rank-set path: apply (+ clear when the colony needs more than one rank group)
    # iter_begin, walk pass 1 + 2, ranking, best copy, iter_end (once per wr_acs_iterate call)
    n = 1 + 2 + rank + 1 + 1.0 / iters
    if sharded:
        n += 1                                                   # gather of the step counts (the barrier is inside)
    warm = 1 if os.environ.get("WR_WALK_WARM", "0") not in ("", "0") else 0   # the L2 warm-up kernel (off by default since round 2)
    if update_mode == 2:
        return n + warm + 2                                      # [L2 warm-up], evaporate, atomic deposits
    if update_mode == 4:                                         # rank sets: [L2 warm-up], gen, evaporate, apply x groups, wipe, serial fallback (both exit at once)
        return n + warm + 1 + 1 + groups + 1 + (2 if sharded else 0)   # sharded: + publish, merge (the barrier is inside)
    n += 1 + sort(slot_bits) + 2                                 # deposit gen, slot sort, tile offsets + fused
    if sharded:
        n += 4 + 1                                               # partition pass, pull of the peers' final values (barrier inside)
    else:
        n += warm                                                # [L2 warm-up]
    return n


# ---------------------------------------------------------------------------------------------------
# the reference's CPU implementation (oracle/_ref = UNMODIFIED reference headers), or the oracle port
# ---------------------------------------------------------------------------------------------------
def reference_worker(args):
    """One process: `warmup + steps` first-iterations of computeSolution (ACSRank_3D.hpp:220-305) with the workload's own colony
    (4096 ants) on the C2 grid, the pheromone field reset between steps (untimed) — the regime of the GPU arm's `e2e` leg
    (fresh searches).  Stops early when the time budget is used up.  Prints {"kind", "ant_steps": [...], "seconds": [...], "init_s"}."""
    from oracle import oracle as O
    wl = build_workload_cpu()
    seed = SEED + 1000 * args.worker
    # the reference sizes its colony as int(0.35*predict/precision) while no path is known (:247)
    predict = (args.cpu_ants + 0.5) * PRECISION / 0.35
    t0 = time.perf_counter()
    use_ref = O.have_ref() and not args.port
    steps, secs = [], []
    budget = args.budget_s
    if use_ref:
        R = O.Ref()
        c0, c1 = wl["cmin"], wl["cmax"]
        dummy = np.array([[0, 0, 1, c0[0], c0[1], c0[2], c1[0], c1[1], c1[2], c0[0], c1[1], c0[2]]], np.float32)
        R.voxelize(dummy, PRECISION, WALL)      # same lattice: cubic box through creatGridMap's own formula
        assert R.dims == (CUBE, CUBE, CUBE), R.dims
        _, xs, ys, zs = R.grid()
        assert np.array_equal(xs, wl["xs"]) and np.array_equal(ys, wl["ys"]) and np.array_equal(zs, wl["zs"])
        R.set_free(wl["isfree"])
        R.acs_init()
        assert R.set_endpoints(wl["start"], wl["goal"])
        init_s = time.perf_counter() - t0
        tb = time.perf_counter()
        for i in range(args.warmup + args.steps):
            t1 = time.perf_counter()
            calls = R.compute(predict, 1, seed + i)    # every successful step draws once (ACSRank_3D.hpp:169)
            secs.append(time.perf_counter() - t1); steps.append(int(calls))
            R.reset()                                  # reset() :307-315, untimed: every step is a fresh search
            if i >= args.warmup and time.perf_counter() - tb > budget:
                break
    else:
        G = O.Grid.from_occupancy(wl["isfree"], wl["xs"], wl["ys"], wl["zs"], PRECISION)
        A = O.Acs(G, seed=seed, rng_mode=O.RNG_SEQUENTIAL, sort_mode=O.SORT_STD)
        A.set_endpoints(wl["start"], wl["goal"])
        init_s = time.perf_counter() - t0
        tb = time.perf_counter()
        for i in range(args.warmup + args.steps):
            before = A.counters()["ant_steps"]
            t1 = time.perf_counter()
            A.begin(predict); A.iterate(1)
            secs.append(time.perf_counter() - t1); steps.append(A.counters()["ant_steps"] - before)
            A.reset()
            if i >= args.warmup and time.perf_counter() - tb > budget:
                break
    print(json.dumps({"kind": "reference" if use_ref else "port", "ant_steps": steps[args.warmup:], "seconds": secs[args.warmup:], "init_s": init_s}))


def run_reference_pool(args, steps, warmup, workers, budget_s):
    """`workers` concurrent single-thread processes (the reference has no threads: independent searches
    are the only parallelism that keeps its arithmetic, SURVEY.md §8d)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--worker-mode", "--steps", str(steps), "--warmup", str(warmup),
           "--cpu-ants", str(args.cpu_ants), "--budget-s", str(budget_s), "--workload", args.workload] + (["--port"] if args.port else [])
    procs = [subprocess.Popen(cmd + ["--worker", str(i)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for i in range(workers)]
    res = []
    for p in procs:
        out, err = p.communicate()
        if p.returncode != 0:
            raise RuntimeError("reference worker failed:\n" + err[-2000:])
        res.append(json.loads(out.strip().splitlines()[-1]))
    done = min(len(r["ant_steps"]) for r in res)            # every process contributes the same number of steps
    tot = sum(sum(r["ant_steps"][:done]) for r in res)
    wall = max(sum(r["seconds"][:done]) for r in res)
    return res, tot, wall, done


def host_workers(args):
    cores = os.cpu_count() or 1
    try:
        with open("/proc/meminfo") as f:
            avail_kb = next(int(l.split()[1]) for l in f if l.startswith("MemAvailable"))
    except Exception:
        avail_kb = 16 << 20
    by_mem = max(1, int(avail_kb * 0.6 / (7 << 20)))    # ~6 GB per unmodified-reference process at 256^3
    return max(1, min(cores, by_mem, args.max_workers))


def cpu_baseline(args):
    """Bounded sample for the default run: ONE process, 1 warm-up + 2 timed first-iterations of the workload's own colony."""
    res, tot, wall, done = run_reference_pool(args, steps=2, warmup=1, workers=1, budget_s=30.0)
    return {"value": tot / wall, "unit": "ant-steps/s", "cores": 1, "kind": res[0]["kind"],
            "sample": "%d first-iterations of computeSolution with the workload's %d ants on the same 256^3 grid (evaporation sweep of the whole field "
                      "included, reset() between them untimed), 1 process — the regime of the `e2e` leg" % (done, args.cpu_ants),
            "seconds": wall, "init_seconds": res[0]["init_s"], "ant_steps": tot}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), min(args.warmup, 1)
    workers = host_workers(args)
    res, tot, wall, done = run_reference_pool(args, steps, warmup, workers, budget_s=150.0)
    value = tot / wall
    print(json.dumps({
        "impl": "reference", "metric": "ant-steps/s", "value": value, "unit": "ant-steps/s", "n_gpus": args.gpus, "steps": done, "warmup": warmup,
        "steps_requested": args.steps, "warmup_requested": args.warmup,
        "ms_per_step": 1e3 * wall / done, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic: same C2 grid as the GPU arm, built on the CPU",
        "config": {"workload": "%s, %d ants/GPU, K=6" % (LABEL, ANTS_PER_GPU),
                   "grid": [CUBE, CUBE, CUBE], "ants": args.cpu_ants, "processes": workers,
                   "step": "one first-iteration of a fresh search with the full colony (the regime of the GPU arm's e2e leg); "
                           "%d of the %d requested steps fit the 150 s budget" % (done, args.steps)},
        "cpu_baseline": {"value": value, "unit": "ant-steps/s", "cores": workers, "kind": res[0]["kind"],
                         "sample": "%d timed first-iterations of computeSolution (ACSRank_3D.hpp:220-305) with %d-ant colonies on the 256^3 grid, "
                                   "%d concurrent single-thread processes (independent searches), evaporation sweep included"
                                   % (done, args.cpu_ants, workers)},
        "e2e": {"value": value, "unit": "ant-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)   # the timed region then is iterations 26-125 of the search, as in the driver's `--steps 20 --warmup 5`
    ap.add_argument("--iters", type=int, default=5, help="ACS iterations per step")
    ap.add_argument("--workload", default="C2", choices=["C2", "C3"], help="C2 = the bench workload; C3 = the 512^3 scaling case (exploration run)")
    ap.add_argument("--ants", type=int, default=0, help="ants per GPU (default: the workload's colony; other values are exploration runs)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--update-mode", type=int, default=4, help="WR_UPDATE_*: 4 = adaptive rank sets | sorted records + fused pass (default), 0 = fused")
    ap.add_argument("--cpu-ants", type=int, default=0, help="colony size of the CPU arm (default: the workload's colony)")
    ap.add_argument("--max-workers", type=int, default=16)
    ap.add_argument("--port", action="store_true", help="time the oracle port instead of oracle/_ref")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-k26", action="store_true", help="skip the K = 26 extension leg")
    ap.add_argument("--no-sub", action="store_true", help="skip the sub-records of the other BASELINE configurations (C3, C4, C5) and the full-search leg")
    ap.add_argument("--no-parity-check", action="store_true", help="N > 1: skip the sharded-vs-single-GPU self-check")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the timed search's best path, counters and a "
                                                          "fixed sample of its pheromone field as DIR/<name>.npy")
    ap.add_argument("--worker-mode", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--worker", type=int, default=0, help=argparse.SUPPRESS)
    ap.add_argument("--budget-s", type=float, default=150.0, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the CUDA path computed (--impl ours)")
    select_workload(args.workload)
    if args.ants <= 0:
        args.ants = ANTS_PER_GPU
    if args.cpu_ants <= 0:
        args.cpu_ants = ANTS_PER_GPU
    if args.workload != "C2":
        args.no_k26 = True
    if args.impl == "reference":
        if args.worker_mode:
            reference_worker(args)
        else:
            run_reference(args)
    else:
        args.warmup = max(args.warmup, 3)
        run_ours(args)


if __name__ == "__main__":
    main()
