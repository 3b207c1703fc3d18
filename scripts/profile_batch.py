"""Short concurrent-search run for ncu captures of the batch walk (k_walk_batch3, pass 2 k_walk2<Batch6>) and the per-query
kernels: C5-shaped queries on a synthetic obstacle grid (256^3 by default), 256 ants each.

    ncu --set full --clock-control none --import-source on -k regex:k_walk_batch -s 4 -c 2 -o gpurun_out/wb python scripts/profile_batch.py 256 512 6
"""
import contextlib
import io
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
import welding_robot_b200 as wr  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 256
nq = int(sys.argv[2]) if len(sys.argv) > 2 else 512
iters = int(sys.argv[3]) if len(sys.argv) > 3 else 6
free = bench.synthetic_boxes(n, 4096 * n ** 3 // 512 ** 3, 4)
axis = np.arange(n, dtype=np.float32)
ids = np.flatnonzero(free)
rng = np.random.default_rng(5)
starts, goals = [], []
while len(starts) < nq:
    s = int(ids[rng.integers(0, len(ids))])
    sz, sy, sx = s // (n * n), (s // n) % n, s % n
    d = int(rng.integers(64, 200))
    a = rng.multinomial(d, [1 / 3] * 3) * rng.choice([-1, 1], 3)
    gz, gy, gx = sz + a[0], sy + a[1], sx + a[2]
    if 0 <= gz < n and 0 <= gy < n and 0 <= gx < n and free[(gz * n + gy) * n + gx]:
        starts.append(s); goals.append(int((gz * n + gy) * n + gx))
g = wr.ACS_Rank(seed=5, fixed_colony=256, step_cap=4096)
g.creatFromOccupancy(free, axis, axis, axis, 1.0)
with contextlib.redirect_stdout(io.StringIO()):
    g.initFromGridMap()
res = g.searchBatch(starts, goals, 300.0, iters, with_paths=False)
g.sync()
print("found", sum(np.isfinite(r[2]) for r in res), "of", nq, g.counters(), g.batchStats())
