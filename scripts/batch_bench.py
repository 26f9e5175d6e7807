"""Grid batches against a loop of single-grid updates: Jacobi5 and HotSpot members of 128^2 .. 2048^2.

For every member size S the batch holds B = 2^26 / S^2 members (every buffer stays above the 126 MB L2),
each filled with the bench.py input of an S x S grid. In one process, alternating, it times
  (a) one batched update of all members, n iterations;
  (b) B single-grid updates of the same members, enqueued without blocking, then one synchronise,
with CUDA events on the runtime's stream around work that ends in a synchronise. Before timing it
checks that (a) and (b) give byte-identical members. For context it also times one 16384^2 grid.

    python scripts/batch_bench.py --out DIR [--iterations 1000] [--repeats 3] [--plan-only]

Writes DIR/batch_bench.json: per workload and member size the GCell-updates/s of (a) and (b) and their
ratio, the plan, the tile efficiency (useful over staged cells of the batch's tiles) and the launch
count, next to the GPU's name, power limit and SM clock read with a read-only nvidia-smi query.
There is no CPU fallback: without a GPU it stops at the first device call (--plan-only prints the
points and stops before it).
"""
from __future__ import annotations

import argparse
import json
import math
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

WORKLOADS = ["jacobi5", "hotspot"]
SIZES = [128, 256, 512, 1024, 2048]
TOTAL_CELLS = 1 << 26
CONTEXT_SIZE = 16384
CW = 4  # columns per thread of both workloads' float planes (Planner.hpp column_group_width)


def points(sizes=SIZES):
    """(member size, members) with members * size^2 = 2^26."""
    return [(s, TOTAL_CELLS // (s * s)) for s in sizes]


def tile_efficiency(stats, rows, cols, n_sub=1, radius=1):
    """Useful cells over staged cells of one full launch over a member of rows x cols cells, and the
    column share of it (tiles wider than the member waste staged columns)."""
    k, tile_h, tile_w = stats.fused_iterations, stats.tile_h, stats.tile_w
    halo = k * n_sub * radius
    staged_cols = stats.block_x * CW
    tiles = math.ceil(rows / tile_h) * math.ceil(cols / tile_w)
    staged = tiles * (tile_h + 2 * halo) * staged_cols
    return rows * cols / staged, cols / (math.ceil(cols / tile_w) * tile_w)


def gpu_info():
    query = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={query}", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True, check=True).stdout.strip()
    return dict(zip(query.split(","), [v.strip() for v in out.split(",")]))


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--out", type=Path, required=True)
    ap.add_argument("--iterations", type=int, default=1000)
    ap.add_argument("--repeats", type=int, default=3, help="timed (a)/(b) pairs per point")
    ap.add_argument("--sizes", type=int, nargs="*", default=SIZES)
    ap.add_argument("--workloads", nargs="*", default=WORKLOADS)
    ap.add_argument("--plan-only", action="store_true", help="print the points, touch no device")
    args = ap.parse_args()
    if args.iterations < 1 or args.repeats < 1:
        raise SystemExit("batch_bench.py: --iterations and --repeats must be positive")
    plan = [(w, s, b) for w in args.workloads for s, b in points(args.sizes)]
    for w, s, b in plan:
        print(f"{w}: {b} members of {s}x{s}, {b * s * s} cells, {args.iterations} iterations")
    if args.plan_only:
        return

    import ctypes as C

    import numpy as np

    import bench
    from stencilstream_b200 import Grid, GridBatch, Params, StencilUpdate, _native

    count = C.c_int()
    if _native.runtime_lib().stst_device_count(C.byref(count)) != 0 or count.value < 1:
        raise SystemExit("batch_bench.py: no CUDA device; this measurement has no CPU fallback")
    args.out.mkdir(parents=True, exist_ok=True)
    timer = bench.StreamTimer(0)
    n = args.iterations
    results = {"iterations": n, "total_cells": TOTAL_CELLS, "points": [], "context": []}

    def params_for(workload, size):
        tf, halo, fill = bench.make_workload(workload, size, size)
        cells = np.empty((size, size), dtype=_native.CELL_DTYPES[workload])
        fill(cells, 0, size, size)
        return tf, halo, cells

    for workload, size, members in plan:
        tf, halo, cells = params_for(workload, size)
        stack = np.broadcast_to(cells, (members, size, size)).copy()
        batch = GridBatch(workload, buffer=stack)
        grids = [Grid(workload, buffer=cells) for _ in range(members)]
        make = lambda: StencilUpdate(workload, Params(transition_function=tf, halo_value=halo,
                                                      n_iterations=n))
        batch_update, loop_update = make(), make()

        def run_batch():
            return batch_update(batch)

        def run_loop():
            return [loop_update(g) for g in grids]

        # warm-up, and the check that both paths compute the same cells
        got = run_batch().to_numpy()
        singles = run_loop()
        for b in (0, members // 2, members - 1):
            if got[b].tobytes() != singles[b].to_numpy().tobytes():
                raise SystemExit(f"batch_bench.py: {workload} {size}^2 member {b}: batch and loop differ")
        del singles
        launches_before = batch_update.get_stats().n_launches
        run_batch()
        stats = batch_update.get_stats()
        batch_launches = stats.n_launches - launches_before
        times = {"batch": [], "loop": []}
        with bench.ClockSampler(0) as clocks:
            for _ in range(args.repeats):
                for name, fn in (("batch", run_batch), ("loop", run_loop)):
                    timer.sync()
                    timer.begin()
                    out = fn()
                    times[name].append(timer.end_ms() * 1e-3)
                    del out
        cell_updates = float(n) * members * size * size
        rate = {k: cell_updates / min(v) / 1e9 for k, v in times.items()}
        eff, col_eff = tile_efficiency(stats, size, size)
        point = {
            "workload": workload, "member": [size, size], "members": members,
            "gcups_batch": rate["batch"], "gcups_loop": rate["loop"],
            "ratio": rate["batch"] / rate["loop"],
            "seconds_batch": times["batch"], "seconds_loop": times["loop"],
            "n_launches_batch": batch_launches,
            "n_launches_loop": members * math.ceil(n / loop_update.get_stats().fused_iterations),
            "plan_batch": {"k": stats.fused_iterations, "tile_h": stats.tile_h, "tile_w": stats.tile_w,
                           "block": [stats.block_x, stats.block_y], "tma": stats.use_tma},
            "plan_loop_tile_h": loop_update.get_stats().tile_h,
            "tile_efficiency": eff, "column_efficiency": col_eff,
            "clocks": clocks.summary(),
        }
        print(json.dumps(point), flush=True)
        results["points"].append(point)
        del batch, grids

    for workload in args.workloads:
        tf, halo, cells = params_for(workload, CONTEXT_SIZE)
        grid = Grid(workload, buffer=cells)
        update = StencilUpdate(workload, Params(transition_function=tf, halo_value=halo, n_iterations=n))
        update(grid)
        best = math.inf
        for _ in range(args.repeats):
            timer.sync()
            timer.begin()
            update(grid)
            best = min(best, timer.end_ms() * 1e-3)
        results["context"].append({"workload": workload, "grid": [CONTEXT_SIZE, CONTEXT_SIZE],
                                   "gcups": float(n) * CONTEXT_SIZE ** 2 / best / 1e9})
        print(json.dumps(results["context"][-1]), flush=True)

    results["gpu"] = gpu_info()
    results["time"] = time.strftime("%Y-%m-%d %H:%M:%S")
    (args.out / "batch_bench.json").write_text(json.dumps(results, indent=1) + "\n")
    print(json.dumps(results["gpu"]))


if __name__ == "__main__":
    main()
