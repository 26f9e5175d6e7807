#!/usr/bin/env python
"""Benchmark of the StencilStream-B200 generation loop.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload jacobi5|jacobi_r2|jacobi_r3|hotspot|fdtd|convection_pt|conway]
                    [--rows R --cols C --iterations I] [--dump-outputs DIR]

Metric (BASELINE.json / reference scripts/benchmark-common.jl:97-98): GCell-updates/s =
rows * cols * n_iterations / time, one "update" being one full iteration (all sub-iterations).
A *step* is one `StencilUpdate` call advancing the whole synthetic grid by `--iterations`
iterations. Default workload at N=1: BASELINE.json configs[1], Jacobi 5-point fp32 16384x16384,
1000 generations, input as the reference generates it (examples/jacobi/jacobi.cpp:111-124).

`value`        grid resident in HBM before the timed region; K steps timed with CUDA events on the
               stream the kernels are launched on, barrier + synchronize on both sides, max over ranks.
`e2e`          the same step through the public Grid/StencilUpdate API starting from cells in pinned
               host memory (GridAccessor image): upload + update + download inside the timed region.
               Its own step count (`e2e.steps`) is min(--steps, 3), and 1 for slabs moved chunk by
               chunk: --steps sets the timed steps of `value`, not of `e2e`.
`roofline`     HBM roofline of the fused sweep kernel: algorithmic bytes (2*sizeof(Cell)*n_sub per
               cell-iteration, the reference's own model) per launch / mean launch duration, against
               the measured copy bandwidth in MEASURED_PEAKS.json.
`cpu_baseline` the CPU oracle (reference-built if available) timed on this box's host cores on a
               bounded sample of the same workload (rank 0, N=1 only).
`parity`       after the end-to-end steps, a window of the step's result (n iterations from the
               synthetic input, as downloaded into host memory) is compared with the CPU oracle run on
               the window's domain of dependence: relative max-norm, bar 1e-5 (Conway: bit-exact).
               The oracle is the checker here, never the thing measured.
`workloads`    (default invocation only) the other BASELINE.json configs measured the same way in the
               same process: HotSpot 16384^2 (strong-scaled at N > 1, plus weak), FDTD max_grid
               (strong), mantle convection 8192 x 65536 cells per GPU (weak).
`--impl reference` times the reference's CPU implementation instead (same metric/config keys).
`--dump-outputs DIR` after the timed steps of every workload measured, writes the cells its last
               timed step returned as DIR/<name>.npy (one file per cell field, float32 or float64) so
               that two builds run with the same arguments can be compared output for output.
               Outputs too large for the 64 MB limit are sampled on rows x columns chosen with a
               fixed seed (see `dump_sample`).

Multi-GPU (torchrun, one rank per GPU): the grid is row-sharded, every rank owns `rows` rows (weak
scaling) or a share of a fixed grid (strong), and exchanges halo rows with its neighbours once per
fused launch.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

WORKLOAD_LABEL = {
    "jacobi5": "Jacobi 5-point fp32 {rows}x{cols}, {iters} generations (BASELINE.json configs[1])",
    "jacobi_r2": "Jacobi radius-2 star (9-point) fp32 {rows}x{cols}, {iters} generations (BASELINE.json configs[1], "
                 "radius-2 variant)",
    "jacobi_r3": "Jacobi radius-3 star (13-point) fp32 {rows}x{cols}, {iters} generations (BASELINE.json configs[1], "
                 "radius-3 variant)",
    "conway": "Conway's Game of Life {rows}x{cols}, {iters} generations (BASELINE.json configs[0] rule on a "
              "bandwidth-sized grid)",
    "hotspot": "Rodinia HotSpot fp32 temp+power {rows}x{cols}, {iters} generations (BASELINE.json configs[2])",
    "fdtd": "FDTD micro-cavity max_grid experiment {rows}x{cols} (coef cells, E/H sub-iterations, tdv source "
            "wave), {iters} time steps (BASELINE.json configs[3])",
    "convection_pt": "Mantle convection pseudo-transient kernel fp64 {rows}x{cols}, {iters} iterations "
                     "(BASELINE.json configs[4])",
}
# (rows per GPU, cols, iterations per step, scaling) used when the command line does not say otherwise
DEFAULTS = {"jacobi_r2": (16384, 16384, 1000, "weak"), "jacobi_r3": (16384, 16384, 1000, "weak"),
            "conway": (16384, 16384, 1000, "weak"),
            "jacobi5": (16384, 16384, 1000, "weak"), "hotspot": (16384, 16384, 1000, "weak"),
            "fdtd": (4608, 4608, 1000, "strong"), "convection_pt": (4096, 8192, 100, "weak")}
DTYPE = {"jacobi_r2": "f32", "jacobi_r3": "f32", "jacobi5": "f32", "hotspot": "f32", "fdtd": "f32", "convection_pt": "f64", "conway": "u8"}


# ---------------------------------------------------------------------------------------------------
# workload set-up
# ---------------------------------------------------------------------------------------------------

def make_workload(name: str, rows: int, cols: int):
    """(params struct, halo cell, function filling an array view with the synthetic input)."""
    from stencilstream_b200 import workloads as W

    if name == "jacobi5":
        return W.jacobi5_params(), 0.0, lambda view, r0, r1, total: fill_jacobi(view, r0, r1, total, cols)
    if name in ("jacobi_r2", "jacobi_r3"):
        return W.jacobi_star_params(int(name[-1])), 0.0, \
            lambda view, r0, r1, total: fill_jacobi(view, r0, r1, total, cols)
    if name == "conway":
        from stencilstream_b200 import _native

        def fill_conway(view, r0, r1, total):
            for lo in range(r0, r1, 1024):  # seeded per row band: slabs generate their own rows
                hi = min(lo + 1024, r1)
                view[lo - r0:hi - r0] = W.conway_soup(hi - lo, cols, seed=42 + lo)
        return _native.ConwayParams(), None, fill_conway
    if name == "hotspot":
        return W.hotspot_params(rows, cols), (0.0, 0.0), \
            lambda view, r0, r1, total: fill_hotspot(view, r0, r1, total, cols)
    if name == "fdtd":
        exp = W.FdtdExperiment(W.FDTD_MAX_GRID)
        if (rows, cols) != (exp.grid_wh(), exp.grid_wh()):
            raise SystemExit(f"bench.py: the max_grid experiment is {exp.grid_wh()} x {exp.grid_wh()}")
        grid0 = {}

        def fill_fdtd(view, r0, r1, total):
            if "cells" not in grid0:
                grid0["cells"] = exp.initial_grid()
            view[...] = grid0["cells"][r0:r1]
        return exp.kernel_params(), None, fill_fdtd
    if name == "convection_pt":
        exp = W.ConvectionExperiment(W.convection_benchmark_config(
            res=cols, n_iters=1, lx=rows / cols, ly=1.0))
        assert exp.grid_shape == (rows, cols), (exp.grid_shape, rows, cols)

        def fill_convection(view, r0, r1, total):
            # Only T is non-zero in the initial state (convection.cpp:380-397). A caller that fills
            # the SAME buffer again and again (the 47 GB slabs are generated chunk by chunk through
            # one pinned buffer) sets `assume_zeroed` after the first chunk, which saves rewriting 80
            # of every 88 bytes.
            if not fill_convection.assume_zeroed:
                view[...] = np.zeros((), dtype=view.dtype)
            for lo in range(r0, r1, 256):
                hi = min(lo + 256, r1)
                view["T"][lo - r0:hi - r0] = exp.initial_temperature(lo, hi)
        fill_convection.assume_zeroed = False
        return exp.pseudo_transient_params(), None, fill_convection
    raise SystemExit(f"bench.py: unsupported workload {name!r}")


def fill_jacobi(view, r0, r1, total_rows, cols):
    """Rows [r0, r1) of the centred unit square of a total_rows x cols grid (jacobi.cpp:111-124)."""
    r = np.arange(r0, r1, dtype=np.float64)[:, None]
    c = np.arange(cols, dtype=np.float64)[None, :]
    inside = (r >= total_rows * 0.25) & (r < total_rows * 0.75) & (c >= cols * 0.25) & (c < cols * 0.75)
    view[...] = inside.astype(np.float32)


def fill_hotspot(view, r0, r1, total_rows, cols):
    """Rows [r0, r1) of the reference's synthetic HotSpot input (data/input_gen.jl:3-15)."""
    view["temp"] = np.float32(30.0)
    view["power"] = np.float32(0.0)
    r_lo, r_hi = total_rows // 4, (3 * total_rows) // 4
    c_lo, c_hi = cols // 4, (3 * cols) // 4
    lo = max(r_lo - 1, r0)
    hi = min(r_hi, r1)
    if hi > lo:
        view["power"][lo - r0:hi - r0, max(c_lo - 1, 0):c_hi] = np.float32(0.5)


# ---------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------

class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU every 100 ms while the timed region runs."""

    REASONS = {
        0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown",
        0x4: "sw_power_cap", 0x80: "hw_power_brake", 0x2: "applications_clocks_setting",
    }

    def __init__(self, device_index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nvml = pynvml
            self._handle = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self._handle, pynvml.NVML_CLOCK_SM)
        except Exception:
            self._nvml = None

    def _loop(self):
        nv = self._nvml
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self._handle, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._handle)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        if self._nvml is not None:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons)}


# ---------------------------------------------------------------------------------------------------
# device-side timing on the runtime's stream
# ---------------------------------------------------------------------------------------------------

class StreamTimer:
    """CUDA events recorded on the stream StencilStream-B200 launches its kernels on."""

    def __init__(self, device: int, record=None, sync=None):
        """`record(event)` / `sync()` override where events are recorded (default: the runtime's
        per-device stream, on which single-GPU updates run; slabs record behind both their streams)."""
        from stencilstream_b200 import _native
        self.rt = _native.runtime_lib()
        self.stream = C.c_void_p()
        self._check(self.rt.stst_default_stream(device, C.byref(self.stream)))
        self._record = record or (lambda ev: self._check(self.rt.stst_event_record(ev, self.stream)))
        self._sync = sync or (lambda: self._check(self.rt.stst_stream_synchronize(self.stream)))
        self.start, self.stop = C.c_void_p(), C.c_void_p()
        self._check(self.rt.stst_event_create(1, C.byref(self.start)))
        self._check(self.rt.stst_event_create(1, C.byref(self.stop)))

    def _check(self, status):
        if status != 0:
            raise RuntimeError(self.rt.stst_last_error().decode())

    def sync(self):
        self._sync()

    def begin(self):
        self._record(self.start)

    def end_ms(self) -> float:
        self._record(self.stop)
        self._check(self.rt.stst_event_synchronize(self.stop))
        ms = C.c_float()
        self._check(self.rt.stst_event_elapsed_ms(self.start, self.stop, C.byref(ms)))
        return float(ms.value)


# ---------------------------------------------------------------------------------------------------
# CPU baseline / reference arm / parity window (the only places the oracle is used; it is the
# checker and the reported baseline, never the product path)
# ---------------------------------------------------------------------------------------------------

def time_cpu_oracle(workload: str, rows: int, cols: int, total_rows: int | None = None,
                    target_seconds: float = 12.0):
    """Time the CPU oracle (reference-built cpu backend if present, else the C port) on a bounded
    sample: a `sample_rows` x cols slab of the workload for `iters` iterations, sized from a short
    calibration run so that it takes roughly `target_seconds`. Uses every host core this process may
    run on, whatever OMP_NUM_THREADS says (torchrun exports OMP_NUM_THREADS=1)."""
    import oracle

    impl = oracle.best()
    cores = oracle.set_threads()
    params, halo, fill = make_workload(workload, total_rows or rows, cols)
    from stencilstream_b200 import _native
    dtype = _native.CELL_DTYPES[workload]
    sample_rows = min(rows, 2048)
    cells = np.empty((sample_rows, cols), dtype=dtype)
    fill(cells, 0, sample_rows, sample_rows)

    impl.run(workload, params, halo, cells, 0, 1)   # first touch, thread start-up
    iters = 4
    while True:  # grow the sample until it runs for most of the target time (short runs are slower
        t0 = time.perf_counter()        # per iteration, so one extrapolation undershoots)
        impl.run(workload, params, halo, cells, 0, iters)
        elapsed = time.perf_counter() - t0
        if elapsed >= 0.6 * target_seconds or iters >= 4000:
            break
        iters = int(min(4000, max(2 * iters, 1.05 * iters * target_seconds / max(elapsed, 1e-4))))
    value = sample_rows * cols * iters / elapsed / 1e9
    return {
        "value": value, "unit": "GCell-updates/s", "cores": cores,
        "kind": "reference" if impl.kind == "reference" else "port",
        "sample": f"{sample_rows}x{cols} slab of the workload grid, {iters} iterations, "
                  f"{elapsed:.1f} s on {cores} host threads (omp_get_max_threads; OpenMP over rows)",
    }, elapsed


def time_rodinia_hotspot(size: int = 2048, iterations: int = 400):
    """Second, independent CPU baseline for HotSpot: the reference's Rodinia OpenMP program
    (examples/hotspot/hotspot_openmp.cpp, compiled in place into oracle/_ref/hotspot_openmp by
    oracle/recipes.py) on a size x size grid. Returns None where the binary does not exist."""
    import re
    import subprocess
    import tempfile
    import oracle

    binary = ROOT / "oracle" / "_ref" / "hotspot_openmp"
    if not binary.exists():
        return None
    cores = oracle.host_threads()
    with tempfile.TemporaryDirectory() as tmp:
        tmp = Path(tmp)
        cells = np.empty((size, size), dtype=[("temp", "f4"), ("power", "f4")])
        fill_hotspot(cells, 0, size, size, size)
        np.savetxt(tmp / "temp", cells["temp"].reshape(-1), fmt="%g")
        np.savetxt(tmp / "power", cells["power"].reshape(-1), fmt="%g")
        env = dict(os.environ, OMP_NUM_THREADS=str(cores))
        proc = subprocess.run([str(binary), str(size), str(size), str(iterations), str(cores),
                               str(tmp / "temp"), str(tmp / "power"), str(tmp / "out")],
                              stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, env=env,
                              timeout=120)
    match = re.search(r"Total time: ([0-9.]+) seconds", proc.stdout)
    if proc.returncode != 0 or not match or float(match.group(1)) <= 0:
        return None
    seconds = float(match.group(1))
    return {"value": size * size * iterations / seconds / 1e9, "unit": "GCell-updates/s",
            "cores": cores, "kind": "reference",
            "sample": f"examples/hotspot/hotspot_openmp.cpp, {size}x{size}, {iterations} iterations, "
                      f"{seconds:.2f} s (its own 'Total time')"}


PARITY_TOLERANCE = 1e-5   # relative max-norm, BASELINE.json north_star (Conway: bit-exact)
STENCIL_SHAPE = {"conway": (1, 1), "jacobi5": (1, 1), "jacobi_r2": (2, 1), "jacobi_r3": (3, 1),
                 "hotspot": (1, 1), "fdtd": (1, 2), "convection_pt": (1, 3)}   # (radius, n_sub)


def parity_window_rows(workload: str, total_rows: int, cols: int):
    """(first row, column range) of the parity window: the north-west corner of the reference
    input's unit square / power block, where the input is not locally constant."""
    q_r, q_c = total_rows // 4, cols // 4
    return q_r, (max(q_c - 32, 0), min(q_c + 32, cols))


def check_parity_window(workload, params, halo, fill, total_rows, cols, iters, row_lo, row_hi, cells,
                        budget_cell_updates: float = 8e9):
    """Compare rows [win_lo, win_hi) x a 64-column range of `cells` (global rows [row_lo, row_hi) of
    the result after `iters` iterations from the synthetic input) with the CPU oracle run on the
    window's domain of dependence. Returns the `parity` record, or a record with a reason when the
    check does not apply (window not in these rows, oracle run beyond the time budget)."""
    import oracle

    radius, n_sub = STENCIL_SHAPE[workload]
    depth = iters * n_sub * radius
    q_r, (c0, c1) = parity_window_rows(workload, total_rows, cols)
    w0, w1 = max(q_r - 32, row_lo), min(q_r + 32, row_hi)
    if w1 <= w0:
        return None
    r0, r1 = max(w0 - depth, 0), min(w1 + depth, total_rows)
    k0, k1 = max(c0 - depth, 0), min(c1 + depth, cols)
    work = float(r1 - r0) * (k1 - k0) * iters
    if work > budget_cell_updates:
        return {"window": [[w0, w1], [c0, c1]], "rel_max_norm": None,
                "skipped": f"domain of dependence {r1 - r0}x{k1 - k0} x {iters} iterations exceeds the "
                           "bench's CPU budget; covered by tests/test_parity_fullsize_gpu.py"}
    # The oracle whose arithmetic matches the build under test: the default build contracts a*b+c into
    # FMAs (as the reference's own icpx build does), so its checker is the reference cpu backend
    # compiled with contraction allowed; STST_STRICT=1 (-fmad=false) is checked against the
    # uncontracted build. The other flavour is reported beside it (`rel_max_norm_vs_*`).
    strict_build = os.environ.get("STST_STRICT", "0") not in ("", "0")
    contracted = None if strict_build else (oracle.reference(fma=True) or
                                            (oracle.port(fma=True) if oracle.cpu_has_fma() else None))
    checker = contracted or oracle.best()
    other = oracle.best() if contracted is not None else None
    cores = oracle.set_threads()
    # (generated from a multiple of 1024 rows on: the Conway soup is seeded per 1024-row band)
    g0 = r0 - r0 % 1024
    band = np.empty((r1 - g0, cols), dtype=cells.dtype)
    fill(band, g0, r1, total_rows)
    crop = np.ascontiguousarray(band[r0 - g0:, k0:k1])
    del band
    t0 = time.perf_counter()
    want = checker.run_window2d(workload, params, halo, crop, r0, k0, total_rows, cols, 0, iters)
    seconds = time.perf_counter() - t0
    want = want[w0 - r0:w1 - r0, c0 - k0:c1 - k0]
    got = np.ascontiguousarray(cells[w0 - row_lo:w1 - row_lo, c0:c1])

    def distance(want):
        if workload == "conway":
            return 0.0 if got.tobytes() == want.tobytes() else 1.0
        err = 0.0
        for name in (got.dtype.names or (None,)):
            a = (got[name] if name else got).astype(np.float64)
            b = (want[name] if name else want).astype(np.float64)
            scale = np.abs(b).max()
            err = max(err, float(np.abs(a - b).max() / scale) if scale > 0 else float(np.abs(a).max()))
        return err

    err = distance(want)
    bar = 0.0 if workload == "conway" else PARITY_TOLERANCE
    extra = {}
    if other is not None and workload != "conway":
        want_other = other.run_window2d(workload, params, halo, crop, r0, k0, total_rows, cols, 0, iters)
        extra = {"rel_max_norm_vs_uncontracted_oracle":
                     distance(want_other[w0 - r0:w1 - r0, c0 - k0:c1 - k0]),
                 "note": "the default build contracts a*b+c into FMAs like the reference's icpx build; "
                         "against the uncontracted oracle it drifts linearly with the iteration count "
                         "(DESIGN.md section 5); STST_STRICT=1 selects the -fmad=false build, which is "
                         "bit-exact against that oracle"}
    return {"window": [[w0, w1], [c0, c1]], "rel_max_norm": err, "tolerance": bar, "ok": err <= bar,
            "bit_exact": bool(got.tobytes() == want.tobytes()),
            "iterations": iters, "oracle": checker.kind,
            "oracle_arithmetic": "g++ -ffp-contract=fast -mfma (contracting, matches -fmad=true)"
            if getattr(checker, "contracts", False) else "g++ -ffp-contract=off (matches -fmad=false)",
            **extra,
            "domain_of_dependence": [r1 - r0, k1 - k0], "oracle_seconds": round(seconds, 2),
            "oracle_threads": cores,
            "build": ("-fmad=false" if strict_build else "default (-fmad=true)") + ", the planner's plan"}


# ---------------------------------------------------------------------------------------------------
# --dump-outputs
# ---------------------------------------------------------------------------------------------------

DUMP_BYTES = 60 << 20   # all files of one invocation: under 64 MB with the .npy headers
DUMP_SEED = 20240607


def dump_dtype(field_dtype: np.dtype) -> np.dtype:
    """float64 for 8-byte fields, float32 for everything narrower (Conway's bool cells included)."""
    return np.dtype(np.float64) if field_dtype.itemsize == 8 else np.dtype(np.float32)


def dump_sample(total_rows: int, cols: int, dtype: np.dtype, budget: int):
    """(row indices, column indices) of the cells --dump-outputs writes: the whole grid where it fits
    `budget` bytes, else a near-square sample of rows x columns. On each axis the sample holds both
    ends (the cells that read the halo, and where e.g. convection's boundary temperatures start) and
    a scatter of the rest drawn with a fixed seed. The choice depends only on its arguments, so every
    run with the same command line dumps the same cells."""
    fields = [dtype[name] for name in dtype.names] if dtype.names else [dtype]
    cell_bytes = sum(dump_dtype(f).itemsize for f in fields)
    cells = max(1, budget // cell_bytes)
    if total_rows * cols <= cells:
        return np.arange(total_rows), np.arange(cols)
    n_rows = min(total_rows, max(1, int(np.sqrt(cells))))
    n_cols = min(cols, max(1, cells // n_rows))
    rng = np.random.default_rng(DUMP_SEED)

    def pick(n_total, n_pick):
        if n_pick >= n_total:
            return np.arange(n_total)
        edge = min(64, n_pick // 4)
        scatter = rng.choice(np.arange(edge, n_total - edge), n_pick - 2 * edge, replace=False)
        return np.sort(np.concatenate([np.arange(edge), np.arange(n_total - edge, n_total), scatter]))
    return pick(total_rows, n_rows), pick(cols, n_cols)


def write_dump(directory: Path, name: str, cells: np.ndarray) -> None:
    """One .npy per cell field (`name.field.npy`), or `name.npy` for single-value cells."""
    directory.mkdir(parents=True, exist_ok=True)
    for field in (cells.dtype.names or (None,)):
        values = cells[field] if field else cells
        np.save(directory / (f"{name}.{field}.npy" if field else f"{name}.npy"),
                np.ascontiguousarray(values, dtype=dump_dtype(values.dtype)))


def workload_config(workload, total_rows, rows, cols, iters, world):
    """The `config` object; identical in both arms (it names the workload, not the implementation)."""
    return {
        "workload": WORKLOAD_LABEL[workload].format(rows=total_rows, cols=cols, iters=iters),
        "rows_per_gpu": rows, "cols": cols, "iterations_per_step": iters,
        "parallelism": f"row-sharded x{world}" if world > 1 else "single GPU",
        "l2": "grid (>= 1 GiB per buffer) exceeds the 126 MB L2; no flush needed",
    }


def resolve_rows(args, world: int, rank: int):
    """(rows of this rank, rows of the whole grid)."""
    if args.scaling == "weak":
        return args.rows, args.rows * world
    from stencilstream_b200.sharding import partition_rows
    lo, hi = partition_rows(args.rows, world, rank)
    return hi - lo, args.rows


def run_reference_arm(args, rank: int, world: int):
    if rank != 0:
        return
    rows, total_rows = resolve_rows(args, world, 0)
    cols, iters = args.cols, args.iterations
    total_steps = args.steps + args.warmup
    budget = 150.0 / max(total_steps, 1)
    results = []
    baseline = None
    for i in range(total_steps):
        baseline, elapsed = time_cpu_oracle(args.workload, rows, cols, total_rows,
                                            target_seconds=min(budget, 15.0))
        if i >= args.warmup:
            results.append((baseline["value"], elapsed))
    value = float(np.mean([v for v, _ in results]))
    ms = float(np.mean([e for _, e in results]) * 1e3)
    baseline["value"] = value
    line = {
        "impl": "reference", "metric": "GCell-updates/s", "value": value, "unit": "GCell-updates/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": DTYPE.get(args.workload, "f32"), "data": "synthetic",
        "config": workload_config(args.workload, total_rows, rows, cols, iters, world),
        "note": "reference StencilStream cpu backend on the host cores; each step is a bounded sample "
                "of the workload (see cpu_baseline.sample)",
        "cpu_baseline": baseline,
        "e2e": {"value": value, "unit": "GCell-updates/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------

def measured_peak_gbs():
    path = ROOT / "MEASURED_PEAKS.json"
    if path.exists():
        try:
            return float(json.loads(path.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_dram_traffic(workload: str, rows: int, cols: int, k: int):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the fused sweep kernel, from the
    `ncu --set full` captures indexed in profiles/dram_traffic.json (written by
    scripts/ncu_summary.py from the committed summaries; a run under ncu is never a bench value, so
    this cannot be measured inside the timed run). None — with the reason — where no capture of this
    exact configuration (grid, fusion depth) exists."""
    index = ROOT / "profiles" / "dram_traffic.json"
    if not index.exists():
        return None, "no profiles/dram_traffic.json"
    for entry in json.loads(index.read_text()):
        if (entry["workload"], entry["rows"], entry["cols"], entry["fused_iterations"]) == \
                (workload, rows, cols, k):
            return float(entry["dram_bytes_per_launch"]), entry["source"]
    return None, f"no ncu capture of {workload} {rows}x{cols} k={k} in profiles/dram_traffic.json"


class Context:
    """Process-wide state shared by the workloads measured in one invocation."""

    def __init__(self, rank, world, local_rank):
        self.rank, self.world, self.device = rank, world, local_rank
        os.environ["STST_DEVICE"] = str(self.device)
        self.dist = None
        self.placement = None
        if world > 1 and os.environ.get("STST_BIND_NUMA", "1") != "0":
            # every rank next to its GPU: host threads (and, by first touch, the pinned cell images)
            # on the cores of the GPU's NUMA node
            from stencilstream_b200.affinity import bind_to_gpu_numa_node
            self.placement = bind_to_gpu_numa_node(self.device)
        if world > 1:
            import torch
            import torch.distributed as dist_mod
            torch.cuda.set_device(self.device)
            dist_mod.init_process_group("nccl", device_id=torch.device("cuda", self.device))
            self.dist = dist_mod

    def max_over_ranks(self, value: float) -> float:
        if self.dist is None:
            return value
        import torch
        t = torch.tensor([value], dtype=torch.float64, device=f"cuda:{self.device}")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def gather(self, obj):
        if self.dist is None:
            return [obj]
        out = [None] * self.world
        self.dist.all_gather_object(out, obj)
        return out

    def close(self):
        if self.dist is not None:
            self.dist.destroy_process_group()


def measure(args, ctx: Context, cpu_seconds: float = 12.0, parity: bool = True, dump=None):
    """One workload, measured as the module docstring says. Collective; rank 0 gets the record.
    `dump` = (directory, name, byte budget): where --dump-outputs writes the last timed step's cells."""
    from stencilstream_b200 import Grid, Params, StencilUpdate, workload_info
    from stencilstream_b200 import _native

    rank, world, device, dist = ctx.rank, ctx.world, ctx.device, ctx.dist
    workload = args.workload
    cols, iters, scaling = args.cols, args.iterations, args.scaling
    rows, total_rows = resolve_rows(args, world, rank)
    info = workload_info(workload)
    params, halo, fill = make_workload(workload, total_rows, cols)
    dtype = _native.CELL_DTYPES[workload]

    runner = None
    # Slabs whose host image would not fit comfortably into (pinned) host memory are generated and
    # transferred in chunks of rows; that path uses the slab object on a single GPU as well.
    slab_bytes = rows * cols * dtype.itemsize
    chunked = slab_bytes > (args.chunk_above_gib << 30)
    chunk_rows = max(1, min(rows, (256 << 20) // (cols * dtype.itemsize)))
    if world > 1 or chunked:
        from stencilstream_b200.sharding import ShardedStencilUpdate
        runner = ShardedStencilUpdate(
            workload, Params(transition_function=params, halo_value=halo, n_iterations=iters,
                             blocking=False, fused_iterations=args.fuse),
            total_rows, cols, rank=rank, world=world, device=device, comm=dist,
            overlap=not args.no_overlap)
        timer = StreamTimer(device, record=runner.slab.record_event, sync=runner.synchronize)
    else:
        timer = StreamTimer(device)

    def barrier():
        timer.sync()
        if dist is not None:
            dist.barrier()
            import torch
            torch.cuda.synchronize()

    host_memory = {"kind": "pinned"}
    pinned_blocks = []

    def pinned_cells(n_rows):
        """A numpy view of pinned host memory for n_rows x cols cells (pageable if the box refuses
        to pin that much)."""
        ptr = C.c_void_p()
        n_bytes = n_rows * cols * dtype.itemsize
        if timer.rt.stst_malloc_host(n_bytes, C.byref(ptr)) != 0:
            host_memory["kind"] = "pageable (cudaHostAlloc failed: " + \
                timer.rt.stst_last_error().decode()[-40:] + ")"
            return np.empty((n_rows, cols), dtype=dtype)
        pinned_blocks.append(ptr)
        raw = (C.c_ubyte * n_bytes).from_address(ptr.value)
        return np.frombuffer(raw, dtype=dtype, count=n_rows * cols).reshape(n_rows, cols)

    # ---- resident-data measurement ------------------------------------------------------------------
    if runner is None:
        grid = Grid(workload, rows, cols, device=device)
        view = grid.accessor("write")
        fill(view, 0, rows, rows)
        del view
        grid.sync_to_device()
        update = StencilUpdate(workload, Params(transition_function=params, halo_value=halo,
                                                n_iterations=iters, blocking=False,
                                                fused_iterations=args.fuse))

        def step():
            return update(grid)

        def n_launches():
            return update.get_n_launches()
    elif chunked:
        host_in = pinned_cells(chunk_rows)

        def generate(lo, hi):
            fill(host_in[:hi - lo], lo, hi, total_rows)
            if hasattr(fill, "assume_zeroed"):   # same buffer next time, only this function wrote it
                fill.assume_zeroed = True
            return host_in[:hi - lo]
        runner.load_chunks(generate, chunk_rows)
        runner.synchronize()
        if hasattr(fill, "assume_zeroed"):
            fill.assume_zeroed = False
    else:
        host_in = pinned_cells(rows)
        fill(host_in, runner.row_lo, runner.row_hi, total_rows)
        runner.load(host_in)
        runner.synchronize()

    if runner is not None:
        def step():
            return runner()

        def n_launches():
            return runner.get_n_launches()

    for _ in range(args.warmup):
        out = step()
    barrier()
    launches_before = n_launches()
    with ClockSampler(device) as clocks:
        timer.begin()
        for _ in range(args.steps):
            out = step()
        elapsed_ms = timer.end_ms()
        barrier()
    launches = n_launches() - launches_before
    if dump is not None:
        dump_dir, dump_name, dump_budget = dump
        rows_idx, cols_idx = dump_sample(total_rows, cols, dtype, dump_budget)
        if runner is None:
            # Grid has no row-range download; the whole result is a temporary here, as it is for the
            # end-to-end phase below, which downloads the same grid
            sample = out.to_numpy()[np.ix_(rows_idx, cols_idx)]
        else:   # only the sampled rows leave the device (a slab may be tens of GB)
            mine = rows_idx[(rows_idx >= runner.row_lo) & (rows_idx < runner.row_hi)]
            owned = np.empty((len(mine), cols), dtype=dtype)
            for i, row in enumerate(mine):
                runner.slab.copy_rows_to_host(int(row) - runner.row_lo, owned[i:i + 1])
            sample = np.concatenate(ctx.gather(owned[:, cols_idx]))
        if rank == 0:
            write_dump(dump_dir, dump_name, sample)
    del out
    elapsed_ms = ctx.max_over_ranks(elapsed_ms)

    total_cells = total_rows * cols
    ms_per_step = elapsed_ms / args.steps
    value = total_cells * iters / (ms_per_step * 1e-3) / 1e9

    stats = update.get_stats() if runner is None else runner.info()
    k = int(stats.fused_iterations)
    plan = {"fused_iterations": k, "tile": [int(stats.tile_h), int(stats.tile_w)],
            "block": [int(stats.block_x), int(stats.block_y)],
            "tma": bool(stats.use_tma), "smem_bytes": int(stats.smem_bytes),
            "passthrough_planes": int(stats.passthrough_planes),
            "speculation_redos": int(stats.speculation_redos if runner is None
                                     else runner.n_speculation_redos)}

    # ---- roofline of the fused sweep kernel -----------------------------------------------------------
    peak, peak_source = measured_peak_gbs()
    # One pass (all launches that together advance the rank's rows by <= k iterations) per k iterations.
    launches_per_step = -(-iters // k)
    # One launch advances this rank's rows*cols cells by (iters / launches_per_step) iterations on average.
    bytes_per_launch = info.bytes_per_cell_iteration * rows * cols * iters / launches_per_step
    launch_ms = ms_per_step / launches_per_step
    achieved = bytes_per_launch / (launch_ms * 1e-3) / 1e9
    traffic, traffic_source = measured_dram_traffic(workload, rows, cols, k)
    roofline = {
        "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "traffic": traffic, "traffic_source": traffic_source,
        "physical_frac": (traffic / (launch_ms * 1e-3) / 1e9 / peak) if traffic else None,
        "algorithmic_bytes_per_launch": bytes_per_launch, "peak_source": peak_source,
        "kernel": "fused_sweep_kernel", "fused_iterations": k,
        "algorithmic_bytes_per_cell_iteration": int(info.bytes_per_cell_iteration),
        "note": "effective fraction: k fused iterations cross HBM once, so it may exceed the physical "
                "DRAM fraction (physical_frac = ncu DRAM bytes per launch / launch time / peak)",
    }

    # ---- end-to-end through the public API, host buffers in pinned memory -----------------------------
    e2e = None
    parity_record = None
    e2e_steps = max(1, min(args.steps, 3))
    if runner is None:
        # Boxes cap pinnable host memory (this pool: ~4 GiB): give the resident grid's pinned image
        # back to the runtime's cache before the end-to-end grids ask for theirs.
        del grid, update
        host_grid = Grid(workload, rows, cols, device=device)
        e2e_update = StencilUpdate(workload, Params(transition_function=params, halo_value=halo,
                                                    n_iterations=iters, blocking=True,
                                                    fused_iterations=args.fuse))
        times = []
        for i in range(1 + e2e_steps):
            view = host_grid.accessor("write")      # pinned host image; marks the device copy stale
            if i == 0:
                fill(view, 0, rows, rows)
            del view
            timer.sync()
            t0 = time.perf_counter()
            result = e2e_update(host_grid)          # H2D upload + layout + all fused launches
            view = result.accessor("read")          # D2H of the whole result grid
            mid = view[rows // 2, cols // 2]
            checksum = float(mid[dtype.names[0]] if dtype.names else mid)
            t1 = time.perf_counter()
            images_pinned = (host_grid.host_image_is_pinned(), result.host_image_is_pinned())
            if i > 0:
                times.append(t1 - t0)
            if i == e2e_steps and parity and rank == 0:
                # the result this step downloaded = `iters` iterations from the synthetic input
                parity_record = check_parity_window(workload, params, halo, fill, total_rows, cols,
                                                    iters, 0, rows, view)
            # `mid` of a struct cell is a numpy.void that references the accessor view, which keeps the
            # result grid and its pinned image alive: drop all of them before the next step allocates
            del mid, view, result
        e2e_value = total_cells * iters / float(np.mean(times)) / 1e9
        e2e = {"value": e2e_value, "unit": "GCell-updates/s", "steps": e2e_steps,
               "h2d_bytes_per_step": int(rows * cols * dtype.itemsize),
               "d2h_bytes_per_step": int(rows * cols * dtype.itemsize),
               "ms_per_step": float(np.mean(times) * 1e3), "checksum": checksum,
               "host_memory": "pinned" if all(images_pinned) else
                              "pageable, staged through the runtime's pinned ring (input pinned: %s, "
                              "result pinned: %s)" % images_pinned}
        del host_grid, e2e_update
    else:
        # Per rank: owned rows from pinned host memory -> slab (H2D + layout + halo exchange), the
        # update, owned rows back into pinned host memory. Wall clock between barriers, max over ranks.
        host_out = host_in  # results overwrite the inputs: one host buffer per rank (boxes cap
        runner.get_params().blocking = True  # pinnable memory at a few GiB per process)
        if chunked:
            e2e_steps = 1
        times = []
        for i in range(1 + e2e_steps):
            if i == e2e_steps and parity and not chunked:
                # the last step starts from the synthetic input again (untimed refill), so that what
                # it downloads is `iters` iterations from a known state: the parity window below
                fill(host_in, runner.row_lo, runner.row_hi, total_rows)
            barrier()
            t0 = time.perf_counter()
            if chunked:  # the same pinned chunk buffer is the source and sink of every chunk
                runner.load_chunks(lambda lo, hi: host_in[:hi - lo], chunk_rows)
                runner()
                for lo in range(0, rows, chunk_rows):
                    n = min(chunk_rows, rows - lo)
                    runner.slab.copy_rows_to_host(lo, host_in[:n])
            else:
                runner.load(host_in)
                runner()
                runner.to_numpy(host_out)
            t1 = time.perf_counter()
            step_seconds = ctx.max_over_ranks(t1 - t0)
            if i > 0:
                times.append(step_seconds)
        mid = host_out[min(rows // 2, host_out.shape[0] - 1), cols // 2]
        checksum = float(mid[dtype.names[0]] if dtype.names else mid)
        e2e = {"value": total_cells * iters / float(np.mean(times)) / 1e9, "unit": "GCell-updates/s",
               "steps": e2e_steps, "h2d_bytes_per_step": int(rows * cols * dtype.itemsize) * world,
               "d2h_bytes_per_step": int(rows * cols * dtype.itemsize) * world,
               "ms_per_step": float(np.mean(times) * 1e3), "checksum": checksum,
               "host_memory": host_memory["kind"]}
        if parity and not chunked:
            # host_out = this rank's rows after `iters` iterations from the synthetic input; the rank
            # that owns the window checks it (its domain of dependence crosses the slab seams)
            mine = check_parity_window(workload, params, halo, fill, total_rows, cols, iters,
                                       runner.row_lo, runner.row_hi, host_out)
            records = [r for r in ctx.gather(mine) if r is not None]
            checked = [r for r in records if r.get("rel_max_norm") is not None]
            parity_record = (checked or records or [None])[0]
            if len(checked) > 1:   # the window straddles a seam: report the worse half
                parity_record = max(checked, key=lambda r: r["rel_max_norm"])
                parity_record["window_parts"] = [r["window"] for r in checked]
        elif parity:
            parity_record = {"rel_max_norm": None,
                             "skipped": "slab moved chunk by chunk through one host buffer; covered by "
                                        "tests/test_parity_fullsize_gpu.py"}
        del mid, host_out
        barrier()
        runner.close()
    for ptr in pinned_blocks:
        timer.rt.stst_free_host(ptr)
    timer.rt.stst_host_cache_trim()

    cpu_baseline = None
    if rank == 0 and world == 1 and cpu_seconds > 0:
        cpu_baseline, _ = time_cpu_oracle(workload, rows, cols, total_rows, target_seconds=cpu_seconds)
        if workload == "hotspot":
            cpu_baseline["rodinia_openmp"] = time_rodinia_hotspot()

    if rank != 0:
        return None
    return {
        "metric": "GCell-updates/s", "value": value, "unit": "GCell-updates/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
        "dtype": DTYPE.get(workload, "f32"), "data": "synthetic",
        "config": workload_config(workload, total_rows, rows, cols, iters, world),
        "plan": plan,
        "roofline": roofline,
        "pct_of_hbm_roofline_8TBps": 100.0 * value * info.bytes_per_cell_iteration / world / 8000.0,
        "cpu_baseline": cpu_baseline,
        "e2e": e2e,
        "parity": parity_record,
        "gpu_launches": int(launches),
        "clocks": clocks.summary(),
        "host_placement": ctx.placement,
    }


# The other BASELINE.json configs, measured after the headline workload by the default invocation:
# (key, workload, rows, cols, iterations per step, scaling, only if world > 1)
SECONDARY = [
    ("hotspot_16384_strong", "hotspot", 16384, 16384, 1000, "strong", False),
    ("hotspot_16384_per_gpu_weak", "hotspot", 16384, 16384, 1000, "weak", True),
    ("fdtd_max_grid_strong", "fdtd", 4608, 4608, 1000, "strong", False),
    ("convection_8192x65536_per_gpu_weak", "convection_pt", 8192, 65536, 20, "weak", False),
]


def dump_target(args, name: str, budget: int):
    return (Path(args.dump_outputs), name, budget) if args.dump_outputs else None


def run_ours(args, ctx: Context, default_invocation: bool):
    secondary = [s for s in SECONDARY if not (s[6] and ctx.world == 1)] \
        if default_invocation and not args.headline_only else []
    budget = DUMP_BYTES // (1 + len(secondary))
    line = measure(args, ctx, dump=dump_target(args, args.workload, budget))
    if secondary:
        import copy
        import gc
        workloads = {}
        for key, workload, rows, cols, iters, scaling, _ in secondary:
            sub = copy.copy(args)
            sub.workload, sub.rows, sub.cols, sub.iterations, sub.scaling = workload, rows, cols, iters, scaling
            sub.fuse = 0
            gc.collect()
            try:
                record = measure(sub, ctx, cpu_seconds=4.0, dump=dump_target(args, key, budget))
            except Exception as exc:  # keep the headline line even if a secondary workload fails
                record = {"error": f"{type(exc).__name__}: {exc}"[:300]}
            if ctx.rank == 0:
                for drop in ("metric", "unit", "higher_is_better", "vs_baseline", "data"):
                    record.pop(drop, None)
                workloads[key] = record
        if ctx.rank == 0:
            line["workloads"] = workloads
    if ctx.rank == 0:
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="", choices=[""] + sorted(WORKLOAD_LABEL),
                    help="measure only this workload (default: the headline Jacobi workload plus the "
                         "other BASELINE.json configs under `workloads`)")
    ap.add_argument("--rows", type=int, default=0,
                    help="rows per GPU (weak scaling) or of the whole grid (strong scaling)")
    ap.add_argument("--cols", type=int, default=0)
    ap.add_argument("--iterations", type=int, default=0, help="iterations per step")
    ap.add_argument("--scaling", default="", choices=["", "weak", "strong"])
    ap.add_argument("--fuse", type=int, default=0, help="fused iterations per launch (0 = planner)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--headline-only", action="store_true",
                    help="default invocation without the `workloads` section")
    ap.add_argument("--chunk-above-gib", type=int, default=4,
                    help="slabs larger than this many GiB are generated/transferred in row chunks")
    ap.add_argument("--no-overlap", action="store_true",
                    help="multi-GPU: one launch per pass instead of boundary-first scheduling")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the cells the last timed step returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the GPU implementation's outputs (--impl ours)")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world and world > 1:
        args.gpus = world

    default_invocation = args.workload == "" and not (args.rows or args.cols or args.iterations)
    args.workload = args.workload or "jacobi5"
    d_rows, d_cols, d_iters, d_scaling = DEFAULTS[args.workload]
    args.rows = args.rows or d_rows
    args.cols = args.cols or d_cols
    args.iterations = args.iterations or d_iters
    args.scaling = args.scaling or d_scaling

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    ctx = Context(rank, world, local_rank)
    try:
        if default_invocation:
            run_ours(args, ctx, True)
        else:
            line = measure(args, ctx, cpu_seconds=0.0 if args.no_cpu_baseline else 12.0,
                           dump=dump_target(args, args.workload, DUMP_BYTES))
            if rank == 0:
                print(json.dumps(line), flush=True)
    finally:
        ctx.close()


if __name__ == "__main__":
    main()
