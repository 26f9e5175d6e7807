"""Host logic of scripts/benchmark.py (the counterpart of the reference's Julia benchmark drivers):
grid-size ladder and roofline model, no GPU."""
import importlib.util
import math
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
spec = importlib.util.spec_from_file_location("stst_benchmark_driver", ROOT / "scripts" / "benchmark.py")
driver = importlib.util.module_from_spec(spec)
spec.loader.exec_module(driver)


def test_max_grid_wh_follows_the_reference_rule():
    # scripts/benchmark-common.jl:186-199 for the A100 (40 GiB): three HotSpot grids in memory,
    # clipped to a power of sqrt(2) / of 2
    assert driver.max_grid_wh(8, 40 * 2 ** 30, clip_to_base=math.sqrt(2)) == 32768
    assert driver.max_grid_wh(8, 40 * 2 ** 30, clip_to_base=2) == 32768
    assert driver.max_grid_wh(8, 40 * 2 ** 30) == int(math.sqrt(40 * 2 ** 30 / 3 / 8))
    # 180 GB of HBM: the 2^31-cell indexing limit binds for 4-byte cells
    assert driver.max_grid_wh(4, 180e9) == int(math.sqrt(2 ** 31))


def test_model_runtime_is_bandwidth_or_launch_bound():
    bw = 6.4e12
    big = driver.model_runtime(16384, 16384, 1000, 4, 1, 1, bw)
    assert math.isclose(big, 1000 * 2 * 4 * 16384 ** 2 / bw)
    fused = driver.model_runtime(16384, 16384, 1000, 4, 1, 6, bw)
    assert math.isclose(fused, math.ceil(1000 / 6) * 2 * 4 * 16384 ** 2 / bw)
    tiny = driver.model_runtime(32, 32, 1000, 4, 1, 1, bw)            # launch-latency bound
    assert math.isclose(tiny, 1000 * driver.SCHEDULING_LATENCY_PER_PASS)


def test_operation_counts_are_the_reference_drivers():
    assert driver.OPERATIONS_PER_CELL == {"jacobi5": 9, "hotspot": 15, "fdtd": 24, "convection_pt": 67}


# ---- bench.py host logic (no GPU) -------------------------------------------------------------------

def _bench():
    spec2 = importlib.util.spec_from_file_location("stst_bench", ROOT / "bench.py")
    mod = importlib.util.module_from_spec(spec2)
    spec2.loader.exec_module(mod)
    return mod


def test_bench_inputs_are_the_reference_recipes_and_slab_wise_generation_agrees():
    """bench.py fills slabs row range by row range; stitched together they must be the whole-grid
    inputs of stencilstream_b200.workloads (which restate the reference's generators)."""
    import numpy as np
    from stencilstream_b200 import _native
    from stencilstream_b200 import workloads as W
    bench = _bench()
    rows, cols = 96, 80
    for workload, whole in (("jacobi5", W.jacobi_input(rows, cols)),
                            ("jacobi_r2", W.jacobi_input(rows, cols)),
                            ("hotspot", W.hotspot_input(rows, cols))):
        _, _, fill = bench.make_workload(workload, rows, cols)
        stitched = np.zeros((rows, cols), dtype=_native.CELL_DTYPES[workload])
        for lo, hi in ((0, 31), (31, 64), (64, 96)):
            fill(stitched[lo:hi], lo, hi, rows)
        assert stitched.tobytes() == whole.tobytes(), workload
    exp = W.ConvectionExperiment(W.convection_benchmark_config(res=64, n_iters=1, lx=1.5, ly=1.0))
    _, _, fill = bench.make_workload("convection_pt", *exp.grid_shape)
    stitched = np.zeros(exp.grid_shape, dtype=_native.CELL_DTYPES["convection_pt"])
    fill(stitched[:40], 0, 40, exp.grid_shape[0])
    fill(stitched[40:], 40, exp.grid_shape[0], exp.grid_shape[0])
    assert stitched.tobytes() == exp.initial_grid().tobytes()


def test_bench_roofline_traffic_comes_from_the_committed_capture():
    bench = _bench()
    traffic, source = bench.measured_dram_traffic("jacobi5", 16384, 16384, 6)
    assert source and (ROOT / source).exists()
    # one read and one write of a 1 GiB grid per launch, within 5 % (halo re-reads hit L2; the last
    # dirty lines are still in L2 when the kernel ends)
    assert abs(traffic / (2 * 2 ** 30) - 1.0) < 0.05
    # a configuration without a capture reports None and says why (never a number of another plan)
    none, why = bench.measured_dram_traffic("jacobi5", 16384, 16384, 4)
    assert none is None and "no ncu capture" in why
    # every index entry points at a committed summary
    import json
    for entry in json.loads((ROOT / "profiles" / "dram_traffic.json").read_text()):
        assert (ROOT / entry["source"]).exists(), entry


def test_bench_parity_window_agrees_with_a_whole_grid_oracle_run(oracle_best, monkeypatch):
    """bench.py's `parity` record: the window check it runs after the end-to-end steps must report
    zero for the oracle's own whole-grid result and a clear failure for a perturbed one. (The result
    handed in here is the UNcontracted oracle's, i.e. what the -fmad=false build produces: with
    STST_STRICT=1 that oracle is the checker; without, it is the one reported beside the contracted
    checker.)"""
    import numpy as np
    import bench
    import oracle

    monkeypatch.setenv("STST_STRICT", "1")

    rows = cols = 256
    iters = 12
    for workload in ("jacobi5", "hotspot"):
        params, halo, fill = bench.make_workload(workload, rows, cols)
        from stencilstream_b200 import _native
        cells = np.empty((rows, cols), dtype=_native.CELL_DTYPES[workload])
        fill(cells, 0, rows, rows)
        whole = oracle_best.run(workload, params, halo, cells, 0, iters)
        record = bench.check_parity_window(workload, params, halo, fill, rows, cols, iters, 0, rows, whole)
        assert record["rel_max_norm"] == 0.0 and record["ok"], record
        assert record["window"] == [[32, 96], [32, 96]]
        # a slab that owns only the lower half of the window checks that half
        half = bench.check_parity_window(workload, params, halo, fill, rows, cols, iters, 64, 128,
                                         whole[64:128])
        assert half["window"][0] == [64, 96] and half["rel_max_norm"] == 0.0
        # rows outside the window: nothing to check
        assert bench.check_parity_window(workload, params, halo, fill, rows, cols, iters, 128, 256,
                                         whole[128:]) is None
        broken = whole.copy()
        field = broken[broken.dtype.names[0]] if broken.dtype.names else broken
        field[64, 64] *= 1.001
        bad = bench.check_parity_window(workload, params, halo, fill, rows, cols, iters, 0, rows, broken)
        assert not bad["ok"] and bad["rel_max_norm"] > 1e-5
    if oracle.cpu_has_fma():
        monkeypatch.setenv("STST_STRICT", "0")
        record = bench.check_parity_window(workload, params, halo, fill, rows, cols, iters, 0, rows, whole)
        assert "contracting" in record["oracle_arithmetic"]
        assert record["rel_max_norm_vs_uncontracted_oracle"] == 0.0
        assert record["rel_max_norm"] <= 1e-5       # FMA vs two roundings after 12 iterations


def test_bench_dump_sample_is_fixed_and_within_the_budget(tmp_path):
    """--dump-outputs: the whole grid where it fits, else a seeded rows x columns sample that is the
    same on every call; files are float32 (float64 for 8-byte fields) and stay under the budget."""
    import numpy as np
    from stencilstream_b200 import _native
    bench = _bench()
    rows, cols = bench.dump_sample(300, 200, _native.CELL_DTYPES["hotspot"], 1 << 20)
    assert (rows == np.arange(300)).all() and (cols == np.arange(200)).all()
    for workload in ("jacobi5", "hotspot", "fdtd", "convection_pt", "conway"):
        dtype = _native.CELL_DTYPES[workload]
        budget = bench.DUMP_BYTES // 4
        rows, cols = bench.dump_sample(16384, 65536, dtype, budget)
        again = bench.dump_sample(16384, 65536, dtype, budget)
        assert (rows == again[0]).all() and (cols == again[1]).all()
        assert len(set(rows)) == len(rows) and (np.diff(rows) > 0).all() and rows[-1] < 16384
        assert (np.diff(cols) > 0).all() and cols[-1] < 65536
        for picked, n in ((rows, 16384), (cols, 65536)):   # both borders of the grid are in it
            assert picked[0] == 0 and picked[-1] == n - 1 and len(picked) < n
        cells = np.zeros((len(rows), len(cols)), dtype=dtype)
        bench.write_dump(tmp_path / workload, workload, cells)
        files = sorted((tmp_path / workload).iterdir())
        assert len(files) == max(1, len(dtype.names or ()))
        assert sum(f.stat().st_size for f in files) <= budget + 128 * len(files)
        for f in files:
            assert np.load(f).dtype in (np.float32, np.float64)
            assert np.load(f).shape == (len(rows), len(cols))
    assert np.load(tmp_path / "convection_pt" / "convection_pt.T.npy").dtype == np.float64
    assert np.load(tmp_path / "conway" / "conway.npy").dtype == np.float32


NCU_CSV = '''==PROF== Connected to process 4242 (/usr/bin/python3.12)
jacobi5 k=6 tile=43x240 call 0: 7.5 ms
==PROF== Profiling "fused_sweep_kernel" - 0: 0%....50%....100% - 9 passes
==PROF== Disconnected from process 4242
"ID","Process ID","Process Name","Host Name","Kernel Name","Context","Stream","Block Size","Grid Size","Device","CC","Section Name","Metric Name","Metric Unit","Metric Value"
"0","4242","python3.12","127.0.0.1","void fused_sweep_kernel<Jacobi5Rule, 4, 1, 64, 256, 1, 0>(...)","1","7","(64, 4, 1)","(26358, 1, 1)","0","10.0","Command line profiler metrics","dram__bytes_read.sum","Gbyte","1.07"
"0","4242","python3.12","127.0.0.1","void fused_sweep_kernel<Jacobi5Rule, 4, 1, 64, 256, 1, 0>(...)","1","7","(64, 4, 1)","(26358, 1, 1)","0","10.0","Command line profiler metrics","dram__bytes_write.sum","Gbyte","1.03"
"0","4242","python3.12","127.0.0.1","void fused_sweep_kernel<Jacobi5Rule, 4, 1, 64, 256, 1, 0>(...)","1","7","(64, 4, 1)","(26358, 1, 1)","0","10.0","Command line profiler metrics","l1tex__t_sectors_pipe_lsu_mem_global_op_ld.sum","sector","0"
"0","4242","python3.12","127.0.0.1","void fused_sweep_kernel<Jacobi5Rule, 4, 1, 64, 256, 1, 0>(...)","1","7","(64, 4, 1)","(26358, 1, 1)","0","10.0","Command line profiler metrics","l1tex__t_requests_pipe_lsu_mem_global_op_ld.sum","","0"
"0","4242","python3.12","127.0.0.1","void fused_sweep_kernel<Jacobi5Rule, 4, 1, 64, 256, 1, 0>(...)","1","7","(64, 4, 1)","(26358, 1, 1)","0","10.0","Command line profiler metrics","l1tex__t_sectors_pipe_lsu_mem_global_op_st.sum","sector","33,554,432"
"0","4242","python3.12","127.0.0.1","void fused_sweep_kernel<Jacobi5Rule, 4, 1, 64, 256, 1, 0>(...)","1","7","(64, 4, 1)","(26358, 1, 1)","0","10.0","Command line profiler metrics","l1tex__t_requests_pipe_lsu_mem_global_op_st.sum","","2,097,152"
"0","4242","python3.12","127.0.0.1","void fused_sweep_kernel<Jacobi5Rule, 4, 1, 64, 256, 1, 0>(...)","1","7","(64, 4, 1)","(26358, 1, 1)","0","10.0","GPU Speed Of Light Throughput","DRAM Throughput","%","27.6"
"0","4242","python3.12","127.0.0.1","void fused_sweep_kernel<Jacobi5Rule, 4, 1, 64, 256, 1, 0>(...)","1","7","(64, 4, 1)","(26358, 1, 1)","0","10.0","GPU Speed Of Light Throughput","L1/TEX Cache Throughput","%","71.2"
"0","4242","python3.12","127.0.0.1","void fused_sweep_kernel<Jacobi5Rule, 4, 1, 64, 256, 1, 0>(...)","1","7","(64, 4, 1)","(26358, 1, 1)","0","10.0","GPU Speed Of Light Throughput","L2 Cache Throughput","%","12.9"
"0","4242","python3.12","127.0.0.1","void fused_sweep_kernel<Jacobi5Rule, 4, 1, 64, 256, 1, 0>(...)","1","7","(64, 4, 1)","(26358, 1, 1)","0","10.0","GPU Speed Of Light Throughput","Compute (SM) Throughput","%","64.5"
"0","4242","python3.12","127.0.0.1","void fused_sweep_kernel<Jacobi5Rule, 4, 1, 64, 256, 1, 0>(...)","1","7","(64, 4, 1)","(26358, 1, 1)","0","10.0","Occupancy","Theoretical Occupancy","%","25"
"0","4242","python3.12","127.0.0.1","void fused_sweep_kernel<Jacobi5Rule, 4, 1, 64, 256, 1, 0>(...)","1","7","(64, 4, 1)","(26358, 1, 1)","0","10.0","Occupancy","Achieved Occupancy","%","24.4"
'''


def test_ncu_scraper_extracts_the_reference_figures():
    """scripts/benchmark.py ncu_metrics: the ten figures of the reference's ncu_profile_command
    (scripts/benchmark-common.jl:246-283) out of ncu's CSV, with the profiled program's own output and
    the ==PROF== lines in front of it."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("benchmark_driver", ROOT / "scripts" / "benchmark.py")
    driver = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(driver)
    rows = driver.parse_ncu_csv(NCU_CSV)
    assert len(rows) == 12 and rows[0]["Metric Name"] == "dram__bytes_read.sum"
    figures = driver.scrape_ncu_metrics(rows)
    assert abs(figures["read_volume"] - 1.07e9) < 1 and abs(figures["write_volume"] - 1.03e9) < 1
    assert figures["achieved_occupancy"] == 24.4 and figures["theoretical_occupancy"] == 25
    assert figures["compute_throughput"] == 64.5 and figures["dram_throughput"] == 27.6
    assert figures["l1_throughput"] == 71.2 and figures["l2_throughput"] == 12.9
    assert figures["sectors_per_store_request"] == 16.0 and figures["sectors_per_load_request"] == 0.0
    cmd = driver.ncu_command("hotspot", 16384, 16384, 48)
    assert cmd[0] == "ncu" and "--csv" in cmd and "regex:fused_sweep_kernel" in cmd
    assert set(figures) >= {"achieved_occupancy", "compute_throughput", "dram_throughput", "l1_throughput",
                            "l2_throughput", "theoretical_occupancy", "read_volume", "write_volume",
                            "sectors_per_load_request", "sectors_per_store_request"}
