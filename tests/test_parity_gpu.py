"""GPU parity tests: the sm_100a generation loop (through the C ABI) against the CPU oracle.

Bars (BASELINE.json north_star): bit-exact for Conway and the integer self-checking functor; fp32/fp64
workloads within 1e-5 relative max-norm in the default build (nvcc contracts a*b+c into FMAs, the
oracle is built with -ffp-contract=off) and bit-exact in the -fmad=false ("strict") build.
"""
import numpy as np
import pytest

import cases
from stencilstream_b200 import Grid, Params, RangeError, StencilUpdate, workload_info

pytestmark = pytest.mark.gpu

FP_TOLERANCE = 1e-5  # relative max-norm, BASELINE.json

BIT_EXACT = {"conway", "kat", "kat_r2"}
ALL = ["conway", "jacobi5", "jacobi9", "jacobi_r2", "jacobi_r3", "hotspot", "fdtd", "convection_pt",
       "convection_thermal", "kat", "kat_r2"]


def run_gpu(workload, params, halo, cells, offset, n, strict=False, **extra):
    grid = Grid(workload, buffer=cells, strict=strict)
    update = StencilUpdate(workload, Params(transition_function=params, halo_value=halo,
                                            iteration_offset=offset, n_iterations=n, blocking=True,
                                            **extra), strict=strict)
    out = update(grid)
    return out.to_numpy(), update


def check(workload, got, want, strict):
    if workload in BIT_EXACT or strict:
        assert got.tobytes() == want.tobytes(), f"{workload}: not bit-exact"
    else:
        err = cases.rel_max_norm(got, want)
        assert err <= FP_TOLERANCE, f"{workload}: relative max-norm {err:g} > {FP_TOLERANCE:g}"


@pytest.mark.parametrize("workload", ALL)
@pytest.mark.parametrize("strict", [False, True], ids=["fma", "strict"])
def test_small_grid_matches_oracle(workload, strict, oracle_best):
    rows, cols = 67, 93  # ragged: not a multiple of any tile or vector width
    params, halo, cells = cases.make_case(workload, rows, cols, seed=1)
    n = 5
    want = oracle_best.run(workload, params, halo, cells, 2 if "kat" not in workload else 0, n)
    got, _ = run_gpu(workload, params, halo, cells, 2 if "kat" not in workload else 0, n, strict)
    check(workload, got, want, strict)


@pytest.mark.parametrize("workload", ["jacobi5", "hotspot", "fdtd", "kat", "conway", "jacobi_r3"])
@pytest.mark.parametrize("fused", [1, 2, 3, 4, 7])
def test_every_fusion_depth_matches_oracle(workload, fused, oracle_best):
    """k = 1 .. 7 fused iterations with n = k, k+1 and n < k (tail launches), mirroring the
    reference's tiling tests (tests/tiling/StencilUpdate.cpp:57-104: n = T, T+1; offsets 0/1)."""
    rows, cols = 150, 530  # several tiles in both directions, ragged edges
    params, halo, cells = cases.make_case(workload, rows, cols, seed=2)
    for n in sorted({fused, fused + 1, max(1, fused - 1), 2 * fused + 1}):
        want = oracle_best.run(workload, params, halo, cells, 0, n)
        got, update = run_gpu(workload, params, halo, cells, 0, n, strict=True, fused_iterations=fused)
        k = update.get_stats().fused_iterations
        assert 1 <= k <= min(fused, n)
        if workload != "fdtd":  # 32-byte cells: depth 7 does not fit into shared memory
            assert k == min(fused, n)
        check(workload, got, want, strict=True)


@pytest.mark.parametrize("shape", [(1, 1), (1, 40), (40, 1), (2, 3), (31, 33), (64, 64), (257, 255)])
def test_degenerate_and_odd_shapes(shape, oracle_best):
    for workload in ("jacobi5", "hotspot", "kat"):
        params, halo, cells = cases.make_case(workload, *shape, seed=3)
        want = oracle_best.run(workload, params, halo, cells, 0, 3)
        got, _ = run_gpu(workload, params, halo, cells, 0, 3, strict=True)
        check(workload, got, want, strict=True)


@pytest.mark.parametrize("split", [False, True])
@pytest.mark.parametrize("case", [(64, 64, 0, 1), (64, 64, 0, 1), (64, 64, 32, 64), (32, 64, 0, 1),
                                  (64, 32, 0, 1)])
def test_reference_stencil_update_cases(case, split):
    """The reference's own cuda StencilUpdate test matrix (tests/cuda/StencilUpdate.cpp:30-50, driven by
    tests/StencilUpdateTest.hpp:30-63). `split` has no effect on this backend; both run."""
    rows, cols, offset, n = case
    cells = cases.kat_input(rows, cols, offset)
    got, update = run_gpu("kat", None, cases.KAT_HALO, cells, offset, n)
    want = cases.kat_expected(rows, cols, offset, n)
    assert got.tobytes() == want.tobytes()
    assert update.get_n_processed_cells() == n * rows * cols


def test_conway_1024_256_generations_bit_exact(oracle_best):
    """BASELINE.json configs[0]: Conway 1024x1024, 256 generations, bit-exact."""
    params, halo, cells = cases.make_case("conway", 1024, 1024)
    want = oracle_best.run("conway", params, halo, cells, 0, 256)
    got, _ = run_gpu("conway", params, halo, cells, 0, 256)
    assert got.tobytes() == want.tobytes()
    assert got.sum() > 0  # the soup is still alive


def test_source_grid_is_not_modified_and_result_is_new():
    params, halo, cells = cases.make_case("jacobi5", 96, 96)
    grid = Grid("jacobi5", buffer=cells)
    update = StencilUpdate("jacobi5", Params(transition_function=params, halo_value=halo,
                                             n_iterations=9, blocking=True))
    out = update(grid)
    assert grid.to_numpy().tobytes() == cells.tobytes()
    assert out.to_numpy().tobytes() != cells.tobytes()


def test_iteration_offset_resume_equals_one_shot(oracle_best):
    """Resuming with iteration_offset (reference :67-73; FDTD snapshots fdtd.cpp:233-242) gives the
    same grid as one call — exercised with the TDV-dependent FDTD functor."""
    params, halo, cells = cases.make_case("fdtd", 80, 76)
    one_shot, _ = run_gpu("fdtd", params, halo, cells, 0, 30, strict=True)
    grid = Grid("fdtd", buffer=cells, strict=True)
    update = StencilUpdate("fdtd", Params(transition_function=params, halo_value=halo,
                                          n_iterations=10, blocking=True), strict=True)
    for _ in range(3):
        grid = update(grid)
        update.get_params().iteration_offset += 10  # live reference, as fdtd.cpp:236 mutates it
    assert grid.to_numpy().tobytes() == one_shot.tobytes()
    want = oracle_best.run("fdtd", params, halo, cells, 0, 30)
    assert one_shot.tobytes() == want.tobytes()


def test_grid_contract():
    """tests/GridTest.hpp of the reference, restated: constructors, buffer round trips,
    make_similar, size-mismatch errors."""
    rows, cols = 128, 128
    info = workload_info("kat")
    assert info.cell_bytes == 20
    cells = cases.kat_input(rows, cols, 7)
    grid = Grid("kat", rows, cols)
    assert grid.get_grid_range() == (rows, cols)
    grid.copy_from_buffer(cells)
    back = np.empty_like(cells)
    grid.copy_to_buffer(back)
    assert back.tobytes() == cells.tobytes()
    similar = grid.make_similar()
    assert similar.get_grid_range() == (rows, cols)
    with pytest.raises(RangeError):
        grid.copy_from_buffer(cells[:-1])
    with pytest.raises(RangeError):
        grid.copy_to_buffer(np.empty((rows, cols + 1), dtype=cells.dtype))
    shared = grid.share()
    shared.copy_from_buffer(cases.kat_input(rows, cols, 9))
    assert grid.to_numpy()["i_iteration"][0, 0] == 9  # handles share storage (Grid.hpp:97)


def test_zero_iterations_returns_same_cells():
    params, halo, cells = cases.make_case("jacobi5", 40, 40)
    got, _ = run_gpu("jacobi5", params, halo, cells, 0, 0)
    assert got.tobytes() == cells.tobytes()


def test_tma_and_cp_async_staging_agree(monkeypatch):
    params, halo, cells = cases.make_case("hotspot", 300, 700, seed=5)
    outs = []
    for tma in ("1", "0"):
        monkeypatch.setenv("STST_TMA", tma)
        got, update = run_gpu("hotspot", params, halo, cells, 0, 6, strict=True)
        assert update.get_stats().use_tma == int(tma)
        outs.append(got)
    assert outs[0].tobytes() == outs[1].tobytes()


# ---- speculative plane pass-through (StencilUpdate::run_detected, run_tile in TileKernel.hpp) ----

def test_passthrough_planes_are_detected():
    """HotSpot never changes `power`, FDTD never changes its four material coefficients: after the
    observing launch the sweeps leave those planes in place (and results stay bit-exact, which every
    other test in this file checks with the speculation active)."""
    params, halo, cells = cases.make_case("hotspot", 200, 300, seed=8)
    _, update = run_gpu("hotspot", params, halo, cells, 0, 12, strict=True)
    stats = update.get_stats()
    assert stats.passthrough_planes == 0b10 and stats.speculation_redos == 0
    params, halo, cells = cases.make_case("fdtd", 120, 130, seed=8)
    _, update = run_gpu("fdtd", params, halo, cells, 0, 6, strict=True)   # before detect_iteration
    assert update.get_stats().passthrough_planes & 0b11110000 == 0b11110000
    # single-plane cells have nothing to pass through
    params, halo, cells = cases.make_case("jacobi5", 64, 64)
    _, update = run_gpu("jacobi5", params, halo, cells, 0, 4)
    assert update.get_stats().passthrough_planes == 0


def test_wrong_speculation_is_repeated_without_it(oracle_best):
    """FDTD's `hz_sum` only starts to change at `detect_iteration` (10 in this case): an updater
    that observed iterations 0..k-1 believes the plane passes through, a later launch reports the
    change, and the call is recomputed from the untouched source grid. Results must equal the
    oracle's bit for bit, for the violating call and for the calls after it."""
    params, halo, cells = cases.make_case("fdtd", 90, 100, seed=12)
    want = oracle_best.run("fdtd", params, halo, cells, 0, 30)
    grid = Grid("fdtd", buffer=cells, strict=True)
    update = StencilUpdate("fdtd", Params(transition_function=params, halo_value=halo,
                                          n_iterations=30, blocking=True, fused_iterations=2),
                           strict=True)
    out = update(grid)
    stats = update.get_stats()
    assert stats.speculation_redos >= 1
    assert stats.passthrough_planes & 0b1000 == 0          # hz_sum (field 3) is no longer trusted
    assert stats.passthrough_planes & 0b11110000 == 0b11110000
    assert out.to_numpy().tobytes() == want.tobytes()
    assert grid.to_numpy().tobytes() == cells.tobytes()     # the source grid survived the repeat
    update.get_params().iteration_offset = 30
    update.get_params().n_iterations = 7
    again = update(out)
    want2 = oracle_best.run("fdtd", params, halo, want, 30, 7)
    assert again.to_numpy().tobytes() == want2.tobytes()
    assert update.get_stats().speculation_redos == stats.speculation_redos


def test_speculation_can_be_switched_off(monkeypatch, oracle_best):
    """STST_SPECULATE=0 is read once per process, so this only checks that both settings give the
    oracle's result in whichever mode this process runs; the mode itself is covered by the stats
    assertions above."""
    params, halo, cells = cases.make_case("convection_pt", 64, 72, seed=2)
    want = oracle_best.run("convection_pt", params, halo, cells, 0, 5)
    got, update = run_gpu("convection_pt", params, halo, cells, 0, 5, strict=True)
    assert got.tobytes() == want.tobytes()
    # 88-byte cells have no pass-through kernels (and T, the only field this kernel never writes,
    # would be 8 of 88 bytes, below the profitability threshold): the plain kernels run
    assert update.get_stats().passthrough_planes == 0
