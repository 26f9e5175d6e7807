"""Grid batches (cuda/GridBatch.hpp, fused_sweep_batch_kernel): B members of one extent advanced by one
launch per fused pass. Every member must come out as its own single-grid update: equal to the oracle
(bit-exact where the parity tests are) and bit for bit equal to the single-grid update in the same
build, with nothing leaking across the seams between stacked members.
"""
import math

import numpy as np
import pytest

import cases
from stencilstream_b200 import Grid, GridBatch, Params, RangeError, StencilUpdate
from stencilstream_b200._native import CELL_DTYPES
from test_paired_sweeps_gpu import has_interior_tile
from test_parity_gpu import ALL, check

pytestmark = pytest.mark.gpu


def member_cases(workload, members, rows, cols, seed0=0):
    """Per-member (params, halo, cells); params and halo are those of the first member."""
    out = [cases.make_case(workload, rows, cols, seed=seed0 + b) for b in range(members)]
    params, halo = out[0][0], out[0][1]
    return params, halo, np.stack([c for _, _, c in out])


def run_batch(workload, params, halo, stack, offset, n, strict=False, **extra):
    batch = GridBatch(workload, buffer=stack, strict=strict)
    update = StencilUpdate(workload, Params(transition_function=params, halo_value=halo,
                                            iteration_offset=offset, n_iterations=n, blocking=True,
                                            **extra), strict=strict)
    return update(batch).to_numpy(), update, batch


def run_single(workload, params, halo, cells, offset, n, strict=False, **extra):
    update = StencilUpdate(workload, Params(transition_function=params, halo_value=halo,
                                            iteration_offset=offset, n_iterations=n, blocking=True,
                                            **extra), strict=strict)
    return update(Grid(workload, buffer=cells, strict=strict)).to_numpy()


@pytest.mark.parametrize("workload", ALL)
@pytest.mark.parametrize("strict", [False, True], ids=["fma", "strict"])
def test_every_workload_matches_oracle_per_member(workload, strict, oracle_best):
    rows, cols, members = 67, 93, 5
    offset = 0 if "kat" in workload else 2
    params, halo, stack = member_cases(workload, members, rows, cols, seed0=11)
    got, update, _ = run_batch(workload, params, halo, stack, offset, 5, strict)
    assert got.shape == (members, rows, cols)
    for b in range(members):
        want = oracle_best.run(workload, params, halo, stack[b], offset, 5)
        check(workload, got[b], want, strict)
        single = run_single(workload, params, halo, stack[b], offset, 5, strict)
        assert got[b].tobytes() == single.tobytes(), f"{workload} member {b} differs from its grid update"


def _seam_stack(workload, members, rows, cols):
    """Member b filled with the constant 1000 * b (member 0: zeros), every field."""
    dtype = CELL_DTYPES[workload]
    stack = np.zeros((members, rows, cols), dtype=dtype)
    for b in range(members):
        if dtype.names:
            for name in dtype.names:
                stack[b][name] = 1000.0 * b
        else:
            stack[b] = 1000.0 * b
    return stack


@pytest.mark.parametrize("workload", ["jacobi5", "hotspot"])
@pytest.mark.parametrize("tma", ["1", "0"], ids=["tma", "cp_async"])
@pytest.mark.parametrize("tile_rows", [0, 7, 1])
def test_no_leakage_across_seams(workload, tma, tile_rows, monkeypatch):
    """Very different constants side by side: after n = 2k+1 iterations every member equals its
    own single-grid update. H = 45 is no multiple of the tile heights tried."""
    monkeypatch.setenv("STST_TMA", tma)
    rows, cols, members = 45, 300, 4
    params, halo, _ = cases.make_case(workload, rows, cols, seed=3)
    stack = _seam_stack(workload, members, rows, cols)
    k = 3
    got, update, _ = run_batch(workload, params, halo, stack, 0, 2 * k + 1, strict=True,
                               fused_iterations=k, tile_rows=tile_rows)
    stats = update.get_stats()
    assert stats.use_tma == (tma == "1")
    if tile_rows:
        assert stats.tile_h <= tile_rows
    for b in range(members):
        single = run_single(workload, params, halo, stack[b], 0, 2 * k + 1, strict=True,
                            fused_iterations=k, tile_rows=tile_rows)
        assert got[b].tobytes() == single.tobytes(), f"{workload} member {b}: seam leakage"


@pytest.mark.parametrize("workload", ["jacobi5", "jacobi9", "hotspot", "fdtd"])
@pytest.mark.parametrize("fused", [1, 2, 3, 5, 6, 8])
def test_fusion_depths_with_interior_tiles(workload, fused, oracle_best):
    rows, cols, members = 300, 1100, 3
    params, halo, stack = member_cases(workload, members, rows, cols, seed0=21)
    for n in (fused, fused + 1, 2 * fused + 1):
        got, update, _ = run_batch(workload, params, halo, stack, 1, n, strict=True,
                                   fused_iterations=fused)
        stats = update.get_stats()
        assert stats.fused_iterations == fused
        if workload != "fdtd":  # (FDTD: two sub-iterations, halo 2k; its plans are checked below)
            assert has_interior_tile(stats, rows, cols), "the plan has no interior tile"
        for b in range(members):
            want = oracle_best.run(workload, params, halo, stack[b], 1, n)
            assert got[b].tobytes() == want.tobytes(), f"{workload} k={fused} n={n} member {b}"


def test_declared_pass_through_keeps_a_batch_asynchronous(oracle_best):
    params, halo, stack = member_cases("hotspot", 4, 200, 300, seed0=5)
    batch = GridBatch("hotspot", buffer=stack, strict=True)
    update = StencilUpdate("hotspot", Params(transition_function=params, halo_value=halo,
                                             n_iterations=12), strict=True)
    out = update(batch)
    stats = update.get_stats()
    assert stats.passthrough_planes == 0b10 and stats.speculation_redos == 0
    got = out.to_numpy()
    for b in range(4):
        assert got[b].tobytes() == oracle_best.run("hotspot", params, halo, stack[b], 0, 12).tobytes()


def test_wrong_speculation_on_a_batch_is_repeated(oracle_best):
    """FDTD's `hz_sum` starts to change at detect_iteration = 10: the batch call is repeated from
    its untouched source batch and comes out bit-exact."""
    params, halo, stack = member_cases("fdtd", 3, 90, 100, seed0=12)
    batch = GridBatch("fdtd", buffer=stack, strict=True)
    update = StencilUpdate("fdtd", Params(transition_function=params, halo_value=halo,
                                          n_iterations=30, blocking=True, fused_iterations=2),
                           strict=True)
    out = update(batch).to_numpy()
    assert update.get_stats().speculation_redos >= 1
    assert batch.to_numpy().tobytes() == stack.tobytes()
    for b in range(3):
        assert out[b].tobytes() == oracle_best.run("fdtd", params, halo, stack[b], 0, 30).tobytes()


def test_resumed_fdtd_batch_equals_one_call():
    params, halo, stack = member_cases("fdtd", 3, 80, 96, seed0=30)
    whole, _, _ = run_batch("fdtd", params, halo, stack, 0, 24, strict=True)
    batch = GridBatch("fdtd", buffer=stack, strict=True)
    update = StencilUpdate("fdtd", Params(transition_function=params, halo_value=halo,
                                          n_iterations=8, blocking=True), strict=True)
    for step in range(3):
        update.get_params().iteration_offset = 8 * step
        batch = update(batch)
    assert batch.to_numpy().tobytes() == whole.tobytes()


@pytest.mark.parametrize("members", [1, 64])
def test_launch_and_cell_counts(members):
    rows, cols, n = 40, 70, 11
    params, halo, stack = member_cases("jacobi5", members, rows, cols)
    _, update, _ = run_batch("jacobi5", params, halo, stack, 0, n, fused_iterations=4)
    stats = update.get_stats()
    assert stats.n_launches == math.ceil(n / stats.fused_iterations)
    assert stats.n_processed_cells == n * members * rows * cols


def test_zero_iterations_return_the_same_cells():
    params, halo, stack = member_cases("hotspot", 3, 20, 30)
    got, update, _ = run_batch("hotspot", params, halo, stack, 0, 0)
    assert got.tobytes() == stack.tobytes()
    assert update.get_stats().n_launches == 0


def test_member_ranges_and_sizes():
    params, halo, stack = member_cases("hotspot", 4, 20, 30)
    batch = GridBatch("hotspot", 4, 20, 30)
    assert batch.shape() == (4, 20, 30) and batch.get_grid_range() == (20, 30)
    batch.copy_from_buffer(stack)
    batch.copy_from_buffer(stack[::-1][1:3], first_member=1)   # members 2, 1 into slots 1, 2
    part = np.empty((2, 20, 30), dtype=stack.dtype)
    batch.copy_to_buffer(part, first_member=1)
    assert part.tobytes() == stack[[2, 1]].tobytes()
    assert batch.field_to_numpy("power").tobytes() == batch.to_numpy()["power"].tobytes()
    m = batch.max_abs([("temp", 20, 30), ("power", 5, 7)], member=3)
    assert m[0] == np.abs(stack[3]["temp"]).max()
    assert m[1] == np.abs(stack[3]["power"][:5, :7]).max()
    with pytest.raises(RangeError):
        batch.copy_from_buffer(stack[:, :19])
    with pytest.raises(RangeError):
        batch.copy_from_buffer(stack[:2], first_member=3)
    with pytest.raises(RangeError):
        batch.copy_to_buffer(np.empty((1, 20, 30), dtype=stack.dtype), first_member=4)
    with pytest.raises(RangeError):
        batch.max_abs([("temp", 20, 30)], member=4)


def test_several_devices_are_rejected():
    params, halo, stack = member_cases("jacobi5", 2, 16, 16)
    with pytest.raises(ValueError):
        run_batch("jacobi5", params, halo, stack, 0, 3, cuda_devices=[0, 0])


@pytest.mark.parametrize("shape", [(1, 1), (1, 40), (40, 1)])
@pytest.mark.parametrize("workload", ["jacobi5", "hotspot", "kat"])
def test_degenerate_members_match_oracle(workload, shape, oracle_best):
    params, halo, stack = member_cases(workload, 3, *shape, seed0=40)
    got, _, _ = run_batch(workload, params, halo, stack, 0, 4, strict=True)
    for b in range(3):
        want = oracle_best.run(workload, params, halo, stack[b], 0, 4)
        assert got[b].tobytes() == want.tobytes(), f"{workload} {shape} member {b}"
