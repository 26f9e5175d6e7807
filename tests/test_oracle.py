"""CPU tests of the parity oracles themselves (no GPU).

The plain-C restatement (oracle/stencil_oracle.c) is pinned three ways:
  1. against the golden vectors in tests/golden/ (outputs of the reference's own cpu backend, built
     in place from /root/reference by tests/golden/generate.py) — bit for bit;
  2. against the reference-built oracle (oracle/_ref) on further seeded cases, where that exists, and
     everywhere against the reference's outputs of those cases stored as digests
     (tests/golden/reference_digests.json);
  3. against the reference's own known-answer test: the self-checking functor of
     /root/reference/tests/TransFuncs.hpp:55-104 with the case matrix of
     tests/cpu/StencilUpdate.cpp:35-41 and tests/cuda/StencilUpdate.cpp:30-50, whose expected output is
     closed-form ({r, c, offset + n, 0, Normal}, tests/StencilUpdateTest.hpp:54-62).
"""
import numpy as np
import pytest

import cases

REFERENCE_KAT_CASES = [(64, 64, 0, 1), (64, 64, 32, 64), (32, 64, 0, 1), (64, 32, 0, 1)]


@pytest.mark.parametrize("workload", cases.GOLDEN_WORKLOADS)
def test_port_reproduces_golden_vectors(workload, oracle_port):
    g = cases.load_golden(workload)
    got = oracle_port.run(workload, g["params"], g["halo"], g["input"], g["iteration_offset"],
                          g["n_iterations"])
    assert got.tobytes() == g["output"].tobytes()


@pytest.mark.parametrize("workload", cases.GOLDEN_WORKLOADS)
def test_reference_build_reproduces_golden_vectors(workload, oracle_ref):
    """Guards the fixtures against drifting from the reference (runs where /root/reference exists)."""
    g = cases.load_golden(workload)
    got = oracle_ref.run(workload, g["params"], g["halo"], g["input"], g["iteration_offset"],
                         g["n_iterations"])
    assert got.tobytes() == g["output"].tobytes()


@pytest.mark.parametrize("workload", cases.GOLDEN_WORKLOADS)
@pytest.mark.parametrize("shape", cases.SEEDED_SHAPES)
def test_port_matches_reference_build(workload, shape, oracle_port, oracle_ref):
    if not cases.seeded_cases(workload, shape):
        pytest.skip("the convection set-up needs at least a 4x4 grid (dx = lx / (nx - 1))")
    digests = cases.load_reference_digests()
    for key, params, halo, cells, offset, n in cases.seeded_cases(workload, shape):
        a = oracle_port.run(workload, params, halo, cells, offset, n)
        b = oracle_ref.run(workload, params, halo, cells, offset, n)
        assert a.tobytes() == b.tobytes(), key
        assert cases.output_digest(b) == digests[key], f"stored digest no longer the reference's: {key}"


@pytest.mark.parametrize("workload", cases.GOLDEN_WORKLOADS)
def test_port_reproduces_the_reference_digests(workload, oracle_port):
    """The seeded cases of test_port_matches_reference_build and the whole-grid run of
    test_window_oracle_equals_the_whole_grid_run, held against the reference build's outputs stored
    as digests (tests/golden/reference_digests.json) — bit for bit, without the reference tree."""
    digests = cases.load_reference_digests()
    runs = [c for shape in cases.SEEDED_SHAPES for c in cases.seeded_cases(workload, shape)]
    runs.append(cases.window_case(workload))
    for key, params, halo, cells, offset, n in runs:
        got = oracle_port.run(workload, params, halo, cells, offset, n)
        assert cases.output_digest(got) == digests[key], key


@pytest.mark.parametrize("case", REFERENCE_KAT_CASES)
@pytest.mark.parametrize("which", ["port", "reference"])
def test_reference_known_answer_cases(case, which, request):
    oracle = request.getfixturevalue("oracle_port" if which == "port" else "oracle_ref")
    rows, cols, offset, n = case
    got = oracle.run("kat", None, cases.KAT_HALO, cases.kat_input(rows, cols, offset), offset, n)
    assert got.tobytes() == cases.kat_expected(rows, cols, offset, n).tobytes()


def test_known_answer_functor_detects_a_wrong_halo(oracle_port):
    """The self-checking functor must actually poison cells: a wrong halo value marks the border."""
    got = oracle_port.run("kat", None, (0, 0, 0, 0, 0), cases.kat_input(16, 16, 0), 0, 1)
    assert (got["status"][0, :] == 1).all() and (got["status"][:, 0] == 1).all()
    assert (got["status"][4:12, 4:12] == 0).all()  # not reached after 2 sweeps of radius 1


def test_known_answer_functor_checks_the_time_dependent_value(oracle_port):
    """tdv == iteration is part of the check: cells claiming another iteration are flagged."""
    cells = cases.kat_input(8, 8, 3)
    got = oracle_port.run("kat", None, cases.KAT_HALO, cells, 4, 1)  # offset disagrees with cells
    assert (got["status"] == 1).all()


def test_zero_iterations_is_identity(oracle_port):
    params, halo, cells = cases.make_case("hotspot", 9, 11)
    assert oracle_port.run("hotspot", params, halo, cells, 0, 0).tobytes() == cells.tobytes()


def test_iteration_offset_resume(oracle_port):
    params, halo, cells = cases.make_case("fdtd", 20, 24)
    one = oracle_port.run("fdtd", params, halo, cells, 0, 12)
    part = oracle_port.run("fdtd", params, halo, cells, 0, 5)
    part = oracle_port.run("fdtd", params, halo, part, 5, 7)
    assert one.tobytes() == part.tobytes()


def test_conway_blinker(oracle_port):
    from stencilstream_b200 import _native
    grid = np.zeros((5, 5), dtype=np.bool_)
    grid[2, 1:4] = True
    once = oracle_port.run("conway", _native.ConwayParams(), None, grid, 0, 1)
    assert once[1:4, 2].all() and once.sum() == 3
    twice = oracle_port.run("conway", _native.ConwayParams(), None, grid, 0, 2)
    assert twice.tobytes() == grid.tobytes()


def test_jacobi_linearity(oracle_port):
    """Size-independent property: with halo 0 the Jacobi sweep is linear in the grid."""
    from stencilstream_b200 import workloads as W
    params = W.jacobi5_params((0.25, 0.25, 0.25, 0.25, 0.0))
    rng = np.random.default_rng(5)
    a = rng.integers(0, 64, (31, 29)).astype(np.float32)  # small integers: sums stay exact in fp32
    b = rng.integers(0, 64, (31, 29)).astype(np.float32)
    fa = oracle_port.run("jacobi5", params, 0.0, a, 0, 3)
    fb = oracle_port.run("jacobi5", params, 0.0, b, 0, 3)
    fab = oracle_port.run("jacobi5", params, 0.0, a + b, 0, 3)
    assert np.array_equal(fab, fa + fb)


WINDOWS = {  # of a 61 x 67 grid: corner, edge, interior, ragged corner, whole grid
    "nw-corner": ((0, 9), (0, 11)), "n-edge": ((0, 7), (30, 41)), "interior": ((25, 33), (28, 40)),
    "se-corner": ((50, 61), (55, 67)), "w-edge": ((20, 31), (0, 5)), "whole": ((0, 61), (0, 67)),
}


@pytest.mark.parametrize("workload", cases.GOLDEN_WORKLOADS)
@pytest.mark.parametrize("which", ["port", "reference"])
def test_window_oracle_equals_the_whole_grid_run(workload, which, request):
    """Pins tests/window_oracle.py (the checker of the full-size GPU parity tests): the oracle run on
    the domain-of-dependence crop of a window — global coordinates through oracle_run_window2d — holds
    bit for bit what the whole-grid run holds in that window; the whole-grid run is the reference
    build's (stored digest), so the windows are too."""
    import window_oracle

    oracle = request.getfixturevalue("oracle_port" if which == "port" else "oracle_ref")
    shape = cases.WINDOW_SHAPE
    key, params, halo, cells, offset, n = cases.window_case(workload)
    whole = oracle.run(workload, params, halo, cells, offset, n)
    assert cases.output_digest(whole) == cases.load_reference_digests()[key], key
    for name, window in WINDOWS.items():
        got = window_oracle.expected_window(
            oracle, workload, params, halo, lambda r0, r1, c0, c1: cells[r0:r1, c0:c1], shape, window,
            offset, n)
        (r0, r1), (c0, c1) = window
        assert got.tobytes() == np.ascontiguousarray(whole[r0:r1, c0:c1]).tobytes(), (workload, name)
