"""Paired sweeps (two generations per shared-memory round trip on interior tiles, TileKernel.hpp
sweep_pair) against the oracle, bit for bit in the strict build.

Every fusion depth from 1 to 8, odd and even, runs with tile heights down to one row, so that row
groups of zero, one and two rows exercise the priming of both register windows, and with n = k, k+1
and 2k+1 generations, so that launches of every depth up to k follow one another (tail launches).
"""
import pytest

import cases
from stencilstream_b200 import Grid, Params, StencilUpdate

pytestmark = pytest.mark.gpu

ROWS, COLS = 300, 1100  # several interior tiles at every depth, ragged edges
CW = 4                  # columns per thread of a float cell


def has_interior_tile(stats, rows, cols):
    """Whether some tile of the plan takes the interior path of fused_sweep_kernel: its staged
    footprint lies inside the grid, with one column to spare on either side."""
    k, tile_h, tile_w = stats.fused_iterations, stats.tile_h, stats.tile_w
    hpad = (stats.block_x * CW - tile_w) // 2
    tile_cols = any(tx * tile_w >= hpad + 1 and (tx + 1) * tile_w + hpad + 1 <= cols
                    for tx in range((cols + tile_w - 1) // tile_w))
    tile_rows = any(ty * tile_h >= k and (ty + 1) * tile_h + k <= rows
                    for ty in range((rows + tile_h - 1) // tile_h))
    return tile_cols and tile_rows


@pytest.mark.parametrize("workload", ["jacobi5", "jacobi9"])
@pytest.mark.parametrize("fused", [1, 2, 3, 5, 6, 8])
@pytest.mark.parametrize("tile_rows", [1, 2, 3, 5, 8, 0])
def test_paired_sweeps_match_oracle(workload, fused, tile_rows, oracle_best):
    params, halo, cells = cases.make_case(workload, ROWS, COLS, seed=4)
    for n in (fused, fused + 1, 2 * fused + 1):
        want = oracle_best.run(workload, params, halo, cells, 1, n)
        grid = Grid(workload, buffer=cells, strict=True)
        update = StencilUpdate(workload, Params(transition_function=params, halo_value=halo,
                                                iteration_offset=1, n_iterations=n, blocking=True,
                                                fused_iterations=fused, tile_rows=tile_rows),
                               strict=True)
        got = update(grid).to_numpy()
        stats = update.get_stats()
        assert stats.fused_iterations == fused
        if tile_rows:
            assert stats.tile_h <= tile_rows
        assert has_interior_tile(stats, ROWS, COLS), "the plan has no interior tile"
        assert got.tobytes() == want.tobytes(), f"{workload} k={fused} tile_rows={tile_rows} n={n}"
