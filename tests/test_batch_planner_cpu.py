"""The planner's small-grid rule (Planner.hpp small_grid_tile_rows) for grid batches, without a GPU:
one member keeps the tile heights the rule gave single grids before batches existed, and many small
members, which fill the GPU together, keep the planner's tall tiles."""
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
BINARY = ROOT / "build" / "own_tests" / "batch_planner"
SLOTS = 148 * 2  # B200 SMs x two CTAs per SM


@pytest.fixture(scope="module")
def rule():
    BINARY.parent.mkdir(parents=True, exist_ok=True)
    pkg = ROOT / "stencilstream_b200"
    subprocess.run(["g++", "-std=c++20", "-O1", "-w", f"-I{pkg / 'include'}", f"-I{pkg / 'compat'}",
                    f"-I{ROOT / 'include'}", "-I/usr/local/cuda/include",
                    str(ROOT / "tests" / "cpp" / "batch_planner.cpp"), "-o", str(BINARY)], check=True)

    def run(tile_h, halo, tile_w, grid_h, grid_w, members, slots=SLOTS):
        out = subprocess.run([str(BINARY)] + [str(v) for v in (tile_h, halo, tile_w, grid_h, grid_w,
                                                                 members, slots)],
                             check=True, capture_output=True, text=True).stdout
        return int(out)
    return run


def single_grid_rule(tile_h, halo, tile_w, grid_h, grid_w, slots=SLOTS):
    """The rule as it stood for single grids (unsigned arithmetic of the original code)."""
    tiles_x = (max(grid_w, 1) + tile_w - 1) // tile_w
    want = max(1, slots * 95 // 100 // tiles_x)
    return min(tile_h, max(2 * halo, (max(grid_h, 1) + want - 1) // want))


# (tile_h, halo, tile_w) of the plans in profiles/r01_s3_sweep_small_grids.log: HotSpot and Jacobi
# at k = 2 and 4, one and two CTAs per SM
PLANS = [(33, 2, 248), (14, 2, 248), (29, 4, 248), (10, 4, 248), (51, 2, 248), (47, 4, 248),
         (19, 4, 248), (43, 6, 240)]


@pytest.mark.parametrize("size", [128, 256, 362, 512, 1024, 2048, 4096, 16384])
def test_one_member_keeps_the_single_grid_tile_height(rule, size):
    for tile_h, halo, tile_w in PLANS:
        assert rule(tile_h, halo, tile_w, size, size, 1) == single_grid_rule(tile_h, halo, tile_w,
                                                                               size, size)


def test_known_single_grid_heights(rule):
    # 1024^2 HotSpot k=4: 29-row tiles shrink to 19 (270 CTAs on 296 slots); 4096^2 stays
    assert rule(29, 4, 248, 1024, 1024, 1) == 19
    assert rule(29, 4, 248, 4096, 4096, 1) == 29


@pytest.mark.parametrize("size,members", [(128, 4096), (256, 1024), (512, 256), (1024, 64)])
def test_many_small_members_keep_tall_tiles(rule, size, members):
    for tile_h, halo, tile_w in PLANS:
        assert rule(tile_h, halo, tile_w, size, size, members) == tile_h
        # the same member alone would have shrunk its tiles
        if size <= 512:
            assert rule(tile_h, halo, tile_w, size, size, 1) < tile_h or tile_h <= 2 * halo


def test_few_members_shrink_less_than_one(rule):
    one = rule(43, 6, 240, 1024, 1024, 1)
    four = rule(43, 6, 240, 1024, 1024, 4)
    assert one <= four <= 43
