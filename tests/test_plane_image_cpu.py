"""The plane image format (cuda/internal/PlaneImage.hpp) and the slab layout built on it
(SlabLayout, cuda/internal/SlabUpdate.hpp), exercised without a GPU: tests/cpp/plane_image.cpp is
host-only code compiled with g++. What is pinned: per-plane pitch (smallest with 128-byte rows),
plane offsets (256-byte aligned) and total bytes, for cells of 1-, 4- and 8-byte and mixed planes
and widths 1, 31, 1030 and 16384. The expected values in tests/golden/plane_image_layouts.jsonl were
recorded from the layout code that grids and slabs each had before the format got one owner; the
device data of existing grids and slabs is therefore laid out byte for byte as before."""
import json
import subprocess
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
BINARY = ROOT / "build" / "own_tests" / "plane_image"
GOLDEN = ROOT / "tests" / "golden" / "plane_image_layouts.jsonl"


@pytest.fixture(scope="module")
def layouts():
    BINARY.parent.mkdir(parents=True, exist_ok=True)
    pkg = ROOT / "stencilstream_b200"
    subprocess.run(["g++", "-std=c++20", "-O1", "-w", f"-I{pkg / 'include'}", f"-I{pkg / 'compat'}",
                    f"-I{ROOT / 'include'}", "-I/usr/local/cuda/include",
                    str(ROOT / "tests" / "cpp" / "plane_image.cpp"), "-o", str(BINARY)], check=True)
    out = subprocess.run([str(BINARY)], check=True, capture_output=True, text=True).stdout
    return [json.loads(line) for line in out.splitlines()]


def test_layouts_match_the_recorded_ones(layouts):
    expected = [json.loads(line) for line in GOLDEN.read_text().splitlines()]
    assert len(layouts) == len(expected)
    for got, want in zip(layouts, expected):
        assert got == want


def test_slab_buffers_have_the_pitches_of_a_grid_of_the_same_width(layouts):
    grid_pitch = {(g["cell"], g["width"]): g["pitch"] for g in layouts if g["kind"] == "grid"}
    slabs = [s for s in layouts if s["kind"] == "slab"]
    assert len(slabs) == 4 * 4 * 2
    for s in slabs:
        assert s["pitch0"] == s["pitch1"] == grid_pitch[(s["cell"], s["width"])]


def test_format_rules(layouts):
    for g in layouts:
        if g["kind"] != "grid":
            continue
        elem = {"u8": [1], "f32": [4], "f64": [8], "mixed": [8, 4, 2, 1, 1]}[g["cell"]]
        for i, (pitch, size) in enumerate(zip(g["pitch"], elem)):
            assert pitch >= g["width"] and pitch * size % 128 == 0
            assert g["offset"][i] % 256 == 0
        ends = g["offset"][1:] + [g["bytes"]]
        for i, size in enumerate(elem):
            plane = g["pitch"][i] * max(g["rows"], 1) * size
            assert ends[i] - g["offset"][i] == (plane + 255) // 256 * 256
