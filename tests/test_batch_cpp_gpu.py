"""tests/cpp/batch_update.cu: GridBatch through the C++ template API with a transition function that is
not in the library (radius 2, two fields), against per-member Grid updates, bit for bit."""
import subprocess
from pathlib import Path

import pytest

pytestmark = pytest.mark.gpu

BINARY = Path(__file__).resolve().parent.parent / "build" / "own_tests" / "unit_test_batch_b200"


def test_grid_batch_with_a_user_functor_equals_per_member_grids(built):
    if not BINARY.exists():
        pytest.skip(f"{BINARY} not built")
    proc = subprocess.run([str(BINARY)], capture_output=True, text=True, timeout=600)
    print(proc.stdout)
    assert proc.returncode == 0, proc.stdout + proc.stderr
    assert sum(line.startswith("[ OK ]") for line in proc.stdout.splitlines()) == 2
