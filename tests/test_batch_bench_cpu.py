"""scripts/batch_bench.py without a GPU: argument parsing and the shape arithmetic (members * S^2 =
2^26 cells for every member size) run up to the first device call."""
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def test_plan_only_prints_every_point(tmp_path):
    out = subprocess.run([sys.executable, str(ROOT / "scripts" / "batch_bench.py"), "--out",
                          str(tmp_path), "--plan-only"], capture_output=True, text=True, check=True)
    lines = out.stdout.strip().splitlines()
    assert len(lines) == 10
    for line in lines:
        members = int(line.split(": ")[1].split(" ")[0])
        size = int(line.split(" of ")[1].split("x")[0])
        assert members * size * size == 1 << 26
    assert not any(tmp_path.iterdir())
