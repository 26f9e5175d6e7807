"""bench.py --dump-outputs on the GPU: what it writes is the result of the last timed step, and
--steps is the number of timed steps.

A resident grid is updated from the same input by every step, so its last step holds `--iterations`
iterations of the synthetic input; `gpu_launches` (launches inside the timed region) shows how many
steps ran. A slab (--chunk-above-gib 0 moves it chunk by chunk, as bench.py does with grids too large
for host memory) advances in place, so its last timed step holds (warmup + steps) x iterations. The
4096 x 4096 grids are larger than the dump budget, so the sampled cells (bench.dump_sample) are
checked; the small ones are dumped whole."""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
STEPS, WARMUP, ITERS = 4, 1, 12


@pytest.mark.parametrize("workload,rows,cols,slab", [
    ("jacobi5", 4096, 4096, False), ("jacobi5", 4096, 4096, True),
    ("hotspot", 320, 256, False), ("hotspot", 320, 256, True),
])
def test_dumped_outputs_are_the_last_timed_step(workload, rows, cols, slab, tmp_path, oracle_best):
    import bench
    from stencilstream_b200 import _native

    proc = subprocess.run(
        [sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--steps", str(STEPS),
         "--warmup", str(WARMUP), "--workload", workload, "--rows", str(rows), "--cols", str(cols),
         "--iterations", str(ITERS), "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "out"),
         *(["--chunk-above-gib", "0"] if slab else [])],
        capture_output=True, text=True, timeout=900, env={**os.environ, "STST_STRICT": "1"})
    assert proc.returncode == 0, proc.stdout + proc.stderr
    record = json.loads(proc.stdout.strip().splitlines()[-1])
    assert record["steps"] == STEPS
    if not slab:
        passes = -(-ITERS // record["plan"]["fused_iterations"])
        assert record["gpu_launches"] == STEPS * passes, record["gpu_launches"]

    dtype = _native.CELL_DTYPES[workload]
    params, halo, fill = bench.make_workload(workload, rows, cols)
    cells = np.empty((rows, cols), dtype=dtype)
    fill(cells, 0, rows, rows)
    n = (WARMUP + STEPS) * ITERS if slab else ITERS
    want = oracle_best.run(workload, params, halo, cells, 0, n)
    rows_idx, cols_idx = bench.dump_sample(rows, cols, dtype, bench.DUMP_BYTES)
    assert (len(rows_idx) < rows) == (rows == 4096)
    want = want[np.ix_(rows_idx, cols_idx)]
    for field in (want.dtype.names or (None,)):
        name = f"{workload}.{field}.npy" if field else f"{workload}.npy"
        got = np.load(tmp_path / "out" / name)
        assert got.dtype == np.float32 and got.shape == (len(rows_idx), len(cols_idx))
        # the -fmad=false build (STST_STRICT=1) against the uncontracted oracle: bit for bit
        assert got.tobytes() == (want[field] if field else want).astype(np.float32).tobytes(), name
