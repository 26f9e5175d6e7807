"""Generate the golden vectors in tests/golden/*.npz from the REFERENCE-BUILT oracle.

Run in the build container (where /root/reference exists):

    python tests/golden/generate.py

For every workload it records small seeded inputs, the raw bytes of the transition-function parameter
block, the halo cell, and the cells the reference's own `stencil::cpu::StencilUpdate`
(/root/reference/StencilStream/cpu/StencilUpdate.hpp:109-223, compiled in place into
oracle/_ref/liboracle_ref.so with -ffp-contract=off) produces after `n_iterations` iterations starting
at `iteration_offset`. The fixtures travel with the repository; /root/reference does not.
They pin (a) the plain-C restatement oracle/stencil_oracle.c on machines without the reference
(tests/test_oracle.py) and (b) the CUDA path in the -fmad=false build (tests/test_parity_gpu.py).
"""
from __future__ import annotations

import ctypes as C
import json
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import cases  # noqa: E402
import oracle  # noqa: E402

# (workload, rows, cols, iteration_offset, n_iterations, seed)
CASES = [
    ("conway", 48, 80, 0, 24, 0),
    ("jacobi5", 33, 47, 3, 6, 1),
    ("jacobi9", 33, 47, 0, 5, 2),
    ("jacobi_r2", 29, 41, 0, 4, 3),
    ("jacobi_r3", 29, 41, 1, 4, 4),
    ("hotspot", 40, 52, 0, 9, 5),
    ("fdtd", 36, 44, 5, 12, 6),
    ("convection_pt", 24, 32, 0, 4, 7),
    ("convection_thermal", 24, 32, 0, 3, 8),
    ("kat", 32, 64, 7, 5, 0),
    ("kat_r2", 19, 23, 0, 3, 0),
]


def main() -> None:
    ref = oracle.reference()
    if ref is None:
        raise SystemExit("the reference-built oracle is not available: nothing generated")
    for workload, rows, cols, offset, n, seed in CASES:
        params, halo, cells = cases.make_case(workload, rows, cols, seed=seed)
        if "kat" in workload:
            cells = cases.kat_input(*cells.shape, offset)
        cells = np.ascontiguousarray(cells)
        want = ref.run(workload, params, halo, cells, offset, n)
        halo_arr = np.zeros((), dtype=cells.dtype)
        if halo is not None:
            halo_arr[()] = halo
        path = HERE / f"{workload}.npz"
        np.savez_compressed(
            path,
            input=cells.view(np.uint8).reshape(cells.shape[0], -1),
            output=want.view(np.uint8).reshape(want.shape[0], -1),
            params=np.frombuffer(bytes(params), dtype=np.uint8) if params is not None
            else np.zeros(0, np.uint8),
            halo=np.frombuffer(halo_arr.tobytes(), dtype=np.uint8),
            has_halo=np.array(halo is not None),
            shape=np.array(cells.shape), iteration_offset=np.array(offset),
            n_iterations=np.array(n), seed=np.array(seed))
        print(f"{workload}: {cells.shape} offset={offset} n={n} -> {path.name} "
              f"({path.stat().st_size} bytes)")
    write_reference_digests(ref, "SHA-256 of the output bytes of the reference build "
                                 "(oracle/_ref/liboracle_ref.so), written by tests/golden/generate.py")


def write_reference_digests(checker, provenance: str) -> None:
    """tests/golden/reference_digests.json: the digest of `checker`'s output for every seeded case of
    tests/test_oracle.py (cases.seeded_cases, cases.window_case)."""
    digests = {}
    for workload in cases.GOLDEN_WORKLOADS:
        runs = [c for shape in cases.SEEDED_SHAPES for c in cases.seeded_cases(workload, shape)]
        runs.append(cases.window_case(workload))
        for key, params, halo, cells, offset, n in runs:
            digests[key] = cases.output_digest(checker.run(workload, params, halo, cells, offset, n))
    path = HERE / "reference_digests.json"
    path.write_text(json.dumps({"provenance": provenance, "digests": digests}, indent=1) + "\n")
    print(f"{len(digests)} digests -> {path.name}")


if __name__ == "__main__":
    main()
