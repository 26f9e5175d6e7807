"""Shared test-case builders: seeded inputs + parameters for every workload."""
from __future__ import annotations

import numpy as np

from stencilstream_b200 import _native
from stencilstream_b200 import workloads as W

KAT_HALO = (0, 0, 0, 0, 2)


def kat_input(rows, cols, iteration_offset):
    """tests/StencilUpdateTest.hpp:38-45 of the reference: Cell{r, c, offset, 0, Normal}."""
    cells = np.zeros((rows, cols), dtype=_native.CELL_DTYPES["kat"])
    cells["r"] = np.arange(rows, dtype=np.int32)[:, None]
    cells["c"] = np.arange(cols, dtype=np.int32)[None, :]
    cells["i_iteration"] = iteration_offset
    cells["i_subiteration"] = 0
    cells["status"] = 0
    return cells


def kat_expected(rows, cols, iteration_offset, n_iterations):
    """tests/StencilUpdateTest.hpp:54-62: {r, c, offset + n, 0, Normal} everywhere."""
    cells = kat_input(rows, cols, iteration_offset + n_iterations)
    return cells


def random_cells(workload, shape, seed=0):
    rng = np.random.default_rng(seed)
    dt = _native.CELL_DTYPES[workload]
    if dt == np.bool_:
        return rng.random(shape) < 0.4
    if dt.names is None:
        return rng.random(shape).astype(dt)
    cells = np.zeros(shape, dtype=dt)
    for name in dt.names:
        cells[name] = rng.random(shape).astype(dt[name])
    return cells


def fdtd_case(rows, cols, seed=0):
    """A small FDTD set-up: reference constants of experiments/default.json, material map centred in
    a rows x cols grid, random initial fields so that every term of the update is exercised."""
    exp = W.FdtdExperiment(W.FDTD_DEFAULT)
    params = exp.kernel_params()
    # Move source and cavity centre into the small grid.
    params.source_r = float(rows // 2)
    params.source_c = float(cols // 2)
    params.source_distance_bound = float(np.float32(0.0) - (np.float32(params.source_c) ** 2
                                                             + np.float32(params.source_r) ** 2))
    params.double_center_rc = float(rows)
    params.cutoff_iteration = 40
    params.detect_iteration = 10
    rng = np.random.default_rng(seed)
    cells = np.zeros((rows, cols), dtype=_native.CELL_DTYPES["fdtd"])
    r = np.arange(rows)[:, None] - rows / 2
    c = np.arange(cols)[None, :] - cols / 2
    inside = (r * r + c * c) < (min(rows, cols) * 0.4) ** 2
    ca, cb, da, db = exp._coefficients(*exp.rings[0][1:])
    for name, v in (("ca", ca), ("cb", cb), ("da", da), ("db", db)):
        cells[name][inside] = v
    for name in ("ex", "ey", "hz"):
        cells[name] = (rng.standard_normal((rows, cols)) * 1e-3).astype(np.float32)
    return params, None, cells


def convection_case(res_x, res_y, seed=0):
    cfg = W.convection_benchmark_config(res=64, n_iters=4, lx=res_x / 64.0, ly=res_y / 64.0)
    exp = W.ConvectionExperiment(cfg)
    cells = exp.initial_grid()
    rng = np.random.default_rng(seed)
    for name in ("Vx", "Vy", "Pt"):
        cells[name] = rng.standard_normal(cells.shape) * 1e-3
    return exp, cells


def make_case(workload, rows, cols, seed=0):
    """Returns (params struct, halo value or None, input cells)."""
    if workload == "conway":
        return _native.ConwayParams(), None, W.conway_soup(rows, cols, seed=seed + 42)
    if workload == "jacobi5":
        return W.jacobi5_params((0.1, 0.2, 0.3, 0.15, 0.25)), 0.5, random_cells(workload, (rows, cols), seed)
    if workload == "jacobi9":
        rng = np.random.default_rng(seed + 1)
        return W.jacobi9_params(rng.random((3, 3)) / 4.5), 0.25, random_cells(workload, (rows, cols), seed)
    if workload in ("jacobi_r2", "jacobi_r3"):
        return W.jacobi_star_params(int(workload[-1])), 1.0, random_cells(workload, (rows, cols), seed)
    if workload == "hotspot":
        cells = W.hotspot_input(rows, cols)
        rng = np.random.default_rng(seed)
        cells["temp"] += rng.random((rows, cols)).astype(np.float32) * 50
        cells["power"] += rng.random((rows, cols)).astype(np.float32) * 0.1
        return W.hotspot_params(rows, cols), (0.0, 0.0), cells
    if workload == "fdtd":
        return fdtd_case(rows, cols, seed)
    if workload == "convection_pt":
        exp, cells = convection_case(rows, cols, seed)
        return exp.pseudo_transient_params(), None, cells
    if workload == "convection_thermal":
        exp, cells = convection_case(rows, cols, seed)
        return exp.thermal_params(1e-6), None, cells
    if workload in ("kat", "kat_r2"):
        return _native.KatParams(), KAT_HALO, kat_input(rows, cols, 0)
    raise KeyError(workload)


def rel_max_norm(a, b):
    """max |a-b| / max |b| per field, reduced with max (BASELINE.json: 1e-5 relative max-norm)."""
    if a.dtype.names is None:
        a64, b64 = a.astype(np.float64), b.astype(np.float64)
        denom = max(np.abs(b64).max(), 1e-300)
        return float(np.abs(a64 - b64).max() / denom)
    worst = 0.0
    for name in a.dtype.names:
        a64, b64 = a[name].astype(np.float64), b[name].astype(np.float64)
        scale = np.abs(b64).max()
        if scale == 0.0:
            worst = max(worst, float(np.abs(a64).max()))
        else:
            worst = max(worst, float(np.abs(a64 - b64).max() / scale))
    return worst


# ---- golden vectors (tests/golden/*.npz, generated from the reference-built oracle) ----------------

GOLDEN_DIR = __import__("pathlib").Path(__file__).resolve().parent / "golden"
GOLDEN_WORKLOADS = ["conway", "jacobi5", "jacobi9", "jacobi_r2", "jacobi_r3", "hotspot", "fdtd",
                    "convection_pt", "convection_thermal", "kat", "kat_r2"]


def load_golden(workload):
    """Returns dict(params=ctypes struct, halo=cell or None, input, output, iteration_offset,
    n_iterations) of the fixture tests/golden/<workload>.npz."""
    import ctypes as C
    data = np.load(GOLDEN_DIR / f"{workload}.npz")
    dtype = _native.CELL_DTYPES[workload]
    shape = tuple(int(x) for x in data["shape"])
    cells_in = np.ascontiguousarray(data["input"]).view(dtype).reshape(shape)
    cells_out = np.ascontiguousarray(data["output"]).view(dtype).reshape(shape)
    params = _native.PARAM_TYPES[workload]()
    raw = data["params"].tobytes()
    assert len(raw) == C.sizeof(params)
    C.memmove(C.addressof(params), raw, len(raw))
    halo = None
    if bool(data["has_halo"]):
        halo = np.frombuffer(data["halo"].tobytes(), dtype=dtype)[0]
    return {"params": params, "halo": halo, "input": cells_in, "output": cells_out,
            "iteration_offset": int(data["iteration_offset"]),
            "n_iterations": int(data["n_iterations"])}


# ---- seeded cases checked against the reference build (tests/test_oracle.py) -----------------------
# Their reference outputs travel with the repository as SHA-256 digests of the output bytes
# (tests/golden/reference_digests.json), so the port is held to them where the reference tree is absent.

SEEDED_SHAPES = [(1, 1), (5, 3), (37, 53)]
WINDOW_SHAPE = (61, 67)


def seeded_cases(workload, shape):
    """[(key, params, halo, cells, iteration_offset, n_iterations)] of one workload and shape: seed 11,
    (offset, n) = (0, 1) and (2, 4). Empty where the workload cannot be set up on that grid."""
    if workload.startswith("convection") and min(shape) < 4:
        return []   # the convection set-up needs at least a 4x4 grid (dx = lx / (nx - 1))
    params, halo, cells = make_case(workload, *shape, seed=11)
    out = []
    for offset, n in ((0, 1), (2, 4)):
        if "kat" in workload:
            cells = kat_input(*shape, offset)
        out.append((f"{workload} {shape[0]}x{shape[1]} seed=11 offset={offset} n={n}",
                    params, halo, cells, offset, n))
    return out


def window_case(workload):
    """(key, params, halo, cells, offset, n): the whole-grid run whose windows
    test_window_oracle_equals_the_whole_grid_run crops (seed 3, offset 1, 3 iterations)."""
    params, halo, cells = make_case(workload, *WINDOW_SHAPE, seed=3)
    offset, n = 1, 3
    if "kat" in workload:
        cells = kat_input(*WINDOW_SHAPE, offset)
    return (f"{workload} {WINDOW_SHAPE[0]}x{WINDOW_SHAPE[1]} seed=3 offset={offset} n={n}",
            params, halo, cells, offset, n)


def output_digest(cells):
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(cells).tobytes()).hexdigest()


def load_reference_digests():
    import json
    return json.loads((GOLDEN_DIR / "reference_digests.json").read_text())["digests"]


# ---- the convection application loop on the oracle (host-side glue as in the reference's main) ----------

def oracle_convection(oracle, config):
    exp = W.ConvectionExperiment(config)
    nx, ny = exp.nx, exp.ny
    cells = exp.initial_grid()
    steps, frames = [], []
    for it in range(1, int(config["nt"]) + 1):
        errV = errP = 2 * config["epsilon"]
        iterations = 0
        while iterations < config["iterMax"] and (errV > config["epsilon"] or errP > config["epsilon"]):
            cells = oracle.run("convection_pt", exp.pseudo_transient_params(), None, cells, 0,
                               config["nerr"])
            norms = {f: float(np.abs(cells[f][:r, :c]).max())
                     for f, r, c in _convection_norm_extents(nx, ny)}
            errV = norms["ErrV"] / (1e-12 + norms["Vy"])
            errP = norms["ErrP"] / (1e-12 + norms["Pt"])
            iterations += config["nerr"]
        with np.errstate(divide="ignore"):
            dt = float(min(exp.dt_diff, min(np.float64(exp.dx) / norms["Vx"],
                                            np.float64(exp.dy) / norms["Vy"]) / 2.1))
        cells = oracle.run("convection_thermal", exp.thermal_params(dt), None, cells, 0, 1)
        steps.append((it, iterations, errV, errP, dt))
        if it % config["nout"] == 0:
            frames.append((it, cells["T"][:nx, :ny].copy()))
    return cells, steps, frames


def _convection_norm_extents(nx, ny):
    from stencilstream_b200.apps import convection_norm_extents
    return convection_norm_extents(nx, ny)
