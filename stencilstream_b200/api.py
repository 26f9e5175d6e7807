"""Host-side mirror of the reference's `Grid` / `StencilUpdate` interface over the C ABI.

Names, argument meaning and error behaviour follow the reference's C++ API for the cuda backend
(reference StencilStream/cuda/Grid.hpp:50-188 and StencilStream/cuda/StencilUpdate.hpp:41-198) so that
tests read like the reference's own (tests/GridTest.hpp, tests/StencilUpdateTest.hpp):

    grid = Grid("hotspot", rows, cols)            # Grid<Cell>(r, c)
    grid.copy_from_buffer(cells)                  # std::range_error  -> RangeError
    update = StencilUpdate("hotspot", Params(transition_function=..., halo_value=...,
                                             n_iterations=100, blocking=True))
    grid = update(grid)                           # operator()(GridImpl&)
    update.get_params().iteration_offset += 100   # live reference, re-read on every call
    update.get_walltime(); update.get_n_processed_cells(); update.get_kernel_runtime()

Every call ends in libstst_workloads.so (sm_100a kernels); nothing is computed in Python.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Any

import numpy as np

from . import _native
from ._native import CELL_DTYPES, PARAM_TYPES, UpdateParams, UpdateStats, WorkloadInfo


class RangeError(ValueError):
    """Counterpart of the `std::range_error` the reference throws on buffer/grid size mismatch
    (reference StencilStream/cuda/Grid.hpp:110-112, 128-130)."""


class StencilStreamError(RuntimeError):
    pass


_ERRORS = {-1: KeyError, -2: ValueError, -3: RangeError, -4: StencilStreamError}


def _check(lib, status: int) -> None:
    if status != 0:
        message = lib.stst_workloads_last_error().decode("utf-8", "replace")
        raise _ERRORS.get(status, StencilStreamError)(message)


def workload_names(strict: bool | None = None) -> list[str]:
    lib = _native.workloads_lib(strict)
    return [lib.stst_workload_name(i).decode() for i in range(lib.stst_workload_count())]


def workload_info(workload: str, strict: bool | None = None) -> WorkloadInfo:
    lib = _native.workloads_lib(strict)
    info = WorkloadInfo()
    _check(lib, lib.stst_workload_get_info(workload.encode(), C.byref(info)))
    return info


class _OwnedView(np.ndarray):
    """ndarray view that keeps the owning Grid (and with it the pinned memory) alive."""
    _owner = None

    def __array_finalize__(self, obj):
        self._owner = getattr(obj, "_owner", None)


class Grid:
    """A two-dimensional grid of cells resident in B200 HBM (mirror of `stencil::cuda::Grid<Cell>`).

    Copying the Python object reference shares the cells, like the reference's copy constructor;
    `share()` creates a second native handle to the same cells.
    """

    dimensions = 2

    def __init__(self, workload: str, rows=None, cols=None, *, buffer=None, device: int = -1,
                 strict: bool | None = None, _handle=None):
        self.workload = workload
        self._lib = _native.workloads_lib(strict)
        self._strict = strict
        self.dtype = CELL_DTYPES[workload]
        if _handle is not None:
            self._handle = _handle
            return
        if buffer is not None:
            buffer = np.asarray(buffer)
            if buffer.ndim != 2:
                raise RangeError("a grid buffer must be two-dimensional")
            rows, cols = buffer.shape
        elif cols is None and rows is not None and not np.isscalar(rows):
            rows, cols = rows  # Grid(range<2>)
        handle = C.c_void_p()
        _check(self._lib, self._lib.stst_grid_create(workload.encode(), int(rows), int(cols),
                                                     int(device), C.byref(handle)))
        self._handle = handle
        if buffer is not None:
            self.copy_from_buffer(buffer)

    def __del__(self):
        handle = getattr(self, "_handle", None)
        if handle:
            self._lib.stst_grid_destroy(handle)
            self._handle = None

    # -- reference API ----------------------------------------------------------------------------
    def get_grid_height(self) -> int:
        return self.get_grid_range()[0]

    def get_grid_width(self) -> int:
        return self.get_grid_range()[1]

    def get_grid_range(self) -> tuple[int, int]:
        rows, cols = C.c_size_t(), C.c_size_t()
        _check(self._lib, self._lib.stst_grid_shape(self._handle, C.byref(rows), C.byref(cols)))
        return (rows.value, cols.value)

    def make_similar(self) -> "Grid":
        handle = C.c_void_p()
        _check(self._lib, self._lib.stst_grid_make_similar(self._handle, C.byref(handle)))
        return Grid(self.workload, strict=self._strict, _handle=handle)

    def copy_from_buffer(self, buffer) -> None:
        """Overwrite the grid with `buffer` (2-D array of the workload's cell dtype, same extent)."""
        arr = np.ascontiguousarray(buffer, dtype=self.dtype)
        if arr.ndim != 2 or tuple(arr.shape) != self.get_grid_range():
            raise RangeError("The target buffer has not the same size as the grid")
        _check(self._lib, self._lib.stst_grid_copy_from_host(
            self._handle, arr.ctypes.data_as(C.c_void_p), arr.nbytes))

    def copy_to_buffer(self, buffer: np.ndarray) -> None:
        """Overwrite `buffer` (C-contiguous, cell dtype, same extent) with the grid contents."""
        if (not isinstance(buffer, np.ndarray) or buffer.dtype != self.dtype or buffer.ndim != 2
                or tuple(buffer.shape) != self.get_grid_range()):
            raise RangeError("The target buffer has not the same size as the grid")
        if not buffer.flags["C_CONTIGUOUS"] or not buffer.flags["WRITEABLE"]:
            raise ValueError("copy_to_buffer needs a writable C-contiguous array")
        _check(self._lib, self._lib.stst_grid_copy_to_host(
            self._handle, buffer.ctypes.data_as(C.c_void_p), buffer.nbytes))

    def accessor(self, mode: str = "read_write") -> np.ndarray:
        """Mirror of `Grid::GridAccessor<mode>` (reference Grid.hpp:145-153): a 2-D numpy view of the
        grid's pinned host image. Waits for device work on the grid; writable modes make the next
        update upload the image. The view keeps this grid object alive."""
        code = {"read": 0, "write": 1, "read_write": 2}[mode]
        ptr = C.c_void_p()
        _check(self._lib, self._lib.stst_grid_host_accessor(self._handle, code, C.byref(ptr)))
        rows, cols = self.get_grid_range()
        n_bytes = rows * cols * self.dtype.itemsize
        raw = (C.c_ubyte * max(n_bytes, 1)).from_address(ptr.value)
        view = np.frombuffer(raw, dtype=self.dtype, count=rows * cols).reshape(rows, cols)
        view = view.view(_OwnedView)
        view._owner = self
        if code == 0:
            view.flags.writeable = False
        return view

    # -- conveniences -------------------------------------------------------------------------------
    def to_numpy(self) -> np.ndarray:
        out = np.empty(self.get_grid_range(), dtype=self.dtype)
        self.copy_to_buffer(out)
        return out

    def host_image_is_pinned(self) -> bool:
        """Whether the accessor's host image is pinned memory (else it is moved through the staged
        pipeline of the runtime; boxes cap how much memory can be pinned)."""
        pinned = C.c_int()
        _check(self._lib, self._lib.stst_grid_host_image_is_pinned(self._handle, C.byref(pinned)))
        return bool(pinned.value)

    # -- B200 extensions: per-field device operations (include/stst_workloads.h) ----------------------
    def max_abs(self, extents) -> list[float]:
        """[(field, rows, cols), ...] -> max |cell.field| over the first rows x cols cells, evaluated
        on the device in one pass (the host loop of reference examples/convection/convection.cpp:412-438
        without migrating the grid). `field` is a member name of the cell struct or its index."""
        extents = list(extents)
        out = (C.c_double * max(len(extents), 1))()
        _check(self._lib, self._lib.stst_grid_max_abs(
            self._handle, _native.field_extents(self.workload, extents), len(extents), out))
        return [float(out[q]) for q in range(len(extents))]

    def field_to_numpy(self, field, out: np.ndarray | None = None) -> np.ndarray:
        """ONE field of every cell as a dense 2-D array (single-plane download), optionally into the
        C-contiguous array `out` (a reused destination avoids first-touch page faults)."""
        dtype = _native.field_dtype(self.workload, field)
        if out is None:
            out = np.empty(self.get_grid_range(), dtype=dtype)
        elif (out.dtype != dtype or tuple(out.shape) != self.get_grid_range()
              or not out.flags["C_CONTIGUOUS"]):
            raise RangeError("The target buffer has not the same size as the grid")
        _check(self._lib, self._lib.stst_grid_copy_field_to_host(
            self._handle, _native.field_index(self.workload, field),
            out.ctypes.data_as(C.c_void_p), out.nbytes))
        return out

    def copy_field_from_buffer(self, field, values) -> None:
        """Overwrite ONE field of every cell; `values` must have the grid's extent (else RangeError)."""
        arr = np.ascontiguousarray(values, dtype=_native.field_dtype(self.workload, field))
        if arr.ndim != 2 or tuple(arr.shape) != self.get_grid_range():
            raise RangeError("The target buffer has not the same size as the grid")
        _check(self._lib, self._lib.stst_grid_copy_field_from_host(
            self._handle, _native.field_index(self.workload, field),
            arr.ctypes.data_as(C.c_void_p), arr.nbytes))

    def share(self) -> "Grid":
        handle = C.c_void_p()
        _check(self._lib, self._lib.stst_grid_share(self._handle, C.byref(handle)))
        return Grid(self.workload, strict=self._strict, _handle=handle)

    def sync_to_device(self) -> None:
        """Upload a pending host image now (so that a following update times only device work)."""
        _check(self._lib, self._lib.stst_grid_sync_to_device(self._handle))


class GridBatch:
    """`members` independent grids of rows x cols cells of one workload on one device (mirror of
    `stencil::cuda::GridBatch<Cell>`), advanced together by `StencilUpdate`: one fused launch per pass
    for all members, each member's result equal to its own grid update. Buffers are (members, rows,
    cols) arrays of the workload's cell dtype."""

    def __init__(self, workload: str, members=None, rows=None, cols=None, *, buffer=None,
                 device: int = -1, strict: bool | None = None, _handle=None):
        self.workload = workload
        self._lib = _native.workloads_lib(strict)
        self._strict = strict
        self.dtype = CELL_DTYPES[workload]
        if _handle is not None:
            self._handle = _handle
            return
        if buffer is not None:
            buffer = np.asarray(buffer)
            if buffer.ndim != 3:
                raise RangeError("a grid batch buffer must be three-dimensional (members, rows, cols)")
            members, rows, cols = buffer.shape
        handle = C.c_void_p()
        _check(self._lib, self._lib.stst_batch_create(workload.encode(), int(members), int(rows),
                                                      int(cols), int(device), C.byref(handle)))
        self._handle = handle
        if buffer is not None:
            self.copy_from_buffer(buffer)

    def __del__(self):
        handle = getattr(self, "_handle", None)
        if handle:
            self._lib.stst_batch_destroy(handle)
            self._handle = None

    def shape(self) -> tuple[int, int, int]:
        """(members, rows, cols)."""
        m, r, c = C.c_size_t(), C.c_size_t(), C.c_size_t()
        _check(self._lib, self._lib.stst_batch_shape(self._handle, C.byref(m), C.byref(r), C.byref(c)))
        return (m.value, r.value, c.value)

    def get_members(self) -> int:
        return self.shape()[0]

    def get_grid_range(self) -> tuple[int, int]:
        """Extent of one member."""
        return self.shape()[1:]

    def copy_from_buffer(self, buffer, first_member: int = 0) -> None:
        """Overwrite members [first_member, first_member + len(buffer)) with `buffer`, a
        (n_members, rows, cols) array; the whole batch by default."""
        arr = np.ascontiguousarray(buffer, dtype=self.dtype)
        if arr.ndim != 3 or tuple(arr.shape[1:]) != self.get_grid_range():
            raise RangeError("The target buffer has not the same size as the grid batch members")
        _check(self._lib, self._lib.stst_batch_copy_from_host(
            self._handle, int(first_member), arr.shape[0], arr.ctypes.data_as(C.c_void_p), arr.nbytes))

    def copy_to_buffer(self, buffer: np.ndarray, first_member: int = 0) -> None:
        """Overwrite `buffer` (C-contiguous (n_members, rows, cols) array of the cell dtype) with
        members [first_member, first_member + n_members)."""
        if (not isinstance(buffer, np.ndarray) or buffer.dtype != self.dtype or buffer.ndim != 3
                or tuple(buffer.shape[1:]) != self.get_grid_range()):
            raise RangeError("The target buffer has not the same size as the grid batch members")
        if not buffer.flags["C_CONTIGUOUS"] or not buffer.flags["WRITEABLE"]:
            raise ValueError("copy_to_buffer needs a writable C-contiguous array")
        _check(self._lib, self._lib.stst_batch_copy_to_host(
            self._handle, int(first_member), buffer.shape[0], buffer.ctypes.data_as(C.c_void_p),
            buffer.nbytes))

    def to_numpy(self) -> np.ndarray:
        """All members as a (members, rows, cols) array."""
        out = np.empty(self.shape(), dtype=self.dtype)
        self.copy_to_buffer(out)
        return out

    def max_abs(self, extents, member: int) -> list[float]:
        """`Grid.max_abs` of member `member`: [(field, rows, cols), ...] in member coordinates."""
        extents = list(extents)
        out = (C.c_double * max(len(extents), 1))()
        _check(self._lib, self._lib.stst_batch_max_abs(
            self._handle, int(member), _native.field_extents(self.workload, extents), len(extents), out))
        return [float(out[q]) for q in range(len(extents))]

    def field_to_numpy(self, field) -> np.ndarray:
        """ONE field of every cell of every member as a (members, rows, cols) array."""
        out = np.empty(self.shape(), dtype=_native.field_dtype(self.workload, field))
        _check(self._lib, self._lib.stst_batch_copy_field_to_host(
            self._handle, _native.field_index(self.workload, field),
            out.ctypes.data_as(C.c_void_p), out.nbytes))
        return out


@dataclass
class Params:
    """Mirror of `StencilUpdate::Params` (reference StencilStream/cuda/StencilUpdate.hpp:54-105);
    the B200-only fields come last, as in the C++ aggregate."""

    transition_function: Any = None  # a ctypes struct from _native.PARAM_TYPES, or a dict of its fields
    halo_value: Any = None           # one cell (numpy scalar / tuple / python scalar); None = Cell()
    iteration_offset: int = 0
    n_iterations: int = 1
    device: Any = None
    blocking: bool = False
    profiling: bool = False
    cuda_device: int = -1
    fused_iterations: int = 0
    tile_rows: int = 0
    cuda_devices: Any = None         # list of CUDA ordinals to shard one update over (None: STST_DEVICES)


def _as_param_struct(workload: str, tf):
    cls = PARAM_TYPES[workload]
    if tf is None:
        return cls()
    if isinstance(tf, cls):
        return tf
    if isinstance(tf, dict):
        obj = cls()
        for key, value in tf.items():
            current = getattr(obj, key)
            if isinstance(current, C.Array):
                flat = np.asarray(value, dtype=np.float32).reshape(-1)
                C.memmove(C.addressof(current), flat.ctypes.data, flat.nbytes)
            else:
                setattr(obj, key, value)
        return obj
    raise TypeError(f"transition_function for {workload!r} must be {cls.__name__} or a dict")


class StencilUpdate:
    """Mirror of `stencil::cuda::StencilUpdate<F>` for the functor named by `workload`."""

    def __init__(self, workload: str, params: Params, *, strict: bool | None = None):
        self.workload = workload
        self._lib = _native.workloads_lib(strict)
        self._strict = strict
        self.params = params
        self._keepalive = None
        handle = C.c_void_p()
        native = self._native_params()
        _check(self._lib, self._lib.stst_update_create(workload.encode(), C.byref(native),
                                                       C.byref(handle)))
        self._handle = handle

    def __del__(self):
        handle = getattr(self, "_handle", None)
        if handle:
            self._lib.stst_update_destroy(handle)
            self._handle = None

    def _native_params(self) -> UpdateParams:
        p = self.params
        tf = _as_param_struct(self.workload, p.transition_function)
        native = UpdateParams()
        native.transition_function = C.addressof(tf)
        native.transition_function_bytes = C.sizeof(tf)
        halo = None
        if p.halo_value is not None:
            halo = np.zeros((), dtype=CELL_DTYPES[self.workload])
            halo[()] = p.halo_value
            native.halo_value = halo.ctypes.data
            native.halo_value_bytes = halo.nbytes
        native.iteration_offset = int(p.iteration_offset)
        native.n_iterations = int(p.n_iterations)
        native.blocking = int(bool(p.blocking))
        native.profiling = int(bool(p.profiling))
        native.cuda_device = int(p.cuda_device)
        native.fused_iterations = int(p.fused_iterations)
        native.tile_rows = int(p.tile_rows)
        devices = None
        if p.cuda_devices:
            devices = (C.c_int * len(p.cuda_devices))(*[int(d) for d in p.cuda_devices])
            native.cuda_devices = devices
            native.n_cuda_devices = len(p.cuda_devices)
        self._keepalive = (tf, halo, devices)
        return native

    def get_params(self) -> Params:
        """Live reference: modifications are used by the next call (reference :152)."""
        return self.params

    def __call__(self, source_grid):
        """operator(): a Grid gives a Grid, a GridBatch a GridBatch (every member advanced)."""
        native = self._native_params()
        _check(self._lib, self._lib.stst_update_set_params(self._handle, C.byref(native)))
        result = C.c_void_p()
        if isinstance(source_grid, GridBatch):
            _check(self._lib, self._lib.stst_update_apply_batch(self._handle, source_grid._handle,
                                                                C.byref(result)))
            return GridBatch(source_grid.workload, strict=self._strict, _handle=result)
        _check(self._lib, self._lib.stst_update_apply(self._handle, source_grid._handle,
                                                      C.byref(result)))
        return Grid(source_grid.workload, strict=self._strict, _handle=result)

    def get_stats(self) -> UpdateStats:
        stats = UpdateStats()
        _check(self._lib, self._lib.stst_update_get_stats(self._handle, C.byref(stats)))
        return stats

    def get_n_processed_cells(self) -> int:
        return int(self.get_stats().n_processed_cells)

    def get_walltime(self) -> float:
        return float(self.get_stats().walltime)

    def get_kernel_runtime(self) -> float:
        return float(self.get_stats().kernel_runtime)

    def get_n_launches(self) -> int:
        return int(self.get_stats().n_launches)
