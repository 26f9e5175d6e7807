"""ctypes bindings for the two C-ABI libraries (include/stst_rt.h, include/stst_workloads.h).

The libraries are built in-tree by `stencilstream_b200._build` and loaded from the package
directory. There is no fallback of any kind: if a library is missing, loading raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

PKG = Path(__file__).resolve().parent


class NativeLibraryMissing(RuntimeError):
    pass


# ---- structs of include/stst_workloads.h ---------------------------------------------------------

class ConwayParams(C.Structure):
    _fields_ = [("reserved", C.c_int32)]


class Jacobi5Params(C.Structure):
    _fields_ = [("coef", C.c_float * 5)]


class Jacobi9Params(C.Structure):
    _fields_ = [("coef", (C.c_float * 3) * 3)]


class JacobiStarParams(C.Structure):
    _fields_ = [("centre", C.c_float), ("arm", C.c_float * 3)]


class HotspotParams(C.Structure):
    _fields_ = [("Rx_1", C.c_float), ("Ry_1", C.c_float), ("Rz_1", C.c_float), ("Cap_1", C.c_float)]


class FdtdParams(C.Structure):
    _fields_ = [
        ("dt", C.c_float), ("t_0", C.c_float), ("tau", C.c_float), ("omega", C.c_float),
        ("cutoff_iteration", C.c_uint64), ("detect_iteration", C.c_uint64),
        ("source_radius_squared", C.c_float), ("source_r", C.c_float), ("source_c", C.c_float),
        ("source_distance_bound", C.c_float), ("double_center_rc", C.c_float),
    ]


class ConvectionPTParams(C.Structure):
    _fields_ = [
        ("nx", C.c_uint64), ("ny", C.c_uint64), ("roh0_g_alpha", C.c_double),
        ("delta_eta_delta_T", C.c_double), ("eta0", C.c_double), ("deltaT", C.c_double),
        ("dx", C.c_double), ("dy", C.c_double), ("delta_tau_iter", C.c_double), ("beta", C.c_double),
        ("rho", C.c_double), ("dampX", C.c_double), ("dampY", C.c_double), ("DcT", C.c_double),
    ]


class ConvectionThermalParams(C.Structure):
    _fields_ = [("nx", C.c_uint64), ("ny", C.c_uint64), ("dx", C.c_double), ("dy", C.c_double),
                ("dt", C.c_double), ("DcT", C.c_double)]


class KatParams(C.Structure):
    _fields_ = [("reserved", C.c_int32)]


class WorkloadInfo(C.Structure):
    _fields_ = [("cell_bytes", C.c_size_t), ("params_bytes", C.c_size_t), ("n_planes", C.c_size_t),
                ("stencil_radius", C.c_size_t), ("n_subiterations", C.c_size_t),
                ("bytes_per_cell_iteration", C.c_size_t)]


class UpdateParams(C.Structure):
    _fields_ = [
        ("transition_function", C.c_void_p), ("transition_function_bytes", C.c_size_t),
        ("halo_value", C.c_void_p), ("halo_value_bytes", C.c_size_t),
        ("iteration_offset", C.c_size_t), ("n_iterations", C.c_size_t),
        ("blocking", C.c_int), ("profiling", C.c_int), ("cuda_device", C.c_int),
        ("fused_iterations", C.c_uint), ("tile_rows", C.c_uint),
        ("cuda_devices", C.POINTER(C.c_int)), ("n_cuda_devices", C.c_size_t),
    ]


class UpdateStats(C.Structure):
    _fields_ = [
        ("n_processed_cells", C.c_size_t), ("walltime", C.c_double), ("kernel_runtime", C.c_double),
        ("n_launches", C.c_size_t), ("fused_iterations", C.c_uint), ("tile_h", C.c_uint),
        ("tile_w", C.c_uint), ("block_x", C.c_uint), ("block_y", C.c_uint), ("use_tma", C.c_uint),
        ("smem_bytes", C.c_size_t), ("passthrough_planes", C.c_uint), ("speculation_redos", C.c_size_t),
        ("n_slabs", C.c_size_t),
    ]


class FieldExtent(C.Structure):
    _fields_ = [("field", C.c_size_t), ("rows", C.c_size_t), ("cols", C.c_size_t)]


class DeviceInfo(C.Structure):
    _fields_ = [
        ("sm_count", C.c_int), ("cc_major", C.c_int), ("cc_minor", C.c_int),
        ("max_smem_per_block_optin", C.c_int), ("max_smem_per_sm", C.c_int), ("l2_bytes", C.c_int),
        ("clock_khz", C.c_int), ("total_mem", C.c_size_t), ("free_mem", C.c_size_t),
        ("name", C.c_char * 128),
    ]


# ---- cell dtypes (array-of-structs images) -----------------------------------------------------------

CELL_DTYPES = {
    "conway": np.dtype(np.bool_),
    "jacobi5": np.dtype(np.float32),
    "jacobi9": np.dtype(np.float32),
    "jacobi_r2": np.dtype(np.float32),
    "jacobi_r3": np.dtype(np.float32),
    "hotspot": np.dtype([("temp", "<f4"), ("power", "<f4")]),
    "fdtd": np.dtype([(n, "<f4") for n in ("ex", "ey", "hz", "hz_sum", "ca", "cb", "da", "db")]),
    "convection_pt": np.dtype([(n, "<f8") for n in (
        "T", "Pt", "Vx", "Vy", "tau_xx", "tau_yy", "sigma_xy", "dVxd_tau", "dVyd_tau", "ErrV", "ErrP")]),
    "kat": np.dtype([(n, "<i4") for n in ("r", "c", "i_iteration", "i_subiteration", "status")]),
}
CELL_DTYPES["convection_thermal"] = CELL_DTYPES["convection_pt"]
CELL_DTYPES["kat_r2"] = CELL_DTYPES["kat"]



def field_index(workload: str, field) -> int:
    """Plane index of `field` (a member name of the workload's cell struct, or already an index)."""
    if isinstance(field, (int, np.integer)):
        return int(field)
    names = CELL_DTYPES[workload].names
    if not names or field not in names:
        raise KeyError(f"workload {workload!r} has no cell field {field!r}")
    return names.index(field)


def field_dtype(workload: str, field) -> np.dtype:
    dtype = CELL_DTYPES[workload]
    if not dtype.names:
        return dtype
    return dtype[dtype.names[field_index(workload, field)]]


def field_extents(workload: str, extents):
    """ctypes array of FieldExtent from [(field, rows, cols), ...]."""
    arr = (FieldExtent * max(len(extents), 1))()
    for q, (field, rows, cols) in enumerate(extents):
        arr[q].field, arr[q].rows, arr[q].cols = field_index(workload, field), int(rows), int(cols)
    return arr


PARAM_TYPES = {
    "conway": ConwayParams,
    "jacobi5": Jacobi5Params,
    "jacobi9": Jacobi9Params,
    "jacobi_r2": JacobiStarParams,
    "jacobi_r3": JacobiStarParams,
    "hotspot": HotspotParams,
    "fdtd": FdtdParams,
    "convection_pt": ConvectionPTParams,
    "convection_thermal": ConvectionThermalParams,
    "kat": KatParams,
    "kat_r2": KatParams,
}

# Every symbol include/stst_rt.h declares (checked by the CPU test-suite against the built library).
RT_SYMBOLS = [
    "stst_rt_abi_version", "stst_last_error", "stst_device_count", "stst_get_device_info",
    "stst_set_device", "stst_malloc", "stst_free", "stst_malloc_ipc", "stst_free_ipc",
    "stst_malloc_host", "stst_free_host", "stst_host_cache_trim", "stst_host_register", "stst_host_unregister",
    "stst_memset_async", "stst_memcpy_h2d_async", "stst_memcpy_d2h_async", "stst_memcpy_d2d_async",
    "stst_memcpy_2d_async", "stst_memcpy_peer_async",
    "stst_memcpy_2d_staged", "stst_memcpy_2d_auto", "stst_host_memcpy", "stst_host_is_pinned", "stst_default_stream", "stst_stream_create",
    "stst_stream_destroy", "stst_stream_synchronize", "stst_stream_wait_event", "stst_event_create",
    "stst_event_destroy", "stst_event_record", "stst_event_synchronize", "stst_event_elapsed_ms",
    "stst_device_synchronize", "stst_stream_write_value32", "stst_stream_wait_value32_geq", "stst_tensor_map_encode_2d", "stst_peer_can_access",
    "stst_peer_enable", "stst_ipc_get_mem_handle", "stst_ipc_open_mem_handle",
    "stst_ipc_close_mem_handle", "stst_ipc_get_event_handle", "stst_ipc_open_event_handle",
    "stst_event_create_ipc", "stst_nccl_available", "stst_nccl_get_unique_id",
    "stst_nccl_comm_init_rank", "stst_nccl_comm_destroy", "stst_nccl_neighbor_exchange",
]

WORKLOADS_SYMBOLS = [
    "stst_workloads_abi_version", "stst_workloads_last_error", "stst_workload_count",
    "stst_workload_name", "stst_workload_get_info", "stst_grid_create", "stst_grid_share",
    "stst_grid_make_similar", "stst_grid_destroy", "stst_grid_shape", "stst_grid_copy_from_host",
    "stst_grid_copy_to_host", "stst_grid_sync_to_device", "stst_grid_host_accessor", "stst_grid_host_image_is_pinned",
    "stst_grid_max_abs", "stst_grid_copy_field_to_host", "stst_grid_copy_field_from_host",
    "stst_slab_max_abs", "stst_slab_copy_field_rows_to_host", "stst_slab_copy_from_slab", "stst_slab_enable_speculation",
    "stst_slab_backup", "stst_slab_restore", "stst_slab_take_violations", "stst_slab_drop_passthrough",
    "stst_update_create",
    "stst_update_set_params", "stst_update_apply", "stst_update_get_stats", "stst_update_destroy",
    "stst_slab_create", "stst_slab_destroy", "stst_slab_get_info", "stst_slab_get_ipc_handle",
    "stst_slab_attach_ipc", "stst_slab_attach_local", "stst_slab_detach", "stst_slab_use_nccl", "stst_slab_copy_from_host",
    "stst_slab_copy_to_host", "stst_slab_copy_rows_from_host", "stst_slab_copy_rows_to_host",
    "stst_slab_exchange_halos", "stst_slab_update", "stst_slab_synchronize",
    "stst_slab_record_event",
    "stst_batch_create", "stst_batch_destroy", "stst_batch_shape", "stst_batch_copy_from_host",
    "stst_batch_copy_to_host", "stst_batch_max_abs", "stst_batch_copy_field_to_host",
    "stst_update_apply_batch",
]

_libs: dict = {}


def _load(path: Path):
    if not path.exists():
        raise NativeLibraryMissing(
            f"{path} is missing. Build it with `python -m stencilstream_b200._build` "
            "(StencilStream-B200 has no CPU or pure-Python fallback).")
    return C.CDLL(str(path), mode=C.RTLD_GLOBAL)


def runtime_lib():
    if "rt" not in _libs:
        lib = _load(PKG / "libstst_rt.so")
        lib.stst_last_error.restype = C.c_char_p
        lib.stst_get_device_info.argtypes = [C.c_int, C.POINTER(DeviceInfo)]
        lib.stst_device_count.argtypes = [C.POINTER(C.c_int)]
        lib.stst_set_device.argtypes = [C.c_int]
        lib.stst_nccl_get_unique_id.argtypes = [C.c_char_p]
        lib.stst_nccl_comm_init_rank.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_char_p, C.c_int]
        lib.stst_nccl_comm_destroy.argtypes = [C.c_void_p]
        _libs["rt"] = lib
    return _libs["rt"]


def workloads_lib(strict: bool | None = None):
    """The workloads library; `strict` selects the -fmad=false build (default: env STST_STRICT)."""
    if strict is None:
        strict = os.environ.get("STST_STRICT", "0") not in ("", "0")
    key = "wl_strict" if strict else "wl"
    if key not in _libs:
        runtime_lib()
        name = "libstst_workloads_strict.so" if strict else "libstst_workloads.so"
        if not strict and os.environ.get("STST_WORKLOADS_LIB"):
            name = os.environ["STST_WORKLOADS_LIB"]  # an experimental build (see _build.build_variant)
        lib = _load(PKG / name)
        vp = C.c_void_p
        lib.stst_workloads_last_error.restype = C.c_char_p
        lib.stst_workload_name.restype = C.c_char_p
        lib.stst_workload_name.argtypes = [C.c_int]
        lib.stst_workload_get_info.argtypes = [C.c_char_p, C.POINTER(WorkloadInfo)]
        lib.stst_grid_create.argtypes = [C.c_char_p, C.c_size_t, C.c_size_t, C.c_int, C.POINTER(vp)]
        lib.stst_grid_share.argtypes = [vp, C.POINTER(vp)]
        lib.stst_grid_make_similar.argtypes = [vp, C.POINTER(vp)]
        lib.stst_grid_destroy.argtypes = [vp]
        lib.stst_grid_shape.argtypes = [vp, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
        lib.stst_grid_copy_from_host.argtypes = [vp, vp, C.c_size_t]
        lib.stst_grid_copy_to_host.argtypes = [vp, vp, C.c_size_t]
        lib.stst_grid_sync_to_device.argtypes = [vp]
        lib.stst_grid_host_accessor.argtypes = [vp, C.c_int, C.POINTER(vp)]
        lib.stst_grid_host_image_is_pinned.argtypes = [vp, C.POINTER(C.c_int)]
        lib.stst_grid_max_abs.argtypes = [vp, C.POINTER(FieldExtent), C.c_size_t,
                                          C.POINTER(C.c_double)]
        lib.stst_grid_copy_field_to_host.argtypes = [vp, C.c_size_t, vp, C.c_size_t]
        lib.stst_grid_copy_field_from_host.argtypes = [vp, C.c_size_t, vp, C.c_size_t]
        lib.stst_slab_max_abs.argtypes = [vp, C.POINTER(FieldExtent), C.c_size_t,
                                          C.POINTER(C.c_double)]
        lib.stst_slab_copy_field_rows_to_host.argtypes = [vp, C.c_size_t, C.c_size_t, C.c_size_t, vp,
                                                          C.c_size_t]
        lib.stst_update_create.argtypes = [C.c_char_p, C.POINTER(UpdateParams), C.POINTER(vp)]
        lib.stst_update_set_params.argtypes = [vp, C.POINTER(UpdateParams)]
        lib.stst_update_apply.argtypes = [vp, vp, C.POINTER(vp)]
        lib.stst_update_get_stats.argtypes = [vp, C.POINTER(UpdateStats)]
        lib.stst_update_destroy.argtypes = [vp]
        lib.stst_batch_create.argtypes = [C.c_char_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int,
                                          C.POINTER(vp)]
        lib.stst_batch_destroy.argtypes = [vp]
        lib.stst_batch_shape.argtypes = [vp, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t),
                                         C.POINTER(C.c_size_t)]
        lib.stst_batch_copy_from_host.argtypes = [vp, C.c_size_t, C.c_size_t, vp, C.c_size_t]
        lib.stst_batch_copy_to_host.argtypes = [vp, C.c_size_t, C.c_size_t, vp, C.c_size_t]
        lib.stst_batch_max_abs.argtypes = [vp, C.c_size_t, C.POINTER(FieldExtent), C.c_size_t,
                                           C.POINTER(C.c_double)]
        lib.stst_batch_copy_field_to_host.argtypes = [vp, C.c_size_t, vp, C.c_size_t]
        lib.stst_update_apply_batch.argtypes = [vp, vp, C.POINTER(vp)]
        _libs[key] = lib
    return _libs[key]
