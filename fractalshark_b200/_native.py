"""ctypes bindings of the two in-tree shared libraries. No fallback: a missing library raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
GPU_LIB_PATH = os.environ.get("FS_GPU_LIB") or os.path.join(_HERE, "libfsgpu.so")  # env override: A/B builds
HOST_LIB_PATH = os.path.join(_HERE, "libfshost.so")


class NativeLibraryMissing(RuntimeError):
    pass


class FsOrbit(C.Structure):  # fs_orbit (include/fs_gpu.h)
    _fields_ = [("elements", C.c_void_p), ("compressed_count", C.c_uint64), ("uncompressed_count", C.c_uint64),
                ("period_maybe_zero", C.c_uint64), ("orbit_x_low", C.c_void_p), ("orbit_y_low", C.c_void_p)]


class FsLaReference(C.Structure):  # fs_la_reference
    _fields_ = [("las", C.c_void_p), ("num_las", C.c_uint64), ("stages", C.c_void_p), ("num_stages", C.c_uint64),
                ("at", C.c_void_p), ("la_stage_count", C.c_uint64), ("use_at", C.c_int32), ("is_valid", C.c_int32)]


class FsBlas(C.Structure):  # fs_blas
    _fields_ = [("levels", C.POINTER(C.c_void_p)), ("level_counts", C.POINTER(C.c_uint64)),
                ("num_levels", C.c_uint32), ("first_level", C.c_uint32), ("lm2", C.c_int32)]


class FsReduction(C.Structure):  # fs_reduction
    _fields_ = [("Min", C.c_uint64), ("Max", C.c_uint64), ("Sum", C.c_uint64)]


DONE_CALLBACK = C.CFUNCTYPE(None, C.c_void_p)

_V, _U32, _I32, _U64 = C.c_void_p, C.c_uint32, C.c_int32, C.c_uint64

# name -> (restype, argtypes); exactly the symbols declared in include/fs_gpu.h
GPU_SYMBOLS = {
    "fs_test_cuda_is_working": (_U32, []),
    "fs_create": (_V, [_I32]),
    "fs_destroy": (None, [_V]),
    "fs_create_group": (_V, [C.POINTER(C.c_int32), _U32]),
    "fs_create_default": (_V, []),
    "fs_device_count": (_U32, [_V]),
    "fs_initialize_memory": (_U32, [_V, _U32, _U32, _U32, _U32, _V, _U32, _U32, _U64, _I32]),
    "fs_initialize_perturb": (_U32, [_V, _U32, _I32, _I32, _U64, C.POINTER(FsOrbit), _I32, _U64, C.POINTER(FsOrbit),
                                     C.POINTER(FsLaReference)]),
    "fs_clear_memory": (None, [_V]),
    "fs_render": (_U32, [_V, _U32, _I32, _V, _V, _V, _V, _U64, _I32]),
    "fs_render_perturb_lav2": (_U32, [_V, _U32, _I32, _I32, _I32, _V, _V, _V, _V, _V, _V, _U64]),
    "fs_render_perturb_lav2_frames": (_U32, [_V, _U32, _I32, _I32, _I32, _U32, _V, _V, _V, _V, _V, _V, _U64]),
    "fs_select_frame": (_U32, [_V, _U32]),
    "fs_render_perturb_lav2_expmap": (_U32, [_V, _U32, _I32, _I32, _I32, _V, _V, _V, _U64]),
    "fs_render_perturb_bla": (_U32, [_V, _U32, _I32, C.POINTER(FsOrbit), C.POINTER(FsBlas), _V, _V, _V, _V, _V, _V,
                                     _U64, _I32]),
    "fs_render_perturb_bla_scaled": (_U32, [_V, _U32, _I32, C.POINTER(FsOrbit), C.POINTER(FsOrbit), _V, _V, _V, _V,
                                            _V, _V, _U64, _I32]),
    "fs_render_current": (_U32, [_V, _U64, _V, _V, C.POINTER(FsReduction), _I32]),
    "fs_render_current_shard": (_U32, [_V, _U64, _V, _V, C.POINTER(FsReduction), _I32]),
    "fs_set_result_sink": (_U32, [_V, _V, _U64]),
    "fs_sync_compute_stream": (_U32, [_V]),
    "fs_sync_display_stream": (_U32, [_V]),
    "fs_query_compute_stream": (_U32, [_V]),
    "fs_enqueue_compute_done_callback": (_U32, [_V, DONE_CALLBACK, _V]),
    "fs_convert_error_to_string": (C.c_char_p, [_U32]),
    "fs_get_width": (_U32, [_V]),
    "fs_get_height": (_U32, [_V]),
    "fs_set_shard": (_U32, [_V, _U32, _U32]),
    "fs_measure_fp32_issue_peak": (_U32, [_I32, C.POINTER(C.c_double)]),
    "fs_measure_fp64_issue_peak": (_U32, [_I32, C.POINTER(C.c_double)]),
    "fs_last_render_ms": (_U32, [_V, C.POINTER(C.c_float)]),
    "fs_enable_step_counter": (_U32, [_V, _I32]),
    "fs_read_step_counter": (_U32, [_V, C.POINTER(_U64)]),
    "fs_read_step_counters": (_U32, [_V, C.POINTER(_U64)]),
    "fs_set_scaled_steps": (_U32, [_V, _I32]),
    "fs_set_split_at": (_U32, [_V, _I32]),
    "fs_set_pool_kernel": (_U32, [_V, _I32]),
    "fs_selftest_numeric_op": (_U32, [_I32, _U32, _V, _V, _V, _U64]),
    "fs_set_la_step2": (_U32, [_V, _I32]),
    "fs_set_at_cycle_detection": (_U32, [_V, _I32]),
    "fs_device_iter_buffer": (_V, [_V]),
    "fs_kernel_launch_count": (_U64, [_V]),
}

HOST_SYMBOLS = {
    "fsh_view_create": (_V, [C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p, _U32, _U32, _U32, _I32]),
    "fsh_view_zoom": (_V, [_V, C.c_char_p]),
    "fsh_view_destroy": (None, [_V]),
    "fsh_view_precision_bits": (_U32, [_V]),
    "fsh_view_coords": (_I32, [_V, _I32, _V, _V, _V, _V, _V, _V]),
    "fsh_view_expmap": (_I32, [_V, _I32, _U32, _V, _V, _V, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "fsh_selftest_numeric_op": (_I32, [_U32, _V, _V, _V, _U64]),
    "fsh_orbit_compute": (_V, [_V, _I32, _U64, _I32]),
    "fsh_orbit_with_bad": (_V, [_V, _I32]),
    "fsh_orbit_compress": (_V, [_V, _I32]),
    "fsh_orbit_uncompressed_count": (_U64, [_V]),
    "fsh_orbit_replay_data": (_V, [_V]),
    "fsh_orbit_destroy": (None, [_V]),
    "fsh_orbit_data": (_V, [_V]),
    "fsh_orbit_count": (_U64, [_V]),
    "fsh_orbit_period": (_U64, [_V]),
    "fsh_orbit_elem_bytes": (_U64, [_V]),
    "fsh_orbit_x_low": (_V, [_V]),
    "fsh_orbit_y_low": (_V, [_V]),
    "fsh_orbit_max_radius": (_V, [_V]),
    "fsh_la_build": (_V, [_V, _U32]),
    "fsh_la_destroy": (None, [_V]),
    "fsh_la_las": (_V, [_V]),
    "fsh_la_num_las": (_U64, [_V]),
    "fsh_la_stages": (_V, [_V]),
    "fsh_la_num_stages": (_U64, [_V]),
    "fsh_la_at": (_V, [_V]),
    "fsh_la_at_bytes": (_U64, [_V]),
    "fsh_la_stage_count": (_U64, [_V]),
    "fsh_la_use_at": (_I32, [_V]),
    "fsh_la_is_valid": (_I32, [_V]),
    "fsh_blas_build": (_V, [_V]),
    "fsh_blas_destroy": (None, [_V]),
    "fsh_blas_num_levels": (_U32, [_V]),
    "fsh_blas_lm2": (_I32, [_V]),
    "fsh_blas_elem_bytes": (_U64, [_V]),
    "fsh_blas_levels": (C.POINTER(C.c_void_p), [_V]),
    "fsh_blas_level_counts": (C.POINTER(C.c_uint64), [_V]),
}


def _load(path: str, symbols: dict) -> C.CDLL:
    if not os.path.exists(path):
        raise NativeLibraryMissing(
            f"{path} is not built. Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C fractalshark_b200/csrc`). There is no CPU fallback for the render path.")
    lib = C.CDLL(path)
    for name, (res, args) in symbols.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing: fail loudly
        fn.restype = res
        fn.argtypes = args
    return lib


_gpu = None
_host = None


def gpu_lib() -> C.CDLL:
    global _gpu
    if _gpu is None:
        _gpu = _load(GPU_LIB_PATH, GPU_SYMBOLS)
    return _gpu


def host_lib() -> C.CDLL:
    global _host
    if _host is None:
        _host = _load(HOST_LIB_PATH, HOST_SYMBOLS)
    return _host
