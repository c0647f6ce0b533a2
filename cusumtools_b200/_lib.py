"""ctypes binding of libcusumtools_b200.so (the C ABI declared in include/cusumtools_b200.h).

There is no CPU fallback: if the library is missing or a call fails, an exception is
raised.  Loading the library does not need a GPU (tests check the exported symbols on
CPU); any compute call without one fails loudly inside CUDA.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CT_LIB_PATH") or os.path.join(_HERE, "libcusumtools_b200.so")   # override: A/B builds

CT_MAX_SECTIONS = 5


class CtFilterCoef(C.Structure):
    _fields_ = [
        ("nsec", C.c_int32),
        ("order", C.c_int32),
        ("na1", C.c_float * CT_MAX_SECTIONS),
        ("na2", C.c_float * CT_MAX_SECTIONS),
        ("ss", C.c_float * CT_MAX_SECTIONS),
        ("fir", C.c_float * (2 * CT_MAX_SECTIONS + 1)),
        ("gain", C.c_float),
    ]


_vp, _i64, _i32, _f32, _u16, _u32 = C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_uint16, C.c_uint32


class CtFilterStats(C.Structure):
    _fields_ = [("origin", C.c_int64), ("block", C.c_int64), ("bmin", C.c_float), ("bmax", C.c_float),
                ("c0", C.c_float), ("shift", C.c_int32), ("cnt", C.c_void_p), ("s1", C.c_void_p), ("s2", C.c_void_p)]


# name -> (restype, argtypes); every symbol include/cusumtools_b200.h declares
SIGNATURES = {
    "ct_version": (C.c_int, []),
    "ct_last_error": (C.c_char_p, []),
    "ct_launch_count": (C.c_uint64, []),
    "ct_launch_count_reset": (None, []),
    "ct_device_info": (C.c_int, [_vp, _vp, _vp, _vp]),
    "ct_filter_seq_tile": (C.c_int, []),
    "ct_filter_decimation": (C.c_int, [C.POINTER(CtFilterCoef), _i64, C.c_int]),
    "ct_filter_summary_count": (_i64, [_i64, _i64, C.c_int]),
    "ct_filtfilt_workspace_bytes": (_i64, [_i64, _i64, C.c_int]),
    "ct_filtfilt_stats_granule": (_i64, [_i64, _i64, C.c_int]),
    "ct_filter_forward_u16": (C.c_int, [_vp, _i64, _i64, _f32, _u16, _f32, C.POINTER(CtFilterCoef), C.c_int, _i64, C.c_int,
                                        _u32, _u32, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _vp]),
    "ct_median_verify": (C.c_int, [_vp, C.c_int, _i64, _i64, _u32, _u32, _f32, _vp, _vp]),
    "ct_filter_forward_ends_u16": (C.c_int, [_vp, _i64, _i64, _f32, _u16, _vp, C.POINTER(CtFilterCoef), C.c_int, _i64, _vp, _i64,
                                             _vp]),
    "ct_filter_backward": (C.c_int, [_i64, _i64, _f32, _f32, _f32, C.POINTER(CtFilterCoef), C.c_int, _i64, _vp, _vp, _i64,
                                     C.POINTER(CtFilterStats), _vp, _vp]),
    "ct_filtfilt_u16": (C.c_int, [_vp, _i64, _i64, _f32, _u16, _f32, _f32, C.POINTER(CtFilterCoef),
                                  C.c_int, C.c_int, _vp, _vp, _i64, C.POINTER(CtFilterStats), _vp]),
    "ct_filtfilt_f32": (C.c_int, [_vp, _i64, _i64, _f32, C.POINTER(CtFilterCoef), C.c_int,
                                  C.c_int, _vp, _vp, _i64, C.POINTER(CtFilterStats), _vp]),
    "ct_hist_sampled_u16": (C.c_int, [_vp, _i64, _i64, _u16, _vp, _vp]),
    "ct_hist_rank": (C.c_int, [_vp, C.c_int, _vp, _vp]),
    "ct_count_window_u16": (C.c_int, [_vp, _i64, _u16, _u32, _u32, _vp, _vp]),
    "ct_count_window4_u16": (C.c_int, [_vp, _i64, _u16, _u32, _u32, _vp, _vp]),
    "ct_block_stats_f32": (C.c_int, [_vp, _i64, _i64, _f32, _f32, _f32, C.c_int, _vp, _vp, _vp, _vp]),
    "ct_detect_run": (C.c_int, []),
    "ct_detect_workspace_bytes": (_i64, [_i64]),
    "ct_detect_f32": (C.c_int, [_vp, _i64, _i64, _vp, _vp, _vp, C.c_int, _vp, _i64, _vp, _i64, _vp, _vp, _i64, _vp, _vp]),
    "ct_welch_workspace_bytes": (_i64, [_i32, _i32]),
    "ct_welch_f32": (C.c_int, [_vp, _i64, _i32, _f32, _i32, _i32, _vp, _i64, _vp, _vp, _vp]),
    "ct_bin_be_f64_to_f32": (C.c_int, [_vp, _i64, _vp, _vp]),
    "ct_i2be_to_f32": (C.c_int, [_vp, _i64, _f32, _vp, _vp]),
    "ct_dequant_u16": (C.c_int, [_vp, _i64, _u16, C.c_double, C.c_double, _vp, _vp]),
    "ct_radix_hist_f32": (C.c_int, [_vp, _i64, _u32, _i32, _i32, _vp, _vp]),
    "ct_baseline_finalize": (C.c_int, [_vp, _vp, _vp, _i64, _f32, C.c_int, _i64, C.c_double, C.c_double, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ct_event_windows": (C.c_int, [_vp, _vp, _vp, _i64, _i64, _i64, _i64, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    "ct_cusum_workspace_bytes": (_i64, [_i64]),
    "ct_welch_single_workspace_bytes": (_i64, [_i64]),
    "ct_welch_single_f32": (C.c_int, [_vp, _i64, C.c_double, C.c_int32, _vp, _i64, _vp, _vp]),
    "ct_event_extrema_f32": (C.c_int, [_vp, _i64, _vp, _vp, _i64, _vp, _vp, _vp, _vp]),
    "ct_event_columns": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, C.c_int, _vp, _vp, _vp]),
    "ct_intra_crossings_f32": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _i64, _vp, _i64, _i64, _vp, _vp, _vp, C.c_int32, _vp, _vp, _vp]),
    "ct_cusum_batch_dev": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _i64, _f32, _f32, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "ct_cusum_batch": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _i64, _f32, _f32, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "ct_stepfit_select": (C.c_int, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _vp]),
    "ct_stepfit_batch": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _i64, _i64, _f32, C.c_int, C.c_int, _vp, _vp, _vp, _vp, _vp,
                                   _vp, _vp, _vp]),
    "ct_stepfit_fallback_select": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp]),
    "ct_stepfit_long_batch": (C.c_int, [_vp, _i64, _vp, _vp, _vp, _vp, _i64, _i64, _f32, C.c_int, C.c_int, _vp, _vp, _vp, _vp,
                                        _vp, _vp, _vp, _vp, _vp]),
}
STEPFIT_MAX_WINDOW = 8192     # CT_STEPFIT_MAX_WINDOW
STEPFIT_LONG_MAX_WINDOW = 131072     # CT_STEPFIT_LONG_MAX_WINDOW
TYPE_STEPFIT_LONG = 8         # CT_TYPE_STEPFIT_LONG

_lib = None


def build(force: bool = False) -> str:
    """Compile the library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    if force or not os.path.exists(LIB_PATH):
        subprocess.check_call([os.path.join(_HERE, "csrc", "build.sh")])
    return LIB_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with cusumtools_b200/csrc/build.sh "
                "(python -c 'import __graft_entry__ as g; g.build()'). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().ct_last_error().decode("utf-8", "replace")
        if rc == -1:
            raise ValueError(f"{what}: {msg}")
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")


def launch_count() -> int:
    return int(lib().ct_launch_count())


def reset_launch_count() -> None:
    lib().ct_launch_count_reset()
