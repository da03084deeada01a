"""ctypes binding of libghostcwt.so (include/ghost_cwt.h).

There is no CPU fallback: if the shared library has not been built the import
of any compute entry point raises, and every compute call needs a CUDA device.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libghostcwt.so")

F32, F64 = 0, 1
OUT_COMPLEX, OUT_AMPLITUDE, OUT_POWER = 0, 1, 2
FLAG_FORCE_GENERIC = 1
FLAG_NO_INTERP = 2
FLAG_NO_GUARD = 4
POOL_MEAN, POOL_MAX = 0, 1
KERNEL_FULL, KERNEL_BANDED, KERNEL_INTERP, KERNEL_WIDE2 = 0, 1, 2, 3

EXPORTS = (
    "gcwt_version", "gcwt_last_error", "gcwt_launch_count", "gcwt_plan_create",
    "gcwt_plan_destroy", "gcwt_plan_levels", "gcwt_plan_classes", "gcwt_plan_workspace_bytes",
    "gcwt_channel_means", "gcwt_execute", "gcwt_execute_host", "gcwt_filter_response",
    "gcwt_morse_kernel", "gcwt_profile_enable", "gcwt_profile_read",
    "gcwt_fastconv", "gcwt_dft", "gcwt_analytic_signal", "gcwt_moments", "gcwt_interp_taps",
    "gcwt_guard_stats", "gcwt_host_stats", "gcwt_pool_rows", "gcwt_execute_host_pooled",
    "gcwt_band_reduce", "gcwt_execute_host_bands", "gcwt_event_reduce", "gcwt_execute_host_events",
)


class GcwtError(RuntimeError):
    pass


class PlanDesc(C.Structure):
    _fields_ = [
        ("n_scales", C.c_int32),
        ("lengths", C.POINTER(C.c_int64)),
        ("k_first", C.POINTER(C.c_int32)),
        ("n_terms", C.POINTER(C.c_int32)),
        ("terms", C.POINTER(C.c_double)),
        ("compute_type", C.c_int32),
        ("out_kind", C.c_int32),
        ("device", C.c_int32),
        ("flags", C.c_int32),
        ("band_tol", C.c_double),
        ("guard_tol", C.c_double),
    ]


class ClassInfo(C.Structure):
    _fields_ = [
        ("level", C.c_int32),
        ("kernel", C.c_int32),
        ("log2u", C.c_int32),
        ("n_scales", C.c_int32),
        ("chunk", C.c_int64),
        ("offset", C.c_int64),
        ("hop", C.c_int64),
    ]


_lib = None


def load():
    """Load the library once; raise loudly if it was never built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GcwtError(
            "ghost_b200: %s is missing. Build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (needs nvcc). There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, dp = C.c_void_p, C.c_int32, C.c_int64, C.POINTER(C.c_double)
    lib.gcwt_version.restype = C.c_int
    lib.gcwt_last_error.restype = C.c_char_p
    lib.gcwt_launch_count.restype = i64
    lib.gcwt_launch_count.argtypes = [i32]
    lib.gcwt_plan_create.argtypes = [C.POINTER(vp), C.POINTER(PlanDesc)]
    lib.gcwt_plan_destroy.argtypes = [vp]
    lib.gcwt_plan_levels.argtypes = [vp, C.POINTER(i32)]
    lib.gcwt_plan_classes.argtypes = [vp, C.POINTER(i32), C.POINTER(ClassInfo), C.POINTER(i32)]
    lib.gcwt_plan_workspace_bytes.restype = C.c_size_t
    lib.gcwt_plan_workspace_bytes.argtypes = [vp]
    lib.gcwt_channel_means.argtypes = [vp, i32, i64, i64, i64, vp, i32, vp]
    lib.gcwt_execute.argtypes = [vp, vp, i32, i64, i64, i64, i64, i64, vp, vp, i64, i64, vp]
    lib.gcwt_execute_host.argtypes = [vp, vp, i32, i64, i64, i64, vp, i32, vp, vp, i64, i64]
    lib.gcwt_host_stats.argtypes = [vp, dp]
    lib.gcwt_pool_rows.argtypes = [vp, i32, i64, i64, i64, i64, i32, i32, vp, i64, i32, vp]
    lib.gcwt_execute_host_pooled.argtypes = [vp, vp, i32, i64, i64, i64, vp, i64, i32, vp, i64, i64]
    lib.gcwt_band_reduce.argtypes = [vp, i32, i32, i64, i64, i64, i64, i32, vp, vp, vp, vp, i64, i64, i32, vp]
    lib.gcwt_execute_host_bands.argtypes = [vp, vp, i32, i64, i64, i64, vp, i32, vp, i32, vp, vp, vp, vp, i64, i64]
    lib.gcwt_event_reduce.argtypes = [vp, i32, i32, i64, i32, i64, i64, i64, i64, vp, i64, i64, i64, vp, vp, i64, i64,
                                      i32, vp]
    lib.gcwt_execute_host_events.argtypes = [vp, vp, i32, i64, i64, i64, vp, i32, vp, vp, i64, i64, i64, vp, vp, i64, i64]
    lib.gcwt_filter_response.argtypes = [i64, i32, i32, dp, i64, i64, i64, dp, i32]
    lib.gcwt_morse_kernel.argtypes = [i64, i32, i32, dp, dp, i32]
    lib.gcwt_fastconv.argtypes = [dp, i32, i64, dp, i32, i64, dp, i32]
    lib.gcwt_dft.argtypes = [dp, i64, i32, dp, i32]
    lib.gcwt_analytic_signal.argtypes = [dp, i64, dp, i32]
    lib.gcwt_moments.argtypes = [vp, i32, i64, i32, dp, i32, vp]
    lib.gcwt_interp_taps.argtypes = [i32, i32, C.c_double, C.POINTER(C.c_float)]
    lib.gcwt_guard_stats.argtypes = [vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), C.POINTER(C.c_ubyte)]
    lib.gcwt_profile_enable.argtypes = [vp, i32]
    lib.gcwt_profile_read.argtypes = [vp, dp, C.POINTER(i64), i32]
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().gcwt_last_error()
        raise GcwtError("ghost_cwt error %d: %s" % (rc, (msg or b"").decode("utf-8", "replace")))


def launch_count(reset=False):
    return int(load().gcwt_launch_count(1 if reset else 0))
