"""ctypes binding of libpriblast_acc.so — every symbol include/priblast_acc.h declares.

Loading the library does not need a GPU (the driver is only touched by prib_acc_create), so symbol
checks run on CPU boxes.  There is no fallback: if the library is missing it is built with nvcc, and if
that is impossible an ImportError-like RuntimeError is raised.
"""
from __future__ import annotations

import ctypes
import os

from . import build as _build

c_i32p = ctypes.POINTER(ctypes.c_int32)
c_i64p = ctypes.POINTER(ctypes.c_int64)
c_f32p = ctypes.POINTER(ctypes.c_float)


class AccParams(ctypes.Structure):
    _fields_ = [
        ("maximal_span", ctypes.c_int32),
        ("min_accessible_length", ctypes.c_int32),
        ("device", ctypes.c_int32),
        ("mode", ctypes.c_int32),
        ("max_batch_bytes", ctypes.c_int64),
    ]


class AccCounters(ctypes.Structure):
    _fields_ = [
        ("sequences", ctypes.c_int64),
        ("nucleotides", ctypes.c_int64),
        ("batches", ctypes.c_int64),
        ("kernel_launches", ctypes.c_int64),
        ("kernel_ms", ctypes.c_double),
        ("h2d_ms", ctypes.c_double),
        ("d2h_ms", ctypes.c_double),
        ("h2d_bytes", ctypes.c_int64),
        ("d2h_bytes", ctypes.c_int64),
        ("dp_state_bytes", ctypes.c_int64),
        ("dp_state_bytes_used", ctypes.c_int64),
        ("phase_ms", ctypes.c_double * 7),
        ("fp64_rerun_sequences", ctypes.c_int64),
        ("fp32_flagged", ctypes.c_int64 * 4),
        ("exact_rerun_sequences", ctypes.c_int64),
    ]


# name -> (restype, argtypes); must list exactly the functions of include/priblast_acc.h
SIGNATURES = {
    "prib_acc_create": (ctypes.c_int, [ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(AccParams)]),
    "prib_acc_create_lengths": (ctypes.c_int, [ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(AccParams),
                                               ctypes.c_int32, c_i32p]),
    "prib_acc_destroy": (None, [ctypes.c_void_p]),
    "prib_acc_run": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_char_p), c_i32p,
                                    ctypes.c_void_p, c_i64p, c_i64p]),
    "prib_acc_stage": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, ctypes.POINTER(ctypes.c_char_p), c_i32p]),
    "prib_acc_compute": (ctypes.c_int, [ctypes.c_void_p]),
    "prib_acc_fetch": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, c_i64p, c_i64p]),
    "prib_acc_sync": (ctypes.c_int, [ctypes.c_void_p]),
    "prib_acc_set_stream": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p]),
    "prib_acc_get_counters": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(AccCounters)]),
    "prib_peak_probe": (ctypes.c_int, [ctypes.c_int32, ctypes.POINTER(ctypes.c_double),
                                       ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)]),
    "prib_device_count": (ctypes.c_int, []),
    "prib_host_alloc": (ctypes.c_void_p, [ctypes.c_size_t]),
    "prib_host_free": (None, [ctypes.c_void_p]),
    "prib_last_error": (ctypes.c_char_p, []),
    "prib_version": (ctypes.c_char_p, []),
    "prib_acc_record_bytes": (ctypes.c_int64, [ctypes.c_int32, ctypes.c_int32]),
    "prib_acc_write_record": (ctypes.c_int64, [c_f32p, c_f32p, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p]),
    "prib_suffix_array": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int32, c_i32p, ctypes.c_int32]),
}

_lib = None


def library_path() -> str:
    return _build.LIB


def load() -> ctypes.CDLL:
    """Load (building first if needed) libpriblast_acc.so.  Raises if it cannot be had."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("PRIB_ACC_LIB")  # experiment builds (profiles/build_variants.py); never set in production
    if not path:
        path = _build.LIB
        # rebuilds when a source is newer than the library (returns at once otherwise); on a box without nvcc a
        # stale library is an error, not something to load silently
        if _build.is_stale():
            _build.build_library()
    lib = ctypes.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


MAX_LENGTHS = 32  # PRIB_MAX_LENGTHS

PHASE_NAMES = ["memset", "inside", "outer_scans", "outside", "biloop_left", "biloop_right", "hairpin_finalize"]


class PribError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libpriblast_acc error {code}: {msg}")
        self.code = code


def check(rc: int) -> None:
    if rc != 0:
        raise PribError(rc, load().prib_last_error().decode(errors="replace"))
