"""ctypes binding of include/acb200.h (libacb200.so).  No torch types cross
this boundary: callers pass raw device pointers (tensor.data_ptr()) and the
raw cudaStream_t."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# ACB200_LIB: another build of the same library (kernel experiments); the default is the in-tree build
LIB_PATH = os.environ.get("ACB200_LIB") or os.path.join(HERE, "libacb200.so")

ACB_OK = 0
ACB_EINVAL, ACB_EBUILD, ACB_EUNSUPPORTED, ACB_ECUDA, ACB_ECAPACITY = -1, -2, -3, -4, -5
ACB_ASCII_CASE_INSENSITIVE = 1   # acb_build_ex flag


class Plan(C.Structure):
    _fields_ = [("n_segments", C.c_uint64), ("n_units", C.c_uint64), ("scratch_words", C.c_uint64),
                ("segment_bytes", C.c_uint32), ("warm_bytes", C.c_uint32), ("lane_stride", C.c_uint32),
                ("task_bytes", C.c_uint32)]


class Workspace(C.Structure):
    _fields_ = [
        ("dev_raw", C.c_void_p), ("dev_raw_seq", C.c_void_p), ("dev_raw_unit", C.c_void_p), ("dev_raw_aux", C.c_void_p),
        ("raw_capacity", C.c_uint64),
        ("dev_unit_counts", C.c_void_p), ("dev_unit_offsets", C.c_void_p), ("dev_seg_info", C.c_void_p),
        ("dev_scratch", C.c_void_p), ("dev_total", C.c_void_p), ("dev_out", C.c_void_p), ("out_capacity", C.c_uint64),
        ("dev_match_offsets", C.c_void_p),
    ]


class Tuning(C.Structure):
    _fields_ = [("kernel", C.c_int), ("hot_rows", C.c_int), ("segment_bytes", C.c_int), ("table", C.c_int)]


class SieveDesc(C.Structure):
    _fields_ = [("window", C.c_uint32), ("last_level", C.c_uint32), ("probes", C.c_uint32), ("bloom_bytes", C.c_uint32),
                ("nodes", C.c_uint32), ("keys", C.c_uint32), ("filter_entries", C.c_uint32), ("table_slots", C.c_uint32)]


class HotDesc(C.Structure):
    _fields_ = [("rows", C.c_uint32), ("rows128", C.c_uint32), ("visited", C.c_uint32), ("reserved", C.c_uint32)]


_lib = None


def lib():
    """The loaded library.  Fails loudly when it has not been built: there is no
    CPU fallback behind the matcher classes."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). ahocorasick_rs_b200 has no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        L.acb_last_error.restype = C.c_char_p
        L.acb_version.restype = C.c_char_p
        L.acb_launch_count.restype = C.c_uint64
        L.acb_set_tuning.argtypes = [C.POINTER(Tuning)]
        L.acb_timing_enable.argtypes = [C.c_int]
        L.acb_timing_read.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_uint64)]
        L.acb_build.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.acb_build_ex.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int, C.c_int, C.c_uint32, C.POINTER(C.c_void_p)]
        L.acb_build_flags.restype = C.c_uint32
        L.acb_build_flags.argtypes = [C.c_void_p]
        L.acb_free.argtypes = [C.c_void_p]
        for name, res in [("acb_num_patterns", C.c_uint64), ("acb_num_states", C.c_uint64),
                          ("acb_num_columns", C.c_uint32), ("acb_max_pattern_len", C.c_uint32),
                          ("acb_min_pattern_len", C.c_uint32), ("acb_match_kind", C.c_int),
                          ("acb_image_bytes", C.c_uint64)]:
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = [C.c_void_p]
        L.acb_image_write.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
        L.acb_plan_scan.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.POINTER(Plan)]
        L.acb_profile.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_uint64, C.c_int,
                                  C.c_void_p, C.c_void_p]
        L.acb_hot_bytes.restype = C.c_uint64
        L.acb_hot_bytes.argtypes = [C.c_void_p, C.c_uint32]
        L.acb_hot_build.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_uint64]
        L.acb_hot_rows.restype = C.c_uint32
        L.acb_hot_rows.argtypes = [C.c_void_p]
        L.acb_hot_describe.argtypes = [C.c_void_p, C.POINTER(HotDesc)]
        L.acb_sieve_build.restype = C.c_uint64
        L.acb_sieve_build.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
        L.acb_sieve_write.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
        L.acb_sieve_describe.argtypes = [C.c_void_p, C.POINTER(SieveDesc)]
        L.acb_select_non_overlapping.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p]
        L.acb_pack_gather_block.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint64, C.c_void_p, C.c_void_p]
        L.acb_scan_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(HotDesc), C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                     C.c_uint64, C.c_int, C.c_int, C.POINTER(Plan), C.POINTER(Workspace), C.c_void_p]
        _lib = L
    return _lib


_tls = __import__("threading").local()


def set_tuning(kernel: int = 0, hot_rows: int = 0, segment_bytes: int = 0, table: int = 0) -> None:
    """acb_set_tuning for the calling thread (the library keeps the knobs per thread); the host layer reads
    the choice back with current_kernel() to decide which device images a scan needs."""
    t = Tuning(kernel, hot_rows, segment_bytes, table)
    if lib().acb_set_tuning(C.byref(t)) != ACB_OK:
        raise RuntimeError(last_error())
    _tls.kernel = kernel


def current_kernel() -> int:
    return getattr(_tls, "kernel", 0)


def last_error() -> str:
    return lib().acb_last_error().decode("utf-8", "replace")


EXPORTS = [
    "acb_last_error", "acb_version", "acb_build", "acb_free", "acb_num_patterns", "acb_num_states",
    "acb_num_columns", "acb_max_pattern_len", "acb_min_pattern_len", "acb_match_kind", "acb_image_bytes",
    "acb_image_write", "acb_plan_scan", "acb_scan_batch",
    "acb_launch_count", "acb_set_tuning", "acb_timing_enable", "acb_timing_read",
    "acb_profile", "acb_hot_bytes", "acb_hot_build", "acb_hot_rows", "acb_hot_describe",
    "acb_sieve_build", "acb_sieve_write", "acb_sieve_describe", "acb_pack_gather_block", "acb_select_non_overlapping",
    "acb_build_ex", "acb_build_flags",
]
