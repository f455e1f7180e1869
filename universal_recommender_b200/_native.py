"""ctypes binding of the C ABI in include/cco_b200.h (libcco_b200.so, built in-tree by
__graft_entry__.build()).  There is no CPU fallback: a missing library or a missing B200 raises."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libcco_b200.so")

OK = 0
E_INVALID_ARG, E_CUDA, E_NCCL, E_OOM, E_SHAPE_MISMATCH, E_UNSUPPORTED = -1, -2, -3, -4, -5, -6
FLAG_ROWRATE_INTDIV = 1
FLAG_ENTROPY_VARARGS = 2
FLAG_ASSUME_CANONICAL = 4
FLAG_RESULT_ON_DEVICE = 8
FLAG_RESULT_NO_COUNT = 16
FLAG_RESULT_NO_LLR = 32
FLAG_INGEST_SHORT_HASH = 64   # tests only: cco_ingest_strings groups ids through its hash-collision path
MAX_TOP_K = 2048


class CcoError(RuntimeError):
    """Any non-zero status of the native library (the JNI shim rethrows these as RuntimeException)."""

    def __init__(self, status: int, message: str):
        super().__init__(f"[cco status {status}] {message}")
        self.status = status


class CcoInvalidArgument(CcoError, ValueError):
    """CCO_E_INVALID_ARG / CCO_E_SHAPE_MISMATCH -- Mahout raises IllegalArgumentException here."""


class CsrT(C.Structure):
    _fields_ = [("n_rows", C.c_int64), ("n_cols", C.c_int32),
                ("row_ptr", C.POINTER(C.c_int64)), ("col_idx", C.POINTER(C.c_int32))]


class ParamsT(C.Structure):
    _fields_ = [("max_interactions", C.c_int32), ("top_k", C.c_int32),
                ("has_min_llr", C.c_int32), ("min_llr", C.c_double)]


class ConfigT(C.Structure):
    _fields_ = [("device", C.c_int32), ("rank", C.c_int32), ("world_size", C.c_int32), ("reserved", C.c_int32),
                ("nccl_unique_id", C.POINTER(C.c_ubyte)), ("result_arena", C.c_void_p), ("result_arena_bytes", C.c_size_t)]


class EventsT(C.Structure):
    _fields_ = [("n_events", C.c_int64), ("user", C.POINTER(C.c_int64)), ("item", C.POINTER(C.c_int32)), ("n_items_raw", C.c_int32)]


class SynthTypeT(C.Structure):
    _fields_ = [("n_events", C.c_int64), ("seed", C.c_uint64), ("n_items", C.c_int32), ("reserved", C.c_int32),
                ("item_cdf", C.POINTER(C.c_double)), ("item_perm", C.POINTER(C.c_int32))]


class DictionaryT(C.Structure):
    _fields_ = [("n", C.c_int64), ("offsets", C.POINTER(C.c_int64)), ("bytes", C.c_char_p)]


class DictionaryRawT(C.Structure):
    """cco_dictionary_t with `bytes` as a plain address (ids may hold NUL bytes; c_char_p would stop at the first)"""
    _fields_ = [("n", C.c_int64), ("offsets", C.POINTER(C.c_int64)), ("bytes", C.c_void_p)]


class StringEventsT(C.Structure):
    _fields_ = [("user", DictionaryRawT), ("item", DictionaryRawT)]


class RankingT(C.Structure):
    _fields_ = [("name", C.c_char_p), ("mode", C.c_int32), ("reserved", C.c_int32), ("start_ms", C.c_int64), ("end_ms", C.c_int64),
                ("item", DictionaryRawT), ("time_ms", C.POINTER(C.c_int64))]


class StatsT(C.Structure):
    _fields_ = [("n_users", C.c_int64), ("nnz_in_total", C.c_int64),
                ("nnz_downsampled", C.c_int64 * 16), ("products", C.c_int64 * 16),
                ("distinct_cells", C.c_int64 * 16), ("out_nnz", C.c_int64 * 16), ("llr_evaluated", C.c_int64 * 16),
                ("ms_h2d", C.c_float), ("ms_prepare", C.c_float), ("ms_cooccurrence", C.c_float),
                ("ms_d2h", C.c_float), ("ms_total", C.c_float), ("ms_indicator", C.c_float * 16),
                ("n_kernel_launches", C.c_int32), ("n_mats", C.c_int32), ("ms_prep_stage", C.c_float * 8)]


# every symbol include/cco_b200.h declares (tests/test_abi.py checks the export table against this)
EXPORTS = [
    "cco_abi_version", "cco_last_error", "cco_status_string", "cco_device_count", "cco_nccl_unique_id",
    "cco_create", "cco_create_group", "cco_destroy", "cco_host_alloc", "cco_host_free", "cco_train", "cco_cooccurrences_idss",
    "cco_dataset_upload", "cco_train_dataset", "cco_dataset_free", "cco_timer_start", "cco_timer_stop",
    "cco_partition_rows", "cco_ingest", "cco_synth_ingest", "cco_dataset_shape", "cco_dataset_download",
    "cco_dataset_copy_to_host", "cco_format_es_bulk", "cco_format_model_bulk", "cco_ingest_strings", "cco_pop_model",
    "cco_result_num_matrices", "cco_result_row_range", "cco_result_matrix", "cco_result_stats", "cco_result_free",
    "cco_debug_cooccurrence", "cco_debug_downsample", "cco_debug_llr", "cco_free",
]

_lib = None


def lib():
    """Load libcco_b200.so; raise (never fall back) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CcoError(E_CUDA, f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(this package has no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    p = C.POINTER
    L.cco_abi_version.restype = C.c_int
    L.cco_last_error.restype = C.c_char_p
    L.cco_status_string.restype = C.c_char_p
    L.cco_status_string.argtypes = [C.c_int]
    L.cco_device_count.restype = C.c_int
    L.cco_nccl_unique_id.argtypes = [p(C.c_ubyte)]
    L.cco_create.argtypes = [p(ConfigT), p(C.c_void_p)]
    L.cco_create_group.argtypes = [C.c_int32, p(C.c_int32), p(C.c_void_p)]
    L.cco_destroy.argtypes = [C.c_void_p]
    L.cco_host_alloc.argtypes = [C.c_void_p, C.c_size_t, p(C.c_void_p)]
    L.cco_host_free.argtypes = [C.c_void_p, C.c_void_p]
    L.cco_train.argtypes = [C.c_void_p, C.c_int32, p(CsrT), p(ParamsT), C.c_int32, C.c_uint32, p(C.c_void_p)]
    L.cco_cooccurrences_idss.argtypes = [C.c_void_p, C.c_int32, p(CsrT), C.c_int32, C.c_int32, C.c_int32, C.c_uint32,
                                         p(C.c_void_p)]
    L.cco_dataset_upload.argtypes = [C.c_void_p, C.c_int32, p(CsrT), C.c_uint32, p(C.c_void_p)]
    L.cco_train_dataset.argtypes = [C.c_void_p, C.c_void_p, p(ParamsT), C.c_int32, C.c_uint32, p(C.c_void_p)]
    L.cco_dataset_free.argtypes = [C.c_void_p]
    L.cco_partition_rows.argtypes = [p(C.c_int64), C.c_int32, C.c_int32, p(C.c_int32)]
    L.cco_ingest.argtypes = [C.c_void_p, C.c_int32, p(EventsT), C.c_int64, C.c_int32, p(C.c_int32), p(p(C.c_int32)), p(C.c_void_p)]
    L.cco_synth_ingest.argtypes = [C.c_void_p, C.c_int32, p(SynthTypeT), C.c_int64, p(C.c_double), p(C.c_int32), C.c_int32, C.c_int32, p(C.c_void_p)]
    L.cco_dataset_copy_to_host.argtypes = [C.c_void_p, C.c_int32, p(C.c_int64), p(C.c_int32)]
    L.cco_format_es_bulk.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, p(C.c_char_p), p(DictionaryT), p(DictionaryT), p(C.c_void_p),
                                     p(C.c_int64)]
    L.cco_format_model_bulk.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, p(C.c_char_p), p(DictionaryRawT), p(DictionaryRawT), C.c_int32,
                                        p(RankingT), p(DictionaryRawT), p(DictionaryRawT), C.c_uint32, p(C.c_void_p), p(C.c_int64)]
    L.cco_ingest_strings.argtypes = [C.c_void_p, C.c_int32, p(StringEventsT), C.c_int32, C.c_uint32, p(DictionaryRawT),
                                     p(DictionaryRawT), p(C.c_void_p)]
    L.cco_pop_model.argtypes = [C.c_void_p, C.c_int32, C.c_int64, p(C.c_int32), p(C.c_int64), C.c_int32, C.c_int64, C.c_int64, p(C.c_double),
                                p(C.c_ubyte)]
    L.cco_dataset_shape.argtypes = [C.c_void_p, C.c_int32, p(C.c_int64), p(C.c_int32), p(C.c_int64)]
    L.cco_dataset_download.argtypes = [C.c_void_p, C.c_int32, p(p(C.c_int64)), p(p(C.c_int32))]
    L.cco_timer_start.argtypes = [C.c_void_p]
    L.cco_timer_stop.argtypes = [C.c_void_p, p(C.c_float)]
    L.cco_result_num_matrices.argtypes = [C.c_void_p]
    L.cco_result_row_range.argtypes = [C.c_void_p, C.c_int32, p(C.c_int64), p(C.c_int64)]
    L.cco_result_matrix.argtypes = [C.c_void_p, C.c_int32, p(C.c_int64), p(C.c_int32), p(p(C.c_int64)),
                                    p(p(C.c_int32)), p(p(C.c_double)), p(p(C.c_int32))]
    L.cco_result_stats.argtypes = [C.c_void_p, p(StatsT)]
    L.cco_result_free.argtypes = [C.c_void_p]
    L.cco_debug_cooccurrence.argtypes = [C.c_void_p, p(CsrT), p(CsrT), p(p(C.c_int64)), p(p(C.c_int32)), p(p(C.c_int32))]
    L.cco_debug_downsample.argtypes = [C.c_void_p, p(CsrT), C.c_int32, C.c_int32, C.c_uint32, p(p(C.c_int64)),
                                       p(p(C.c_int32)), p(C.c_int32), p(C.c_int32)]
    L.cco_debug_llr.argtypes = [C.c_void_p, C.c_int64, p(C.c_int64), p(C.c_int64), p(C.c_int64), p(C.c_int64), C.c_uint32,
                                p(C.c_double)]
    L.cco_free.argtypes = [C.c_void_p]
    L.cco_free.restype = None
    _lib = L
    return L


def check(status: int):
    if status == OK:
        return
    msg = lib().cco_last_error().decode(errors="replace")
    if status in (E_INVALID_ARG, E_SHAPE_MISMATCH):
        raise CcoInvalidArgument(status, msg)
    raise CcoError(status, msg)


def as_csr_t(n_rows: int, n_cols: int, row_ptr: np.ndarray, col_idx: np.ndarray) -> CsrT:
    assert row_ptr.dtype == np.int64 and col_idx.dtype == np.int32
    return CsrT(n_rows, n_cols, row_ptr.ctypes.data_as(C.POINTER(C.c_int64)),
                col_idx.ctypes.data_as(C.POINTER(C.c_int32)))
