"""ctypes binding of the C ABI declared in include/dbsp_b200.h.

`CApi(lib, prefix)` binds every entry point of the header.  The product
runtime (`runtime.Runtime`) instantiates it on `libdbsp_b200.so` with the
prefix ``dbsp_``; this module itself contains no compute and no fallback.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

MAX_LANES = 8
MAX_PREDS = 4

OK = 0
ERR_NAMES = {1: "DBSP_ERR_INVALID", 2: "DBSP_ERR_CUDA", 3: "DBSP_ERR_NO_DEVICE", 4: "DBSP_ERR_UNSUPPORTED"}

U64, I64 = 0, 1
SRC_KEY, SRC_LVAL, SRC_RVAL, SRC_CONST = 0, 1, 2, 3
OP_COPY, OP_NEG, OP_ADD, OP_SUB, OP_MUL, OP_DIV = range(6)
CMP_EQ, CMP_NE, CMP_LT, CMP_LE, CMP_GT, CMP_GE, CMP_IN = range(7)
AGG_MAX, AGG_MIN, AGG_FOLD_COUNT, AGG_FOLD_SUM, AGG_WCOUNT, AGG_WCOUNT2 = range(6)
WEIGH_LINEAR, WEIGH_AVG = 0, 1


class CSchema(C.Structure):
    _fields_ = [("n_key_lanes", C.c_uint8), ("n_val_lanes", C.c_uint8), ("lane_types", C.c_uint8 * MAX_LANES)]


class CSrc(C.Structure):
    _fields_ = [("kind", C.c_uint8), ("idx", C.c_uint8), ("pad_", C.c_uint8 * 6), ("cst", C.c_int64)]


class CExpr(C.Structure):
    _fields_ = [("op", C.c_uint8), ("pad_", C.c_uint8 * 7), ("a", CSrc), ("b", CSrc)]


class CPred(C.Structure):
    _fields_ = [("cmp", C.c_uint8), ("is_signed", C.c_uint8), ("pad_", C.c_uint8 * 6), ("a", CSrc), ("b", CSrc)]


class CProj(C.Structure):
    _fields_ = [
        ("out_schema", CSchema),
        ("n_pred", C.c_uint8),
        ("pad_", C.c_uint8 * 5),
        ("out", CExpr * MAX_LANES),
        ("pred", CPred * MAX_PREDS),
    ]


class CTableJob(C.Structure):
    _fields_ = [
        ("cols", C.c_void_p),
        ("weights", C.c_void_p),
        ("n", C.c_uint64),
        ("upload", C.c_void_p),
        ("proj", C.POINTER(CProj)),
        ("n_cols", C.c_uint32),
        ("on_device", C.c_int32),
    ]


class DbspError(RuntimeError):
    pass


_P = C.c_void_p
_PP = C.POINTER(C.c_void_p)
_U64P = C.POINTER(C.c_uint64)
_I64P = C.POINTER(C.c_int64)

# name -> argtypes (restype is int32 unless noted)
_SIGS = {
    "ctx_create": [C.c_int32, _PP],
    "ctx_destroy": [_P],
    "ctx_sync": [_P],
    "ctx_stats": [_P, _U64P, _U64P, _U64P, C.c_int32],
    "ctx_profile": [_P, C.c_int32],
    "ctx_profile_read": [_P, C.c_int32, C.c_char_p, _U64P, C.POINTER(C.c_double), _U64P],
    "batch_from_tuples": [_P, C.POINTER(CSchema), _PP, _P, C.c_uint64, C.c_int32, _PP],
    "batch_from_table": [_P, _PP, C.c_uint32, _P, C.c_uint64, C.c_int32, C.POINTER(CProj), _PP],
    "batch_from_sorted": [_P, C.POINTER(CSchema), _PP, _P, C.c_uint64, C.c_int32, _PP],
    "upload_begin": [_P, _PP, C.c_uint32, C.c_uint32, _P, C.c_uint64, _PP],
    "batch_from_upload": [_P, _P, C.POINTER(CProj), _PP],
    "upload_free": [_P],
    "batch_empty": [_P, C.POINTER(CSchema), _PP],
    "batch_merge": [_P, _P, _P, _PP],
    "batcher_new": [_P, C.POINTER(CSchema), _PP],
    "batcher_push": [_P, _P, _PP, _P, C.c_uint64, C.c_int32],
    "batcher_push_consolidated": [_P, _P, _PP, _P, C.c_uint64, C.c_int32],
    "batcher_tuples": [_P, _U64P],
    "batcher_seal": [_P, _P, _PP],
    "batcher_free": [_P],
    "batch_merge_bounded": [_P, _P, _P, _U64P, _PP],
    "merger_new": [_P, _P, _P, _U64P, _PP],
    "merger_work": [_P, _P, _I64P],
    "merger_done": [_P, _P, _PP],
    "merger_free": [_P],
    "batch_truncate_keys_below": [_P, _P, _U64P, _PP],
    "batch_neg": [_P, _P, _PP],
    "batch_reindex": [_P, _P, C.c_uint32, _PP],
    "batch_len": [_P, _U64P],
    "batch_key_count": [_P, _P, _U64P],
    "batch_schema": [_P, C.POINTER(CSchema)],
    "batch_download_csr": [_P, _P, _PP, _P, _PP, _P],
    "batch_download_begin": [_P, _P, _PP, _P, _PP],
    "download_finish": [_P],
    "ctx_sync_stats": [_P, _U64P, C.POINTER(C.c_double), C.c_int32],
    "batch_device_columns": [_P, _PP, _PP],
    "batch_last_key": [_P, _P, _U64P, C.POINTER(C.c_int32)],
    "batch_clone": [_P, _PP],
    "batch_free": [_P],
    "spine_new": [_P, C.POINTER(CSchema), _PP],
    "spine_insert": [_P, _P, _P],
    "spine_consolidate": [_P, _P, _PP],
    "spine_truncate_keys_below": [_P, _P, _U64P],
    "spine_truncate_values_below": [_P, _P, _U64P],
    "spine_exert": [_P, _P, _I64P],
    "spine_len": [_P, _U64P, C.POINTER(C.c_uint32)],
    "spine_free": [_P],
    "spine_save": [_P, _P, C.c_char_p],
    "spine_load": [_P, C.c_char_p, _PP],
    "join_delta_trace": [_P, _P, _P, C.POINTER(CProj), C.c_int32, _PP],
    "join_batches": [_P, _P, _P, C.POINTER(CProj), _PP],
    "semijoin": [_P, _P, _P, _PP],
    "aggregate_delta": [_P, _P, _P, _P, C.c_int32, _PP],
    "weigh": [_P, _P, C.POINTER(CExpr), C.c_int32, _PP],
    "distinct_delta": [_P, _P, _P, _PP],
    "stream_distinct": [_P, _P, _PP],
    "window_delta": [_P, _P, _P, C.c_int32, _U64P, _U64P, _U64P, _U64P, _PP],
    "map_index": [_P, _P, C.POINTER(CProj), _PP],
    "shard_partition": [_P, _P, C.c_uint32, _PP],
    "comm_create": [_P, C.c_int32, C.c_int32, C.c_uint64, _P],
    "comm_connect": [_P, _P],
    "comm_destroy": [_P],
    "comm_info": [_P, C.POINTER(C.c_int32), C.POINTER(C.c_int32), _U64P],
    "shard": [_P, _P, _PP],
    "shard2": [_P, _P, _P, _PP, _PP],
    "gather": [_P, _P, C.c_int32, _PP],
    "allreduce_max_u64": [_P, _U64P],
}
# The grouped calls that run on the CUDA library's two execution lanes.  A library without them (the CPU oracle)
# leaves them unbound and `zset.Backend` issues the same sequence of single calls instead.
_GROUPED_SIGS = {
    "batches_from_tables": [_P, C.c_uint32, C.POINTER(CTableJob), _PP],
    "join_step": [_P, _P, _P, _P, _P, C.POINTER(CProj), _PP],
}
COMM_BLOB_BYTES = 128


class CApi:
    """Thin, typed view of a shared library exporting the dbsp_b200.h ABI."""

    def __init__(self, lib: C.CDLL, prefix: str, require_grouped: bool = False):
        self.lib = lib
        self.prefix = prefix
        for name, argtypes in _SIGS.items():
            fn = getattr(lib, prefix + name)  # AttributeError if a symbol is missing
            fn.argtypes = argtypes
            fn.restype = C.c_int32
            setattr(self, "_" + name, fn)
        for name, argtypes in _GROUPED_SIGS.items():
            fn = getattr(lib, prefix + name) if require_grouped else getattr(lib, prefix + name, None)
            if fn is not None:
                fn.argtypes = argtypes
                fn.restype = C.c_int32
            setattr(self, "_" + name, fn)
        self._last_error = getattr(lib, prefix + "last_error")
        self._last_error.restype = C.c_char_p
        self._last_error.argtypes = []
        self._ctx_stream = getattr(lib, prefix + "ctx_stream")
        self._ctx_stream.restype = C.c_void_p
        self._ctx_stream.argtypes = [_P]
        self._proj_table_mask = getattr(lib, prefix + "proj_table_mask")
        self._proj_table_mask.restype = C.c_uint32
        self._proj_table_mask.argtypes = [C.POINTER(CProj)]

    @staticmethod
    def symbols(prefix: str = "dbsp_"):
        return [prefix + n for n in list(_SIGS) + list(_GROUPED_SIGS) + ["last_error", "ctx_stream", "proj_table_mask"]]

    def check(self, rc: int, what: str):
        if rc != OK:
            msg = self._last_error()
            raise DbspError(f"{self.prefix}{what} failed: {ERR_NAMES.get(rc, rc)}: {msg.decode() if msg else ''}")

    def call(self, name: str, *args):
        self.check(getattr(self, "_" + name)(*args), name)


def col_ptrs(cols):
    """Array of void* from a list of numpy arrays / raw integer addresses."""
    arr = (C.c_void_p * max(len(cols), 1))()
    for i, c in enumerate(cols):
        if c is None:
            arr[i] = None
        elif isinstance(c, int):
            arr[i] = c
        else:
            arr[i] = c.ctypes.data
    return arr


def as_u64(a, n=None):
    """Contiguous uint64 view of integer data (i64 lanes are bit-cast)."""
    a = np.asarray(a)
    if a.dtype == np.int64:
        a = a.view(np.uint64)
    elif a.dtype != np.uint64:
        a = a.astype(np.int64).view(np.uint64)
    return np.ascontiguousarray(a)
