"""The product backend: the CUDA library behind include/dbsp_b200.h.

There is deliberately no fallback here.  If `libdbsp_b200.so` is missing or
no CUDA device is usable, construction raises — the hot path never runs on
the CPU (the CPU oracle under oracle/ is test infrastructure and is not
reachable from this package).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from ._capi import CApi, DbspError
from .zset import Backend, Batch, Schema

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DBSP_B200_LIB") or os.path.join(_HERE, "libdbsp_b200.so")

_lib = None


def load_library() -> C.CDLL:
    """dlopen the in-tree CUDA library (built by __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise DbspError(
                f"{LIB_PATH} not found: build it with `python __graft_entry__.py` "
                "(nvcc, sm_100a). There is no CPU fallback for the hot path."
            )
        _lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    return _lib


class _DevArray:
    """__cuda_array_interface__ view of library-owned device memory."""

    def __init__(self, ptr, n, typestr, owner):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 3}
        self._owner = owner


class Runtime(Backend):
    """One GPU + one CUDA stream (one circuit replica, runtime.rs:137-180)."""

    name = "cuda"

    def __init__(self, device: int = 0):
        super().__init__(CApi(load_library(), "dbsp_", require_grouped=True), device)

    @property
    def stream_ptr(self) -> int:
        return self.api._ctx_stream(self.ctx) or 0

    def batch_device_columns(self, b: Batch):
        cols = (C.c_void_p * 8)()
        w = C.c_void_p()
        self.api.call("batch_device_columns", b.h, cols, C.byref(w))
        return [cols[i] or 0 for i in range(b.schema.nl)], (w.value or 0)

    def batch_flat_tensors(self, b: Batch, synced: bool = False):
        import torch

        n = len(b)
        cols, w = self.batch_device_columns(b)
        dev = torch.device("cuda", self.device)
        if n == 0:
            return [torch.empty(0, dtype=torch.int64, device=dev) for _ in cols], torch.empty(0, dtype=torch.int64, device=dev)
        if not synced:
            self.sync()
        ts = [torch.as_tensor(_DevArray(p, n, "<i8", b), device=dev) for p in cols]
        return ts, torch.as_tensor(_DevArray(w, n, "<i8", b), device=dev)

    def batch_from_flat_tensors(self, schema: Schema, cols, weights, synced: bool = False) -> Batch:
        import torch

        n = int(weights.numel())
        if n == 0:
            return self.batch_empty(schema)
        if not synced:
            torch.cuda.current_stream(self.device).synchronize()
        return self.batch_from_sorted(schema, [int(c.data_ptr()) for c in cols], int(weights.data_ptr()), n, True)

    def batch_from_device_tensors(self, schema: Schema, cols, weights) -> Batch:
        """Batch::from_tuples over unsorted device-resident torch columns."""
        import torch

        n = int(weights.numel())
        if n == 0:
            return self.batch_empty(schema)
        torch.cuda.current_stream(self.device).synchronize()
        b = self.batch_from_columns(schema, [int(c.data_ptr()) for c in cols], int(weights.data_ptr()), n=n, on_device=True)
        self.sync()   # the torch tensors may be freed as soon as this returns
        return b
