"""ctypes front of oracle/nexmark_workers.cpp — the native (C++ threads, no interpreter between steps) CPU arm.

TEST / BASELINE INFRASTRUCTURE (lives under oracle/): used only by bench.py's `cpu_baseline` / `--impl reference`
legs and by tests/test_oracle_workers.py.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
QUERY_ID = {"q3": 3, "q4": 4, "q7": 7}
_libs = {}
_tmpdirs = []   # keeps the native build's directory alive while its library is loaded


def load(native: bool = False):
    """native=True: rebuild with -march=native on THIS machine, into a temporary directory removed at exit (the
    source tree may be read-only); falls back to the portable build."""
    key = "native" if native else "portable"
    if key in _libs:
        return _libs[key]
    path, how = os.path.join(HERE, "liborc_workers.so"), "portable (-O3)"
    if native:
        try:
            out = tempfile.TemporaryDirectory(prefix="dbsp_orc_native_")
            _tmpdirs.append(out)
            subprocess.check_call(["make", "-C", HERE, "native", f"NATIVE={out.name}", "-s"],
                                  stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
            path, how = os.path.join(out.name, "liborc_workers.so"), "-O3 -march=native, built on this host"
        except Exception:
            pass
    if not os.path.exists(path):
        subprocess.check_call(["make", "-C", HERE, "-s"])
    lib = C.CDLL(path)
    lib.orcw_run.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64),
                             C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    lib.orcw_run.restype = C.c_int32
    _libs[key] = (lib, how)
    return _libs[key]


def run(query: str, n_threads: int, steps: list[dict], native: bool = False):
    """steps: list of NexmarkGenerator.tables() dicts.  Returns (seconds per step, output rows per step,
    output fingerprint per step, build description)."""
    lib, how = load(native)
    n = len(steps)
    ptrs = (C.c_void_p * (n * 15))()
    counts = (C.c_uint64 * (n * 3))()
    for s, t in enumerate(steps):
        for ti, name in enumerate(("person", "auction", "bid")):
            cols = t.get(name)
            counts[s * 3 + ti] = 0 if cols is None else len(cols[0])
            for c in range(5):
                ptrs[(s * 3 + ti) * 5 + c] = None if cols is None else cols[c].ctypes.data
    secs = (C.c_double * n)()
    rows = (C.c_uint64 * n)()
    fps = (C.c_uint64 * n)()
    rc = lib.orcw_run(QUERY_ID[query], n_threads, n, ptrs, counts, secs, rows, fps)
    if rc != 0:
        raise RuntimeError(f"orcw_run failed: {rc}")
    return list(secs), list(rows), list(fps), how


def _mix64(x):
    x = x + np.uint64(0x9E3779B97F4A7C15)
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def fingerprint(flat_cols, weights) -> int:
    """Order-independent fingerprint of a Z-set given its flat rows (same function as nexmark_workers.cpp)."""
    n = len(weights)
    if n == 0:
        return 0
    with np.errstate(over="ignore"):
        h = np.full(n, 0x243F6A8885A308D3, dtype=np.uint64)
        for c in flat_cols:
            h = _mix64(h ^ np.asarray(c).view(np.uint64))
        return int((h * np.asarray(weights).view(np.uint64)).sum(dtype=np.uint64))
