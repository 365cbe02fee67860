"""Host-side handles: Schema, row expressions, Batch, Spine, and the backend.

A *backend* is a `CApi` plus one context; the product backend is
`runtime.Runtime` (CUDA library, fails loudly if it cannot load).  The
test-suite injects a second implementation of the same C ABI (the CPU
oracle, prefix ``orc_``) through `Backend` to check host logic without a
GPU — product code never constructs it.

Mirrors, on the host, the reference's `OrdZSet` / `OrdIndexedZSet` values
(crates/dbsp/src/trace/ord/zset_batch.rs:28-31, indexed_zset_batch.rs:27-41)
and the `zset!` / `indexed_zset!` literals (algebra/zset/zset_macro.rs:7-44).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Iterable, Sequence

import numpy as np

from . import _capi as capi
from ._capi import CApi, CExpr, CPred, CProj, CSchema, CSrc, CTableJob, as_u64, col_ptrs


@dataclass(frozen=True)
class Schema:
    """Row type: key lanes then value lanes, each 'u' (u64) or 'i' (i64)."""

    key: str
    val: str = ""

    @property
    def nk(self):
        return len(self.key)

    @property
    def nv(self):
        return len(self.val)

    @property
    def nl(self):
        return len(self.key) + len(self.val)

    @property
    def lanes(self):
        return self.key + self.val

    def c(self) -> CSchema:
        s = CSchema()
        s.n_key_lanes, s.n_val_lanes = self.nk, self.nv
        for i, t in enumerate(self.lanes):
            s.lane_types[i] = capi.I64 if t == "i" else capi.U64
        return s

    @staticmethod
    def from_c(s: CSchema) -> "Schema":
        t = "".join("i" if s.lane_types[i] == capi.I64 else "u" for i in range(s.n_key_lanes + s.n_val_lanes))
        return Schema(t[: s.n_key_lanes], t[s.n_key_lanes :])

    def reindex(self, nk: int) -> "Schema":
        return Schema(self.lanes[:nk], self.lanes[nk:])


# ---- declarative row expressions (stand in for the Rust closures) --------
class Src:
    def __init__(self, kind, idx=0, cst=0):
        self.kind, self.idx, self.cst = kind, idx, cst

    def c(self) -> CSrc:
        s = CSrc()
        s.kind, s.idx, s.cst = self.kind, self.idx, self.cst
        return s

    # arithmetic sugar -> Expr
    def __neg__(self):
        return Expr(capi.OP_NEG, self)

    def __add__(self, o):
        return Expr(capi.OP_ADD, self, _src(o))

    def __sub__(self, o):
        return Expr(capi.OP_SUB, self, _src(o))

    def __mul__(self, o):
        return Expr(capi.OP_MUL, self, _src(o))

    def __floordiv__(self, o):
        return Expr(capi.OP_DIV, self, _src(o))

    # comparison sugar -> Pred (unsigned unless .signed())
    def _cmp(self, op, o):
        return Pred(op, self, _src(o))

    def eq(self, o):
        return self._cmp(capi.CMP_EQ, o)

    def ne(self, o):
        return self._cmp(capi.CMP_NE, o)

    def lt(self, o):
        return self._cmp(capi.CMP_LT, o)

    def le(self, o):
        return self._cmp(capi.CMP_LE, o)

    def gt(self, o):
        return self._cmp(capi.CMP_GT, o)

    def ge(self, o):
        return self._cmp(capi.CMP_GE, o)

    def isin(self, codes):
        """membership in a set of small codes (< 64)"""
        mask = 0
        for c in codes:
            assert 0 <= c < 64
            mask |= 1 << c
        if mask >= 1 << 63:
            mask -= 1 << 64
        return self._cmp(capi.CMP_IN, mask)


def _src(x):
    return x if isinstance(x, Src) else Src(capi.SRC_CONST, 0, int(x))


def key(i):
    return Src(capi.SRC_KEY, i)


def lval(i):
    return Src(capi.SRC_LVAL, i)


def rval(i):
    return Src(capi.SRC_RVAL, i)


val = lval  # single-input operators (map_index / weigh): the batch's value lanes
col = lval  # raw event tables: column index


def const(c):
    return Src(capi.SRC_CONST, 0, int(c))


class Expr:
    def __init__(self, op, a, b=None):
        self.op, self.a, self.b = op, a, b if b is not None else Src(capi.SRC_CONST)

    def c(self) -> CExpr:
        e = CExpr()
        e.op, e.a, e.b = self.op, self.a.c(), self.b.c()
        return e


def _expr(x) -> Expr:
    if isinstance(x, Expr):
        return x
    return Expr(capi.OP_COPY, _src(x))


class Pred:
    def __init__(self, cmp, a, b, is_signed=False):
        self.cmp, self.a, self.b, self.is_signed = cmp, a, b, is_signed

    def signed(self):
        return Pred(self.cmp, self.a, self.b, True)

    def c(self) -> CPred:
        p = CPred()
        p.cmp, p.is_signed, p.a, p.b = self.cmp, int(self.is_signed), self.a.c(), self.b.c()
        return p


class Proj:
    """join_func / flat_map closure: output lanes + conjunctive filter."""

    def __init__(self, schema: Schema, out: Sequence, where: Sequence[Pred] = ()):
        assert len(out) == schema.nl, "one expression per output lane"
        assert len(where) <= capi.MAX_PREDS
        self.schema, self.out, self.where = schema, [_expr(o) for o in out], list(where)
        p = CProj()
        p.out_schema = schema.c()
        p.n_pred = len(self.where)
        for i, e in enumerate(self.out):
            p.out[i] = e.c()
        for i, w in enumerate(self.where):
            p.pred[i] = w.c()
        self._c = p

    def c(self):
        return C.byref(self._c)


class Batch:
    """Owning handle of an immutable device (or oracle) batch."""

    def __init__(self, be: "Backend", handle: int, schema: Schema | None = None):
        self.be, self.h = be, handle
        if schema is None:
            cs = CSchema()
            be.api.call("batch_schema", handle, C.byref(cs))
            schema = Schema.from_c(cs)
        self.schema = schema

    def __del__(self):
        try:
            if self.h:
                self.be.api._batch_free(self.h)
                self.h = None
        except Exception:
            pass

    def __len__(self):
        n = C.c_uint64()
        self.be.api.call("batch_len", self.h, C.byref(n))
        return n.value

    def key_count(self):
        n = C.c_uint64()
        self.be.api.call("batch_key_count", self.be.ctx, self.h, C.byref(n))
        return n.value

    def download(self):
        """Canonical vectors: dict(keys=[..], offs=.., vals=[..], diffs=..)."""
        s = self.schema
        n, nkeys = len(self), self.key_count()
        keys = [np.zeros(nkeys, np.uint64) for _ in range(s.nk)]
        vals = [np.zeros(n, np.uint64) for _ in range(s.nv)]
        offs = np.zeros(nkeys + 1, np.uint64) if s.nv else None
        diffs = np.zeros(n, np.int64)
        self.be.api.call(
            "batch_download_csr", self.be.ctx, self.h, col_ptrs(keys),
            offs.ctypes.data if offs is not None else None, col_ptrs(vals), diffs.ctypes.data,
        )
        for i, t in enumerate(s.key):
            if t == "i":
                keys[i] = keys[i].view(np.int64)
        for i, t in enumerate(s.val):
            if t == "i":
                vals[i] = vals[i].view(np.int64)
        return {"keys": keys, "offs": offs, "vals": vals, "diffs": diffs}

    def rows(self):
        """Flat list of (lane.., weight) python tuples (small batches)."""
        d = self.download()
        s = self.schema
        out = []
        if s.nv == 0:
            for i in range(len(d["diffs"])):
                out.append(tuple(int(k[i]) for k in d["keys"]) + (int(d["diffs"][i]),))
            return out
        nkeys = len(d["offs"]) - 1
        for k in range(nkeys):
            for v in range(int(d["offs"][k]), int(d["offs"][k + 1])):
                out.append(tuple(int(c[k]) for c in d["keys"]) + tuple(int(c[v]) for c in d["vals"]) + (int(d["diffs"][v]),))
        return out

    def last_key(self):
        k = (C.c_uint64 * capi.MAX_LANES)()
        valid = C.c_int32()
        self.be.api.call("batch_last_key", self.be.ctx, self.h, k, C.byref(valid))
        if not valid.value:
            return None
        out = []
        for i, t in enumerate(self.schema.key):
            v = int(k[i])
            out.append(v - (1 << 64) if (t == "i" and v >= 1 << 63) else v)
        return tuple(out)

    def __eq__(self, other):
        if not isinstance(other, Batch) or self.schema != other.schema:
            return False
        a, b = self.download(), other.download()
        eq = all(np.array_equal(x, y) for x, y in zip(a["keys"], b["keys"]))
        eq = eq and all(np.array_equal(x, y) for x, y in zip(a["vals"], b["vals"]))
        eq = eq and np.array_equal(a["diffs"], b["diffs"])
        if a["offs"] is not None:
            eq = eq and np.array_equal(a["offs"], b["offs"])
        return bool(eq)

    def __repr__(self):
        n = len(self)
        body = self.rows() if n <= 32 else f"{n} tuples"
        return f"Batch<{self.schema.key}|{self.schema.val}>({body})"


class Upload:
    """In-flight H2D copy of a raw table (keeps the host arrays alive)."""

    def __init__(self, be, handle, cols, weights):
        self.be, self.h, self._cols, self._w = be, handle, cols, weights

    def __del__(self):
        try:
            if self.h:
                self.be.api._upload_free(self.h)
                self.h = None
        except Exception:
            pass


class Download:
    """In-flight D2H copy of a batch's flat rows (keeps the destination arrays alive)."""

    def __init__(self, be, handle, n, cols, diffs):
        self.be, self.h, self.n, self.cols, self.diffs = be, handle, n, cols, diffs

    def finish(self):
        """Wait for the copy; returns (cols trimmed to n rows, diffs trimmed)."""
        if self.h:
            h, self.h = self.h, None
            self.be.api.call("download_finish", h)
        return [None if c is None else c[: self.n] for c in self.cols], None if self.diffs is None else self.diffs[: self.n]

    def __del__(self):
        try:
            if self.h:
                self.be.api._download_finish(self.h)
                self.h = None
        except Exception:
            pass


class Spine:
    """Owning handle of a trace (trace/spine_fueled.rs:107-119)."""

    def __init__(self, be: "Backend", schema: Schema, _handle=None):
        self.be, self.schema = be, schema
        if _handle is not None:
            self.h = _handle
            return
        h = C.c_void_p()
        be.api.call("spine_new", be.ctx, C.byref(schema.c()), C.byref(h))
        self.h = h.value

    def save(self, path: str):
        """Checkpoint the trace to `path` (dbsp_spine_save)."""
        self.be.api.call("spine_save", self.be.ctx, self.h, str(path).encode())

    @staticmethod
    def load(be: "Backend", path: str, schema: Schema) -> "Spine":
        """Resume a trace from a checkpoint written by save() — by this library or by the oracle."""
        h = C.c_void_p()
        be.api.call("spine_load", be.ctx, str(path).encode(), C.byref(h))
        return Spine(be, schema, _handle=h.value)

    def __del__(self):
        try:
            if self.h:
                self.be.api._spine_free(self.h)
                self.h = None
        except Exception:
            pass

    def insert(self, b: Batch):
        self.be.api.call("spine_insert", self.be.ctx, self.h, b.h)

    def consolidate(self) -> Batch:
        out = C.c_void_p()
        self.be.api.call("spine_consolidate", self.be.ctx, self.h, C.byref(out))
        return Batch(self.be, out.value, self.schema)

    def truncate_keys_below(self, key: Sequence[int]):
        k = (C.c_uint64 * capi.MAX_LANES)(*[int(x) & ((1 << 64) - 1) for x in key])
        self.be.api.call("spine_truncate_keys_below", self.be.ctx, self.h, k)

    def truncate_values_below(self, val: Sequence[int]):
        """Trace::truncate_values_below (spine_fueled.rs:644-656)."""
        v = (C.c_uint64 * capi.MAX_LANES)(*[int(x) & ((1 << 64) - 1) for x in val])
        self.be.api.call("spine_truncate_values_below", self.be.ctx, self.h, v)

    def exert(self, effort: int) -> int:
        """Trace::exert (spine_fueled.rs:627-634); returns the effort left."""
        e = C.c_int64(int(effort))
        self.be.api.call("spine_exert", self.be.ctx, self.h, C.byref(e))
        return e.value

    def stats(self):
        n, nb = C.c_uint64(), C.c_uint32()
        self.be.api.call("spine_len", self.h, C.byref(n), C.byref(nb))
        return n.value, nb.value


class Merger:
    """The fuelled Merger (trace/mod.rs:371-396): new_merger / work / done."""

    def __init__(self, be: "Backend", a: Batch, b: Batch, val_lower_bound: Sequence[int] | None = None):
        self.be, self.schema = be, a.schema
        self._keep = (a, b)
        h = C.c_void_p()
        be.api.call("merger_new", be.ctx, a.h, b.h, _lanes(val_lower_bound), C.byref(h))
        self.h = h.value

    def work(self, fuel: int) -> int:
        """Spend up to `fuel`; the returned fuel is > 0 iff the merge is complete."""
        f = C.c_int64(int(fuel))
        self.be.api.call("merger_work", self.be.ctx, self.h, C.byref(f))
        return f.value

    def done(self) -> Batch:
        out = C.c_void_p()
        h, self.h = self.h, None   # freed by the library on success
        try:
            self.be.api.call("merger_done", self.be.ctx, h, C.byref(out))
        except Exception:
            self.h = h
            raise
        return Batch(self.be, out.value, self.schema)

    def __del__(self):
        try:
            if self.h:
                self.be.api._merger_free(self.h)
                self.h = None
        except Exception:
            pass


class Batcher:
    """Batcher (trace/mod.rs:316-335) = MergeBatcher (merge_batcher/mod.rs:22-81)."""

    def __init__(self, be: "Backend", schema: Schema):
        self.be, self.schema = be, schema
        h = C.c_void_p()
        be.api.call("batcher_new", be.ctx, C.byref(schema.c()), C.byref(h))
        self.h = h.value

    def _push(self, fn, cols, weights):
        cols = [as_u64(c) for c in cols]
        n = len(cols[0]) if cols else 0
        w = np.ascontiguousarray(np.asarray(weights, dtype=np.int64)) if weights is not None else None
        self.be.api.call(fn, self.be.ctx, self.h, col_ptrs(cols), w.ctypes.data if w is not None else None, n, 0)

    def push_batch(self, cols: Sequence, weights=None):
        """Unsorted tuples, column-major host arrays (weights None = all +1)."""
        self._push("batcher_push", cols, weights)

    def push_rows(self, rows: Iterable[Sequence[int]]):
        rows = list(rows)
        if not rows:
            return
        arr = [[_wrap(r[l]) for r in rows] for l in range(self.schema.nl)]
        self.push_batch([np.array(a, dtype=np.uint64) for a in arr], [r[-1] for r in rows])

    def push_consolidated_batch(self, cols: Sequence, weights):
        """Rows already sorted, unique and non-zero."""
        self._push("batcher_push_consolidated", cols, weights)

    def tuples(self) -> int:
        n = C.c_uint64()
        self.be.api.call("batcher_tuples", self.h, C.byref(n))
        return n.value

    def seal(self) -> Batch:
        out = C.c_void_p()
        h, self.h = self.h, None   # consumed by the library
        self.be.api.call("batcher_seal", self.be.ctx, h, C.byref(out))
        return Batch(self.be, out.value, self.schema)

    def __del__(self):
        try:
            if self.h:
                self.be.api._batcher_free(self.h)
                self.h = None
        except Exception:
            pass


def _wrap(x):
    return int(x) & ((1 << 64) - 1)


def _lanes(vals: Sequence[int] | None):
    if vals is None:
        return None
    return (C.c_uint64 * capi.MAX_LANES)(*[int(x) & ((1 << 64) - 1) for x in vals])


class Backend:
    """One C-ABI library + one context.  Operator-level calls, 1:1 with the
    header (see include/dbsp_b200.h for the reference file:line of each)."""

    name = "abstract"

    def __init__(self, api: CApi, device: int = 0):
        self.api = api
        ctx = C.c_void_p()
        api.call("ctx_create", device, C.byref(ctx))
        self.ctx = ctx.value
        self.device = device

    def close(self):
        if getattr(self, "ctx", None):
            self.api._ctx_destroy(self.ctx)
            self.ctx = None

    def sync(self):
        self.api.call("ctx_sync", self.ctx)

    def stats(self, reset=False):
        a, b, c = C.c_uint64(), C.c_uint64(), C.c_uint64()
        self.api.call("ctx_stats", self.ctx, C.byref(a), C.byref(b), C.byref(c), int(reset))
        n, us = C.c_uint64(), C.c_double()
        self.api.call("ctx_sync_stats", self.ctx, C.byref(n), C.byref(us), int(reset))
        return {"kernel_launches": a.value, "h2d_bytes": b.value, "d2h_bytes": c.value,
                "host_waits": n.value, "host_wait_ms": us.value / 1e3}

    def download_begin(self, batch: "Batch", cols: Sequence, diffs):
        """Queue the D2H copy of `batch`'s flat rows into caller-owned (pinned) arrays: cols[l] takes lane l,
        diffs the weights, each with room for len(batch) entries.  Returns a Download; .finish() waits."""
        cols = [None if c is None else as_u64(c) for c in cols]
        n = len(batch)
        for c in cols:
            assert c is None or len(c) >= n
        assert diffs is None or len(diffs) >= n
        ptrs = col_ptrs(cols)
        h = C.c_void_p()
        self.api.call("batch_download_begin", self.ctx, batch.h, ptrs, diffs.ctypes.data if diffs is not None else None,
                      C.byref(h))
        return Download(self, h.value, n, cols, diffs)

    def profile(self, enable=True):
        self.api.call("ctx_profile", self.ctx, int(enable))

    def profile_pause(self):
        """Stop recording per-kernel events; what was collected stays readable (a sampling window)."""
        self.api.call("ctx_profile", self.ctx, 2)

    def profile_read(self):
        """{kernel name: dict(launches, ms, alg_bytes)} since profile(True)."""
        out, i = {}, 0
        while True:
            name = C.create_string_buffer(32)
            n, ms, b = C.c_uint64(), C.c_double(), C.c_uint64()
            rc = self.api._ctx_profile_read(self.ctx, i, name, C.byref(n), C.byref(ms), C.byref(b))
            if rc != 0:
                break
            if n.value:
                out[name.value.decode()] = {"launches": n.value, "ms": ms.value, "alg_bytes": b.value}
            i += 1
        return out

    # -- construction ------------------------------------------------------
    def _out(self):
        return C.c_void_p()

    def batch_from_columns(self, schema: Schema, cols: Sequence, weights=None, n=None, on_device=False) -> Batch:
        """Batch::from_tuples over column-major inputs.  Host inputs are numpy
        arrays; device inputs are raw integer addresses (on_device=True)."""
        if not on_device:
            cols = [as_u64(c) for c in cols]
            n = len(cols[0]) if cols else (len(weights) if weights is not None else 0)
            if weights is not None:
                weights = np.ascontiguousarray(np.asarray(weights, dtype=np.int64))
            wptr = weights.ctypes.data if weights is not None else None
        else:
            wptr = weights
        out = self._out()
        self.api.call("batch_from_tuples", self.ctx, C.byref(schema.c()), col_ptrs(cols), wptr, n, int(on_device), C.byref(out))
        return Batch(self, out.value, schema)

    def batch_from_rows(self, schema: Schema, rows: Iterable[Sequence[int]]) -> Batch:
        """rows: (lane.., weight) tuples — the `zset!` literal."""
        rows = list(rows)
        if not rows:
            return self.batch_empty(schema)
        arr = np.array([[int(x) & ((1 << 64) - 1) for x in r] for r in rows], dtype=np.uint64)
        cols = [np.ascontiguousarray(arr[:, i]) for i in range(schema.nl)]
        w = np.ascontiguousarray(arr[:, schema.nl]).view(np.int64)
        return self.batch_from_columns(schema, cols, w)

    def batch_from_table(self, cols: Sequence, proj: Proj, weights=None, n=None, on_device=False) -> Batch:
        if not on_device:
            cols = [as_u64(c) for c in cols]
            n = len(cols[0])
            if weights is not None:
                weights = np.ascontiguousarray(np.asarray(weights, dtype=np.int64))
            wptr = weights.ctypes.data if weights is not None else None
        else:
            wptr = weights
        out = self._out()
        self.api.call("batch_from_table", self.ctx, col_ptrs(cols), len(cols), wptr, n, int(on_device), proj.c(), C.byref(out))
        return Batch(self, out.value, proj.schema)

    def upload_begin(self, cols: Sequence, col_mask: int = 0xFF, weights=None):
        """Start the H2D copy of a future step's table (pinned host columns)."""
        cols = [as_u64(c) for c in cols]
        n = len(cols[0])
        if weights is not None:
            weights = np.ascontiguousarray(np.asarray(weights, dtype=np.int64))
        up = C.c_void_p()
        self.api.call("upload_begin", self.ctx, col_ptrs(cols), len(cols), col_mask,
                      weights.ctypes.data if weights is not None else None, n, C.byref(up))
        return Upload(self, up.value, cols, weights)

    def batch_from_upload(self, up: "Upload", proj: Proj) -> Batch:
        out = self._out()
        self.api.call("batch_from_upload", self.ctx, up.h, proj.c(), C.byref(out))
        return Batch(self, out.value, proj.schema)

    def batches_from_tables(self, tables: Sequence) -> list[Batch]:
        """flat_map_index of several raw tables in one call: `tables` holds
        (table, proj) pairs, a table being ("host", cols, weights, None),
        ("dev", ptrs, weights, n) or ("upload", Upload, None, None) as
        `TableHandle` takes them.  Returns what `batch_from_table` /
        `batch_from_upload` would return for each pair; the CUDA library runs
        the tables side by side on its two execution lanes."""
        if self.api._batches_from_tables is None:   # a library without the grouped calls: the single calls in turn
            return [self.batch_from_upload(t[1], p) if t[0] == "upload"
                    else self.batch_from_table(t[1], p, weights=t[2], n=t[3], on_device=(t[0] == "dev")) for t, p in tables]
        k = len(tables)
        jobs = (CTableJob * max(k, 1))()
        keep = []   # host arrays and C structs must outlive the call
        for i, ((kind, cols, w, n), proj) in enumerate(tables):
            j = jobs[i]
            j.proj = C.pointer(proj._c)
            if kind == "upload":
                j.upload = cols.h
                continue
            if kind == "host":
                cols = [as_u64(c) for c in cols]
                n = len(cols[0])
                if w is not None:
                    w = np.ascontiguousarray(np.asarray(w, dtype=np.int64))
                    keep.append(w)
                    w = w.ctypes.data
            ptrs = col_ptrs(cols)
            keep.append((cols, ptrs))
            j.cols = C.cast(ptrs, C.c_void_p)
            j.weights = w
            j.n = n
            j.n_cols = len(cols)
            j.on_device = int(kind == "dev")
        outs = (C.c_void_p * max(k, 1))()
        self.api.call("batches_from_tables", self.ctx, k, jobs, outs)
        return [Batch(self, outs[i], tables[i][1].schema) for i in range(k)]

    def proj_table_mask(self, proj: Proj) -> int:
        return int(self.api._proj_table_mask(proj.c()))

    def batch_from_sorted(self, schema: Schema, cols: Sequence, weights, n: int, on_device: bool) -> Batch:
        out = self._out()
        if not on_device:
            cols = [as_u64(c) for c in cols]
            weights = np.ascontiguousarray(np.asarray(weights, dtype=np.int64))
            wptr = weights.ctypes.data
        else:
            wptr = weights
        self.api.call("batch_from_sorted", self.ctx, C.byref(schema.c()), col_ptrs(cols), wptr, n, int(on_device), C.byref(out))
        return Batch(self, out.value, schema)

    def batch_empty(self, schema: Schema) -> Batch:
        out = self._out()
        self.api.call("batch_empty", self.ctx, C.byref(schema.c()), C.byref(out))
        return Batch(self, out.value, schema)

    # -- batch algebra -----------------------------------------------------
    def merge(self, a: Batch, b: Batch, val_lower_bound: Sequence[int] | None = None) -> Batch:
        out = self._out()
        if val_lower_bound is None:
            self.api.call("batch_merge", self.ctx, a.h, b.h, C.byref(out))
        else:
            self.api.call("batch_merge_bounded", self.ctx, a.h, b.h, _lanes(val_lower_bound), C.byref(out))
        return Batch(self, out.value, a.schema)

    def batcher(self, schema: Schema) -> "Batcher":
        return Batcher(self, schema)

    def merger(self, a: Batch, b: Batch, val_lower_bound: Sequence[int] | None = None) -> "Merger":
        return Merger(self, a, b, val_lower_bound)

    def truncate_keys_below(self, b: Batch, key: Sequence[int]) -> Batch:
        out = self._out()
        self.api.call("batch_truncate_keys_below", self.ctx, b.h, _lanes(key), C.byref(out))
        return Batch(self, out.value, b.schema)

    def neg(self, a: Batch) -> Batch:
        out = self._out()
        self.api.call("batch_neg", self.ctx, a.h, C.byref(out))
        return Batch(self, out.value, a.schema)

    def reindex(self, a: Batch, nk: int) -> Batch:
        out = self._out()
        self.api.call("batch_reindex", self.ctx, a.h, nk, C.byref(out))
        return Batch(self, out.value, a.schema.reindex(nk))

    # -- operators ---------------------------------------------------------
    def join_delta_trace(self, delta: Batch, trace: Spine, proj: Proj, delta_is_left=True) -> Batch:
        out = self._out()
        self.api.call("join_delta_trace", self.ctx, delta.h, trace.h, proj.c(), int(delta_is_left), C.byref(out))
        return Batch(self, out.value, proj.schema)

    def join_step(self, dl: Batch, dr: Batch, lt: Spine, rt: Spine, proj: Proj) -> Batch:
        """One step of the incremental join (operator/join.rs:180-292):
        rt.insert(dr); o1 = dl |x| rt; o2 = dr |x| lt; lt.insert(dl); o1 + o2.
        The CUDA library runs the two halves side by side."""
        if self.api._join_step is None:   # a library without the grouped calls: the single calls in turn
            rt.insert(dr)
            o1 = self.join_delta_trace(dl, rt, proj, delta_is_left=True)
            o2 = self.join_delta_trace(dr, lt, proj, delta_is_left=False)
            lt.insert(dl)
            return self.merge(o1, o2)
        out = self._out()
        self.api.call("join_step", self.ctx, dl.h, dr.h, lt.h, rt.h, proj.c(), C.byref(out))
        return Batch(self, out.value, proj.schema)

    def join_batches(self, left: Batch, right: Batch, proj: Proj) -> Batch:
        out = self._out()
        self.api.call("join_batches", self.ctx, left.h, right.h, proj.c(), C.byref(out))
        return Batch(self, out.value, proj.schema)

    def semijoin(self, pairs: Batch, keys: Batch) -> Batch:
        out = self._out()
        self.api.call("semijoin", self.ctx, pairs.h, keys.h, C.byref(out))
        return Batch(self, out.value, Schema(pairs.schema.lanes))   # OrdZSet<(K, V)> (semijoin.rs:47)

    def aggregate_delta(self, delta: Batch, in_trace: Spine, out_trace: Spine, kind: int) -> Batch:
        out = self._out()
        self.api.call("aggregate_delta", self.ctx, delta.h, in_trace.h, out_trace.h, kind, C.byref(out))
        return Batch(self, out.value, out_trace.schema)

    def weigh(self, b: Batch, f, mode: int) -> Batch:
        out = self._out()
        e = _expr(f).c()
        self.api.call("weigh", self.ctx, b.h, C.byref(e), mode, C.byref(out))
        return Batch(self, out.value)

    def distinct_delta(self, delta: Batch, integral: Spine) -> Batch:
        out = self._out()
        self.api.call("distinct_delta", self.ctx, delta.h, integral.h, C.byref(out))
        return Batch(self, out.value, delta.schema)

    def stream_distinct(self, b: Batch) -> Batch:
        out = self._out()
        self.api.call("stream_distinct", self.ctx, b.h, C.byref(out))
        return Batch(self, out.value, b.schema)

    def window_delta(self, trace: Spine, delta: Batch, prev, cur) -> Batch:
        def arr(k):
            return (C.c_uint64 * capi.MAX_LANES)(*[int(x) & ((1 << 64) - 1) for x in k])

        s0, e0 = (arr(prev[0]), arr(prev[1])) if prev is not None else (arr(cur[0]), arr(cur[1]))
        out = self._out()
        self.api.call("window_delta", self.ctx, trace.h, delta.h, int(prev is not None), s0, e0, arr(cur[0]), arr(cur[1]), C.byref(out))
        return Batch(self, out.value, delta.schema)

    def map_index(self, b: Batch, proj: Proj) -> Batch:
        out = self._out()
        self.api.call("map_index", self.ctx, b.h, proj.c(), C.byref(out))
        return Batch(self, out.value, proj.schema)

    def shard_partition(self, b: Batch, n_shards: int):
        outs = (C.c_void_p * n_shards)()
        self.api.call("shard_partition", self.ctx, b.h, n_shards, outs)
        return [Batch(self, outs[i], b.schema) for i in range(n_shards)]

    # -- communication between replicas (include/dbsp_b200.h "communication") ------
    def comm_create(self, rank: int, world: int, slot_bytes: int = 0) -> bytes:
        blob = (C.c_uint8 * capi.COMM_BLOB_BYTES)()
        self.api.call("comm_create", self.ctx, rank, world, slot_bytes, blob)
        return bytes(blob)

    def comm_connect(self, blobs: bytes):
        buf = (C.c_uint8 * len(blobs)).from_buffer_copy(blobs)
        self.api.call("comm_connect", self.ctx, buf)

    def comm_destroy(self):
        if getattr(self, "ctx", None):
            self.api.call("comm_destroy", self.ctx)

    def comm_info(self):
        r, w, b = C.c_int32(), C.c_int32(), C.c_uint64()
        self.api.call("comm_info", self.ctx, C.byref(r), C.byref(w), C.byref(b))
        return r.value, w.value, b.value

    def shard(self, b: Batch) -> Batch:
        out = self._out()
        self.api.call("shard", self.ctx, b.h, C.byref(out))
        return Batch(self, out.value, b.schema)

    def shard2(self, a: Batch, b: Batch):
        oa, ob = self._out(), self._out()
        self.api.call("shard2", self.ctx, a.h, b.h, C.byref(oa), C.byref(ob))
        return Batch(self, oa.value, a.schema), Batch(self, ob.value, b.schema)

    def gather(self, b: Batch, root: int = 0) -> Batch:
        out = self._out()
        self.api.call("gather", self.ctx, b.h, root, C.byref(out))
        return Batch(self, out.value, b.schema)

    def allreduce_max(self, x: int) -> int:
        v = C.c_uint64(int(x) & ((1 << 64) - 1))
        self.api.call("allreduce_max_u64", self.ctx, C.byref(v))
        return v.value

    # -- flat column access for the exchange (overridden per backend) -------
    def batch_flat_tensors(self, b: Batch):
        """(list of per-lane torch tensors, weight tensor) of the flat rows."""
        raise NotImplementedError

    def batch_from_flat_tensors(self, schema: Schema, cols, weights) -> Batch:
        raise NotImplementedError
