"""Stream / operator API for the Z-set delta hot path.

Host-side mirror of the reference's `RootCircuit` + `Stream` operator surface
(crates/dbsp/src/circuit/circuit_builder.rs:1403-1433, operator/*.rs) for the
operators on the hot path.  A circuit is a static DAG built once; `step()`
evaluates every node once in creation (= dependency) order, exactly like the
reference's schedulers (circuit/schedule/static_scheduler.rs:52-87).  All
data work is done by the backend (the CUDA library behind include/dbsp_b200.h).

Rust closures become declarative `Proj` / expression objects (zset.py).
Stateful operators own their traces; the `z^-1` delays of the reference's
feedback loops are realised by the order of trace inserts inside `eval`.
"""
from __future__ import annotations

from typing import Callable, Sequence

import numpy as np

from . import _capi as capi
from .zset import Backend, Batch, Proj, Schema, Spine, key, lval, rval


class Max:  # operator/aggregate/max.rs:36-55
    kind = capi.AGG_MAX


class Min:  # operator/aggregate/min.rs:38-57
    kind = capi.AGG_MIN


class FoldCount:  # Fold counting distinct values (aggregate/mod.rs:908-916)
    kind = capi.AGG_FOLD_COUNT


class FoldSum:  # Fold summing distinct values (aggregate/mod.rs:918-929)
    kind = capi.AGG_FOLD_SUM


class Node:
    table_proj = None   # set on the flat_map_index of a raw table, which `RootCircuit.step` evaluates in groups

    def __init__(self, circuit: "RootCircuit", inputs: Sequence["Node"], fn: Callable | None, name: str):
        self.circuit, self.inputs, self.fn, self.name = circuit, list(inputs), fn, name
        self.value = None
        circuit.nodes.append(self)

    def eval(self):
        self.value = self.fn(*[i.value for i in self.inputs])


class InputHandle:
    """CollectionHandle (operator/input.rs:664-703): rows appended between
    steps form the next step's batch."""

    def __init__(self, circuit, schema: Schema):
        self.circuit, self.schema, self.pending = circuit, schema, []

    def append(self, rows):
        """rows: iterable of (lane.., weight)."""
        self.pending.extend(rows)

    def push(self, *row):
        """push(k.., w) (operator/input.rs:676-681): one (lane.., weight) update."""
        self.pending.append(tuple(row))

    def clear_input(self):
        """clear_input (operator/input.rs:697-703): drop the updates buffered since the last step."""
        self.pending = []

    def _take(self) -> Batch:
        rows, self.pending = self.pending, []
        return self.circuit.be.batch_from_rows(self.schema, rows)


class TableHandle:
    """Input of a raw column-major event table (no order, optional weights).
    `set(cols, weights=None)` with host numpy columns, or
    `set_device(ptrs, n)` with resident device columns."""

    def __init__(self):
        self.cur = None

    def set(self, cols, weights=None):
        self.cur = ("host", list(cols), weights, None)

    def set_device(self, ptrs, n, weights=None):
        self.cur = ("dev", list(ptrs), weights, int(n))

    def set_upload(self, upload):
        """upload: an `Upload` started with Backend.upload_begin for this step
        (pipelined ingest; its column mask must cover `TableStream.table_mask()`)."""
        self.cur = ("upload", upload, None, None)

    def _take(self):
        cur, self.cur = self.cur, None
        return cur


class RootCircuit:
    """RootCircuit::build + CircuitHandle::step
    (circuit_builder.rs:1403-1433, 3658-3663)."""

    def __init__(self, backend: Backend | None = None, comm=None):
        if backend is None:
            from .runtime import Runtime  # the CUDA library; raises if unavailable

            backend = Runtime()
        self.be = backend
        self.comm = comm  # parallel.Comm or None (single worker)
        if comm is not None and getattr(comm, "native", None) is None and hasattr(comm, "attach") and comm.world_size > 1:
            comm.attach(backend)   # CUDA backend: the exchange moves into the library (csrc/comm.cu)
        self.nodes: list[Node] = []

    # -- sources -------------------------------------------------------------
    def add_input_zset(self, schema: Schema):
        """add_input_zset / add_input_indexed_zset (operator/input.rs:75-86)."""
        h = InputHandle(self, schema)
        node = Node(self, [], h._take, "input")
        return Stream(self, node, schema), h

    add_input_indexed_zset = add_input_zset

    def add_input_table(self, n_cols: int):
        h = TableHandle()
        node = Node(self, [], h._take, "table")
        return TableStream(self, node, n_cols), h

    def add_source(self, gen: Callable[[], object], schema: Schema | None = None):
        """Generator source (operator/generator.rs): gen() each step."""
        node = Node(self, [], gen, "source")
        return Stream(self, node, schema)

    def step(self):
        done = set()
        for n in self.nodes:
            if id(n) in done:
                continue
            if n.table_proj is not None:
                # every table projection whose table is already evaluated, in one call: the library ingests the
                # tables side by side on its two execution lanes
                group = [m for m in self.nodes if m.table_proj is not None and id(m) not in done and id(m.inputs[0]) in done]
                self._eval_tables(group)
                done.update(id(m) for m in group)
            else:
                n.eval()
                done.add(id(n))

    def _eval_tables(self, group):
        live = [(m, m.table_proj) for m in group if m.inputs[0].value is not None]
        outs = self.be.batches_from_tables([(m.inputs[0].value, p) for m, p in live]) if live else []
        got = {id(m): b for (m, _), b in zip(live, outs)}
        for m in group:
            m.value = got[id(m)] if id(m) in got else self.be.batch_empty(m.table_proj.schema)

    @property
    def workers(self):
        return self.comm.world_size if self.comm is not None else 1


class TableStream:
    def __init__(self, circuit, node, n_cols):
        self.circuit, self.node, self.n_cols = circuit, node, n_cols
        self.projs = []   # projections consuming this table, in creation order

    def table_mask(self) -> int:
        """Columns read by any consumer of this table (bit l = column l)."""
        m = 0
        for p in self.projs:
            m |= self.circuit.be.proj_table_mask(p)
        return m

    def flat_map_index(self, proj: Proj) -> "Stream":
        """flat_map_index on the event stream (filter_map.rs:143-152,700-724):
        filter + project + from_tuples, straight from the raw columns
        (evaluated by `RootCircuit.step` together with the circuit's other
        table projections)."""
        self.projs.append(proj)
        node = Node(self.circuit, [self.node], None, "flat_map_index")
        node.table_proj = proj
        return Stream(self.circuit, node, proj.schema)


class Stream:
    """Stream<RootCircuit, Batch> for Batch in {OrdZSet, OrdIndexedZSet}, or a
    host scalar stream (schema None)."""

    def __init__(self, circuit: RootCircuit, node: Node, schema: Schema | None, sharded=False):
        self.circuit, self.node, self.schema, self.sharded = circuit, node, schema, sharded

    # -- plumbing ------------------------------------------------------------
    def _unary(self, fn, name, schema, sharded=False) -> "Stream":
        return Stream(self.circuit, Node(self.circuit, [self.node], fn, name), schema, sharded)

    def _binary(self, other, fn, name, schema, sharded=False) -> "Stream":
        return Stream(self.circuit, Node(self.circuit, [self.node, other.node], fn, name), schema, sharded)

    def inspect(self, cb: Callable) -> "Stream":
        """inspect (operator/inspect.rs)."""

        def fn(v):
            cb(v)
            return v

        return self._unary(fn, "inspect", self.schema, self.sharded)

    def output(self):
        """OutputHandle: .value after each step."""
        return self.node

    def apply(self, f: Callable) -> "Stream":
        """apply (operator/apply.rs): host function on the stream's value."""
        return self._unary(f, "apply", None)

    # -- linear / stateless --------------------------------------------------
    def index(self, nk: int) -> "Stream":
        """index() (operator/index.rs:128-157): OrdZSet<(K,V)> -> OrdIndexedZSet<K,V>."""
        be = self.circuit.be
        return self._unary(lambda b: be.reindex(b, nk), "index", self.schema.reindex(nk))

    def map_index(self, proj: Proj) -> "Stream":
        """map_index / flat_map_index / map / filter (filter_map.rs:563-577,700-724)."""
        be = self.circuit.be
        return self._unary(lambda b: be.map_index(b, proj), "map_index", proj.schema)

    # the reference's closure-taking variants all lower to one projection + filter in the row language:
    # map / flat_map produce an OrdZSet, map_index / flat_map_index / index_with an OrdIndexedZSet — the output
    # schema of `proj` says which (filter_map.rs:40-215, index.rs:38-62)
    map = map_index
    flat_map = map_index
    flat_map_index = map_index
    index_with = map_index

    def filter(self, *preds) -> "Stream":
        """filter (operator/filter_map.rs:40-54): keep the rows satisfying every predicate; schema unchanged."""
        from .zset import key, val

        s = self.schema
        ident = [key(i) for i in range(s.nk)] + [val(i) for i in range(s.nv)]
        return self.map_index(Proj(s, ident, list(preds)))

    def sum(self, others: Sequence["Stream"]) -> "Stream":
        """sum (operator/sum.rs:20-40): self + every stream of `others` (aliases allowed)."""
        out = self
        for o in others:
            out = out.plus(o)
        return out

    def neg(self) -> "Stream":
        be = self.circuit.be
        return self._unary(lambda b: be.neg(b), "neg", self.schema, self.sharded)

    def plus(self, other: "Stream") -> "Stream":
        """plus (operator/plus.rs:127-143) = batch merge."""
        be = self.circuit.be
        return self._binary(other, lambda a, b: be.merge(a, b), "plus", self.schema, self.sharded and other.sharded)

    def minus(self, other: "Stream") -> "Stream":
        be = self.circuit.be
        return self._binary(other, lambda a, b: be.merge(a, be.neg(b)), "minus", self.schema)

    def stream_distinct(self) -> "Stream":
        """stream_distinct (operator/distinct.rs:40-52)."""
        be = self.circuit.be
        s = self.shard()
        return s._unary(lambda b: be.stream_distinct(b), "stream_distinct", self.schema, True)

    def stream_join(self, other: "Stream", proj: Proj) -> "Stream":
        """stream_join (operator/join.rs:52-84): stateless Join::eval."""
        be = self.circuit.be
        l, r = self.shard_with(other)
        return l._binary(r, lambda a, b: be.join_batches(a, b, proj), "stream_join", proj.schema)

    def semijoin_stream(self, keys: "Stream") -> "Stream":
        """semijoin_stream (operator/semijoin.rs:38-62)."""
        be = self.circuit.be
        l, r = self.shard(), keys.shard()
        return l._binary(r, lambda a, b: be.semijoin(a, b), "semijoin", Schema(self.schema.lanes), True)

    # -- stateful ------------------------------------------------------------
    def integrate(self) -> "Stream":
        """integrate (operator/integrate.rs): running sum of deltas."""
        be = self.circuit.be
        state = {"acc": None}

        def fn(b):
            state["acc"] = b if state["acc"] is None else be.merge(state["acc"], b)
            return state["acc"]

        return self._unary(fn, "integrate", self.schema, self.sharded)

    def differentiate(self) -> "Stream":
        """differentiate (operator/differentiate.rs): x[t] - x[t-1]."""
        be = self.circuit.be
        state = {"prev": None}

        def fn(b):
            out = b if state["prev"] is None else be.merge(b, be.neg(state["prev"]))
            state["prev"] = b
            return out

        return self._unary(fn, "differentiate", self.schema, self.sharded)

    def join(self, other: "Stream", proj: Proj) -> "Stream":
        """join / join_index / join_generic (operator/join.rs:180-292):
        delta_L |x| trace(R) + delta_R |x| z^-1 trace(L), both sides sharded."""
        be = self.circuit.be
        left, right = self.shard_with(other)
        lt, rt = Spine(be, left.schema), Spine(be, right.schema)

        def fn(dl: Batch, dr: Batch):
            # rt.insert(dr) (right.trace()); o1 = dl |x| rt; o2 = dr |x| z^-1(lt); lt.insert(dl) (left.trace());
            # o1 + o2 (left.plus(&right)) — the halves run side by side in the library
            return be.join_step(dl, dr, lt, rt, proj)

        return left._binary(right, fn, "join", proj.schema)

    join_index = join

    def antijoin(self, other: "Stream") -> "Stream":
        """antijoin (operator/join.rs:294-320): the rows of `self` whose key is
        absent from `other` = self - self |x| distinct(other) with the identity
        closure (k, v1)."""
        s1 = self.shard()
        s2 = other.distinct().shard()
        nk, nv = self.schema.nk, self.schema.nv
        ident = Proj(self.schema, [key(i) for i in range(nk)] + [lval(i) for i in range(nv)])
        out = s1.minus(s1.join(s2, ident))
        out.sharded = True   # mark_sharded (join.rs:316)
        return out

    def join_incremental(self, other: "Stream", proj: Proj) -> "Stream":
        """join_incremental (operator/join.rs:136-155):
        I(a) |x| I(b) - z^-1(I(a)) |x| z^-1(I(b)), via stateless joins."""
        be = self.circuit.be
        l, r = self.shard(), other.shard()
        st = {"a": None, "b": None}

        def fn(da, db):
            a = da if st["a"] is None else be.merge(st["a"], da)
            b = db if st["b"] is None else be.merge(st["b"], db)
            cur = be.join_batches(a, b, proj)
            if st["a"] is not None:
                cur = be.merge(cur, be.neg(be.join_batches(st["a"], st["b"], proj)))
            st["a"], st["b"] = a, b
            return cur

        return l._binary(r, fn, "join_incremental", proj.schema)

    def aggregate(self, aggregator, local: bool = False) -> "Stream":
        """aggregate (operator/aggregate/mod.rs:204-244): AggregateIncremental
        over stream.trace(), then upsert into the output trace.
        `local=True` skips the shard(): every worker aggregates its own rows —
        the first level of a two-level aggregate for semigroup aggregators
        (MinSemigroup / MaxSemigroup, aggregate/min.rs:17-27), whose partial
        results are then aggregated again after a shard of <= P rows per key."""
        be = self.circuit.be
        s = Stream(self.circuit, self.node, self.schema, True) if local else self.shard()
        kind = aggregator.kind
        if kind in (capi.AGG_MAX, capi.AGG_MIN):
            out_schema = s.schema
        else:
            out_schema = Schema(s.schema.key, "u")
        in_tr, out_tr = Spine(be, s.schema), Spine(be, out_schema)

        def fn(d: Batch):
            in_tr.insert(d)
            out = be.aggregate_delta(d, in_tr, out_tr, kind)
            out_tr.insert(out)
            return out

        return s._unary(fn, "aggregate", out_schema, not local)

    def stream_aggregate(self, aggregator) -> "Stream":
        """stream_aggregate (operator/aggregate/mod.rs:172-196): Aggregate::eval
        (:362-376) — the aggregate of every key of *this step's* batch with
        weight +1; no state.  Runs the same kernels as `aggregate` on a trace
        holding only the batch and an empty output trace."""
        be = self.circuit.be
        s = self.shard()
        kind = aggregator.kind
        out_schema = s.schema if kind in (capi.AGG_MAX, capi.AGG_MIN) else Schema(s.schema.key, "u")

        def fn(d: Batch):
            if len(d) == 0:
                return be.batch_empty(out_schema)
            tin, tout = Spine(be, s.schema), Spine(be, out_schema)
            tin.insert(d)
            return be.aggregate_delta(d, tin, tout, kind)

        return s._unary(fn, "stream_aggregate", out_schema, True)

    def weigh(self, f, mode=capi.WEIGH_LINEAR) -> "Stream":
        """weigh (operator/aggregate/mod.rs:285-323)."""
        be = self.circuit.be
        sch = Schema(self.schema.key + ("u" if mode == capi.WEIGH_AVG else ""), "")
        return self._unary(lambda b: be.weigh(b, f, mode), "weigh", sch, self.sharded)

    def aggregate_linear(self, f) -> "Stream":
        """aggregate_linear (aggregate/mod.rs:253-273) = weigh(f).aggregate(WeightedCount)."""
        be = self.circuit.be
        w = self.weigh(f).shard()   # weigh first (linear): only one row per key crosses the exchange
        out_schema = Schema(self.schema.key, "i")
        in_tr, out_tr = Spine(be, w.schema), Spine(be, out_schema)

        def fn(d: Batch):
            in_tr.insert(d)
            out = be.aggregate_delta(d, in_tr, out_tr, capi.AGG_WCOUNT)
            out_tr.insert(out)
            return out

        return w._unary(fn, "aggregate_linear", out_schema, True)

    def average(self, f) -> "Stream":
        """average (operator/aggregate/average.rs:227-246): aggregate_linear
        with the (sum,count) pair weight, then apply_average (:266-307) —
        truncating signed division of the value column.  The pair weight is
        carried as two rows (K,0)->sum and (K,1)->count of an OrdZSet (see
        include/dbsp_b200.h, DBSP_AGG_WCOUNT2).  Unlike apply_average the
        result is re-consolidated, which only removes +1/-1 pairs that the
        reference's downstream map/from_tuples would cancel anyway."""
        be = self.circuit.be
        # weigh first (linear): <= 2 rows per key cross the exchange; shard on K only so that
        # the (K,0) and (K,1) rows of a key meet on one worker (index() is a zero-copy view)
        nk0 = self.schema.nk
        w = self.weigh(f, capi.WEIGH_AVG).index(nk0).shard().index(nk0 + 1)
        pair_schema = Schema(self.schema.key, "ii")
        out_schema = Schema(self.schema.key, "i")
        in_tr, out_tr = Spine(be, w.schema), Spine(be, pair_schema)
        nk = self.schema.nk
        avg = Proj(out_schema, [key(i) for i in range(nk)] + [lval(0) // lval(1)])

        def fn(d: Batch):
            in_tr.insert(d)
            out = be.aggregate_delta(d, in_tr, out_tr, capi.AGG_WCOUNT2)
            out_tr.insert(out)
            return be.map_index(out, avg)

        return w._unary(fn, "average", out_schema, True)

    def distinct(self) -> "Stream":
        """distinct (operator/distinct.rs:64-106): DistinctIncrementalTotal
        against the delayed integral of the sharded input."""
        be = self.circuit.be
        s = self.shard()
        integral = Spine(be, s.schema)

        def fn(d: Batch):
            out = be.distinct_delta(d, integral)
            integral.insert(d)
            return out

        return s._unary(fn, "distinct", s.schema, True)

    def window(self, bounds: "Stream") -> "Stream":
        """window (operator/time_series/window.rs:75-86): the trace is delayed
        and truncated below the previous lower bound (operator/trace.rs:578-605)."""
        be = self.circuit.be
        trace = Spine(be, self.schema)
        st = {"prev": None}
        nk = self.schema.nk

        def norm(b):
            lo, hi = b
            lo = tuple(lo) if isinstance(lo, (tuple, list)) else (lo,)
            hi = tuple(hi) if isinstance(hi, (tuple, list)) else (hi,)
            assert len(lo) == nk and len(hi) == nk
            return lo, hi

        def fn(d: Batch, b):
            cur = norm(b)
            out = be.window_delta(trace, d, st["prev"], cur)
            trace.insert(d)
            trace.truncate_keys_below(cur[0])
            st["prev"] = cur
            return out

        out = self._binary(bounds, fn, "window", self.schema, self.sharded)
        out.window_trace = trace   # the bounded trace of the operator (window.rs:454-486 asserts that it stays small)
        return out

    def watermark_monotonic(self, f: Callable[[int], int]) -> "Stream":
        """watermark_monotonic (operator/time_series/watermark.rs:33-74): max of
        the previous watermark and f(last key of the batch); all-reduced (max)
        across workers."""
        comm = self.circuit.comm
        st = {"wm": 0}

        def fn(b: Batch):
            k = b.last_key()
            if k is not None:
                st["wm"] = max(st["wm"], f(k[0] if len(k) == 1 else k))
            if comm is not None and comm.world_size > 1:
                st["wm"] = comm.allreduce_max(st["wm"])
            return st["wm"]

        return self._unary(fn, "watermark_monotonic", None)

    # -- communication -------------------------------------------------------
    def shard(self) -> "Stream":
        """shard (operator/communication/shard.rs:89-162): hash-partition by
        key, all-to-all, merge at the receiver.  Identity with one worker
        (shard.rs:111-114) or when already sharded."""
        comm = self.circuit.comm
        if comm is None or comm.world_size == 1 or self.sharded:
            return Stream(self.circuit, self.node, self.schema, True)
        be = self.circuit.be
        return self._unary(lambda b: comm.shard(be, b), "shard", self.schema, True)

    def shard_with(self, other: "Stream") -> tuple["Stream", "Stream"]:
        """shard() of both inputs of a binary operator (join.rs:265-266) in ONE
        exchange round: same result as (self.shard(), other.shard())."""
        comm = self.circuit.comm
        if comm is None or comm.world_size == 1 or self.sharded or other.sharded:
            return self.shard(), other.shard()
        be = self.circuit.be
        pair = Node(self.circuit, [self.node, other.node], lambda a, b: comm.shard_many(be, [a, b]), "shard2")
        left = Stream(self.circuit, Node(self.circuit, [pair], lambda t: t[0], "shard2.0"), self.schema, True)
        right = Stream(self.circuit, Node(self.circuit, [pair], lambda t: t[1], "shard2.1"), other.schema, True)
        return left, right

    def gather(self, root: int = 0) -> "Stream":
        """gather (operator/communication/gather.rs:41-103)."""
        comm = self.circuit.comm
        if comm is None or comm.world_size == 1:
            return self
        be = self.circuit.be
        return self._unary(lambda b: comm.gather(be, b, root), "gather", self.schema)
