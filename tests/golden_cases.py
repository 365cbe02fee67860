"""The reference's own golden vectors for the hot path (SURVEY.md §8c), written
once against the Stream API and run against any backend: the CPU oracle
(`-m "not gpu"`, pins the oracle) and the CUDA library (`-m gpu`, parity).

Strings in the reference literals are replaced by order-preserving integer
codes (single letters -> ord(), decimal strings -> their value, names ->
rank in a sorted dictionary).  Paths are relative to /root/reference/crates.
"""
import numpy as np

from dbsp_b200 import FoldCount, FoldSum, Max, Min, Proj, RootCircuit, Schema, key, lval, rval
from dbsp_b200.nexmark import queries as nq


def zset(be, schema, rows):
    return be.batch_from_rows(schema, rows)


def rows_of(b):
    return b.rows()


# ---- consolidation (dbsp/src/trace/consolidation/tests/mod.rs:14-163) -------
def consolidation_cases():
    a, b = ord("a"), ord("b")
    cases = [
        ([(a, -1), (b, -2), (a, 1)], [(b, -2)]),
        ([(a, -1), (b, 0), (a, 1)], []),
        ([(a, 0)], []),
        ([(a, 0), (b, 0)], []),
        ([(a, 1), (b, 1)], [(a, 1), (b, 1)]),
    ]
    return cases


def run_consolidation(be):
    s = Schema("u")
    for inp, out in consolidation_cases():
        assert rows_of(zset(be, s, inp)) == out
    # consolidate_paired_slices_corpus (tests/mod.rs:103-163)
    corpus = [((0, 0), 0)] * 10 + [((1107, 0), 0)] + [((0, 0), 0)] * 4 + [((1107, 0), 0)] + [
        ((0, 0), 1), ((0, 0), 1), ((0, 0), -1), ((0, 0), -1), ((0, 0), 1)]
    got = rows_of(zset(be, Schema("uu"), [(k[0], k[1], w) for k, w in corpus]))
    assert got == [(0, 0, 1)]
    # empty input
    assert rows_of(zset(be, s, [])) == []


# ---- join (dbsp/src/operator/join.rs:887-1017) ------------------------------
def run_join_test(be):
    o = ord
    input1 = [
        [(1, o("a"), 1), (1, o("b"), 2), (2, o("c"), 3), (2, o("d"), 4), (3, o("e"), 5), (3, o("f"), -2)],
        [(1, o("a"), 1)],
        [(1, o("a"), 1)],
        [(4, o("n"), 2)],
        [(1, o("a"), 0)],
    ]
    input2 = [
        [(2, o("g"), 3), (2, o("h"), 4), (3, o("i"), 5), (3, o("j"), -2), (4, o("k"), 5), (4, o("l"), -2)],
        [(1, o("b"), 1)],
        [(4, o("m"), 1)],
        [],
        [],
    ]
    outputs = [
        [(2, o("c"), o("g"), 9), (2, o("c"), o("h"), 12), (2, o("d"), o("g"), 12), (2, o("d"), o("h"), 16),
         (3, o("e"), o("i"), 25), (3, o("e"), o("j"), -10), (3, o("f"), o("i"), -10), (3, o("f"), o("j"), 4)],
        [(1, o("a"), o("b"), 1)],
        [], [], [],
    ]
    inc_outputs = [
        outputs[0],
        [(1, o("a"), o("b"), 2), (1, o("b"), o("b"), 2)],
        [(1, o("a"), o("b"), 1)],
        [(4, o("n"), o("k"), 10), (4, o("n"), o("l"), -4), (4, o("n"), o("m"), 2)],
        [],
    ]
    c = RootCircuit(be)
    pair = Schema("uu")
    it1, it2 = iter(input1), iter(input2)
    index1 = c.add_source(lambda: zset(be, pair, next(it1)), pair).index(1)
    index2 = c.add_source(lambda: zset(be, pair, next(it2)), pair).index(1)
    proj = Proj(Schema("uuu"), [key(0), lval(0), rval(0)])   # (k, format!("{} {}", s1, s2))
    got = {"stream": [], "inc": [], "join": []}
    index1.stream_join(index2, proj).gather(0).inspect(lambda b: got["stream"].append(rows_of(b)))
    index1.join_incremental(index2, proj).gather(0).inspect(lambda b: got["inc"].append(rows_of(b)))
    index1.join(index2, proj).gather(0).inspect(lambda b: got["join"].append(rows_of(b)))
    for _ in range(5):
        c.step()
    assert got["stream"] == outputs
    assert got["inc"] == inc_outputs
    assert got["join"] == inc_outputs


# ---- merge batcher (dbsp/src/trace/ord/merge_batcher/tests.rs:26-125) ---------
def run_merge_batcher(be):
    """The literal MergeSorter tests, observed through push / seal (the chunk
    structure of the reference's expected values is flattened)."""
    def cols(rows, nl):
        return [np.array([r[l] for r in rows], dtype=np.uint64) for l in range(nl)], np.array([r[-1] for r in rows], dtype=np.int64)

    one, two = Schema("u"), Schema("uu")
    # merge_empty_inputs
    b = be.batcher(one)
    assert b.tuples() == 0 and b.seal().rows() == []
    # small_push: queue [[(0,0):1], [(45,0):-1]] then push [(45,1):1]
    b = be.batcher(two)
    b.push_consolidated_batch(*cols([(0, 0, 1), (45, 0, -1)], 2))
    b.push_batch(*cols([(45, 1, 1)], 2))
    assert b.seal().rows() == [(0, 0, 1), (45, 0, -1), (45, 1, 1)]
    # merge_by
    b = be.batcher(one)
    b.push_consolidated_batch(*cols([(0, 1), (1, 6), (24, 5), (54, -23)], 1))
    b.push_consolidated_batch(*cols([(0, 7), (1, 6), (24, -5), (25, 12), (89, 1)], 1))
    assert b.seal().rows() == [(0, 8), (1, 12), (25, 12), (54, -23), (89, 1)]
    # push_with_excess_stashes
    b = be.batcher(one)
    b.push_batch(*cols([(0, 1), (1, 6), (24, 5), (54, -23)], 1))
    assert b.tuples() == 4
    assert b.seal().rows() == [(0, 1), (1, 6), (24, 5), (54, -23)]
    # force_finish_merge / force_merge_on_push
    expected = [(0, 9), (1, 18), (23, 54), (24, 5), (25, 12), (54, -46), (89, 1), (97, -102)]
    for last_is_push in (False, True):
        b = be.batcher(one)
        b.push_consolidated_batch(*cols([(0, 1), (1, 6), (24, 5), (54, -23)], 1))
        b.push_consolidated_batch(*cols([(89, 1)], 1))
        b.push_consolidated_batch(*cols([(0, 8), (1, 12), (25, 12), (54, -23)], 1))
        if last_is_push:
            b.push_batch(*cols([(97, -102), (23, 54)], 1))
        else:
            b.push_consolidated_batch(*cols([(23, 54), (97, -102)], 1))
        assert b.seal().rows() == expected


# ---- antijoin (dbsp/src/operator/join.rs:1335-1385) --------------------------
def run_antijoin(be):
    input1 = [[(1, 0, 1), (1, 1, 2), (2, 0, 1), (2, 1, 1)], [(3, 1, 1)], [], [(2, 2, 1), (4, 1, 1)]]
    input2 = [[], [], [(1, 1, 3)], [(2, 5, 1)]]
    outputs = [
        [(1, 0, 1), (1, 1, 2), (2, 0, 1), (2, 1, 1)],
        [(3, 1, 1)],
        [(1, 0, -1), (1, 1, -2)],
        [(2, 0, -1), (2, 1, -1), (4, 1, 1)],
    ]
    c = RootCircuit(be)
    pair = Schema("uu")
    it1, it2 = iter(input1), iter(input2)
    in1 = c.add_source(lambda: zset(be, pair, next(it1)), pair).index(1)
    in2 = c.add_source(lambda: zset(be, pair, next(it2)), pair).index(1)
    got = []
    in1.antijoin(in2).gather(0).inspect(lambda b: got.append(rows_of(b)))
    for _ in range(4):
        c.step()
    assert got == outputs


# ---- aggregate (dbsp/src/operator/aggregate/mod.rs:878-998) -----------------
def run_count_test(be):
    c = RootCircuit(be)
    inp, h = c.add_input_indexed_zset(Schema("u", "u"))
    outs = {}
    inp.aggregate_linear(lambda_one()).gather(0).inspect(lambda b: outs.__setitem__("count_weighted", rows_of(b)))
    inp.aggregate_linear(lval(0)).gather(0).inspect(lambda b: outs.__setitem__("sum_weighted", rows_of(b)))
    inp.aggregate(FoldCount).gather(0).inspect(lambda b: outs.__setitem__("count_distinct", rows_of(b)))
    inp.aggregate(FoldSum).gather(0).inspect(lambda b: outs.__setitem__("sum_distinct", rows_of(b)))

    h.append([(1, 1, 1), (1, 2, 2)])
    c.step()
    assert outs["count_distinct"] == [(1, 2, 1)]
    assert outs["sum_distinct"] == [(1, 3, 1)]
    assert outs["count_weighted"] == [(1, 3, 1)]
    assert outs["sum_weighted"] == [(1, 5, 1)]

    h.append([(2, 2, 1), (2, 4, 1), (1, 2, -1)])
    c.step()
    assert outs["count_distinct"] == [(2, 2, 1)]
    assert outs["sum_distinct"] == [(2, 6, 1)]
    assert outs["count_weighted"] == [(1, 2, 1), (1, 3, -1), (2, 2, 1)]
    assert outs["sum_weighted"] == [(1, 3, 1), (1, 5, -1), (2, 6, 1)]

    h.append([(1, 3, 1), (1, 2, -1)])
    c.step()
    assert outs["count_distinct"] == []
    assert outs["sum_distinct"] == [(1, 3, -1), (1, 4, 1)]
    assert outs["count_weighted"] == []
    assert outs["sum_weighted"] == [(1, 3, -1), (1, 4, 1)]


def lambda_one():
    from dbsp_b200 import const

    return const(1)


# ---- average (dbsp/src/operator/aggregate/average.rs:317-331) ----------------
def run_average(be):
    c = RootCircuit(be)
    inp, h = c.add_input_indexed_zset(Schema("u", "i"))
    out = []
    inp.average(lval(0)).inspect(lambda b: out.append(rows_of(b)))
    # Avg(1000,10) -> 100 ; Avg(200,20) -> 10
    h.append([(1, 100, 10), (2, 10, 20)])
    c.step()
    assert out[-1] == [(1, 100, 1), (2, 10, 1)]
    # truncating signed division: (-7)/2 = -3
    h.append([(3, -7, 1), (3, 0, 1)])
    c.step()
    assert out[-1] == [(3, -3, 1)]


# ---- distinct (dbsp/src/operator/distinct.rs:825-890) ------------------------
def run_distinct_indexed(be):
    c = RootCircuit(be)
    inp, h = c.add_input_indexed_zset(Schema("u", "u"))
    o1, o2 = [], []
    inp.integrate().stream_distinct().gather(0).inspect(lambda b: o2.append(rows_of(b)))
    inp.distinct().integrate().gather(0).inspect(lambda b: o1.append(rows_of(b)))
    h.append([(1, 0, 1), (1, 1, 2), (2, 0, 1), (2, 1, 1)])
    c.step()
    assert o1[-1] == [(1, 0, 1), (1, 1, 1), (2, 0, 1), (2, 1, 1)] and o1[-1] == o2[-1]
    h.append([(3, 1, 1), (2, 1, 1)])
    c.step()
    assert o1[-1] == [(1, 0, 1), (1, 1, 1), (2, 0, 1), (2, 1, 1), (3, 1, 1)] and o1[-1] == o2[-1]
    h.append([(1, 1, 3), (2, 1, -3)])
    c.step()
    assert o1[-1] == [(1, 0, 1), (1, 1, 1), (2, 0, 1), (3, 1, 1)] and o1[-1] == o2[-1]


# ---- window (dbsp/src/operator/time_series/window.rs:250-451) ----------------
def _window_run(be, inputs, outputs, bounds_fn, steps):
    c = RootCircuit(be)
    pair = Schema("uu")
    it = iter(inputs)
    st = {"i": 0}

    def bgen():
        r = bounds_fn(st["i"])
        st["i"] += 1
        return r

    bounds = c.add_source(bgen)
    index1 = c.add_source(lambda: zset(be, pair, [(t, t, w) for t, w in next(it)]), pair).index(1)
    got = []
    index1.window(bounds).inspect(lambda b: got.append(rows_of(b)))
    for _ in range(steps):
        c.step()
    exp = [sorted((t, t, w) for t, w in o) for o in outputs]
    assert got == exp


def run_window_sliding(be):
    inputs = [
        [(800, 1), (900, 1), (950, 1), (999, 1), (1000, 1)],
        [(700, 1), (900, 1), (901, 1), (999, 1), (1000, 1), (1001, 1), (1002, 1), (1003, 1)],
        [(1004, 1)], [], [], [],
    ]
    outputs = [
        [(900, 1), (950, 1), (999, 1)],
        [(900, -1), (901, 1), (999, 1), (1000, 2)],
        [(901, -1), (1001, 1)],
        [(1002, 1)], [(1003, 1)], [(1004, 1)],
    ]
    _window_run(be, inputs, outputs, lambda i: (1000 + i - 100, 1000 + i), 6)


def run_window_tumbling(be):
    inputs = [
        [(700, 1), (995, 1), (996, 1), (999, 1), (1000, 1)],
        [(995, 1), (1000, 1), (1001, 1)],
        [(999, 1)], [(1002, 1)], [(1003, 1)], [(996, 1)], [(999, 1)], [(1004, 1)], [(1005, 1)], [(1010, 1)], [(1005, 1)],
    ]
    outputs = [
        [(995, 1), (996, 1), (999, 1)],
        [(995, 1)],
        [(999, 1)],
        [], [],
        [(1000, 2), (1001, 1), (1002, 1), (1003, 1), (995, -2), (996, -1), (999, -2)],
        [],
        [(1004, 1)],
        [], [],
        [(1000, -2), (1001, -1), (1002, -1), (1003, -1), (1004, -1), (1005, 2)],
    ]

    def b(i):
        clock = 1000 + i
        start = (clock // 5) * 5 - 5
        return (start, start + 5)

    _window_run(be, inputs, outputs, b, 11)


def run_window_shrinking(be):
    inputs = [
        [(800, 1), (900, 1), (950, 1), (990, 1), (999, 1), (1000, 1)],
        [(700, 1), (900, 1), (901, 1), (915, 1), (940, 1), (985, 1), (999, 1), (1000, 1), (1001, 1), (1002, 1), (1003, 1)],
        [(1004, 1), (1010, 1), (1020, 1), (1039, 1)],
        [], [], [],
    ]
    outputs = [
        [(900, 1), (950, 1), (990, 1), (999, 1)],
        [(900, -1), (915, 1), (940, 1), (985, 1), (990, -1), (999, -1)],
        [(915, -1), (985, -1)],
        [(1000, 2), (1001, 1), (1002, 1), (1003, 1), (1004, 1), (1010, 1), (1020, 1), (1039, 1), (985, 1), (990, 1), (999, 2)],
        [(1039, -1), (940, -1)],
        [(1020, -1), (950, -1)],
    ]
    windows = [(900, 1000), (910, 990), (920, 980), (940, 1040), (950, 1030), (960, 1020)]
    _window_run(be, inputs, outputs, lambda i: windows[i], 6)


# ---- watermark (dbsp/src/operator/time_series/watermark.rs:81-120) -----------
def run_watermark(be):
    c = RootCircuit(be)
    inp, h = c.add_input_zset(Schema("u"))
    got = []
    inp.watermark_monotonic(lambda ts: ts + 5).inspect(lambda w: got.append(w))
    for batch in ([(100, 1), (110, 1), (50, 1)], [(90, 1), (90, 1), (50, 1)], [(110, 1), (120, 1), (100, 1)], [(130, 1), (140, 1), (0, 1)]):
        h.append(batch)
        c.step()
    assert got == [115, 115, 125, 145]


# ---- Nexmark q3 / q4 / q7 (nexmark/src/queries/{q3,q4,q7}.rs tests) ----------
def _make_person(**kw):   # generator/mod.rs:161-172 make_person()
    d = dict(id=1, name="AAA BBBB", city="Phoenix", state="OR", date_time=0)
    d.update(kw)
    return d


def _make_auction(**kw):  # generator/mod.rs:186-199
    d = dict(id=1, seller=1, category=1, date_time=0, expires=2000)
    d.update(kw)
    return d


def _make_bid(**kw):      # generator/mod.rs:174-184
    d = dict(auction=1, bidder=1, price=99, date_time=0, extra=0)
    d.update(kw)
    return d


def _feed(handles, events, dicts):
    """events: list of ('person'|'auction'|'bid', dict).  Sets the three tables."""
    P = [e for k, e in events if k == "person"]
    A = [e for k, e in events if k == "auction"]
    B = [e for k, e in events if k == "bid"]
    u = lambda xs: np.array(xs, dtype=np.uint64)
    handles["person"].set([u([p["id"] for p in P]), u([dicts["name"][p["name"]] for p in P]),
                           u([dicts["city"][p["city"]] for p in P]), u([dicts["state"][p["state"]] for p in P]),
                           u([p["date_time"] for p in P])])
    handles["auction"].set([u([a[k] for a in A]) for k in ("id", "seller", "category", "date_time", "expires")])
    handles["bid"].set([u([b[k] for b in B]) for k in ("auction", "bidder", "price", "date_time", "extra")])


def run_q3(be):
    """queries/q3.rs:75-220 test_q3_people."""
    names = sorted(["NL Seller", "CA Seller", "ID Seller", "OR Seller", "AAA BBBB"])
    states = sorted(["NL", "CA", "ID", "OR"])
    dicts = {"name": {s: i for i, s in enumerate(names)}, "city": {"Phoenix": 0}, "state": {s: i for i, s in enumerate(states)}}
    steps = [
        [("person", _make_person(id=1, name="NL Seller", state="NL")),
         ("person", _make_person(id=2, name="CA Seller", state="CA")),
         ("person", _make_person(id=3, name="ID Seller", state="ID")),
         ("auction", _make_auction(id=999, seller=2, category=10)),
         ("auction", _make_auction(id=452, seller=3, category=10))],
        [("person", _make_person(id=4, name="OR Seller", state="OR")),
         ("auction", _make_auction(id=999, seller=4, category=11)),
         ("person", _make_person(id=5, name="OR Seller", state="OR")),
         ("auction", _make_auction(id=333, seller=5, category=10))],
    ]
    N, S = dicts["name"], dicts["state"]
    expected = [
        [(N["CA Seller"], 0, S["CA"], 999, 1), (N["ID Seller"], 0, S["ID"], 452, 1)],
        [(N["OR Seller"], 0, S["OR"], 333, 1)],
    ]
    c = RootCircuit(be)
    inp, handles = nq.add_nexmark_input(c)
    got = []
    nq.q3(inp, states_of_interest=[S["OR"], S["ID"], S["CA"]]).inspect(lambda b: got.append(rows_of(b)))
    for ev in steps:
        _feed(handles, ev, dicts)
        c.step()
    assert got == expected


def run_q4(be):
    """queries/q4.rs:95-237 test_q4_average_final_bids_per_category."""
    steps = [
        [("auction", _make_auction(id=1, category=1, date_time=1000, expires=2000)),
         ("auction", _make_auction(id=2, category=1)),
         ("auction", _make_auction(id=3, category=2)),
         ("bid", _make_bid(auction=1, date_time=1100, price=80)),
         ("bid", _make_bid(price=100, auction=1, date_time=1500)),
         ("bid", _make_bid(price=500, auction=1, date_time=2500)),
         ("bid", _make_bid(price=300, auction=2)),
         ("bid", _make_bid(price=200, auction=2)),
         ("bid", _make_bid(price=20, auction=3))],
        [("bid", _make_bid(price=30, auction=3))],
        [("auction", _make_auction(id=4, category=2)),
         ("bid", _make_bid(price=60, auction=4))],
    ]
    expected = [
        [(1, 200, 1), (2, 20, 1)],
        [(2, 20, -1), (2, 30, 1)],
        [(2, 30, -1), (2, 45, 1)],
    ]
    c = RootCircuit(be)
    inp, handles = nq.add_nexmark_input(c)
    got = []
    nq.q4(inp).inspect(lambda b: got.append(rows_of(b)))
    for ev in steps:
        _feed(handles, ev, {"name": {}, "city": {}, "state": {}})
        c.step()
    assert got == expected


Q7_CASES = {   # queries/q7.rs:108-147 (rstest cases)
    "latest_bid_determines_window": (
        [[(9_000, 1_000_000), (11_000, 50), (14_000, 90), (16_000, 70), (21_000, 1_000_000), (32_000, 1_000_000)]],
        [[(1, 1, 90, 14_000, 0, 1)]]),
    "window_boundary_below": ([[(9_999, 50), (32_000, 1_000_000)]], [[]]),
    "window_boundary_lower": ([[(10_000, 50), (32_000, 1_000_000)]], [[(1, 1, 50, 10_000, 0, 1)]]),
    "window_boundary_upper": ([[(19_999, 50), (32_000, 1_000_000)]], [[(1, 1, 50, 19_999, 0, 1)]]),
    "window_boundary_above": ([[(20_000, 50), (32_000, 1_000_000)]], [[]]),
    "tumble_into_new_window": (
        [[(9_000, 1_000_000), (11_000, 50), (14_000, 90), (16_000, 70), (21_000, 1_000_000)], [(32_000, 10)], [(42_000, 10)]],
        [[(1, 1, 1_000_000, 9_000, 0, 1)],
         [(1, 1, 90, 14_000, 0, 1), (1, 1, 1_000_000, 9_000, 0, -1)],
         [(1, 1, 90, 14_000, 0, -1), (1, 1, 1_000_000, 21_000, 0, 1)]]),
    "multiple_max_bids": (
        [[(11_000, 90), (14_000, 90), (16_000, 90), (21_000, 1_000_000), (32_000, 1_000_000)]],
        [[(1, 1, 90, 11_000, 0, 1), (1, 1, 90, 14_000, 0, 1), (1, 1, 90, 16_000, 0, 1)]]),
}


def run_q7(be, case):
    batches, expected = Q7_CASES[case]
    c = RootCircuit(be)
    inp, handles = nq.add_nexmark_input(c)
    got = []
    nq.q7(inp).inspect(lambda b: got.append(rows_of(b)))
    for batch in batches:
        _feed(handles, [("bid", _make_bid(date_time=dt, price=p)) for dt, p in batch], {"name": {}, "city": {}, "state": {}})
        c.step()
    assert got == [sorted(e) for e in expected]


ALL_CASES = {
    "consolidation": run_consolidation,
    "join_test": run_join_test,
    "count_test": run_count_test,
    "average": run_average,
    "distinct_indexed": run_distinct_indexed,
    "window_sliding": run_window_sliding,
    "window_tumbling": run_window_tumbling,
    "antijoin": run_antijoin,
    "merge_batcher": run_merge_batcher,
    "window_shrinking": run_window_shrinking,
    "watermark": run_watermark,
    "q3": run_q3,
    "q4": run_q4,
}
for _name in Q7_CASES:
    ALL_CASES["q7_" + _name] = (lambda be, _n=_name: run_q7(be, _n))


# ---- window bounded_memory (dbsp/src/operator/time_series/window.rs:453-486) ----
# 100 fresh timestamps per step under the window (watermark - 1000, watermark): the trace behind the window must
# not grow with the stream (the reference asserts < 20 000 bytes over 10 000 steps; here: rows, over 1 500 steps).
def run_window_bounded_memory(be, steps=1500):
    c = RootCircuit(be)
    inp, h = c.add_input_zset(Schema("i"))
    bounds = inp.watermark_monotonic(lambda ts: ts).apply(lambda ts: (ts - 1000, ts))
    w = inp.window(bounds)
    out = w.output()
    worst = 0
    for i in range(steps):
        h.append((j, 1) for j in range(i * 100, (i + 1) * 100))   # input_handle.push(j, 1)
        c.step()
        worst = max(worst, w.window_trace.stats()[0])   # rows held by the trace (all layers)
    assert worst <= 1200, worst          # the window (1000 timestamps) + the step that just arrived
    assert len(out.value) <= 200


# run on the oracle by test_oracle_golden.py and on the CUDA library by test_zz_gpu_late.py
ORACLE_ONLY_CASES = {"window_bounded_memory": run_window_bounded_memory}
