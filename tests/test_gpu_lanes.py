"""The two execution lanes: dbsp_batches_from_tables and dbsp_join_step return what the single calls return in
sequence, on CUDA and on the oracle; an error detected on lane 1 comes back as the call's status; batches made on
lane 1 download like any other."""
import zlib

import numpy as np
import pytest

from dbsp_b200 import Schema, Spine
from dbsp_b200._capi import DbspError
from dbsp_b200.zset import Proj, col, key, lval, rval
from parity_util import assert_batches_equal

pytestmark = pytest.mark.gpu

STATES = (1, 2, 3)


def _table(name):
    """(5 raw u64 columns, weights or None, projection) of one catalogue table."""
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    cols = lambda n: [rng.integers(0, 1 << 40, n).astype(np.uint64) for _ in range(5)]   # noqa: E731
    if name == "empty":
        return [np.empty(0, np.uint64)] * 5, None, Proj(Schema("u", "u"), [col(0), col(1)])
    if name == "all_filtered":
        return cols(5000), None, Proj(Schema("u", "u"), [col(0), col(1)], where=[col(2).eq(7)])
    if name == "id_ordered":   # already canonical: the projected rows are adopted without a sort
        c = cols(40_000)
        c[0] = np.arange(1000, 41_000, dtype=np.uint64)
        c[3] = rng.integers(0, 6, 40_000).astype(np.uint64)
        return c, None, Proj(Schema("u", "uuu"), [col(0), col(1), col(2), col(3)], where=[col(3).isin(STATES)])
    if name == "unordered_60k":   # two-pass sort
        c = cols(60_000)
        c[1] = rng.integers(0, 20_000, 60_000).astype(np.uint64)
        return c, rng.integers(-2, 3, 60_000), Proj(Schema("u", "u"), [col(1), col(0)])
    if name == "big_300k":   # splitter mode
        c = cols(300_000)
        c[0] = rng.integers(0, 1 << 20, 300_000).astype(np.uint64)
        return c, None, Proj(Schema("u", "uu"), [col(0), col(2), col(3)])
    if name == "two_word_i64":
        c = cols(80_000)
        c[0] = rng.integers(-500, 500, 80_000).astype(np.int64).view(np.uint64)
        c[1] = rng.integers(-(1 << 40), 1 << 40, 80_000).astype(np.int64).view(np.uint64)
        return c, rng.integers(-1, 2, 80_000), Proj(Schema("ii", "iu"), [col(0), col(1), col(1), col(4)])
    if name == "hot_key":   # most rows share a key: the sort raises its fallback flag
        n = 200_000
        c = cols(n)
        c[0] = np.where(rng.random(n) < 0.7, 12345, rng.integers(0, 1 << 30, n)).astype(np.uint64)
        return c, rng.integers(-1, 2, n), Proj(Schema("u", "u"), [col(0), col(1)])
    raise KeyError(name)


GROUPS = [
    ["empty"], ["all_filtered"], ["id_ordered"], ["unordered_60k"], ["big_300k"], ["two_word_i64"], ["hot_key"],
    ["big_300k", "hot_key"],   # the hot key lands on lane 1 (fewer rows)
    ["unordered_60k", "id_ordered"],
    ["empty", "all_filtered"],
    ["two_word_i64", "unordered_60k"],
    ["big_300k", "two_word_i64", "empty"],
    ["hot_key", "all_filtered", "id_ordered"],
]


def _device(cols, w):
    import torch

    dc = [torch.from_numpy(c.view(np.int64).copy()).cuda() for c in cols]
    dw = torch.from_numpy(np.asarray(w, np.int64).copy()).cuda() if w is not None else None
    return dc, dw


@pytest.mark.parametrize("source", ["dev", "upload", "host"])
@pytest.mark.parametrize("group", GROUPS, ids=lambda g: "+".join(g))
def test_batches_from_tables_equal_single_calls(cuda, oracle, group, source):
    import torch

    specs = [_table(n) for n in group]
    keep, jobs, singles = [], [], []
    for cols, w, proj in specs:
        n = len(cols[0])
        if source == "dev":
            dc, dw = _device(cols, w)
            keep.append((dc, dw))
            ptrs = [int(x.data_ptr()) for x in dc]
            wp = int(dw.data_ptr()) if dw is not None else None
            jobs.append((("dev", ptrs, wp, n), proj))
            singles.append(cuda.batch_from_table(ptrs, proj, weights=wp, n=n, on_device=True))
        elif source == "upload":
            if w is not None:   # uploads of weighted tables are covered by the host source
                w = None
            jobs.append((("upload", cuda.upload_begin(cols, cuda.proj_table_mask(proj)), None, None), proj))
            singles.append(cuda.batch_from_upload(cuda.upload_begin(cols, cuda.proj_table_mask(proj)), proj))
        else:
            jobs.append((("host", cols, w, None), proj))
            singles.append(cuda.batch_from_table(cols, proj, weights=w))
        specs[len(jobs) - 1] = (cols, w, proj)
    torch.cuda.synchronize()
    got = cuda.batches_from_tables(jobs)
    assert len(got) == len(group)
    for name, g, s, (cols, w, proj) in zip(group, got, singles, specs):
        assert_batches_equal(g, s, f"{name} ({source}) vs the single call")
        assert_batches_equal(g, oracle.batch_from_table(cols, proj, weights=w), f"{name} ({source}) vs the oracle")


def test_lane1_error_is_the_calls_error(cuda):
    cols, _, proj = _table("unordered_60k")
    bad = [np.zeros(10, np.uint64)] * 9   # nine columns: rejected, on lane 1 (the smaller job)
    with pytest.raises(DbspError, match="1..8 columns"):
        cuda.batches_from_tables([(("host", cols, None, None), proj), (("host", bad, None, None), proj)])
    got = cuda.batches_from_tables([(("host", cols, None, None), proj), (("host", cols, None, None), proj)])
    ref = cuda.batch_from_table(cols, proj)
    for g in got:
        assert_batches_equal(g, ref, "after a lane-1 error")


def test_download_begin_of_lane1_batch(cuda):
    big, _, pb = _table("big_300k")
    small, _, ps = _table("unordered_60k")
    a, b = cuda.batches_from_tables([(("host", big, None, None), pb), (("host", small, None, None), ps)])
    for x in (a, b):   # b was made on lane 1
        n = len(x)
        cols = [np.empty(n, np.uint64) for _ in range(x.schema.nl)]
        d = cuda.download_begin(x, cols, np.empty(n, np.int64))
        got_cols, got_w = d.finish()
        want = x.download()
        offs = np.asarray(want["offs"]).astype(np.int64) if want["offs"] is not None else None
        keys = [np.asarray(k).view(np.uint64) for k in want["keys"]]
        if offs is not None:
            keys = [np.repeat(k, np.diff(offs)) for k in keys]
        flat = keys + [np.asarray(v).view(np.uint64) for v in want["vals"]]
        for l, c in enumerate(flat):
            assert np.array_equal(got_cols[l], c), f"lane {l}"
        assert np.array_equal(got_w, np.asarray(want["diffs"]))


LS, RS = Schema("u", "u"), Schema("u", "uu")
JPROJ = Proj(Schema("u", "uu"), [key(0), lval(0), rval(1)], where=[rval(0).ge(lval(0))])


def _deltas(n_steps, seed):
    """Per step (dl rows, dr rows): first sizes that shrink geometrically, so each batch takes a spine layer of
    its own and the traces grow past 16 batches; then equal sizes on both sides, so merges fall due in both
    spines in the same step; empty deltas on either side and on both."""
    rng = np.random.default_rng(seed)
    sizes = [(1 << k, 1 << k) for k in range(17, 0, -1)]
    sizes += [(3000, 3000)] * 6 + [(0, 2000), (2000, 0), (0, 0), (50_000, 40_000)]
    out = []
    for nl, nr in sizes[:n_steps]:
        dl = ([rng.integers(0, 1 << 20, nl).astype(np.uint64), rng.integers(0, 1 << 30, nl).astype(np.uint64)],
              rng.integers(-1, 3, nl))
        dr = ([rng.integers(0, 1 << 20, nr).astype(np.uint64), rng.integers(0, 1 << 30, nr).astype(np.uint64),
               rng.integers(0, 1 << 30, nr).astype(np.uint64)], rng.integers(-1, 3, nr))
        out.append((dl, dr))
    return out


def _sequential(be, lt, rt, dl, dr):
    rt.insert(dr)
    o1 = be.join_delta_trace(dl, rt, JPROJ, delta_is_left=True)
    o2 = be.join_delta_trace(dr, lt, JPROJ, delta_is_left=False)
    lt.insert(dl)
    return be.merge(o1, o2)


def test_join_step_equals_sequential(cuda, oracle):
    steps = _deltas(100, 7)
    st = {be: {"step": (Spine(be, LS), Spine(be, RS)), "seq": (Spine(be, LS), Spine(be, RS))} for be in (cuda, oracle)}
    max_batches = 0
    o2_only = 0   # output rows of steps with an empty left delta: o2 alone
    for i, ((lc, lw), (rc, rw)) in enumerate(steps):
        outs = {}
        for be in (cuda, oracle):
            dl, dr = be.batch_from_columns(LS, lc, lw), be.batch_from_columns(RS, rc, rw)
            lt, rt = st[be]["step"]
            outs[be, "step"] = be.join_step(dl, dr, lt, rt, JPROJ)
            slt, srt = st[be]["seq"]
            outs[be, "seq"] = _sequential(be, slt, srt, dl, dr)
        assert_batches_equal(outs[cuda, "step"], outs[cuda, "seq"], f"step {i}: CUDA join_step vs sequential")
        assert_batches_equal(outs[oracle, "step"], outs[oracle, "seq"], f"step {i}: oracle join_step vs sequential")
        assert_batches_equal(outs[cuda, "step"], outs[oracle, "step"], f"step {i}: CUDA vs oracle")
        for side in (0, 1):
            a, b = st[cuda]["step"][side], st[cuda]["seq"][side]
            assert a.stats() == b.stats(), f"step {i}: trace {side} layout differs"
        if len(lw) == 0:
            o2_only += len(outs[cuda, "step"])
        max_batches = max(max_batches, st[cuda]["step"][0].stats()[1], st[cuda]["step"][1].stats()[1])
    for side in (0, 1):
        assert_batches_equal(st[cuda]["step"][side].consolidate(), st[oracle]["step"][side].consolidate(), f"trace {side}")
    assert max_batches > 16
    assert o2_only > 0
