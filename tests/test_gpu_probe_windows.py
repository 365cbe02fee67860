"""Join probes against traces whose batches cover disjoint key ranges, against the oracle.

The probe bounds, per tile of sorted delta rows and per trace batch, the window of batch rows between the tile's
first and last key, and settles every key of the tile for a batch whose window is empty.  These cases put delta
tiles wholly above, below, between and inside the batches' key ranges (q3's shape: fresh keys that only the newest
batch can hold), one key whose delta rows span several tiles and match in several batches, signed keys with
negative values, two-lane keys, a one-row batch and a batch whose rows all share one key."""
import numpy as np
import pytest

from dbsp_b200 import Schema, Spine
from dbsp_b200.zset import Proj, key, lval, rval
from parity_util import assert_batches_equal

pytestmark = pytest.mark.gpu

GAP = 10_000      # batch j holds keys in [lo_j, lo_j + HALF); [lo_j + HALF, lo_j + GAP) is a gap no batch covers
HALF = 5_000
SIZES = (20_000, 8_000, 3_000, 900, 200, 1)   # decreasing: the spine keeps them in separate batches


def key_lanes(keys, kt):
    """Split int64 keys over the key lanes of type string kt, order preserving."""
    if len(kt) == 1:
        return [keys if kt == "i" else (keys + (1 << 40)).astype(np.uint64)]
    hi, lo = np.divmod(keys, 97)
    return [hi if kt[0] == "i" else (hi + (1 << 40)).astype(np.uint64), lo.astype(np.uint64)]


def base(j, kt):
    return (j - 3) * GAP if kt[0] == "i" else j * GAP   # signed keys: the older batches hold negative keys


def delta_keys(rng, mode, nd, kt):
    nb = len(SIZES)
    top = base(nb - 1, kt)
    if mode == "newest":     # q3: every key at or past the newest batches' ranges
        return base(nb - 3, kt) + rng.integers(0, 3 * GAP, nd)
    if mode == "above":      # past every batch but a few hits in the newest one
        k = top + HALF + rng.integers(0, 3 * GAP, nd)
        k[: nd // 50 + 1] = top
        return k
    if mode == "below":      # below every batch but a few hits in the oldest one
        k = base(0, kt) - 3 * GAP + rng.integers(0, 3 * GAP, nd)
        k[: nd // 50 + 1] = base(0, kt)
        return k
    if mode == "gaps":       # between batches' ranges, one hit per batch
        j = rng.integers(0, nb, nd)
        k = np.array([base(x, kt) for x in j]) + HALF + rng.integers(0, GAP - HALF, nd)
        k[: min(nb, nd)] = [base(x, kt) + 7 for x in range(min(nb, nd))]
        return k
    return base(0, kt) + rng.integers(0, nb * GAP, nd)   # mixed


def run_join(be, kt, mode, nd, left, hot_rows=0):
    s = Schema(kt, "u")
    rng = np.random.default_rng(nd * 31 + len(kt) * 7 + left + hot_rows + sum(map(ord, mode + kt)))
    tr = Spine(be, s)
    for j, m in enumerate(SIZES):
        k = base(j, kt) + rng.integers(0, HALF, m)
        if m == 200:
            k[:] = base(j, kt) + 7   # every row of this batch shares one key
        if m == 1:
            k[:] = base(j, kt)
        tr.insert(be.batch_from_columns(s, key_lanes(k, kt) + [rng.integers(0, 1 << 16, m).astype(np.uint64)], rng.choice([-1, 1, 2], m)))
    dk = delta_keys(rng, mode, nd, kt)
    if hot_rows:   # one key with hot_rows delta rows (spanning tiles), held by every batch but the one-row one
        dk = np.concatenate([dk, np.full(hot_rows, base(len(SIZES) - 2, kt) + 7)])
        extra = [base(j, kt) + 7 for j in range(len(SIZES) - 2)]
        for k in extra:   # the hot key in the older batches too: one more row each, merged into the spine
            tr.insert(be.batch_from_columns(s, key_lanes(np.array([k]), kt) + [np.array([5], np.uint64)], np.array([1])))
    n = len(dk)
    d = be.batch_from_columns(s, key_lanes(dk, kt) + [rng.integers(0, 64, n).astype(np.uint64)], rng.integers(1, 3, n))
    pj = Proj(Schema(kt, "uu"), [key(i) for i in range(len(kt))] + [lval(0), rval(0)], [])
    return be.join_delta_trace(d, tr, pj, left), tr.stats()


@pytest.mark.parametrize("left", [True, False])
@pytest.mark.parametrize("nd", [1, 700, 5000])
@pytest.mark.parametrize("mode", ["newest", "above", "below", "gaps", "mixed"])
@pytest.mark.parametrize("kt", ["u", "i", "uu", "iu"])
def test_probe_windows(cuda, oracle, kt, mode, nd, left):
    got, st = run_join(cuda, kt, mode, nd, left)
    want, _ = run_join(oracle, kt, mode, nd, left)
    assert st[1] >= 3, f"trace has {st[1]} batches"
    if nd > 1:
        assert len(want) > 0
    assert_batches_equal(got, want, f"probe windows kt={kt} mode={mode} nd={nd} left={left}")


@pytest.mark.parametrize("kt", ["u", "i", "uu"])
@pytest.mark.parametrize("hot_rows", [2500, 5000])
def test_probe_key_spans_tiles(cuda, oracle, kt, hot_rows):
    """one key's delta rows cover three or more 1024-row tiles and match rows of several batches"""
    got, _ = run_join(cuda, kt, "gaps", 3000, True, hot_rows)
    want, _ = run_join(oracle, kt, "gaps", 3000, True, hot_rows)
    assert len(want) > hot_rows
    assert_batches_equal(got, want, f"hot key kt={kt} rows={hot_rows}")
