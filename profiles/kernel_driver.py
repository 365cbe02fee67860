"""Driver for the ncu captures of round 2: runs one hot path at a bench-like size so that a single launch of the
kernel of interest can be profiled in isolation, e.g.

    ncu --set full --clock-control none --import-source on -k regex:k_rs_pass -s 2 -c 1 \
        -o gpurun_out/r2_rs_pass python profiles/kernel_driver.py sort

what:  sort   Batch::from_tuples of 4.6 M unsorted 3-lane rows (q4's bids_by_auction shape): k_props, k_pack12,
              k_sample, k_rs_hist_all, k_rs_pass, k_bucket_ids, k_chunk_sort, k_reduce_emit
       sort2  the same with 6-lane rows (two key words, q7's bids_by_price shape)
       join   q4's probe shape: a 300 k-row delta against a 3-batch trace of 30 M rows with keys spread over the whole
              trace: k_probe_ranges, k_probe_fill
       join3  q3's probe shape: a 60 k-row delta whose keys lie past all but the newest of a 10-batch, 4 M-row trace
              (sellers among the newest persons): k_probe_ranges, k_probe_fill
       merge  2 x 20 M-row OrdIndexedZSet<u64,u64,i64> merge: k_merge_partition, k_merge_tiles
       merge1 the same with OrdZSet<u64,i64> rows (one lane + staged weights)
       project  flat_map_index of a 40 M-row table with a 50 % filter, output ordered on arrival: k_project_rows, k_props
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from dbsp_b200 import Proj, Schema, Spine, key, lval, rval  # noqa: E402
from dbsp_b200.runtime import Runtime  # noqa: E402


def join_q4_shape(be, rng):
    """(delta, trace, proj) of the `join` mode"""
    ts, ds = Schema("u", "uu"), Schema("u", "uuu")
    tr = Spine(be, ts)
    for m in (20_000_000, 7_000_000, 3_000_000):
        tr.insert(be.batch_from_columns(ts, [rng.integers(0, 6_000_000, m).astype(np.uint64), rng.integers(0, 1 << 27, m).astype(np.uint64),
                                             rng.integers(0, 1 << 20, m).astype(np.uint64)], np.ones(m, np.int64)))
    nd = 300_000
    d = be.batch_from_columns(ds, [rng.integers(0, 6_000_000, nd).astype(np.uint64), rng.integers(10, 15, nd).astype(np.uint64),
                                   rng.integers(0, 1 << 20, nd).astype(np.uint64), rng.integers(1 << 20, 1 << 21, nd).astype(np.uint64)],
                              np.ones(nd, np.int64))
    proj = Proj(Schema("uu", "u"), [key(0), lval(0), rval(0)], where=[rval(1).ge(lval(1)), rval(1).le(lval(2))])
    return d, tr, proj


def join_q3_shape(be, rng):
    """(delta, trace, proj) of the `join3` mode: q3's auction-by-seller delta against the person-by-id trace"""
    ts, ds = Schema("u", "uuu"), Schema("u", "u")
    tr = Spine(be, ts)
    first = 1000
    for lg in range(21, 11, -1):   # oldest (largest) batch first, ids increasing: one batch per spine level
        m = 1 << lg
        ids = np.arange(first, first + m, dtype=np.uint64)
        first += m
        tr.insert(be.batch_from_columns(ts, [ids, rng.integers(0, 1 << 30, m).astype(np.uint64), rng.integers(0, 1 << 30, m).astype(np.uint64),
                                             rng.integers(1, 4, m).astype(np.uint64)], np.ones(m, np.int64)))
    nd = 60_000
    d = be.batch_from_columns(ds, [(first - 1 - rng.integers(0, 1000, nd)).astype(np.uint64), rng.integers(0, 1 << 32, nd).astype(np.uint64)],
                              np.ones(nd, np.int64))
    proj = Proj(Schema("uuuu"), [rval(0), rval(1), rval(2), lval(0)])
    return d, tr, proj


def main():
    what = sys.argv[1] if len(sys.argv) > 1 else "sort"
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    be = Runtime(0)
    rng = np.random.default_rng(7)
    n = 4_600_000
    if what in ("sort", "sort2"):
        price = np.ceil(np.power(10.0, rng.random(n) * 6.0) * 100.0).astype(np.uint64)
        auction = rng.integers(1000, 300_000, n).astype(np.uint64)
        dt = np.uint64(1436918400000) + rng.integers(0, 5000, n).astype(np.uint64)
        if what == "sort":
            s, cols = Schema("u", "uu"), [auction, price, dt]
        else:
            s, cols = Schema("u", "uuuuu"), [price, auction, rng.integers(1000, 100_000, n).astype(np.uint64), price, dt,
                                             rng.integers(0, 1 << 32, n).astype(np.uint64)]
        for _ in range(reps):
            b = be.batch_from_columns(s, cols, np.ones(n, np.int64))
        be.sync()
        print(what, len(b))
    elif what in ("join", "join3"):
        d, tr, proj = (join_q4_shape if what == "join" else join_q3_shape)(be, rng)
        for _ in range(reps):
            o = be.join_delta_trace(d, tr, proj, delta_is_left=True)
        be.sync()
        print(what, len(o), tr.stats())
    elif what in ("merge", "merge1"):
        import bench

        print(bench.merge_sweep(0, rows=20_000_000, n_val_lanes=1 if what == "merge" else 0, reps=reps))
    elif what == "project":
        from dbsp_b200 import col

        m = 40_000_000   # bid-table shape: (auction, bidder, price, date_time), filter on price, key by auction
        cols = [rng.integers(1000, 300_000, m).astype(np.uint64), rng.integers(1000, 100_000, m).astype(np.uint64),
                rng.integers(0, 1 << 24, m).astype(np.uint64), np.arange(m, dtype=np.uint64)]
        proj = Proj(Schema("u", "uu"), [col(3), col(0), col(2)], where=[col(2).lt(1 << 23)])
        for _ in range(reps):
            b = be.batch_from_table(cols, proj)
        be.sync()
        print(what, len(b))
    else:
        raise SystemExit("unknown " + what)


if __name__ == "__main__":
    main()
