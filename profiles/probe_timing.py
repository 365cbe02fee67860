"""Device time of one join probe (join_delta_trace) per kernel class, at q3's and q4's shapes, from the library's
per-kernel CUDA events over many repetitions; and the batch count of q3's two join traces at the bench's size.

    python profiles/probe_timing.py [reps] [q3 bench steps]

Prints one JSON line: per shape, µs per probe for each kernel class (`probe_ranges`, `probe_fill`, and the
consolidation behind the fill) and the wall time per probe (host clock over `reps` probes ending in a synchronise,
read-backs included); then, for q3 run as bench.py runs it (5 M events per circuit step, default 25 bench steps),
the rows and batches (Spine.stats()) of the trace each probe of the last circuit step searched.
"""
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from kernel_driver import join_q3_shape, join_q4_shape  # noqa: E402

from dbsp_b200.runtime import Runtime  # noqa: E402


def time_probe(be, d, tr, proj, reps):
    for _ in range(5):
        o = be.join_delta_trace(d, tr, proj, delta_is_left=True)
    be.sync()
    t0 = time.perf_counter()
    for _ in range(reps):
        o = be.join_delta_trace(d, tr, proj, delta_is_left=True)
    be.sync()
    wall = (time.perf_counter() - t0) / reps
    be.profile(True)
    for _ in range(reps):
        o = be.join_delta_trace(d, tr, proj, delta_is_left=True)
    be.sync()
    prof = be.profile_read()
    be.profile(False)
    return {"delta_rows": len(d), "trace": tr.stats(), "out_rows": len(o), "wall_us_per_probe": round(wall * 1e6, 1),
            "us_per_probe": {k: round(v["ms"] * 1e3 / reps, 2) for k, v in sorted(prof.items())},
            "launches_per_probe": {k: v["launches"] / reps for k, v in sorted(prof.items())}}


def q3_trace_stats(be, bench_steps):
    """(delta rows, trace rows, trace batches) of each probe of q3's last circuit step, fed as bench.py feeds it"""
    import bench
    import dbsp_b200
    from dbsp_b200.nexmark import queries as nq

    S = bench.CIRCUIT_STEPS["q3"]
    seen = []
    join = be.join_delta_trace

    def recording(delta, trace, proj, delta_is_left=True):
        n, nb = trace.stats()
        seen.append({"delta_is_left": delta_is_left, "delta_rows": len(delta), "trace_rows": n, "trace_batches": nb})
        return join(delta, trace, proj, delta_is_left)

    be.join_delta_trace = recording
    c = dbsp_b200.RootCircuit(be, None)
    inp, handles = nq.add_nexmark_input(c)
    nq.QUERIES["q3"](inp).output()
    for t in bench.gen_steps("q3", 0, 1, bench_steps * S, 5_000_000, pinned=False):
        for k in ("person", "auction", "bid"):
            handles[k].set(t[k] if t[k] is not None else bench.empty_cols())
        c.step()
    be.sync()
    be.join_delta_trace = join
    return {"circuit_steps": bench_steps * S, "last_step_probes": seen[-2:],
            "max_trace_batches": max(x["trace_batches"] for x in seen)}


def main():
    reps = int(sys.argv[1]) if len(sys.argv) > 1 else 200
    bench_steps = int(sys.argv[2]) if len(sys.argv) > 2 else 25
    be = Runtime(0)
    res = {}
    for name, shape in (("q3", join_q3_shape), ("q4", join_q4_shape)):
        d, tr, proj = shape(be, np.random.default_rng(7))
        res[name] = time_probe(be, d, tr, proj, reps if name == "q3" else max(1, reps // 10))
        del d, tr
    res["q3_bench_traces"] = q3_trace_stats(Runtime(0), bench_steps)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
