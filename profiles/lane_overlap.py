"""Overlap of the two execution lanes on q3, from a torch.profiler trace with CUDA activities.

    python profiles/lane_overlap.py [--events 5000000] [--warmup 5] [--steps 4] [--out lane_overlap.json]

Runs q3 on device-resident Nexmark tables like bench.py (its own run: tracing slows the host, so its times are not
bench numbers) and records `--steps` circuit steps, each followed by a device synchronise.  Per step it reports the
kernel intervals on each stream, the union of each stream's busy time, the time both streams run kernels at once,
and the main lane's critical path (first kernel start to last kernel end on lane 0, the stream bench.py times).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def union(iv):
    """Merge [start, end) intervals; returns the merged list."""
    out = []
    for a, b in sorted(iv):
        if out and a <= out[-1][1]:
            out[-1][1] = max(out[-1][1], b)
        else:
            out.append([a, b])
    return out


def intersect_len(x, y):
    i = j = 0
    t = 0.0
    while i < len(x) and j < len(y):
        a, b = max(x[i][0], y[j][0]), min(x[i][1], y[j][1])
        if b > a:
            t += b - a
        if x[i][1] < y[j][1]:
            i += 1
        else:
            j += 1
    return t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--events", type=int, default=5_000_000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--out", default="lane_overlap.json")
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile, record_function

    import dbsp_b200  # noqa: F401
    from dbsp_b200.nexmark import NexmarkGenerator
    from dbsp_b200.runtime import Runtime
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from parity_util import build_query

    os.environ.setdefault("DBSP_POOL_RESERVE_GB", "24")
    dev = torch.device("cuda", 0)
    be = Runtime(0)
    lane0 = be.stream_ptr
    gen = NexmarkGenerator()
    E = args.events
    n_total = args.warmup + args.steps
    tables = []
    for s in range(n_total):
        t = gen.tables(s * E, E)
        tables.append({k: [torch.from_numpy(c.view(np.int64)).to(dev) for c in t[k]] for k in ("person", "auction")})
    torch.cuda.synchronize()
    c, handles, out = build_query(be, "q3")
    empty = [np.empty(0, np.uint64)] * 5

    def feed(d):
        for k in ("person", "auction"):
            handles[k].set_device([int(x.data_ptr()) for x in d[k]], int(d[k][0].numel()))
        handles["bid"].set(empty)

    for s in range(args.warmup):
        feed(tables[s])
        c.step()
    be.sync()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for s in range(args.warmup, n_total):
            feed(tables[s])
            with record_function(f"circuit_step_{s - args.warmup}"):
                c.step()
                be.sync()
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "trace.json")
        prof.export_chrome_trace(path)
        trace = json.load(open(path))
    evs = trace["traceEvents"] if isinstance(trace, dict) else trace
    windows = sorted((e["ts"], e["ts"] + e["dur"], e["name"]) for e in evs
                     if e.get("ph") == "X" and str(e.get("name", "")).startswith("circuit_step_") and e.get("cat") == "user_annotation")
    kernels = [e for e in evs if e.get("ph") == "X" and e.get("cat") == "kernel"]
    streams = sorted({k["args"].get("stream") for k in kernels})
    # lane 0 is the stream of the context (its handle is the cudaStream_t; the trace names streams by id): take the
    # stream that ran the most kernels over the window as lane 0 and the other library stream as lane 1
    per_stream = {s: sum(1 for k in kernels if k["args"].get("stream") == s) for s in streams}
    ranked = sorted(streams, key=lambda s: -per_stream[s])
    res = {"card": torch.cuda.get_device_name(0), "events_per_circuit_step": E, "streams": per_stream,
           "lane0_stream": ranked[0] if ranked else None, "lane1_stream": ranked[1] if len(ranked) > 1 else None,
           "lane0_handle": hex(lane0 or 0), "steps": []}
    for a, b, name in windows:
        ks = [k for k in kernels if a <= k["ts"] < b]
        by = {}
        for k in ks:
            by.setdefault(k["args"].get("stream"), []).append((k["ts"], k["ts"] + k["dur"], k["name"]))
        l0 = by.get(res["lane0_stream"], [])
        l1 = by.get(res["lane1_stream"], [])
        u0, u1 = union([(x, y) for x, y, _ in l0]), union([(x, y) for x, y, _ in l1])
        step = {
            "step": name,
            "lane0_kernels": len(l0), "lane1_kernels": len(l1),
            "lane0_busy_us": sum(y - x for x, y in u0), "lane1_busy_us": sum(y - x for x, y in u1),
            "overlap_us": intersect_len(u0, u1),
            "lane0_critical_path_us": (max(y for _, y, _ in l0) - min(x for x, _, _ in l0)) if l0 else 0.0,
            "lane1_span_us": (max(y for _, y, _ in l1) - min(x for x, _, _ in l1)) if l1 else 0.0,
            "lane0_intervals": [[round(x - a, 1), round(y - a, 1), n[:48]] for x, y, n in sorted(l0)],
            "lane1_intervals": [[round(x - a, 1), round(y - a, 1), n[:48]] for x, y, n in sorted(l1)],
        }
        res["steps"].append(step)
        print(f"{name}: lane0 {step['lane0_kernels']} kernels busy {step['lane0_busy_us']:.1f} us, critical path "
              f"{step['lane0_critical_path_us']:.1f} us; lane1 {step['lane1_kernels']} kernels busy "
              f"{step['lane1_busy_us']:.1f} us; overlapped {step['overlap_us']:.1f} us")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
