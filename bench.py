#!/usr/bin/env python
"""bench.py — Nexmark events/s through the B200 Z-set hot path.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--query q3|q4|q7] [--dump-outputs DIR]

Workload.  A *circuit step* is one `Circuit::step()` of the query over E = 5 M synthetic Nexmark events per
GPU.  A *bench step* (what --steps / --warmup count) is S consecutive circuit steps (S per query below), so that
the timed region of the driver's `--steps 20` is hundreds of circuit steps instead of 20 sub-millisecond ones.
The primary line at N=1 is BASELINE.json configs[1]: Nexmark q3 (person |x| auction incremental join); q4, q7 and
the config[4] merge sweep ride along under `queries` / `merge_sweep` unless --query pins one query.

`value`    : events/s, the step's input columns already resident in HBM (device-timed, CUDA events on the library's
             stream, max over ranks).  `rows_per_s` next to it counts only the table rows the query ingests (q3 reads
             the 8 % of events that are persons/auctions).
`e2e`      : the same steps through the C ABI with HOST (pinned) columns: the H2D copy of every step's inputs and
             the D2H download of every step's output Z-set are inside the timed region.
`roofline` : the dominant kernel class of the timed region: algorithmic bytes / device time from CUDA events the
             library records on its own stream (dbsp_ctx_profile), against MEASURED_PEAKS.json; `traffic` from the
             committed ncu --set full capture of that kernel (profiles/r2_ncu_traffic.json), scaled by bytes.
`--impl reference` / `cpu_baseline`: the CPU arm = oracle/nexmark_workers.cpp — the C++ restatement of the
             reference's algorithms run as N worker threads with hash-shard + in-process exchange and no interpreter
             between steps (the Rust reference cannot be built here: no rustc), rebuilt with -march=native on the box
             it is timed on.  `--impl reference` runs the SAME circuit steps as the GPU arm (same E, same S, same
             K and W); the in-line `cpu_baseline` of a default run is a bounded sample (fewer steps, stated).
`--dump-outputs DIR`: after the timed steps, the primary query's output Z-set of the last timed circuit step goes to
             DIR as float64 .npy files (see dump_outputs), so that two builds run with the same arguments (hence the
             same seeded inputs) can be compared output for output.

bench.py writes nothing into the source tree (which may be read-only): the CPU arm's -march=native build goes to a
temporary directory and no bytecode is cached.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
DUMP_LIMIT_BYTES = 64 << 20

METRIC = "nexmark_events_per_sec"
UNIT = "events/s"
QUERY_COLS = {   # tables each query reads (the others are not generated / copied)
    "q3": ("person", "auction"),
    "q4": ("auction", "bid"),
    "q7": ("bid",),
    "q0": ("bid",),
}
FULL_EVENTS = {"q3": 100_000_000, "q4": 100_000_000, "q7": 1_000_000_000}
# circuit steps per bench step
CIRCUIT_STEPS = {"q3": 8, "q4": 2, "q7": 2}
# NexmarkConfig::first_event_rate (crates/nexmark/src/config.rs:51,134).  q3/q4 never look at event time.  q7's 10 s
# tumbling windows (q7.rs:43) hold 100 M events at the reference default of 10 M events/s: none would close before
# event 140 M.  At 1 M events/s a window closes every second circuit step, so the run does the same work per event
# as configs[3] (1 B events at the default rate: every bid enters one window and leaves it once), ten windows deep.
EVENT_RATE = {"q3": 0, "q4": 0, "q7": 1_000_000}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (NVML, ~2 ms period)."""

    HW_SLOWDOWN, SW_THERMAL, HW_THERMAL, SW_POWER_CAP = 0x8, 0x20, 0x40, 0x4

    def __init__(self, gpu_index=0):
        self.idx, self.rows, self.stop, self.t = gpu_index, [], False, None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            # CUDA_VISIBLE_DEVICES may remap indices: NVML enumerates physical devices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[gpu_index]) if vis and vis.split(",")[gpu_index].isdigit() else gpu_index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        while not self.stop:
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((sm, rs))
            except Exception:
                pass
            time.sleep(0.002)

    def __enter__(self):
        if self.nv is not None:
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()
        return self

    def __exit__(self, *a):
        self.stop = True
        if self.t is not None:
            self.t.join(timeout=1)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = [r[0] for r in self.rows]
        bits = 0
        for r in self.rows:
            bits |= r[1]
        names = [("hw_slowdown", self.HW_SLOWDOWN), ("hw_thermal_slowdown", self.HW_THERMAL),
                 ("sw_thermal_slowdown", self.SW_THERMAL), ("sw_power_cap", self.SW_POWER_CAP)]
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(self.max_sm), "reasons": [n for n, b in names if bits & b],
                "samples": len(sm)}


def gen_steps(query, rank, world, n_steps, events_per_step, pinned, rate=None):
    """Host column tables of n_steps circuit steps for this rank.  Rank r's step s is the contiguous event range
    [(s*world + r) * E, +E) (round-robin input distribution at batch granularity, operator/input.rs:664-703)."""
    from dbsp_b200.nexmark import NexmarkGenerator

    gen = NexmarkGenerator(threads=max(1, (os.cpu_count() or 8) // max(world, 1)),
                           first_event_rate=EVENT_RATE[query] if rate is None else rate)
    want = QUERY_COLS[query]
    if pinned:
        import torch

        def alloc(k):
            return torch.empty(k, dtype=torch.int64).pin_memory().numpy().view(np.uint64)
    else:
        alloc = None
    return [gen.tables((s * world + rank) * events_per_step, events_per_step, want=want, alloc=alloc) for s in range(n_steps)]


def rows_in(steps, lo, hi):
    return sum(len(t[k][0]) for t in steps[lo:hi] for k in t if t[k] is not None)


def empty_cols():
    return [np.empty(0, np.uint64) for _ in range(5)]


def make_comm(device, be=None):
    from dbsp_b200.parallel import Comm

    return Comm(device)


def workload_cfg(query, E, S, W, K, world):
    total = world * E * S * (W + K)
    cfg = {"workload": f"Nexmark {query}: {E} events per circuit step per GPU, {S} circuit steps per bench step, "
                       f"{K} timed + {W} warm-up bench steps = {total} events over {world} GPU(s); "
                       f"BASELINE configs full size {FULL_EVENTS.get(query)}",
           "query": query, "events_per_circuit_step_per_gpu": E, "circuit_steps_per_bench_step": S,
           "timed_circuit_steps": K * S, "total_events": total,
           "first_event_rate": EVENT_RATE[query] or 10_000_000,
           "l2": "inputs larger than L2 (every circuit step streams fresh event columns); traces grow past L2",
           "parallelism": f"key-hash shard x{world}" if world > 1 else "single GPU"}
    return cfg


def flat_rows(batch):
    """A batch's rows as flat uint64 lanes (keys, then values) and int64 weights, in the batch's canonical order."""
    d = batch.download()
    lanes = [np.asarray(k).view(np.uint64) for k in d["keys"]]
    if d["offs"] is not None:
        counts = np.diff(d["offs"].astype(np.int64))
        lanes = [np.repeat(k, counts) for k in lanes] + [np.asarray(v).view(np.uint64) for v in d["vals"]]
    return lanes, d["diffs"]


def dump_outputs(out_dir, prefix, lanes, weights, limit_bytes):
    """Writes one output Z-set as float64 .npy files: every uint64 lane as its two 32-bit halves
    (`<prefix>lane<i>_hi`, `<prefix>lane<i>_lo`; float64 holds them exactly) and `<prefix>weight`.  An output larger
    than `limit_bytes` is cut to a fixed, seeded sample of rows whose indices go to `<prefix>row_index`."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {}
    row_bytes = 8 * (2 * len(lanes) + 2)
    if len(weights) * row_bytes > limit_bytes:
        idx = np.sort(np.random.default_rng(0).choice(len(weights), limit_bytes // row_bytes, replace=False))
        lanes, weights = [c[idx] for c in lanes], weights[idx]
        arrays["row_index"] = idx
    for i, c in enumerate(lanes):
        arrays[f"lane{i}_hi"] = c >> np.uint64(32)
        arrays[f"lane{i}_lo"] = c & np.uint64(0xFFFFFFFF)
    arrays["weight"] = weights
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{prefix}{name}.npy"), a.astype(np.float64))


def run_b200(args, query, rank, world, comm, device, do_e2e=True, keep_output=False):
    """Returns dict with value / e2e / profile for `query` on this rank; with keep_output, also `output`: the flat
    rows of the last timed circuit step's output Z-set."""
    import torch

    import dbsp_b200
    from dbsp_b200.nexmark import queries as nq
    from dbsp_b200.runtime import Runtime

    E, S = args.events_per_step, args.circuit_steps or CIRCUIT_STEPS[query]
    W, K = args.warmup * S, args.steps * S          # in circuit steps
    steps = gen_steps(query, rank, world, W + K, E, pinned=True)
    res = {"circuit_steps_per_bench_step": S}

    def build(be):
        c = dbsp_b200.RootCircuit(be, comm)
        inp, handles = nq.add_nexmark_input(c)
        out = nq.QUERIES[query](inp).output()
        build.tables = inp
        return c, handles, out

    def sync_all(be):
        be.sync()
        if comm is not None:
            torch.cuda.synchronize(device)
            comm.barrier()

    def max_over_ranks(x):
        if comm is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=device)
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        return float(t.item())

    # ---- (1) device-resident inputs -------------------------------------------
    os.environ.setdefault("DBSP_POOL_RESERVE_GB", "24")   # pool growth (cudaMalloc of slabs) stays out of the timed region
    be = Runtime(device.index)
    if comm is not None and hasattr(comm, "attach"):
        comm.attach(be)
    ext = torch.cuda.ExternalStream(be.stream_ptr, device=device)
    dev_steps = []
    for t in steps:
        d = {}
        for k, cols in t.items():
            d[k] = None if cols is None else [torch.from_numpy(c.view(np.int64)).to(device, non_blocking=True) for c in cols]
        dev_steps.append(d)
    torch.cuda.synchronize(device)
    c, handles, out = build(be)

    def feed_dev(d):
        for k in ("person", "auction", "bid"):
            if d[k] is None:
                handles[k].set(empty_cols())
            else:
                handles[k].set_device([int(x.data_ptr()) for x in d[k]], int(d[k][0].numel()))

    for s in range(W):
        feed_dev(dev_steps[s])
        c.step()
    sync_all(be)
    be.stats(reset=True)
    # per-kernel CUDA events (two per kernel class scope) cost host time on a launch-bound step (q3: 0.61 ms with
    # them on every step, 0.48 ms without): they are recorded over the last quarter of the timed region (whole bench
    # steps, at least one; the traces are at their largest there), live, inside the timed region
    prof_steps = min(K, max(S, (K // 4) // S * S))
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    with ClockSampler(device.index) as clk:
        t0 = time.perf_counter()
        evs[0].record(ext)
        for s in range(W, W + K):
            if s - W == K - prof_steps:
                be.profile(True)     # the per-kernel events are a sampling window: the steps before it run without them
            feed_dev(dev_steps[s])
            c.step()
            evs[s - W + 1].record(ext)
        sync_all(be)
        wall = time.perf_counter() - t0
    dev_ms = evs[0].elapsed_time(evs[K])
    per_step = sorted(evs[i].elapsed_time(evs[i + 1]) for i in range(K))
    ms = max_over_ranks(dev_ms)
    st = be.stats()
    prof = be.profile_read()
    be.profile(False)
    out_rows = len(out.value)
    if keep_output:
        res["output"] = flat_rows(out.value)
    in_rows = rows_in(steps, W, W + K)
    res.update(value=world * E * K / (ms / 1e3), rows_per_s=world * in_rows / (ms / 1e3), ms_per_step=ms / args.steps,
               ms_per_circuit_step=ms / K, wall_ms_per_circuit_step=wall * 1e3 / K,
               circuit_step_ms_p50=per_step[K // 2], circuit_step_ms_p99=per_step[min(K - 1, int(K * 0.99))],
               circuit_step_ms_max=per_step[-1], timed_region_ms=ms,
               gpu_launches=st["kernel_launches"], profile=prof, clocks=clk.summary(), last_step_out_rows=out_rows,
               profile_window_circuit_steps=min(prof_steps, K),
               launches_per_circuit_step=st["kernel_launches"] / K,
               host_readbacks_per_circuit_step=st["host_waits"] / K,      # counts the device publishes to the host mailbox
               host_wait_ms_per_circuit_step=st["host_wait_ms"] / K)      # time the host spent waiting for them
    del c, handles, out, dev_steps
    be.sync()

    # ---- (2) end to end: host columns in, output Z-set out -----------------------------
    if do_e2e:
        c, handles, out = build(be)
        tabs = {"person": build.tables.person, "auction": build.tables.auction, "bid": build.tables.bid}
        masks = {k: tabs[k].table_mask() for k in tabs}

        def start_uploads(t):
            """H2D of one step's tables on the copy stream (only the columns the query reads)."""
            return {k: (be.upload_begin(t[k], masks[k]) if (t[k] is not None and masks[k]) else None) for k in tabs}

        def feed_uploads(ups):
            for k in tabs:
                if ups[k] is None:
                    handles[k].set(empty_cols())
                else:
                    handles[k].set_upload(ups[k])

        # D2H of a step's output Z-set: flat lanes + weights into pinned host columns on the copy stream, drained
        # while the next step runs (two buffer sets); the last one is drained inside the timed region
        import torch as _t
        host_out = [None, None]

        def start_download(slot):
            b = out.value
            n, nl = len(b), b.schema.nk + b.schema.nv
            if host_out[slot] is None or len(host_out[slot][0]) < n:
                cap = max(2 * n, 1 << 16)
                host_out[slot] = [_t.empty(cap, dtype=_t.int64).pin_memory().numpy() for _ in range(nl + 1)]
            hb = host_out[slot]
            return be.download_begin(b, [x.view(np.uint64) for x in hb[:nl]], hb[nl])

        for s in range(W):
            feed_uploads(start_uploads(steps[s]))
            c.step()
            start_download(s & 1).finish()
        sync_all(be)
        be.stats(reset=True)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(ext)
        pending = None
        nxt = start_uploads(steps[W])             # every step's H2D copy is inside the timed region ...
        for s in range(W, W + K):
            cur = nxt
            nxt = start_uploads(steps[s + 1]) if s + 1 < W + K else None   # ... and overlaps the previous step's kernels
            feed_uploads(cur)
            c.step()
            dl = start_download(s & 1)            # D2H of the step's result Z-set ...
            if pending is not None:
                pending.finish()                  # ... read by the host while the next step runs
            pending = dl
        pending.finish()
        e1.record(ext)
        sync_all(be)
        wall2 = time.perf_counter() - t0
        ms2 = max_over_ranks(max(e0.elapsed_time(e1), wall2 * 1e3))   # host copies are part of the path: take the larger clock
        st2 = be.stats()
        res["e2e"] = {"value": world * E * K / (ms2 / 1e3), "unit": UNIT, "h2d_bytes_per_step": st2["h2d_bytes"] // args.steps,
                      "d2h_bytes_per_step": st2["d2h_bytes"] // args.steps, "ms_per_step": ms2 / args.steps,
                      "ms_per_circuit_step": ms2 / K}
        del c, handles, out
    be.sync()
    import gc

    if comm is not None:
        res["nvlink_bytes_sent"] = getattr(comm, "bytes_sent", None)
        if hasattr(comm, "detach"):
            comm.detach()
    gc.collect()
    be.close()
    return res


def parity_check(rank, world, comm, device, queries=("q3", "q4", "q7"), events=100_000, n_steps=5):
    """N > 1 only, outside every timed region: the sharded circuit's output, gathered to rank 0, must equal —
    bit for bit, every step — the output of a single-GPU circuit fed the union of all ranks' inputs.  The driver's
    1-GPU test box cannot run tests/test_multigpu.py, so the multi-GPU CUDA path is verified here."""
    import torch

    import dbsp_b200
    from dbsp_b200.nexmark import queries as nq
    from dbsp_b200.runtime import Runtime

    be = Runtime(device.index)
    if hasattr(comm, "attach"):
        comm.attach(be)
    report = {"steps": n_steps, "events_per_step_per_gpu": events, "queries": {}}
    ok_all = True
    try:
        for q in queries:
            rate = 20_000 if q == "q7" else 0             # q7: 10 s of event time = 200 k events: windows close from step 2 on
            mine = gen_steps(q, rank, world, n_steps, events, pinned=False, rate=rate)
            c = dbsp_b200.RootCircuit(be, comm)
            inp, handles = nq.add_nexmark_input(c)
            out = nq.QUERIES[q](inp).gather(0).output()
            if rank == 0:
                c1 = dbsp_b200.RootCircuit(be, None)
                inp1, handles1 = nq.add_nexmark_input(c1)
                out1 = nq.QUERIES[q](inp1).output()
                union = gen_steps(q, 0, 1, n_steps, events * world, pinned=False, rate=rate)
            ok, rows = True, 0
            for s in range(n_steps):
                for k in ("person", "auction", "bid"):
                    handles[k].set(mine[s][k] if mine[s][k] is not None else empty_cols())
                c.step()
                if rank == 0:
                    for k in ("person", "auction", "bid"):
                        handles1[k].set(union[s][k] if union[s][k] is not None else empty_cols())
                    c1.step()
                    a, b = out.value.download(), out1.value.download()
                    same = len(a["diffs"]) == len(b["diffs"]) and np.array_equal(a["diffs"], b["diffs"])
                    same = same and all(np.array_equal(x, y) for x, y in zip(a["keys"], b["keys"]))
                    same = same and all(np.array_equal(x, y) for x, y in zip(a["vals"], b["vals"]))
                    if a["offs"] is not None:
                        same = same and np.array_equal(a["offs"], b["offs"])
                    ok = ok and bool(same)
                    rows += len(b["diffs"])
            t = torch.tensor([1 if ok else 0, rows], dtype=torch.int64, device=device)
            torch.distributed.broadcast(t, 0)
            ok, rows = bool(t[0].item()), int(t[1].item())
            report["queries"][q] = {"equal_every_step": ok, "output_rows_compared": rows}
            ok_all = ok_all and ok and (rows > 0)
            del c, handles, out
            if rank == 0:
                del c1, handles1, out1
    finally:
        be.sync()
        if hasattr(comm, "detach"):
            comm.detach()
        import gc

        gc.collect()
        be.close()
    report["ok"] = ok_all
    return report


ROOFLINE_NOTES = {
    "q3": "q3 reads only Person/Auction events (8% of the stream): a 5M-event circuit step is ~60k-row batches, so its "
          "kernels are launch-latency bound and sit far below the HBM roofline; see queries.q4.roofline, "
          "queries.q7.roofline and merge_sweep[*].roofline for the bandwidth-bound kernels",
}


def ncu_traffic(kernel, alg_bytes_per_launch):
    """dram bytes per launch of `kernel` from the committed ncu --set full capture, scaled by algorithmic bytes."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")))[kernel]
        return t["dram_bytes"] * alg_bytes_per_launch / t["alg_bytes"], t["source"]
    except Exception:
        return None, None


def roofline_from_profile(prof, query=None):
    peak, how = peaks()
    if not prof:
        return None
    name = max(prof, key=lambda k: prof[k]["ms"])
    p = prof[name]
    total_ms = sum(v["ms"] for v in prof.values())
    achieved = p["alg_bytes"] / (p["ms"] / 1e3) / 1e9 if p["ms"] > 0 else 0.0
    traffic, src = ncu_traffic(name, p["alg_bytes"] / p["launches"])
    return {"bound": "hbm", "kernel": name, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": traffic, "traffic_source": src, "launches": p["launches"], "avg_launch_us": 1e3 * p["ms"] / p["launches"],
            "alg_bytes_per_launch": p["alg_bytes"] / p["launches"], "share_of_kernel_time": p["ms"] / total_ms if total_ms else None,
            "peak_source": how, **({"note": ROOFLINE_NOTES[query]} if query in ROOFLINE_NOTES else {})}


def kernel_table(prof):
    peak, _ = peaks()
    return {k: {"launches": v["launches"], "ms": round(v["ms"], 3), "alg_GB": round(v["alg_bytes"] / 1e9, 4),
                "frac_of_hbm_peak": round(v["alg_bytes"] / (v["ms"] / 1e3) / 1e9 / peak, 4) if v["ms"] > 0 else None}
            for k, v in prof.items()}


def merge_sweep(device_index, rows=50_000_000, n_val_lanes=1, reps=5):
    """BASELINE.json configs[4]: merge of two consolidated batches of `rows` rows each — OrdIndexedZSet<u64,u64,i64>
    (n_val_lanes=1) or OrdZSet<u64,i64> (n_val_lanes=0) — Zipf(1) keys; algorithmic GB/s of the merge kernel
    (every input row read once, every output row written once) vs the HBM peak."""
    import torch

    from dbsp_b200 import Schema
    from dbsp_b200.runtime import Runtime

    be = Runtime(device_index)
    dev = torch.device("cuda", device_index)
    g = torch.Generator(device=dev)
    g.manual_seed(0x7FC359184519C0AA & 0x7FFFFFFF)
    s = Schema("u", "u" * n_val_lanes)
    batches = []
    for _ in range(2):
        # Zipf(s=1) keys over a domain of rows/4: inverse-CDF of a log-uniform draw
        u = torch.rand(rows, generator=g, device=dev, dtype=torch.float64)
        dom = max(rows // 4, 2)
        keys = torch.exp(u * np.log(dom)).to(torch.int64).clamp_(1, dom)
        del u
        if n_val_lanes == 0:   # OrdZSet<u64>: spread the Zipf keys so that consolidation keeps most rows
            keys = keys * 1024 + torch.randint(0, 1024, (rows,), generator=g, device=dev, dtype=torch.int64)
        vals = [torch.randint(0, 1 << 40, (rows,), generator=g, device=dev, dtype=torch.int64) for _ in range(n_val_lanes)]
        w = torch.randint(0, 4, (rows,), generator=g, device=dev, dtype=torch.int64)
        w = torch.where(w >= 2, w - 1, w - 2)   # {-2,-1,1,2}
        torch.cuda.synchronize(dev)
        batches.append(be.batch_from_columns(s, [int(keys.data_ptr())] + [int(v.data_ptr()) for v in vals], int(w.data_ptr()), n=rows, on_device=True))
        be.sync()
        del keys, vals, w
        torch.cuda.empty_cache()
    a, b = batches
    for _ in range(2):
        be.merge(a, b)
    be.profile(True)
    for _ in range(reps):
        m = be.merge(a, b)
    prof = be.profile_read()
    be.profile(False)
    peak, how = peaks()
    p = prof["merge_tiles"]
    ach = p["alg_bytes"] / (p["ms"] / 1e3) / 1e9
    traffic, src = ncu_traffic("merge_tiles", p["alg_bytes"] / p["launches"])
    ty = "OrdZSet<u64,i64>" if n_val_lanes == 0 else f"OrdIndexedZSet<u64,{'(' + ','.join(['u64'] * n_val_lanes) + ')' if n_val_lanes > 1 else 'u64'},i64>"
    res = {"workload": f"merge 2 x {ty}, {len(a)}+{len(b)} rows -> {len(m)}", "rows_per_s": (len(a) + len(b)) / (p["ms"] / reps / 1e3),
           "roofline": {"bound": "hbm", "kernel": "merge_tiles", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                        "traffic": traffic, "traffic_source": src,
                        "alg_bytes_per_launch": p["alg_bytes"] / p["launches"], "avg_launch_us": 1e3 * p["ms"] / p["launches"], "peak_source": how},
           "inputs_larger_than_l2": (len(a) + len(b)) * 8 * (2 + n_val_lanes) > 126e6,
           "consolidate_kernels": {k: v for k, v in kernel_table(prof).items() if k != "merge_tiles"}}
    del a, b, m, batches
    be.sync()
    be.close()
    return res


def run_reference(args, query, bench_steps=None, warmup=None, n_workers=None, gpus=1):
    """The CPU arm: the oracle port as native C++ worker threads (oracle/nexmark_workers.cpp), rebuilt with
    -march=native on this host.  Runs the same circuit steps (same E and S) as the GPU arm; `bench_steps` / `warmup`
    bound the number of bench steps (the in-line cpu_baseline is a bounded sample)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import native_workers as nw

    T = n_workers or min(os.cpu_count() or 1, args.cpu_threads)
    E, S = args.events_per_step * gpus, args.circuit_steps or CIRCUIT_STEPS[query]
    Kb = args.steps if bench_steps is None else bench_steps
    Wb = args.warmup if warmup is None else warmup
    # bounded sample: the whole CPU run stays below ~2.4 G generated events (minutes, a few GB of host columns) by
    # running fewer circuit steps per bench step — the circuit step itself (E events) is never shrunk
    S_full = S
    S = max(1, min(S, 2_400_000_000 // max(1, (Wb + Kb) * E)))
    W, K = Wb * S, Kb * S
    steps = gen_steps(query, 0, 1, W + K, E, pinned=False)
    secs, rows, fps, how = nw.run(query, T, steps, native=True)
    timed = float(sum(secs[W:]))
    in_rows = rows_in(steps, W, W + K)
    return {"value": E * K / timed, "rows_per_s": in_rows / timed, "cores": T, "kind": "port", "ms_per_step": 1e3 * timed / Kb,
            "bench_steps": Kb, "warmup": Wb, "build": how, "last_step_out_rows": rows[-1],
            "circuit_steps_per_bench_step": S, "circuit_steps_per_bench_step_full": S_full, "timed_events": E * K,
            "sample": f"{query}: {Wb}+{Kb} bench steps x {S} circuit steps{'' if S == S_full else f' (of {S_full}: bounded sample)'} of {E} events on {T} native oracle worker threads "
                      f"(C++ port of the reference's algorithms, hash-shard + in-process exchange, {how})"}


def main():
    sys.dont_write_bytecode = True   # no __pycache__ of the in-tree modules the runs import
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--query", default=None, help="q3 | q4 | q7 (default: q3 primary + q4, q7 riding along)")
    ap.add_argument("--events-per-step", type=int, default=5_000_000, help="events per circuit step per GPU")
    ap.add_argument("--circuit-steps", type=int, default=0, help="circuit steps per bench step (0 = per-query default)")
    ap.add_argument("--cpu-threads", type=int, default=16)
    ap.add_argument("--no-extras", action="store_true", help="skip q4/q7, the merge sweep and the in-line cpu_baseline")
    ap.add_argument("--sweep-rows", default="10000000,100000000,1000000000", help="config[4] total rows per merge")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the primary query's output of the last timed circuit step to DIR as .npy files")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs the GPU arm: the CPU arm returns only a fingerprint per step")
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    primary = args.query or "q3"
    E, W, K = args.events_per_step, args.warmup, args.steps
    S = args.circuit_steps or CIRCUIT_STEPS[primary]

    if args.impl == "reference":
        if rank != 0:
            return
        # same workload as the GPU arm at --gpus N: N x E events per circuit step, all on this host's cores
        r = run_reference(args, primary, gpus=max(args.gpus, 1))
        cfg = workload_cfg(primary, E, S, W, K, max(args.gpus, 1))
        if r["circuit_steps_per_bench_step"] != r["circuit_steps_per_bench_step_full"]:
            # same circuit steps (events per step, query, generator) as the GPU arm, fewer of them per bench step
            cfg["reference_sample"] = {"circuit_steps_per_bench_step_run": r["circuit_steps_per_bench_step"],
                                       "timed_circuit_steps_run": r["circuit_steps_per_bench_step"] * K,
                                       "timed_events_run": r["timed_events"]}
        line = {"impl_note": f"CPU arm: every circuit step's {max(args.gpus, 1) * E} events on one host, {r['cores']} worker threads; the Rust "
                             "reference cannot be built here (no rustc): this is the C++ port under oracle/ (kind: port)",
                "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
                "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64",
                "data": "synthetic", "impl": "reference", "config": cfg, "rows_per_s": r["rows_per_s"],
                "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
                "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import torch

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the hot path has no CPU fallback (use --impl reference for the CPU arm)"}))
        sys.exit(2)
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    comm = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=device)
        comm = make_comm(device)

    res = run_b200(args, primary, rank, world, comm, device, keep_output=bool(args.dump_outputs))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, f"{primary}_" if world == 1 else f"{primary}_rank{rank}_", *res.pop("output"),
                     limit_bytes=DUMP_LIMIT_BYTES // world)
    cfg = workload_cfg(primary, E, S, W, K, world)
    line = {"metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int64", "data": "synthetic", "config": cfg, "clocks": res["clocks"], "e2e": res.get("e2e"),
            "gpu_launches": res["gpu_launches"], "rows_per_s": res["rows_per_s"],
            "ms_per_circuit_step": res["ms_per_circuit_step"], "timed_region_ms": res["timed_region_ms"],
            "circuit_step_latency_ms": {"p50": res["circuit_step_ms_p50"], "p99": res["circuit_step_ms_p99"], "max": res["circuit_step_ms_max"]},
            "roofline": roofline_from_profile(res["profile"], primary), "kernel_profile": kernel_table(res["profile"]),
            "host_sync": {k: res[k] for k in ("launches_per_circuit_step", "host_readbacks_per_circuit_step", "host_wait_ms_per_circuit_step")},
            "kernel_profile_window": f"per-kernel CUDA events recorded over the last {res['profile_window_circuit_steps']} of the {K * S} timed circuit steps"}
    if comm is not None:
        line["nvlink_bytes_sent_rank0"] = res.get("nvlink_bytes_sent")

    if not args.no_extras and args.query is None and world == 1:
        # the circuit step size is DBSP's throughput / latency knob (the reference's --batch-size): q3 at larger steps
        import copy
        sweep_steps = []
        for e_big in (20_000_000, 80_000_000):
            a2 = copy.copy(args)
            a2.events_per_step, a2.circuit_steps, a2.steps, a2.warmup = e_big, 1, 6, 3
            r = run_b200(a2, "q3", rank, world, comm, device)
            cb = run_reference(a2, "q3", bench_steps=4, warmup=2)
            sweep_steps.append({"events_per_circuit_step": e_big, "value": r["value"], "unit": UNIT, "ms_per_circuit_step": r["ms_per_circuit_step"],
                                "e2e": r.get("e2e"), "gpu_launches": r["gpu_launches"],
                                "cpu_baseline": {"value": cb["value"], "unit": UNIT, "cores": cb["cores"], "kind": cb["kind"], "sample": cb["sample"]}})
        line["q3_step_size_sweep"] = sweep_steps

    if not args.no_extras and args.query is None:
        extras = {}
        for q in ("q4", "q7"):
            r = run_b200(args, q, rank, world, comm, device)
            extras[q] = {"value": r["value"], "unit": UNIT, "rows_per_s": r["rows_per_s"], "ms_per_step": r["ms_per_step"],
                         "ms_per_circuit_step": r["ms_per_circuit_step"], "timed_region_ms": r["timed_region_ms"],
                         "circuit_step_latency_ms": {"p50": r["circuit_step_ms_p50"], "p99": r["circuit_step_ms_p99"], "max": r["circuit_step_ms_max"]},
                         "e2e": r.get("e2e"), "gpu_launches": r["gpu_launches"], "roofline": roofline_from_profile(r["profile"]),
                         "kernel_profile": kernel_table(r["profile"]), "config": workload_cfg(q, E, r["circuit_steps_per_bench_step"], W, K, world),
                         "last_step_out_rows": r["last_step_out_rows"],
                         "host_sync": {k: r[k] for k in ("launches_per_circuit_step", "host_readbacks_per_circuit_step", "host_wait_ms_per_circuit_step")}}
        line["queries"] = extras
        # configs[4]: every rank merges its own replica (no exchange); rank 0 reports its own and the aggregate
        sweep = []
        for total in [int(x) for x in args.sweep_rows.split(",") if x]:
            for nv in (1, 0):
                if nv == 0 and total != 100_000_000:
                    continue
                try:
                    m = merge_sweep(local, rows=total // 2, n_val_lanes=nv)
                except Exception as e:   # e.g. out of memory on a shared box: report, do not hide
                    m = {"workload": f"merge sweep {total} rows nv={nv}", "error": str(e)[:200]}
                if world > 1 and "roofline" in m:
                    t = torch.tensor([m["roofline"]["achieved"]], dtype=torch.float64, device=device)
                    torch.distributed.all_reduce(t)
                    m["aggregate_GBps_all_gpus"] = float(t.item())
                    m["replicas"] = world
                sweep.append(m)
        line["merge_sweep"] = sweep

    if comm is not None:
        try:
            par = parity_check(rank, world, comm, device)
        except Exception as e:
            par = {"ok": False, "error": repr(e)[:300]}
        line["parity_checked"] = bool(par.get("ok"))
        line["parity"] = par

    if rank == 0 and world == 1 and not args.no_extras:
        cb = run_reference(args, primary, bench_steps=4, warmup=1)
        line["cpu_baseline"] = {"value": cb["value"], "unit": UNIT, "cores": cb["cores"], "kind": cb["kind"], "sample": cb["sample"]}
        if "queries" in line:
            for q in ("q4", "q7"):
                c2 = run_reference(args, q, bench_steps=3, warmup=1)
                line["queries"][q]["cpu_baseline"] = {"value": c2["value"], "unit": UNIT, "cores": c2["cores"], "kind": c2["kind"], "sample": c2["sample"]}
    elif rank == 0 and world == 1:
        cb = run_reference(args, primary, bench_steps=2, warmup=1)
        line["cpu_baseline"] = {"value": cb["value"], "unit": UNIT, "cores": cb["cores"], "kind": cb["kind"], "sample": cb["sample"]}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
