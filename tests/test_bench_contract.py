"""The CPU arm of bench.py (`--impl reference`) honours the driver's JSON contract, runs the same circuit steps as the
GPU arm and spells out a bounded sample; the GPU arm refuses to run without a device (no CPU fallback)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600, env=e)
    lines = [ln for ln in p.stdout.strip().splitlines() if ln.startswith("{")]
    return p.returncode, (json.loads(lines[-1]) if lines else None)


def test_reference_arm_line():
    rc, d = run_bench("--impl", "reference", "--gpus", "2", "--steps", "3", "--warmup", "3", "--events-per-step", "20000")
    assert rc == 0
    assert d["impl"] == "reference" and d["metric"] == "nexmark_events_per_sec" and d["unit"] == "events/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 2 and d["steps"] == 3 and d["warmup"] == 3
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": "events/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "40000 events" in cb["sample"]
    assert d["config"]["query"] == "q3" and d["config"]["events_per_circuit_step_per_gpu"] == 20000
    assert "reference_sample" not in d["config"]   # small run: nothing was cut


def test_reference_arm_bounded_sample_is_declared():
    # 8 x 3 M events per circuit step, (5 + 20) bench steps: 8 circuit steps per bench step would be 4.8 G events
    sys.path.insert(0, ROOT)
    import bench

    class A:
        events_per_step, circuit_steps, steps, warmup, cpu_threads = 3_000_000, 0, 20, 5, 2

    calls = {}

    def fake_gen(query, rank, world, n_steps, E, pinned, rate=None):
        calls["n_steps"], calls["E"] = n_steps, E
        raise RuntimeError("stop before generating")

    orig = bench.gen_steps
    bench.gen_steps = fake_gen
    try:
        try:
            bench.run_reference(A, "q3", gpus=8)
        except RuntimeError:
            pass
    finally:
        bench.gen_steps = orig
    assert calls["E"] == 24_000_000
    assert calls["n_steps"] * calls["E"] <= 2_400_000_000 and calls["n_steps"] == 25 * 4   # 4 of 8 circuit steps per bench step


def test_gpu_arm_refuses_without_device():
    rc, d = run_bench("--steps", "1", env={"CUDA_VISIBLE_DEVICES": ""})
    assert rc != 0 and "no CUDA device" in d["error"]


def load_dump(d, prefix, n_lanes):
    """(lanes, weights, row indices or None) of a --dump-outputs directory, lanes reassembled from their halves."""
    lanes = [(np.load(os.path.join(d, f"{prefix}lane{i}_hi.npy")).astype(np.uint64) << np.uint64(32))
             | np.load(os.path.join(d, f"{prefix}lane{i}_lo.npy")).astype(np.uint64) for i in range(n_lanes)]
    idx = os.path.join(d, f"{prefix}row_index.npy")
    return lanes, np.load(os.path.join(d, f"{prefix}weight.npy")), (np.load(idx).astype(np.int64) if os.path.exists(idx) else None)


@pytest.mark.parametrize("limit", [64 << 20, 8 * 8 * 100], ids=["whole", "sampled"])
def test_dump_outputs_exact_and_bounded(tmp_path, oracle, limit):
    # lanes above 2**53 must survive the float64 files bit for bit; an output over the limit becomes a seeded sample
    sys.path.insert(0, ROOT)
    import bench
    import dbsp_b200

    rng = np.random.default_rng(3)
    b = oracle.batch_from_columns(dbsp_b200.Schema("u", "uu"), [rng.integers(0, 50, 4000).astype(np.uint64),
                                  rng.integers(0, 1 << 62, 4000).astype(np.uint64), rng.integers(0, 9, 4000).astype(np.uint64)],
                                  rng.integers(-2, 3, 4000))
    lanes, w = bench.flat_rows(b)
    ref_lanes, ref_w = oracle.flat(b)
    assert all(np.array_equal(x, y) for x, y in zip(lanes, ref_lanes)) and np.array_equal(w, ref_w)
    for d in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(str(d), "q_", lanes, w, limit)
    got, gw, idx = load_dump(tmp_path / "a", "q_", 3)
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= limit + 8 * 128   # + the .npy headers
    if limit == 64 << 20:
        assert idx is None
        idx = np.arange(len(w))
    else:
        assert len(idx) == 100 and np.all(np.diff(idx) > 0)
        assert np.array_equal(idx, load_dump(tmp_path / "b", "q_", 3)[2])
    assert all(np.array_equal(g, c[idx]) for g, c in zip(got, lanes)) and np.array_equal(gw, w[idx].astype(np.float64))


@pytest.mark.gpu
def test_gpu_dump_outputs_match_oracle(tmp_path, oracle):
    # --steps K times K bench steps, and --dump-outputs holds the output of the last of them: the oracle circuit fed
    # the same seeded warm-up + timed circuit steps ends on the same Z-set
    sys.path.insert(0, ROOT)
    import bench
    import dbsp_b200
    from dbsp_b200.nexmark import queries as nq

    E, W, K = 100_000, 3, 2
    rc, d = run_bench("--query", "q3", "--no-extras", "--steps", str(K), "--warmup", str(W), "--circuit-steps", "1",
                      "--events-per-step", str(E), "--dump-outputs", str(tmp_path))
    assert rc == 0 and d["steps"] == K and d["config"]["timed_circuit_steps"] == K
    c = dbsp_b200.RootCircuit(oracle, None)
    inp, handles = nq.add_nexmark_input(c)
    out = nq.QUERIES["q3"](inp).output()
    for t in bench.gen_steps("q3", 0, 1, W + K, E, pinned=False):
        for k in ("person", "auction", "bid"):
            handles[k].set(t[k] if t[k] is not None else bench.empty_cols())
        c.step()
    lanes, w = bench.flat_rows(out.value)
    got, gw, idx = load_dump(tmp_path, "q3_", len(lanes))
    assert len(w) > 0 and idx is None
    assert all(np.array_equal(g, x) for g, x in zip(got, lanes)) and np.array_equal(gw, w.astype(np.float64))
