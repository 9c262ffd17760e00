"""bench.py contract.  Without a GPU: the reference arm (the reference's algorithm on host cores, here the reference-shaped
restatement) prints ONE JSON line with the keys a consumer of the line reads, and the --dump-outputs writer stores exact
values within its size budget.  On the GPU: --dump-outputs writes what the last timed pass returned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra, env=None):
    e = dict(os.environ)
    e.update(env or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--cpu-sample-runs", "300"] + extra, capture_output=True, text=True, timeout=300, env=e, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return out.stdout.strip().splitlines()


def test_reference_arm_prints_one_contract_line():
    lines = _run([])
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "evals/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("step ready-evals/sec") and d["steps"] == 2 and d["value"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "refshape" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and d["vs_baseline"] is None and "workload" in d["config"]


def test_reference_arm_non_zero_ranks_stay_silent():
    """under torchrun only rank 0 runs and prints the reference arm; the other ranks exit 0 without work"""
    assert _run(["--gpus", "2"], env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}) == []


def test_dump_outputs_exact_values_and_seeded_sample_within_budget(tmp_path):
    import bench
    rng = np.random.default_rng(5)
    arrays = {"result": rng.integers(0, 256, (5000, 80), dtype=np.uint8), "counts": np.array([7, 3, 0, 2 ** 40], np.int64),
              "expansion": rng.integers(0, 2 ** 32, (3000, 3), dtype=np.uint32)}
    budget = 200_000
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, budget)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["counts.npy", "expansion.npy", "result.npy", "result_rows.npy"]
    got = {n[:-4]: np.load(tmp_path / "a" / n) for n in names}
    assert sum(a.nbytes for a in got.values()) <= budget
    assert got["counts"].dtype == np.float64 and got["counts"].tolist() == [7, 3, 0, 2 ** 40]
    assert got["expansion"].dtype == np.float64 and np.array_equal(got["expansion"], arrays["expansion"])
    rows = got["result_rows"].astype(np.int64)
    assert len(rows) > 300 and np.all(np.diff(rows) > 0) and rows[-1] < 5000
    assert got["result"].dtype == np.float32 and np.array_equal(got["result"], arrays["result"][rows])
    for n in names:
        assert np.array_equal(np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n))


@pytest.mark.gpu
def test_gpu_arm_dumps_what_the_last_timed_pass_returned(tmp_path):
    """with one input set every timed pass evaluates the seeded batch of set 0, so the dump must equal the oracle on it"""
    from bobrapet_b200 import synth
    from bobrapet_b200.records import layout_py
    from oracle import packed as PK
    n, S = 3000, 256
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--runs", str(n), "--rot", "1",
                          "--reps", "1", "--no-e2e", "--no-cpu", "--no-extra", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["steps"] == 3 and d["timing"]["region_ms"] and sorted(os.listdir(tmp_path)) == ["counts.npy", "result.npy"]
    counts, res = np.load(tmp_path / "counts.npy"), np.load(tmp_path / "result.npy")
    assert counts.dtype == np.float64 and counts.tolist() == [d["counts_last_pass"][k] for k in ("ready", "skip", "expansion", "evals")]
    L = layout_py(S, 0, 0)
    slots = np.arange(n, dtype=np.uint32)
    ts = synth.topologies(3, 0, n, S)
    want, wc = PK.evaluate(PK.PackedTopologies(ts, slots), L, synth.state(3, 0, n, L, slots, ts), threads=4)
    assert res.dtype == np.float32 and np.array_equal(res, want.astype(np.float32))
    assert counts.tolist() == [wc["ready"], wc["skip"], wc["expansion"], wc["evals"]]
