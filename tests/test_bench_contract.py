"""bench.py's output contract: exactly one JSON line on stdout with the keys the driver reads.
The reference arm runs on the host cores (no GPU needed); the product arm is checked on the GPU box."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e"}


def run_bench(*args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=900,
                       cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.split("\n") if l.strip()]
    assert len(lines) == 1, lines          # one JSON line, nothing else on stdout
    return json.loads(lines[0])


def test_reference_arm_line():
    d = run_bench("--impl", "reference", "--db", "3000", "--steps", "2", "--warmup", "1")
    assert BASE_KEYS <= set(d)
    assert d["impl"] == "reference" and d["unit"] == "GCUPS" and d["higher_is_better"] is True
    assert d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0
    assert d["vs_baseline"] is None and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_dumps_its_results(tmp_path, oracle, blosum62):
    d = run_bench("--impl", "reference", "--db", "3000", "--steps", "1", "--warmup", "0", "--dump-outputs", str(tmp_path))
    assert d["steps"] == 1
    assert sorted(os.listdir(tmp_path)) == ["end_query.npy", "end_ref.npy", "score.npy"]
    import bench
    query, cat, off = bench.make_inputs(3000)
    exp = oracle.align_batch(query, np.array([0, len(query)]), cat, off, blosum62, mode=oracle.SW, open=bench.OPEN,
                             gap=bench.GAP, shared_query=True, threads=0)
    for k in ("score", "end_query", "end_ref"):
        got = np.load(tmp_path / f"{k}.npy")
        assert got.dtype == np.float64 and np.array_equal(got, exp[k]), k


def test_dump_outputs_samples_large_results(tmp_path):
    import bench
    n, limit = 100000, 256 << 10
    arrays = {"score": np.arange(n, dtype=np.int32) * 3, "end_ref": np.arange(n, dtype=np.int32) - 7}
    bench.dump_outputs(str(tmp_path / "a"), arrays, limit=limit)
    bench.dump_outputs(str(tmp_path / "b"), arrays, limit=limit)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["end_ref.npy", "sample_index.npy", "score.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= limit
    idx = np.load(tmp_path / "a" / "sample_index.npy").astype(np.int64)
    assert len(idx) > 1000 and np.all(np.diff(idx) > 0) and idx[-1] < n
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f   # the same sample every run
    for k, v in arrays.items():
        assert np.array_equal(np.load(tmp_path / "a" / f"{k}.npy"), v[idx]), k
    bench.dump_outputs(str(tmp_path / "c"), arrays)                       # fits: everything, no index
    assert sorted(os.listdir(tmp_path / "c")) == ["end_ref.npy", "score.npy"]
    assert np.array_equal(np.load(tmp_path / "c" / "score.npy"), arrays["score"])


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--db", "3000",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_product_arm_line():
    d = run_bench("--db", "20000", "--steps", "3", "--warmup", "3", "--e2e-steps", "2", "--cpu-sample", "2000")
    assert BASE_KEYS | {"gpu_launches", "clocks", "roofline", "cpu_baseline"} <= set(d)
    assert "impl" not in d or d["impl"] != "reference"
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["warmup"] >= 3 and d["value"] > 0
    assert d["gpu_launches"] >= 3
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] != d["value"]
    rf = d["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(rf) and 0 < rf["frac"] < 1.5
    cb = d["cpu_baseline"]
    assert {"value", "unit", "cores", "kind", "sample"} <= set(cb) and cb["kind"] == "port"
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])


@pytest.mark.gpu
def test_product_arm_dumps_its_results(tmp_path, oracle, blosum62):
    d = run_bench("--db", "20000", "--steps", "2", "--warmup", "3", "--e2e-steps", "1", "--no-cpu", "--dump-outputs", str(tmp_path))
    assert d["steps"] == 2
    got = {k: np.load(tmp_path / f"{k}.npy") for k in ("score", "end_query", "end_ref")}
    assert all(v.dtype == np.float64 and v.shape == (20000,) for v in got.values())
    import bench
    query, cat, off = bench.make_inputs(20000)
    exp = oracle.align_batch(query, np.array([0, len(query)]), cat, off[:501], blosum62, mode=oracle.SW, open=bench.OPEN,
                             gap=bench.GAP, shared_query=True, threads=0)
    for k, v in got.items():
        assert np.array_equal(v[:500], exp[k]), k
