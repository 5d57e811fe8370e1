"""The reference arm of bench.py runs without a GPU: its JSON line must keep the driver's contract (keys, units, the
`impl` / `cpu_baseline` / `e2e` objects).  One bounded step on the host cores."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "images/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["steps"] == 1 and d["warmup"] == 0 and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_bench_rejects_meaningless_step_counts_and_dump_targets():
    for extra in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "unused"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert r.returncode == 2 and "error" in r.stderr and r.stdout == "", extra


def test_dump_sample_of_the_default_batch():
    import numpy as np
    import bench
    keep = bench.dump_sample(bench.BATCH)
    assert np.array_equal(keep, bench.dump_sample(bench.BATCH))                       # the same images on every run
    assert keep.size < bench.BATCH and np.all(np.diff(keep) > 0) and 0 <= keep[0] and keep[-1] < bench.BATCH
    # what --dump-outputs writes: the images as float32 and the index as float64, each with a .npy header
    assert keep.size * 3 * bench.OUT * bench.OUT * 4 + keep.size * 8 + 2 * 128 < 64e6
    assert np.array_equal(bench.dump_sample(8), np.arange(8))                         # a small batch is kept whole


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""
