"""bench.py --dump-outputs: the arrays written are what the timed path computed, so that two builds of the project can be
compared output for output on the benchmark's own (seeded) inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    batch = 8
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0", "--batch", str(batch),
                        "--no-secondary", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert d["steps"] == 2
    out = np.load(tmp_path / "c2_output.npy")
    idx = np.load(tmp_path / "c2_output_sample_index.npy")
    assert out.dtype == np.float32 and out.shape == (batch, 3, 224, 224) and np.array_equal(idx, np.arange(batch))
    # the same seeded batch through the pipeline in this process
    import bench
    from dali_b200.hotpath import ImagePipelineC2
    streams = bench.make_batch(batch, 0, 4)
    mirror = np.random.default_rng(0).integers(0, 2, batch)
    want = ImagePipelineC2(batch).run(streams, mirror).float().cpu().numpy()
    assert np.array_equal(out, want)
