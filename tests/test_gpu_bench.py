"""bench.py on a small workload: --steps sets the number of timed steps, and --dump-outputs writes the last timed step's
outputs as float32 / float64 .npy files (at most 64 MB) that are identical from run to run with the same inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(steps, out_dir, *extra):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
           "--images", "20000", "--no-cpu-baseline", "--no-hbm-kernels", "--dump-outputs", str(out_dir), *extra]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_bench_steps_and_dump_outputs(tmp_path):
    one = _bench(1, tmp_path / "one")
    two = _bench(2, tmp_path / "two", "--no-verify")
    assert one["verified"] is True and one["steps"] == 1 and two["steps"] == 2
    assert two["gpu_launches"] == 2 * one["gpu_launches"] > 0           # every timed step launches the same kernels
    names = sorted(os.listdir(tmp_path / "one"))
    assert names == ["images_sample.npy", "recovered_vectors_sample.npy", "topk_ids.npy", "topk_scores.npy"]
    assert sorted(os.listdir(tmp_path / "two")) == names
    total = 0
    for name in names:
        a, b = np.load(tmp_path / "one" / name), np.load(tmp_path / "two" / name)
        assert a.dtype in (np.float32, np.float64) and a.size > 0 and np.isfinite(a).all(), name
        np.testing.assert_array_equal(a, b, err_msg=name)
        total += os.path.getsize(tmp_path / "one" / name)
    assert total <= 64 << 20
    img = np.load(tmp_path / "one" / "images_sample.npy")
    att = np.load(tmp_path / "one" / "recovered_vectors_sample.npy")
    ids = np.load(tmp_path / "one" / "topk_ids.npy")
    assert img.shape[1:] == (1, 32, 32) and att.shape == (img.shape[0], 100) and img.shape[0] == 8192
    assert ids.shape == (4096, 20) and ids.min() >= 0 and ids.max() < 20000 and (ids == np.rint(ids)).all()
