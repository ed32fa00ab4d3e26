"""bench.py contract, GPU part: `--steps` sets the number of timed steps, and `--dump-outputs` writes the same arrays
for the same arguments, so that two builds of the project can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ["--n-envs", "64", "--warmup", "1", "--no-cpu-baseline", "--no-e2e", "--no-consensus"]


def run_bench(steps, dump_dir=None):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps)] + SMALL
    if dump_dir is not None:
        cmd += ["--dump-outputs", str(dump_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout)


def test_steps_set_the_timed_work_and_dumped_outputs_repeat(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    one = run_bench(1)
    a = run_bench(2, tmp_path / "a")
    b = run_bench(2, tmp_path / "b")
    assert one["steps"] == 1 and a["steps"] == 2
    assert a["gpu_launches"] == 2 * one["gpu_launches"] > 0          # every step launches the same kernels
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b"))
    assert {"est_returns.npy", "true_returns.npy", "critic_loss.npy", "actor.npy", "buffer_sa.npy"} <= set(names)
    total = 0
    for name in names:
        x, y = np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name)
        assert x.dtype in (np.float32, np.float64) and x.size > 0, name
        assert np.isfinite(x).all(), name
        np.testing.assert_array_equal(x, y, err_msg=name)
        total += x.nbytes
    assert total <= 64 << 20
