"""bench.py --dump-outputs: the arrays the timed update computed in its last step, for comparing two builds run with
the same arguments."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(out_dir, steps):
    cmd = [sys.executable, os.path.join(REPO, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "2",
           "--config", "halfcheetah", "--batch", "256", "--replay-size", "20000", "--no-cpu-baseline",
           "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    return {f[:-len(".npy")]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_dump_outputs_repeat_with_the_same_arguments_and_follow_steps(tmp_path):
    a, b, c = run_bench(tmp_path / "a", 3), run_bench(tmp_path / "b", 3), run_bench(tmp_path / "c", 4)
    for want in ("tb_info", "log_alpha", "q1.q.0.weight", "q2_target.q.4.bias", "policy.policy.4.weight"):
        assert want in a, want
    assert a["tb_info"].shape == (14,) and np.isfinite(a["tb_info"]).all()
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    # same inputs: only the summation order of the kernels' float atomics may differ between the runs
    assert a.keys() == b.keys() == c.keys()
    for k in a:
        np.testing.assert_allclose(a[k], b[k], rtol=1e-4, atol=1e-6, err_msg=k)
    # one more timed step is one more Adam update (learning rate 1e-4)
    assert np.abs(c["q1.q.0.weight"] - a["q1.q.0.weight"]).max() > 1e-5
