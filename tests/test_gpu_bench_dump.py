"""bench.py --dump-outputs: the last timed step's loss and predictions are written as float32 .npy files, --steps is
the number of timed steps, and two runs with the same arguments (seeded inputs) compute the same outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--workload", "small", "--steps", "7",
           "--warmup", "3", "--no-cpu-baseline", "--no-kernel-prof", "--e2e-steps", "-1", "--dump-outputs", str(out_dir)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, res.stdout[-2000:]
    return json.loads(lines[0])


def test_dump_outputs_of_the_last_timed_step(tmp_path):
    runs = []
    for name in ("a", "b"):
        r = _bench(tmp_path / name)
        assert r["steps"] == 7 and r["config"]["local_batch"] == 128
        loss = np.load(tmp_path / name / "loss.npy")
        pred = np.load(tmp_path / name / "predictions.npy")
        assert loss.dtype == np.float32 and loss.shape == ()
        assert pred.dtype == np.float32 and pred.shape == (128, 1)
        assert np.isfinite(loss) and loss > 0 and np.all((pred >= 0) & (pred <= 1))    # BCE of sigmoid outputs
        runs.append((loss, pred))
    np.testing.assert_allclose(runs[1][0], runs[0][0], rtol=1e-5)
    np.testing.assert_allclose(runs[1][1], runs[0][1], rtol=1e-5, atol=1e-7)
