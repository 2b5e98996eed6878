"""bench.py --dump-outputs: the last timed step's outputs are written as float .npy files, 64 MB at most, and two runs
with the same arguments (the same seeded tokens, weights and dropout keys) give the same outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "small", "--steps", str(steps),
                        "--warmup", "3", "--no-cpu-baseline", "--no-gpu-baseline", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout)


def test_dump_outputs_of_the_last_timed_step_are_reproducible(tmp_path):
    a, b = tmp_path / "a", tmp_path / "b"
    line = _bench(a, 4)
    assert line["steps"] == 4
    _bench(b, 4)
    names = sorted(os.listdir(a))
    assert names == sorted(os.listdir(b))
    assert {"loss.npy", "norm.npy", "state_h0.npy", "state_c1.npy", "param_embed.W.npy", "param_fc.b.npy"} <= set(names)
    # the loss in the dump is the one the bench line reports for the last timed step
    assert float(np.load(a / "loss.npy")) == line["final_loss"]
    total = 0
    for n in names:
        x, y = np.load(a / n), np.load(b / n)
        assert x.dtype in (np.float32, np.float64) and x.shape == y.shape, n
        assert np.isfinite(x).all(), n
        # same inputs; fp32 atomics (embedding-gradient scatter, split-K GEMMs) may add in another order per run
        np.testing.assert_allclose(x, y, rtol=0, atol=1e-4 * max(1.0, float(np.abs(y).max())), err_msg=n)
        total += x.nbytes
    assert total <= 64 << 20
