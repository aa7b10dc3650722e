"""bench.py --dump-outputs: the headline's output planes after the timed steps, identical from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
M2_PLANES = {"theta", "strength", "g2", "h2", "e", "magnitude", "phase"}


def _bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "0",
                        "--quick", "--no-e2e", "--no-cpu", "--configs", "", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_dump_outputs_repeatable(tmp_path):
    a, b = tmp_path / "a", tmp_path / "b"
    la, lb = _bench(a, 2), _bench(b, 3)
    for line, steps in ((la, 2), (lb, 3)):
        assert line["steps"] == steps and line["gpu_launches"] == steps, line
    names = {f[:-4] for f in os.listdir(a)}
    assert names == M2_PLANES and {f[:-4] for f in os.listdir(b)} == names
    assert sum(os.path.getsize(a / (n + ".npy")) for n in names) <= 64 << 20
    for n in names:
        x, y = np.load(a / (n + ".npy")), np.load(b / (n + ".npy"))
        assert x.dtype == np.float32 and x.shape == (1 << 20,) and np.isfinite(x).all(), n
        assert np.array_equal(x, y), n
