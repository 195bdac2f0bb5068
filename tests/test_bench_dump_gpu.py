"""GPU: bench.py end to end on the tiny model -- one JSON line whose `steps` is the --steps asked for, and
--dump-outputs writes the last timed step's loss and weights as float32 .npy."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_tiny_dump_outputs(tmp_path):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--model", "tiny", "--batch", "2", "--t_txt", "32",
           "--steps", "5", "--warmup", "0", "--no-cpu-baseline", "--no-gpu-eager-ref", "--dump-outputs", str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    line = json.loads(lines[0])
    assert line["steps"] == 5 and line["value"] > 0
    assert sorted(os.listdir(tmp_path)) == ["loss.npy", "params.npy"]
    loss, params = np.load(tmp_path / "loss.npy"), np.load(tmp_path / "params.npy")
    assert loss.dtype == np.float32 and loss.shape == () and np.isfinite(loss) and loss > 0
    assert params.dtype == np.float32 and params.ndim == 1
    assert params.size >= line["config"]["trainable_params"] and np.isfinite(params).all()
