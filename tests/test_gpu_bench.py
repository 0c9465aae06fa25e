"""bench.py --dump-outputs on the GPU: the last timed step's outputs, the same in every run with
the same arguments (seeded inputs and model, deterministic kernels)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ["--gpus", "1", "--steps", "3", "--warmup", "1", "--batch", "16", "--layers", "2",
         "--hidden", "32", "--no-e2e", "--no-roofline", "--no-stock-gpu", "--no-cpu-baseline"]


@pytest.mark.gpu
def test_dump_outputs_repeat_bit_for_bit(tmp_path):
    for d in ("a", "b"):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + SMALL
                           + ["--dump-outputs", str(tmp_path / d)],
                           cwd=ROOT, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 3
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(os.listdir(tmp_path / "b"))
    assert {"loss.npy", "pred.npy"} <= set(files)
    assert any(f.startswith("param.") for f in files) and any(f.startswith("grad.") for f in files)
    assert np.load(tmp_path / "a" / "pred.npy").shape == (16, 1)
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype in (np.float32, np.float64) and np.isfinite(a).all(), f
        assert np.array_equal(a, b), f
