"""GPU: bench.py --dump-outputs writes the loss the last timed training step returned (small batch, auxiliary legs off)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from gpu_util import ROOT

pytestmark = pytest.mark.gpu


def test_dump_outputs_of_the_timed_step(tmp_path):
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "3",
                        "--batch", "64", "--no-profile", "--no-decode", "--no-eager", "--no-cpu-baseline",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout)
    assert line["steps"] == 2 and line["warmup"] == 3 and line["value"] > 0
    arrays = {p.stem: np.load(p) for p in out.iterdir()}
    assert sorted(arrays) == ["loss"]
    loss = arrays["loss"]
    assert loss.dtype == np.float32 and loss.shape == (1,) and np.isfinite(loss).all() and loss[0] > 0
