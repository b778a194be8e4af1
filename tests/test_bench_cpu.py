"""CPU: bench.py keeps stdout to the one JSON line the driver parses, even when a library printf()s to fd 1."""
import json
import os
import subprocess
import sys

from gpu_util import ROOT


def test_stdout_carries_only_the_json_line():
    code = ("import ctypes, os, sys; sys.path.insert(0, %r); import bench; os.environ['NCCL_DEBUG'] = 'VERSION'; "
            "bench._protect_stdout(); libc = ctypes.CDLL(None); libc.printf(b'NCCL version banner\\n'); "
            "libc.fflush(None); print('python-level chatter'); bench.emit({'metric': 'x', 'value': 1}); "
            "assert 'NCCL_DEBUG' not in os.environ" % ROOT)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert r.stdout.count("\n") == 1 and json.loads(r.stdout) == {"metric": "x", "value": 1}
    assert "NCCL version banner" in r.stderr and "python-level chatter" in r.stderr


def test_arguments_it_cannot_honour_are_refused():
    """--steps sets the number of timed steps, so no step count below one is silently raised; --dump-outputs is the
    training step's"""
    bench = os.path.join(ROOT, "bench.py")
    for extra in (["--steps", "0"], ["--warmup", "-1"], ["--mode", "decode", "--dump-outputs", "out"],
                  ["--impl", "reference", "--dump-outputs", "out"]):
        r = subprocess.run([sys.executable, bench] + extra, capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and r.stdout == "" and "error" in r.stderr, (extra, r.stderr[-500:])


def test_reference_arm_line_has_the_contract_keys():
    """--impl reference: the oracle port on the host cores, same metric / config keys as the CUDA arm (tiny sample)"""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "1", "--cpu-batch", "1"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout)
    assert d["impl"] == "reference" and d["metric"] == "train_bars_per_sec" and d["unit"] == "bars/s"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["value"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and "workload" in d["config"]
