"""bench.py on the GPU: --dump-outputs writes the same arrays for the same arguments, and --steps sets the timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _bench(out, steps, warmup):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1", "--steps", str(steps), "--warmup", str(warmup),
           "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    return json.loads(lines[0])


def test_dump_outputs_repeat_and_steps(tmp_path):
    steps, warmup = 3, 1
    a = _bench(tmp_path / "a", steps, warmup)
    _bench(tmp_path / "b", steps, warmup)
    assert a["steps"] == steps and a["warmup"] == warmup
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(os.listdir(tmp_path / "b")) and {"tree_tok.npy", "roots_tok.npy", "counters.npy", "sigma.npy"} <= set(files)
    for f in files:
        x, y = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert x.dtype == np.float64 and np.array_equal(x, y, equal_nan=True), f
    # the dump is the state after warm-up and timed steps: every chain ran sweeps_per_step sweeps in each of them
    cfg = a["config"]
    cnt = np.load(tmp_path / "a" / "counters.npy")
    assert cnt.shape == (cfg["chains_per_gpu"], 8)
    assert (cnt[:, 7] == cfg["sweeps_per_step"] * (steps + warmup)).all()
    assert (cnt[:, 0] == cfg["K"] * cfg["sweeps_per_step"] * (steps + warmup)).all()
