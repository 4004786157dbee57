"""bench.py on the GPU: `--steps` sets the timed steps and `--dump-outputs` writes what the last of them computed."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_dumps_the_last_timed_step(tmp_path):
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "c2", "--steps", "2", "--warmup", "1",
                           "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True,
                          timeout=900, cwd=ROOT)
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [ln for ln in proc.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, proc.stdout
    d = json.loads(lines[0])
    assert d["steps"] == 2
    out = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert sorted(out) == ["grad_norm", "logits", "loss", "weights"]
    assert float(out["loss"]) == d["last_loss"] and float(out["grad_norm"]) == d["last_grad_norm"]
    assert out["logits"].shape == (64, 1, 28, 28) and out["logits"].dtype == np.float32
    assert out["weights"].dtype == np.float32 and out["weights"].size > 0
    assert all(np.isfinite(a).all() for a in out.values())
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64 << 20
