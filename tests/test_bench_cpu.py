"""The reference arm of bench.py runs on the host CPU (oracle port): one JSON line with the contract's keys."""

import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "c1",
                           "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [ln for ln in proc.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, proc.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "images/sec" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_dump_outputs_writes_the_step_results_and_a_fixed_weight_sample(tmp_path):
    import numpy as np
    import torch

    import bench

    model = torch.nn.Linear(3000, 2)  # weight: 6000 elements, sampled down to per_tensor; bias: kept whole
    logits = torch.randn(2, 3, 4, 4, dtype=torch.bfloat16)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), (1.25, 3.5), logits, model)
    assert sorted(os.listdir(tmp_path / "a")) == ["grad_norm.npy", "logits.npy", "loss.npy", "weights.npy"]
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    assert got["loss"].dtype == got["grad_norm"].dtype == np.float64 and got["loss"] == 1.25 and got["grad_norm"] == 3.5
    assert got["logits"].dtype == np.float32 and np.array_equal(got["logits"], logits.float().numpy())
    w = got["weights"]
    assert w.dtype == np.float32 and w.shape == (4096 + 2,)
    assert np.isin(w[:4096], model.weight.detach().numpy()).all() and np.array_equal(w[4096:], model.bias.detach().numpy())
    assert np.array_equal(w, np.load(tmp_path / "b" / "weights.npy"))  # the same positions on every run
    bench.dump_outputs(str(tmp_path / "c"), (1.25, 3.5), logits, model, max_logits=2 * 3 * 4 * 4 - 1)
    assert np.array_equal(np.load(tmp_path / "c" / "logits.npy"), logits[:1].float().numpy())  # leading images only


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                          capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert proc.returncode == 0 and proc.stdout.strip() == ""
