"""CPU: the reference arm of bench.py (the oracle port timed on host cores) prints the contract's JSON line; the
argument checks and the --dump-outputs writer."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "samples/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]


def test_steps_below_one_are_rejected():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=60,
                         cwd=ROOT)
    assert out.returncode == 2 and "--steps" in out.stderr


def test_dump_outputs_writes_the_losses_and_a_fixed_parameter_sample(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_PARAMS", 1000)
    losses = torch.randn(3, 8)
    params = torch.arange(3 * 2000, dtype=torch.float32).view(3, 2000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), losses, params)
    got = {d: {f: np.load(str(tmp_path / d / (f + ".npy"))) for f in ("losses", "params")} for d in ("a", "b")}
    assert got["a"]["losses"].dtype == np.float32 and np.array_equal(got["a"]["losses"], losses.numpy())
    sample = got["a"]["params"]
    assert sample.dtype == np.float32 and sample.shape == (1000,) and np.all(np.diff(sample) >= 0)
    assert np.array_equal(sample, got["b"]["params"])  # same indices in every run
    bench.dump_outputs(str(tmp_path / "c"), losses[:1], params[:1, :500])  # fits: written whole
    assert np.array_equal(np.load(str(tmp_path / "c" / "params.npy")), params[0, :500].numpy())
