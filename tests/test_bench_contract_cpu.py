"""bench.py contract checks that need no GPU: the reference arm (`--impl reference`) runs the reference's CPU path and prints
ONE JSON line with the keys the driver reads; the default arm refuses to run without a CUDA device (no CPU fallback)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line(tmp_path):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--dump-outputs", str(tmp_path / "out")], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.strip().splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    for k in ("metric", "value", "unit", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
              "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["unit"] == "tokens/s" and d["higher_is_better"] is True and d["value"] > 0
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == ("reference" if oracle.ref_ggml() is not None else "port") and cb["cores"] >= 1 and cb["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # --dump-outputs: the last timed token's matmul outputs, float32
    logits = np.load(tmp_path / "out" / "logits.npy")
    assert logits.dtype == np.float32 and logits.shape == (1, 32000) and np.isfinite(logits).all()
    assert np.load(tmp_path / "out" / "last_layer_w2.npy").shape == (1, 4096)


def test_default_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA device present")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"], capture_output=True, text=True,
                       timeout=300, cwd=ROOT)
    assert p.returncode != 0                                  # fails loudly ...
    assert not [ln for ln in p.stdout.splitlines() if ln.startswith("{")]   # ... and reports no number
