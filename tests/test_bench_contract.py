"""bench.py contract, the part that runs without a GPU: the reference arm prints exactly ONE JSON line on
stdout with the keys the driver reads (metric, value, unit, n_gpus, steps, warmup, ms_per_step, ...)."""
import json
import os
import subprocess
import sys

import numpy as np

from conftest import ROOT


def test_reference_arm_emits_one_json_line(tmp_path):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-800:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, p.stdout[:400]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "ecdsa_verifies_per_sec" and d["unit"] == "verifies/s"
    for key in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["value"] > 0 and d["steps"] == 1 and d["config"]["workload"].startswith("ECDSA verify batch 2^20")
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    # --dump-outputs: the verify result of the last timed step, every 16th row corrupted by construction
    ok = np.load(tmp_path / "ecdsa_verify_ok.npy")
    assert ok.dtype == np.float32 and ok.ndim == 1 and len(ok) >= 4096
    assert set(np.unique(ok)) == {0.0, 1.0} and ok.sum() == len(ok) - len(ok) // 16


def test_dump_outputs_samples_a_large_array(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 4000)
    big = np.arange(5000) % 3 == 0
    bench.dump_outputs(str(tmp_path), {"v": big})
    v, rows = np.load(tmp_path / "v.npy"), np.load(tmp_path / "v_rows.npy")
    assert v.dtype == np.float32 and rows.dtype == np.float64 and len(v) == len(rows) == 4000 // 12
    assert np.array_equal(v, big[rows.astype(np.int64)]) and np.all(np.diff(rows) > 0)
    bench.dump_outputs(str(tmp_path / "again"), {"v": big})
    assert np.array_equal(np.load(tmp_path / "again" / "v_rows.npy"), rows)


def test_own_arm_fails_loudly_without_a_gpu():
    """No CPU fallback: on a box without a CUDA device the product arm must exit non-zero, not print numbers."""
    import torch
    if torch.cuda.is_available():
        return
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode != 0
    assert not [ln for ln in p.stdout.splitlines() if ln.strip().startswith("{")]
