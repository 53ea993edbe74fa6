"""bench.py contract on the CPU arm (`--impl reference`): exactly ONE JSON line on stdout with the keys the driver reads."""
import json
import os
import subprocess
import sys

import numpy as np

from _util import ROOT


def test_reference_arm_prints_one_json_line(tmp_path):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "3",
                        "--batch", "1", "--dump-outputs", str(tmp_path / "out")], capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "images/s" and d["value"] > 0 and d["higher_is_better"] is True
    # "reference" = the unmodified reference shipped in oracle/_ref (make -C oracle), "port" = the oracle when that tree is absent
    expect = "reference" if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "ultralytics", "nn", "tasks.py")) else "port"
    assert d["cpu_baseline"]["kind"] == expect and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]
    # --dump-outputs: the (B, 300, 6) detections of the last timed step, float32
    det = np.load(tmp_path / "out" / "detections.npy")
    assert det.dtype == np.float32 and det.shape == (1, 300, 6) and np.isfinite(det).all()
