"""CPU: the bench.py contract that can be checked without a GPU -- the reference arm prints exactly one JSON line
with the agreed keys, and the product arm refuses to run (loudly) when there is no CUDA device."""
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "ROIs/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["gpu_launches"] == 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "ROIs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("configs[1]")
    # --dump-outputs: the last timed step's outputs, float32 / float64, within 64 MB
    files = sorted(os.listdir(tmp_path))
    assert files == sorted(n + ".npy" for n in ("proposal_boxes", "proposal_logits", "proposal_valid", "box_feats",
                                               "det_boxes", "det_scores", "det_classes", "det_valid", "mask_feats"))
    assert sum(os.path.getsize(os.path.join(tmp_path, f)) for f in files) <= 64 << 20
    assert all(np.load(os.path.join(tmp_path, f)).dtype in (np.float32, np.float64) for f in files)


def test_product_arm_needs_a_gpu():
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True,
                       timeout=600, cwd=ROOT)
    assert r.returncode != 0
    assert "no CUDA device" in (r.stderr + r.stdout)
    assert r.stdout.strip() == ""  # nothing that could be mistaken for a result line
