"""GPU: `bench.py --dump-outputs DIR` writes what the timed step computed -- the same files whatever `--steps` is,
within 64 MB, float32 / float64 only -- and the GPU arm's files equal the reference arm's (the CPU oracle's step on
the same seeded inputs), name for name."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu
NAMES = ["box_feats", "det_boxes", "det_classes", "det_scores", "det_valid", "mask_feats", "proposal_boxes",
         "proposal_logits", "proposal_valid"]


def _bench(out, steps, *extra):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                        "--dump-outputs", str(out)] + list(extra), capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == steps
    files = sorted(os.listdir(out))
    assert files == [n + ".npy" for n in NAMES]
    assert sum(os.path.getsize(os.path.join(out, f)) for f in files) <= 64 << 20
    return {f[:-4]: np.load(os.path.join(out, f)) for f in files}


def test_dump_outputs_are_the_oracle_step(cuda, tmp_path):
    fast = ("--no-cpu", "--no-extras", "--no-e2e")
    a = _bench(tmp_path / "a", 1, *fast)
    b = _bench(tmp_path / "b", 6, *fast)
    want = _bench(tmp_path / "ref", 1, "--impl", "reference")
    for k in NAMES:
        assert a[k].dtype in (np.float32, np.float64) and a[k].dtype == want[k].dtype, k
        assert np.array_equal(a[k], b[k]), k
        if k.endswith("_feats"):
            w = want[k]
            assert a[k].shape == w.shape and np.abs(a[k] - w).max() <= 1e-5 * max(np.abs(w).max(), 1e-30), k
        else:
            assert np.array_equal(a[k], want[k]), k
