"""GPU: `bench.py --dump-outputs DIR` writes what the last timed training step computed, consistent with the step's own
inputs, and two runs with the same arguments write identical arrays (seeded inputs, weights and dropout masks; every
float reduction of the library has a fixed order), so the outputs of two builds can be compared one to one."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
B, S = 4, 64


def _bench(out_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--batch", str(B), "--size", str(S),
           "--no-extras", "--no-cpu-baseline", "--no-eager-baseline", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    return json.loads(lines[0]), {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_dump_outputs_are_the_last_timed_step_and_repeat_exactly(tmp_path):
    from tools.synthetic import synthetic_batch
    rec, a = _bench(tmp_path / "a")
    assert rec["steps"] == 2 and len(rec["ms_each_step"]) == 2
    assert sorted(a) == ["bn_running_stats", "confusion_counts", "grads", "loss", "params", "probs"]
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 * 10 ** 6
    p = a["probs"].astype(np.float64)
    assert p.shape == (B, 1, S, S) and ((p >= 0) & (p <= 1)).all()
    # the loss and the confusion counts are those of the dumped probabilities on the bench's inputs
    y = synthetic_batch(B, 3, S, S, seed=123)[1].numpy().astype(np.float64)
    with np.errstate(divide="ignore"):                 # saturated probabilities: log 0 = -inf, clamped like nn.BCELoss
        bce = -np.mean(y * np.maximum(np.log(p), -100) + (1 - y) * np.maximum(np.log1p(-p), -100))
    assert abs(float(a["loss"]) - bce) <= 1e-4 * bce
    pos = p > 0.5
    want = np.stack([(pos & (y == 1)).sum((1, 2, 3)), (pos & (y == 0)).sum((1, 2, 3)), (~pos & (y == 1)).sum((1, 2, 3)),
                     (~pos & (y == 0)).sum((1, 2, 3))], 1)
    assert np.array_equal(a["confusion_counts"], want)
    # 40.9 M parameters: a fixed seeded sample of 4 Mi values
    assert a["grads"].shape == a["params"].shape == (1 << 22,)
    assert np.isfinite(a["grads"]).all() and np.isfinite(a["params"]).all() and np.isfinite(a["bn_running_stats"]).all()
    _, b = _bench(tmp_path / "b")
    assert sorted(b) == sorted(a)
    for k in a:
        diff = np.abs(a[k].astype(np.float64) - b[k])
        assert np.array_equal(a[k], b[k]), f"{k}: {int((diff > 0).sum())} of {diff.size} differ, max {diff.max()}"
