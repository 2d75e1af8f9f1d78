"""bench.py --dump-outputs on the GPU arm: the last timed step's outputs, loss and parameter gradient as float32 .npy files
inside 64 MB, the loss equal to the one in the JSON line, and the same arrays again from a second run with the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1", "--batch", "4",
           "--no-cpu-baseline", "--no-module-api", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    return json.loads(lines[0]), {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_dump_outputs_of_the_timed_step(tmp_path):
    from vilbert_b200.engine import BERT_OUT_NAMES, HEAD_NAMES
    d, arrays = _bench(tmp_path / "a")
    assert d["steps"] == 2
    assert set(arrays) == {f"VQA.{n}" for n in BERT_OUT_NAMES + HEAD_NAMES} | {"VQA.loss", "param_grad"}
    assert all(a.dtype == np.float32 for a in arrays.values())
    assert sum(os.path.getsize(p) for p in (tmp_path / "a").iterdir()) <= 64 * 2 ** 20
    assert arrays["VQA.vil_prediction"].shape == (4, 3129)                 # small arrays keep their shape
    assert arrays["VQA.linguisic_prediction"].ndim == 1                    # 4 x 36 x 30522 logits: a fixed sample
    assert arrays["VQA.loss"].shape == (1,) and arrays["VQA.loss"][0] == np.float32(d["config"]["loss"])
    assert all(np.isfinite(a).all() for a in arrays.values()) and np.abs(arrays["param_grad"]).max() > 0
    _, again = _bench(tmp_path / "b")
    for k, a in arrays.items():
        # same inputs, weights and dropout masks; only the order of the gradient atomics may differ
        assert np.abs(again[k] - a).max() <= 1e-4 * np.abs(a).max() + 1e-30, k
