"""`bench.py --dump-outputs` on the tiny model: the last timed step's outputs land as float32 .npy files within 64 MB, the
same arguments give the same outputs bit for bit, and --steps sets how many training steps produced them."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--model", "tiny", "--seq", "512", "--lora-r", "16",
           "--steps", str(steps), "--warmup", "3", "--no-cpu-baseline", "--no-gpu-baseline", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
    return {f[:-len(".npy")]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def _rel(a, b):
    return float(np.linalg.norm(a.astype(np.float64) - b) / np.linalg.norm(b.astype(np.float64)))


def test_dump_outputs_repeatable_and_follow_steps(tmp_path):
    a = _bench(tmp_path / "a", 2)
    assert set(a) == {"loss", "lora_weights", "lora_grads"}
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert a["loss"].shape == (1,) and a["lora_weights"].shape == a["lora_grads"].shape
    b = _bench(tmp_path / "b", 2)
    for name in a:   # seq 512 spans four 128-token key blocks of the attention backward: bit-equal all the same
        assert np.array_equal(b[name], a[name]), name
    # each step trains on the next of 8 seeded batches: one more timed step ends on another batch
    c = _bench(tmp_path / "c", 3)
    assert _rel(c["lora_grads"], a["lora_grads"]) > 0.1
    assert _rel(c["lora_weights"], a["lora_weights"]) > 1e-3   # two more AdamW updates of lr 2e-4
