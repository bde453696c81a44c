"""bench.py --dump-outputs: the last timed step's results are written as float arrays, small enough to
keep beside a benchmark result, and two runs with the same arguments compute the same thing (the inputs
are seeded; PCM_DETERMINISTIC=1 makes the LoRA gradients bit-reproducible)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = {"loss", "optimizer_state", "lora_params", "adam_exp_avg", "adam_exp_avg_sq"}


def _bench(out, steps, warmup):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
           "--warmup", str(warmup), "--batch", "1", "--latent", "16", "--no-cpu-baseline",
           "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT,
                       env=dict(os.environ, PCM_DETERMINISTIC="1"))
    assert r.returncode == 0, r.stderr[-4000:]
    line = json.loads([s for s in r.stdout.splitlines() if s.startswith("{")][-1])
    return line, {n: np.load(os.path.join(out, n + ".npy")) for n in NAMES}


def test_dump_outputs_are_the_last_timed_step(cuda, tmp_path):
    steps, warmup = 3, 2
    line, a = _bench(tmp_path / "a", steps, warmup)
    assert sorted(os.listdir(tmp_path / "a")) == sorted(n + ".npy" for n in NAMES)
    assert all(v.dtype == np.float32 for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert line["steps"] == steps
    assert a["loss"].shape == (1,) and float(a["loss"][0]) == line["loss"]
    assert a["optimizer_state"][1] == warmup + steps      # AdamW step count: no extra or missing steps
    assert a["lora_params"].shape == a["adam_exp_avg"].shape == a["adam_exp_avg_sq"].shape
    assert all(np.isfinite(v).all() for v in a.values())
    assert np.abs(a["adam_exp_avg"]).max() > 0 and a["adam_exp_avg_sq"].min() >= 0
    _, b = _bench(tmp_path / "b", steps, warmup)
    for n in NAMES:
        assert np.array_equal(a[n], b[n]), n
