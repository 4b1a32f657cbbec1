"""bench.py --dump-outputs: the CUDA arm writes what its last timed step computed (loss, grad-norm, sampled updated
fp32 weights) as float32 / float64 .npy files within 64 MB, and the same arguments give the same outputs, so that
two builds can be compared output for output. Runs a 2-layer model of Llama-2-7B width to keep the test short."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(out_dir, steps):
    cmd = [sys.executable, "bench.py", "--gpus", "1", "--steps", str(steps), "--warmup", "1", "--layers", "2",
           "--per-device-batch", "1", "--micro-batch", "1", "--no-cpu", "--no-decode", "--dump-outputs", str(out_dir)]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-1500:]
    assert json.loads(p.stdout)["steps"] == steps
    return {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_dump_outputs_are_reproducible_and_follow_steps(tmp_path):
    a = _run(tmp_path / "a", 2)
    b = _run(tmp_path / "b", 2)
    one = _run(tmp_path / "one", 1)
    assert {"loss", "grad_norm", "model.embed_tokens.weight", "lm_head.weight", "model.norm.weight",
            "model.layers.0.mlp.down_proj.weight", "model.layers.1.self_attn.q_proj.weight"} <= set(a)
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert np.isfinite(float(a["loss"])) and float(a["grad_norm"]) > 0
    assert set(a) == set(b) == set(one)
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    # one timed step fewer: the weights were updated one step fewer
    assert not np.array_equal(a["model.layers.0.mlp.down_proj.weight"], one["model.layers.0.mlp.down_proj.weight"])
