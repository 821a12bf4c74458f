"""bench.py --dump-outputs on a small workload: the last timed step's rollout buffer, parameters and update statistics
come out as float .npy files within 64 MB, and two runs with the same arguments, or with one more timed step, write
the same arrays (the update's to rounding)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROLLOUT = ("obs", "actions", "rewards", "episode_starts", "values", "log_probs", "advantages", "returns")


def _bench(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
           "--envs-per-gpu", "256", "--n-steps", "32", "--batch", "1024", "--no-cpu-baseline", "--no-extras",
           "--dump-outputs", str(out_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    return {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_dump_outputs_are_reproducible(cuda_lib, tmp_path):
    a = _bench(tmp_path / "a", 2)
    assert set(a) == {f"rollout_{k}" for k in ROLLOUT} | {"policy_params", "train_stats", "sample_env_index"}
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert a["rollout_obs"].shape == (32, 256, 14) and a["rollout_actions"].shape == (32, 256, 2)
    assert np.array_equal(a["sample_env_index"], np.arange(256))
    assert np.isfinite(a["policy_params"]).all() and np.abs(a["rollout_advantages"]).max() > 0

    # every timed step starts from the seeded state the model was built in: the rollout is the same bit for bit;
    # the update adds the CTAs' partial gradients in L2 in no fixed order, so its outputs agree to rounding
    b = _bench(tmp_path / "b", 2)
    for k in a:
        if k in ("policy_params", "train_stats"):
            np.testing.assert_allclose(b[k], a[k], rtol=1e-4, atol=1e-5, err_msg=k)
        else:
            np.testing.assert_array_equal(b[k], a[k], err_msg=k)

    # ... and a third timed step computes what the second one did
    c = _bench(tmp_path / "c", 3)
    np.testing.assert_array_equal(c["rollout_obs"], a["rollout_obs"])
    np.testing.assert_allclose(c["policy_params"], a["policy_params"], rtol=1e-4, atol=1e-5)
