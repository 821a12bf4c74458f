"""2-GPU NCCL run: sharded update == single-GPU update (skipped on a 1-GPU box)."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sharded_update_matches_single_gpu(cuda_lib):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29511", os.path.join(ROOT, "tests", "dist_worker_gpu.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    assert "DIST_RESULT" in out.stdout and "ok=True" in out.stdout
