"""Checkpoint and resume of data-parallel train() on two processes and GPUs: scripts/check_dp_checkpoint.py under
torchrun.  Needs >= 2 GPUs on the box."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dp_resume_is_bit_identical(cuda_device):
    """Both exchanges, replicated and sharded learned table: an interrupted and resumed train() equals an uninterrupted
    one on both ranks; a W = 2 sharded checkpoint evaluated by one process gives the W = 2 scores."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29567", os.path.join(ROOT, "scripts", "check_dp_checkpoint.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=1800)
    assert res.returncode == 0, res.stdout[-6000:] + res.stderr[-3000:]
    assert "dp checkpoint ok" in res.stdout
