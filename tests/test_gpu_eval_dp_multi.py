"""Data-parallel evaluation across two processes and GPUs (``evaluate(..., group=...)``, layer 2 over NVLink peer memory):
scripts/check_dp_eval.py under torchrun.  Needs >= 2 GPUs on the box."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_data_parallel_evaluation_matches_one_gpu(cuda_device):
    """Full-batch and mini-batch scores equal one-GPU evaluate(), window logits bit-identical, mini-batch predictions
    reassembled, a forced mapping failure on one rank falls back on every rank, train() the same with and without
    shard_eval."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29551", os.path.join(ROOT, "scripts", "check_dp_eval.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-6000:] + res.stderr[-3000:]
    assert "dp eval ok" in res.stdout
