"""Data parallelism with dropout in the classifier GCN (``--dropout`` under torchrun): per-rank masks, the mean of the
ranks' masked gradients, identical replicas.  Needs >= 2 GPUs on the box."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dropout_data_parallel_matches_oracle(cuda_device):
    """scripts/check_dp_dropout.py under torchrun, both exchanges, with and without --embed_nodes: each rank's masks equal
    the numpy restatement for its rank and differ across ranks; the exchanged gradient equals the mean of the ranks'
    float64 oracle gradients taken through their own masks; replicas bit-identical after eager and graph-replayed steps."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29551", os.path.join(ROOT, "scripts", "check_dp_dropout.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-6000:] + res.stderr[-3000:]
    assert "dp dropout ok" in res.stdout
