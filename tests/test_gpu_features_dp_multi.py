"""A feature table sharded across two processes and GPUs (``train(shard_features=True)``, rows gathered over NVLink peer
memory): scripts/check_dp_features.py under torchrun.  Needs >= 2 GPUs on the box."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sharded_features_match_replicated(cuda_device):
    """Shards hold their rows and ~1/W of the bytes; full-batch (F <= D, F > D, bf16) and mini-batch scores equal the
    replicated evaluation; train() with and without shard_features gives bit-identical parameters and the same scores;
    an allocation failure on one rank raises on every rank."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29553", os.path.join(ROOT, "scripts", "check_dp_features.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-6000:] + res.stderr[-3000:]
    assert "dp features ok" in res.stdout
