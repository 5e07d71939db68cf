"""A learned node-feature table sharded across two processes and GPUs (``train(shard_embeddings=True)``: each rank
updates its own rows and reads the others over NVLink peer memory): scripts/check_dp_embed_sharded.py under torchrun.
Needs >= 2 GPUs on the box."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sharded_learned_table_matches_replicated(cuda_device):
    """Both exchanges: train() with and without shard_embeddings gives bit-identical parameters, table and moments and
    the same scores, with about 1/W of the table bytes per rank; a delayed merge stays bit-identical with the epoch wait
    and differs without it; a missing epoch post is flagged and its step is not applied."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29561", os.path.join(ROOT, "scripts", "check_dp_embed_sharded.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=1200)
    assert res.returncode == 0, res.stdout[-6000:] + res.stderr[-3000:]
    assert "dp embed sharded ok" in res.stdout
