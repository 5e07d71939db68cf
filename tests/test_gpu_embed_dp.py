"""Data parallelism with learned node features (``--embed_nodes`` under torchrun; /root/reference/main.py:89-100,116):
row-sparse exchange of the table gradient and the same dense table Adam on every rank.  Needs >= 2 GPUs on the box."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_embed_data_parallel_matches_oracle_and_one_gpu(cuda_device):
    """scripts/check_dp_embed.py under torchrun, both exchanges: first-step union rows and mean table gradient against
    the float64 oracle, three steps against the data-parallel oracle, bit-identical table / moments / parameters across
    ranks (eager and graph replay), bit-identical to one GPU when both ranks run the same batches, a failed peer exchange
    leaves everything untouched, peer vs NCCL within the sign-flip bound, and train() end to end."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29547", os.path.join(ROOT, "scripts", "check_dp_embed.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-6000:] + res.stderr[-3000:]
    assert "dp embed ok" in res.stdout
