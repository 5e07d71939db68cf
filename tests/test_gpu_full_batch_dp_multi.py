"""Data-parallel full-graph training across two processes and GPUs (``full_batch.train(..., group=...)``, the backward's
transposed aggregations over NVLink peer memory): scripts/check_dp_full_batch.py under torchrun.  Needs >= 2 GPUs."""
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_data_parallel_full_batch_training(cuda_device):
    """Parameters bit-identical across ranks after every epoch and to the emulated two-rank run, test F1 equal to one
    process's evaluate(), the window structure built once, an unmappable row table refused on both ranks."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29557", os.path.join(ROOT, "scripts", "check_dp_full_batch.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-6000:] + res.stderr[-3000:]
    assert "dp full batch ok" in res.stdout
