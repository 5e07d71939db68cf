"""CLI with the reference's behaviour (/root/reference/main.py:367-390):
``python -m grapes_b200.main --config_file configs/gflownet/cora.txt [--flag value ...]``.

``GRAPES_CHECKPOINT_DIR=<dir>`` (the ``Arguments`` stay the reference's): run r of ``--runs`` writes a checkpoint into
``<dir>/run<r>`` at the end of every epoch and, when that directory holds a complete checkpoint, resumes from it."""
import os

import numpy as np
import torch

from .args import parse_cli
from .train import train


def main(argv=None):
    args = parse_cli(argv)
    results = torch.empty(args.runs)
    mem1, mem2, mem3 = [], [], []
    ckpt = os.environ.get("GRAPES_CHECKPOINT_DIR")
    for r in range(args.runs):
        kw = dict(checkpoint_dir=os.path.join(ckpt, f"run{r}"), resume=True) if ckpt else {}
        test_f1, m1, m2, m3 = train(args, **kw)
        results[r] = test_f1
        mem1.extend(m1); mem2.extend(m2); mem3.extend(m3)
    print(f'Memory point 1: {np.mean(mem1)} MB ± {np.std(mem1):.2f}')
    print(f'Memory point 2: {np.mean(mem2)} MB ± {np.std(mem2):.2f}')
    print(f'Memory point 2: {np.mean(mem3)} MB ± {np.std(mem3):.2f}')
    print(f'Acc: {100 * results.mean():.2f} ± {100 * results.std():.2f}')


if __name__ == "__main__":
    main()
