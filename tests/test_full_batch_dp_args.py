"""CPU tests of the data-parallel full-graph training driver (grapes_b200.full_batch): the per-rank working-set
estimate, the refusals decided from the arguments alone, the window loss shares and the rank-order reduction."""
import pytest
import torch


def test_per_rank_working_set():
    """Arithmetic only: the papers100M shape (bf16 table as stored) fits a 180 GB device per rank at W = 8, not at
    W = 1; W = 1 keeps the one-GPU estimate."""
    from grapes_b200.full_batch import working_set_bytes
    from grapes_b200.synth import SHAPES
    s = SHAPES["papers"]
    args = (s["N"], s["E_dir"], s["F"], 256, s["C"])
    assert working_set_bytes(*args, world=8, x_itemsize=2) < 180e9
    assert working_set_bytes(*args, world=1, x_itemsize=2) > 180e9
    assert working_set_bytes(*args, world=1) == working_set_bytes(*args)
    per = [working_set_bytes(*args, world=W, x_itemsize=2) for W in (2, 4, 8)]
    assert per[0] > per[1] > per[2]
    c = SHAPES["cora"]                                   # F > D: the [N, D] product P on every rank is counted
    assert working_set_bytes(c["N"], c["E_dir"], c["F"], 64, c["C"], world=2) > \
        working_set_bytes(c["N"], c["E_dir"], 32, 64, c["C"], world=2)


def test_refusal_reasons():
    from grapes_b200.args import Arguments
    from grapes_b200.full_batch import data_parallel_refusal
    from grapes_b200.synth import make_synth
    d = make_synth("tiny", seed=0)
    assert data_parallel_refusal(Arguments(hidden_dim=16), d, d.num_classes) is None
    assert "embed_nodes" in data_parallel_refusal(Arguments(hidden_dim=16, embed_nodes=True), d, d.num_classes)
    assert "dropout" in data_parallel_refusal(Arguments(hidden_dim=16, dropout=0.1), d, d.num_classes)
    assert "hidden width" in data_parallel_refusal(Arguments(hidden_dim=d.num_classes), d, d.num_classes)
    d.x = d.x.double()
    assert "fp32 or bf16" in data_parallel_refusal(Arguments(hidden_dim=16), d, d.num_classes)


def test_one_gpu_refusal_names_the_data_parallel_form(monkeypatch):
    from grapes_b200 import full_batch as fb
    from grapes_b200._lib import GrapesError
    from grapes_b200.args import Arguments
    monkeypatch.setenv("WORLD_SIZE", "2")
    with pytest.raises(GrapesError, match="group="):
        fb.train(Arguments(dataset="synth:tiny"))


@pytest.mark.parametrize("multilabel", [False, True])
@pytest.mark.parametrize("reg_param", [0., 1e-2])
def test_window_losses_add_up_to_the_classifier_loss(multilabel, reg_param):
    from grapes_b200.full_batch import classifier_loss, window_loss
    gen = torch.Generator().manual_seed(1)
    N, C = 97, 5
    logits = torch.randn(N, C, generator=gen, dtype=torch.float64)
    y = (torch.rand(N, C, generator=gen) < 0.3).double() if multilabel else torch.randint(0, C, (N,), generator=gen)
    mask = torch.rand(N, generator=gen) < 0.4
    whole = classifier_loss(logits, y, mask, reg_param)
    bounds = [0, 10, 10, 61, N]                                       # an empty window included
    parts = [window_loss(logits[a:b], y[a:b], mask[a:b], int(mask.sum()), reg_param) for a, b in zip(bounds, bounds[1:])]
    assert torch.allclose(sum(parts), whole, rtol=1e-12, atol=0)


def test_sum_in_rank_order():
    from grapes_b200.full_batch import sum_in_rank_order
    parts = [torch.tensor([1e8, 1.], dtype=torch.float32), torch.tensor([-1e8, 1.]), torch.tensor([1., 1.])]
    got = sum_in_rank_order(parts)
    assert torch.equal(got, (parts[0] + parts[1]) + parts[2])
    assert torch.equal(parts[0], torch.tensor([1e8, 1.]))                # the inputs are left as they were
