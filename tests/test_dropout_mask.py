"""CPU tests (no GPU): the numpy restatement of the engine's dropout masks (tests/dropout_utils.py) and the replay of
given masks inside the CPU oracle, which the GPU parity tests of dropout rest on."""
import numpy as np
import pytest
import torch

from dropout_utils import keep_mask, philox4x32_10, replay_masks, tag, threshold
from grapes_b200.synth import make_synth
from oracle import ref_import
from oracle import reference_port as rp

needs_reference = pytest.mark.skipif(not ref_import.reference_available(),
                                     reason="needs GRAPES_REFERENCE_ROOT: a checkout of the reference GRAPES project")


@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF, 0xFFFFFFFF), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox_known_answers(ctr, key, want):
    """Random123's known-answer vectors for Philox4x32-10"""
    assert tuple(int(w) for w in philox4x32_10(ctr, key)) == want


@pytest.mark.parametrize("p", [0.1, 0.5, 0.9])
def test_keep_fraction_within_5_sigma(p):
    rows, width = 4096, 256                     # 1,048,576 entries
    k = keep_mask(12345, 7, tag(0), threshold(p), rows, width)
    n, q = k.size, 1.0 - p
    assert abs(k.sum() - n * q) < 5.0 * np.sqrt(n * q * (1 - q))


def test_masks_differ_across_step_rank_and_site():
    thr = threshold(0.5)
    base = keep_mask(3, 10, tag(0, 0), thr, 64, 47)
    for other in (keep_mask(3, 11, tag(0, 0), thr, 64, 47),          # next step
                  keep_mask(3, 10, tag(0, 1), thr, 64, 47),          # next rank
                  keep_mask(3, 10, tag(1, 0), thr, 64, 47),          # logits site
                  keep_mask(4, 10, tag(0, 0), thr, 64, 47)):         # another seed
        assert (base != other).mean() > 0.4
    assert np.array_equal(base, keep_mask(3, 10, tag(0, 0), thr, 64, 47))
    # row-major entry index: a wider site is not a reshaped narrower one, but its first row-major entries are the same
    assert np.array_equal(keep_mask(3, 10, 1, thr, 8, 4).reshape(-1), keep_mask(3, 10, 1, thr, 4, 8).reshape(-1))
    # steps beyond 2**32 use the high counter word
    assert not np.array_equal(keep_mask(3, 1 << 32, 1, thr, 64, 47), keep_mask(3, 0, 1, thr, 64, 47))


def test_threshold_edges():
    assert threshold(0.0) == 1 << 24 and threshold(1.0) == 0 and threshold(0.5) == 1 << 23
    assert keep_mask(1, 2, 1, threshold(0.0), 100, 40).all()
    assert not keep_mask(1, 2, 1, threshold(1.0), 100, 40).any()


@pytest.fixture
def single_thread():
    """one CPU thread: reductions in a fixed order, so two runs of the same arithmetic agree bit for bit"""
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(threads)


def _recorded_dropout_masks():
    """Wraps torch's dropout so each call also reports the Bernoulli draw it made (same RNG consumption, same output)."""
    real = rp.F_
    masks = []

    class _Rec:
        def __getattr__(self, name):
            return getattr(real, name)

        @staticmethod
        def dropout(x, p=0.5, training=True, inplace=False):
            if training and 0 < p < 1:
                state = torch.get_rng_state()
                masks.append(real.dropout(torch.ones_like(x), p=p, training=True) != 0)
                torch.set_rng_state(state)
            return real.dropout(x, p=p, training=training, inplace=inplace)

    return _Rec(), masks


@pytest.mark.parametrize("p,dtype", [(0.5, torch.float64), (0.1, torch.float64), (0.3, torch.float32)])
def test_replayed_masks_equal_torch_dropout(single_thread, p, dtype):
    """OracleGCN in training mode with torch's own dropout, then the same forward / backward with the masks that dropout
    drew replayed: logits and gradients equal bit for bit."""
    d = make_synth("tiny", seed=0)
    st = rp.OracleState(d, seed=100, dtype=dtype, dropout=p, hidden_dim=64)
    x = d.x.to(dtype)
    edges = [d.edge_index[:, :900], d.edge_index[:, 900:]]

    def run():
        st.gcn_c.zero_grad()
        logits, _ = st.gcn_c(x, edges)
        logits.square().sum().backward()
        return logits.detach().clone(), [q.grad.clone() for q in st.gcn_c.parameters()]

    rec, masks = _recorded_dropout_masks()
    real = rp.F_
    torch.manual_seed(9)
    rp.F_ = rec
    try:
        want, want_g = run()
    finally:
        rp.F_ = real
    assert len(masks) == 2 and 0 < masks[0].float().mean() < 1
    with replay_masks(lambda site, shape: masks[site]):
        got, got_g = run()
    assert torch.equal(got, want)
    assert all(torch.equal(a, b) for a, b in zip(got_g, want_g))
    # without the block the oracle is torch's dropout again
    assert rp.F_ is real


def test_replay_at_p_one_gives_zeros():
    d = make_synth("tiny", seed=0)
    st = rp.OracleState(d, seed=100, dtype=torch.float64, dropout=1.0, hidden_dim=32)
    with replay_masks(lambda site, shape: torch.ones(shape, dtype=torch.bool)):
        logits, _ = st.gcn_c(d.x.double(), d.edge_index)
    assert torch.equal(logits, torch.zeros_like(logits))


@needs_reference
def test_oracle_dropout_matches_live_reference_train(single_thread):
    """The reference's own ``train(args)`` with ``dropout=0.5`` against the oracle's batch loop over one epoch, both
    consuming the global RNG in the same order (DataLoader seed, Gumbel draws, dropout draws): every batch's loss_c /
    loss_gfn bit for bit and the weights after the epoch to 1e-7.  Training quantities only: whether the reference
    evaluates in training mode is not compared (the product evaluates without dropout)."""
    d = make_synth("tiny", seed=5)
    B, k, hops, seed, rng_seed = 32, 8, 2, 5, 4247
    _, logs, nets = ref_import.run_reference_train(d, weight_seed=seed + 100, rng_seed=rng_seed, batch_size=B,
                                                   num_samples=k, sampling_hops=hops, dropout=0.5)
    st = rp.OracleState(d, sampling_hops=hops, num_samples=k, seed=seed + 100, dtype=torch.float32, dropout=0.5)
    torch.manual_seed(rng_seed)
    tr = d.train_mask.nonzero().squeeze(1)
    recs = [rp.reference_step(st, b[0], stable_ties=False)
            for b in torch.utils.data.DataLoader(torch.utils.data.TensorDataset(tr), batch_size=B)]
    assert len(recs) == len(logs) >= 2
    for r, l in zip(recs, logs):
        assert float(r["loss_c"]) == l["batch_loss_c"]
        assert float(r["loss_gfn"]) == float(l["batch_loss_gfn"])
    for key, net, mine in zip(("gcn_c", "gcn_gf", "gcn_z"), nets, (st.gcn_c, st.gcn_gf, st.gcn_z)):
        for (n, a), (_, b) in zip(net.named_parameters(), mine.named_parameters()):
            assert torch.allclose(b, a, rtol=0, atol=1e-7 * float(a.abs().max())), f"{key}.{n}"
