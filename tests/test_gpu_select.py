"""Selection parity (SURVEY.md section 8 row a8): the sampled SET is bit-exact when the kernel is fed
the reference's keys or its logits + Gumbel noise; log-probs / stats within fp32 tolerance."""
import pytest
import torch

from oracle import reference_port as rp

pytestmark = pytest.mark.gpu
RTOL = 1e-5


def _run(logits, nb, k, dev, **kw):
    from grapes_b200.utils import sample_neighborhoods_from_probs
    return sample_neighborhoods_from_probs(logits.to(dev), nb, k, **kw)


@pytest.mark.parametrize("n,k,seed", [(1000, 16, 0), (1135, 16, 1), (63407, 256, 2), (300, 299, 3), (40000, 1, 4)])
def test_sampled_set_bit_exact_given_gumbel_noise(cuda_device, n, k, seed):
    g = torch.Generator().manual_seed(seed)
    logits = torch.randn(n, 1, generator=g) * 2
    nb = torch.sort(torch.randperm(5 * n, generator=g)[:n]).values
    noise = rp.draw_gumbel_like_reference(n, g)
    ref_nodes, ref_lp, ref_stats = rp.sample_neighborhoods_from_probs(logits, nb, k, gumbel_noise=noise)
    # the k-th / (k+1)-th key gap must exceed fp32 evaluation noise for the set to be well defined
    keys = rp.perturbed_keys(logits.squeeze(-1), noise)
    srt = torch.sort(keys, descending=True).values
    assert (srt[k - 1] - srt[k]) > 2e-6 * srt.abs().max()
    nodes, lp, stats = _run(logits, nb, k, cuda_device, gumbel_noise=noise)
    assert torch.equal(nodes.cpu(), ref_nodes)
    torch.testing.assert_close(lp.cpu(), ref_lp, rtol=RTOL, atol=1e-6)
    for key in ("min_prob", "max_prob", "mean_entropy", "std_entropy"):
        torch.testing.assert_close(stats[key].cpu(), ref_stats[key], rtol=1e-4, atol=1e-6)


def test_exact_given_keys_with_ties_lowest_index(cuda_device):
    from grapes_b200.utils import NOISE_KEYS
    n, k = 5000, 100
    g = torch.Generator().manual_seed(7)
    keys = torch.randint(0, 50, (n,), generator=g).float()            # massive ties
    keys[::97] = float("-inf")
    logits = torch.zeros(n, 1)
    nb = torch.arange(n) * 3
    nodes, _, _ = _run(logits, nb, k, cuda_device, gumbel_noise=keys, noise_mode=NOISE_KEYS)
    want = nb[torch.sort(rp.stable_topk_indices(keys, k)).values]
    assert torch.equal(nodes.cpu(), want)


def test_take_all_branch(cuda_device):
    """k >= n: every neighbour kept, log_prob = logsigmoid(logits), empty stats (utils.py:31-33)."""
    n = 37
    logits = torch.randn(n, 1, generator=torch.Generator().manual_seed(0))
    nb = torch.arange(n) * 2 + 1
    for k in (n, n + 5):
        nodes, lp, stats = _run(logits, nb, k, cuda_device)
        assert torch.equal(nodes.cpu(), nb) and stats == {}
        torch.testing.assert_close(lp.cpu(), torch.nn.functional.logsigmoid(logits.squeeze(-1)), rtol=RTOL, atol=1e-6)


def test_log_prob_gradient(cuda_device):
    n, k = 2000, 64
    g = torch.Generator().manual_seed(5)
    logits = (torch.randn(n, 1, generator=g) * 3).requires_grad_(True)
    nb = torch.arange(n)
    noise = rp.draw_gumbel_like_reference(n, g)
    _, ref_lp, _ = rp.sample_neighborhoods_from_probs(logits, nb, k, gumbel_noise=noise)
    ref_lp.sum().backward()
    lg = logits.detach().to(cuda_device).requires_grad_(True)
    from grapes_b200.utils import sample_neighborhoods_from_probs
    _, lp, _ = sample_neighborhoods_from_probs(lg, nb, k, gumbel_noise=noise)
    lp.sum().backward()
    torch.testing.assert_close(lg.grad.cpu(), logits.grad, rtol=RTOL, atol=1e-6)


def test_philox_sampler_is_uniform_when_logits_constant(cuda_device):
    """random_sampling=True: constant logits 100 -> uniform k-subsets (main.py:207).  Property test at
    a size no oracle loop is needed for: each node's inclusion frequency ~ k/n."""
    from grapes_b200.utils import sample_neighborhoods_from_probs
    n, k, trials = 512, 64, 400
    logits = torch.full((n, 1), 100.0, device=cuda_device)
    nb = torch.arange(n)
    hits = torch.zeros(n)
    rng = torch.tensor([1234, 0], dtype=torch.int64, device=cuda_device)
    for _ in range(trials):
        nodes, _, _ = sample_neighborhoods_from_probs(logits, nb, k, rng_state=rng)
        assert nodes.numel() == k and torch.all(nodes[1:] > nodes[:-1])
        hits[nodes.cpu()] += 1
    freq = hits / trials
    assert abs(freq.mean().item() - k / n) < 1e-6
    assert freq.min() > 0.04 and freq.max() < 0.25          # k/n = 0.125, sd ~ 0.0165


def _check_log_probs_and_stats(logits, nb, k, nodes, lp, stats):
    """Log-probs against the float64 Bernoulli log-probability of the selected mask (utils.py:71); statistics against
    the oracle's, which depend only on the logits."""
    mask = torch.isin(nb, nodes.cpu()).double()
    ref_lp = -torch.nn.functional.binary_cross_entropy_with_logits(logits.squeeze(-1).double(), mask, reduction="none")
    torch.testing.assert_close(lp.cpu(), ref_lp.float(), rtol=RTOL, atol=1e-6)
    _, _, ref_stats = rp.sample_neighborhoods_from_probs(logits, nb, k, gumbel_noise=torch.zeros(nb.numel()))
    assert stats.keys() == ref_stats.keys()
    for key in ref_stats:
        torch.testing.assert_close(stats[key].cpu(), ref_stats[key], rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("n,k,levels", [(40000, 1000, 1), (70001, 256, 3), (9000, 8999, 2), (150000, 256, 100000)])
def test_crowded_threshold_bucket_matches_oracle(cuda_device, n, k, levels):
    """Massive ties (few distinct keys, so the threshold bucket holds far more members than the on-chip list): the
    radix-select fallback finds the exact threshold; ties go to the LOWEST candidate index.  Log-probs and statistics
    match the oracle."""
    from grapes_b200.utils import NOISE_KEYS
    g = torch.Generator().manual_seed(n + k)
    keys = torch.randint(0, levels, (n,), generator=g).float() * 0.25 - 3.0
    logits = torch.randn(n, 1, generator=g)
    nb = torch.arange(n) * 2 + 1
    want = nb[torch.sort(rp.stable_topk_indices(keys, k)).values]
    nodes, lp, stats = _run(logits, nb, k, cuda_device, gumbel_noise=keys, noise_mode=NOISE_KEYS)
    assert torch.equal(nodes.cpu(), want)
    _check_log_probs_and_stats(logits, nb, k, nodes, lp, stats)


def test_selection_matches_oracle_on_gumbel_keys(cuda_device):
    """Gumbel noise in -> the oracle's sampled set, log-probs and statistics, at the frontier sizes of the BASELINE
    shapes (products ~65 k, Reddit ~150 k candidates) and at sizes around the block boundaries."""
    for n, k in ((65000, 256), (150000, 256), (511, 16), (513, 16), (75777, 256), (1, 1), (2, 1)):
        g = torch.Generator().manual_seed(n)
        logits = torch.randn(n, 1, generator=g) * 2
        nb = torch.sort(torch.randperm(3 * n, generator=g)[:n]).values
        noise = rp.draw_gumbel_like_reference(n, g)
        nodes, lp, stats = _run(logits, nb, k, cuda_device, gumbel_noise=noise)
        if k < n:
            ref_nodes, _, _ = rp.sample_neighborhoods_from_probs(logits, nb, k, gumbel_noise=noise)
            keys = rp.perturbed_keys(logits.squeeze(-1), noise)
            srt = torch.sort(keys, descending=True).values
            if (srt[k - 1] - srt[k]) > 2e-6 * srt.abs().max():
                assert torch.equal(nodes.cpu(), ref_nodes), (n, k)
        _check_log_probs_and_stats(logits, nb, k, nodes, lp, stats)
