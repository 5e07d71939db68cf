"""The CUDA path against the committed golden fixtures (tests/golden/*.npz), i.e. against outputs of the reference's OWN code
(tests/golden/make_golden.py ran the reference's modules/utils.py, the mask statements of main.py:183-195 and eval.py's
``evaluate`` from a checkout of the reference project, which this repository does not contain).  The other GPU tests compare with the oracle, which
tests/test_oracle.py holds to the same fixtures; here the fixtures are the checker directly.

hoploop_*.npz  one batch of the hop loop through the drop-in callables (grapes_b200.utils): CSR, get_neighborhoods, mask dedup,
               TensorMap, sample_neighborhoods_from_probs given the reference's Gumbel noise, slice_adjacency -- integer outputs
               bit-exact, log-probs / statistics at 1e-5 / 1e-4.
eval_*.npz     grapes_b200.eval.evaluate (full-batch and mini-batch on the engine) with the fixture's weights: logits at 1e-5 of
               the reference run's fp32 logits, scores equal up to argmax flips of near-tied rows.

This file sorts last on purpose: it was written after the round's GPU budget was spent.  Every device call below follows the
usage of an older, GPU-verified test, and both test bodies were dry-run on the CPU with the oracle's functions standing in for
the device calls (fixture keys, shapes, index handling and the assertions themselves are exercised that way)."""
import glob
import os
import types

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _t(a):
    return torch.from_numpy(np.asarray(a))


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "hoploop_*.npz"))))
def test_hop_loop_callables_against_reference_golden(cuda_device, path):
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.utils import TensorMap, get_neighborhoods, sample_neighborhoods_from_probs, slice_adjacency
    dev = cuda_device
    z = np.load(path)
    N, k, hops = int(z["N"]), int(z["k"]), int(z["hops"])
    g = DeviceGraph.from_edge_index(_t(z["edge_index"]), N, device=dev)                 # main.py:134-136
    assert np.array_equal(g.indptr.cpu().numpy(), z["csr_indptr"].astype(np.int64))
    assert np.array_equal(g.indices.cpu().numpy(), z["csr_indices"].astype(np.int32))
    target = _t(z["target_nodes"])
    node_map = TensorMap(size=N, device=dev)
    prev = target.clone()
    all_mask = torch.zeros(N, dtype=torch.bool, device=dev)
    all_mask[target.to(dev)] = True
    for hop in range(hops):
        p = f"hop{hop}_"
        assert torch.equal(prev, _t(z[p + "prev"]))
        nb = get_neighborhoods(prev, g)                                                  # utils.py:74-82
        assert nb.device == prev.device                                                  # host ids in -> host ids out
        assert torch.equal(nb.cpu(), _t(z[p + "neighborhoods"])), f"hop {hop}: neighborhoods"
        nb = nb.to(dev)
        pm = torch.zeros(N, dtype=torch.bool, device=dev)
        bm = torch.zeros(N, dtype=torch.bool, device=dev)
        pm[prev.to(dev)] = True                                                          # main.py:183-190
        bm[nb.view(-1)] = True
        batch_nodes = node_map.values[bm]
        neighbor_nodes = node_map.values[bm & ~pm]
        assert torch.equal(batch_nodes.cpu(), _t(z[p + "batch_nodes"])), f"hop {hop}: batch_nodes"
        assert torch.equal(neighbor_nodes.cpu(), _t(z[p + "neighbor_nodes"])), f"hop {hop}: neighbor_nodes"
        node_map.update(batch_nodes)                                                     # utils.py:98-120
        assert torch.equal(node_map.map(nb).cpu(), _t(z[p + "local_neighborhoods"])), f"hop {hop}: TensorMap"
        logits = _t(z[p + "logits"])
        noise = _t(z[p + "gumbel"]) if z[p + "gumbel"].size else None                     # empty: k >= n, nothing was drawn
        nbc = neighbor_nodes.cpu()
        if noise is not None:
            sampled, lp, stats = sample_neighborhoods_from_probs(logits.to(dev), nbc, k, gumbel_noise=noise)
        else:
            sampled, lp, stats = sample_neighborhoods_from_probs(logits.to(dev), nbc, k)
        assert torch.equal(sampled.cpu(), _t(z[p + "sampled"])), f"hop {hop}: sampled set"
        torch.testing.assert_close(lp.detach().cpu(), _t(z[p + "log_prob"]), rtol=1e-5, atol=1e-6)
        ref_stats = z[p + "stats"]
        if ref_stats.size:
            for i, key in enumerate(("min_prob", "max_prob", "mean_entropy", "std_entropy")):
                assert abs(float(stats[key]) - float(ref_stats[i])) <= 1e-4 * max(1.0, abs(float(ref_stats[i]))), key
        else:
            assert stats == {}
        all_mask[sampled.to(dev)] = True
        nxt = torch.cat([target, sampled.cpu()])
        blk = slice_adjacency(g, nxt, prev)                                              # utils.py:85-95, main.py:241
        assert torch.equal(blk.cpu(), _t(z[p + "block_edges"])), f"hop {hop}: block"
        prev = nxt
    all_nodes = node_map.values[all_mask]                                                # main.py:252-253
    node_map.update(all_nodes)
    assert torch.equal(all_nodes.cpu(), _t(z["all_nodes"]))
    assert torch.equal(node_map.map(target).cpu(), _t(z["local_target_ids"]))


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "eval_*.npz"))))
def test_evaluate_against_reference_golden(cuda_device, path):
    from grapes_b200.eval import evaluate
    from grapes_b200.gcn import GCN
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import make_synth
    dev = cuda_device
    z = np.load(path)
    name, seed, B, k, hops = str(z["name"]), int(z["seed"]), int(z["B"]), int(z["k"]), int(z["hops"])
    d = make_synth(name, seed=seed)
    mask = _t(z["mask"])
    assert torch.equal(mask, d.test_mask)
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    num_ind = hops + 1
    gcn_c = GCN(d.num_features, [256, d.num_classes]).to(dev)
    gcn_c.load_state_dict({n: _t(z[f"w_gcn_c.{n}"]).float() for n in gcn_c.state_dict()})
    gcn_gf = GCN(d.num_features + num_ind, [256, 1]).to(dev)
    gcn_gf.load_state_dict({n: _t(z[f"w_gcn_gf.{n}"]).float() for n in gcn_gf.state_dict()})
    args = types.SimpleNamespace(sampling_hops=hops, num_samples=k, use_indicators=True)
    n_eval = max(int(mask.sum()), 1)
    # ---- full batch (eval.py:47-70) ----
    ref = _t(z["full_logits"]).double()
    acc, f1, logits = evaluate(gcn_c, gcn_gf, d, args, g, None, num_ind, dev, mask=mask, full_batch=True,
                               return_predictions=True)
    err = ((logits.double().cpu() - ref).abs().max() / ref.abs().max()).item()
    assert err < 1e-5, f"full-batch logits: {err:.3e}"
    top2 = ref[mask].topk(2, dim=1).values
    unsafe = int(((top2[:, 0] - top2[:, 1]) <= 1e-4 * ref.abs().max()).sum())          # rows whose argmax fp32 rounding may flip
    assert abs(acc - float(z["full_accuracy"])) <= unsafe / n_eval + 1e-6 and acc == f1
    # ---- mini batch on the engine (eval.py:71-163) ----
    idx = mask.nonzero().squeeze(1)
    loader = [(b,) for b in torch.split(idx, B)]
    assert len(loader) == int(z["mini_batches"])
    acc_m, f1_m, pred = evaluate(gcn_c, gcn_gf, d, args, g, None, num_ind, dev, mask=mask, loader=loader,
                                 full_batch=False, return_predictions=True)
    assert pred.numel() == idx.numel() and acc_m == f1_m
    assert abs(acc_m - float(z["mini_accuracy"])) <= 1.0 / n_eval + 1e-6
