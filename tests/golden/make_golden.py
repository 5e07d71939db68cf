"""Generates the golden fixtures in this directory FROM THE REFERENCE ITSELF: imports the reference's
modules/utils.py (through the scipy tensor-index shim of oracle/ref_import.py) and runs
its own get_neighborhoods / slice_adjacency / TensorMap / sample_neighborhoods_from_probs and the mask
dedup statements of main.py:183-195 on seeded synthetic graphs; and the reference's eval.py ``evaluate``
(full-batch and mini-batch) for the eval_*.npz fixtures and its main.py ``train`` for train_*.npz.  Needs a checkout of
the reference GRAPES project, which this repository does not contain; the .npz outputs are committed.

    GRAPES_REFERENCE_ROOT=<reference checkout> python tests/golden/make_golden.py
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from grapes_b200.synth import make_synth            # noqa: E402
from oracle import ref_import                       # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
CASES = [("tiny", 0, 32, 8, 2), ("tiny", 1, 50, 4, 3), ("cora", 0, 512, 16, 2)]


def main():
    ru = ref_import.load_reference_utils()
    for name, seed, B, k, hops in CASES:
        d = make_synth(name, seed=seed)
        N = d.num_nodes
        adj = ref_import.reference_adjacency(d.edge_index, N)
        train_idx = d.train_mask.nonzero().squeeze(1)
        target_nodes = train_idx[:B]
        out = {"N": N, "edge_index": d.edge_index.numpy(), "target_nodes": target_nodes.numpy(), "k": k, "hops": hops,
               "csr_indptr": adj.m.indptr.astype(np.int64), "csr_indices": adj.m.indices.astype(np.int64)}
        # ---- the hop loop's integer statements, verbatim from main.py:161-247 with random-but-seeded logits
        node_map = ru.TensorMap(size=N)
        prev_nodes_mask = torch.zeros(N, dtype=torch.bool)
        batch_nodes_mask = torch.zeros(N, dtype=torch.bool)
        previous_nodes = target_nodes.clone()
        all_nodes_mask = torch.zeros_like(prev_nodes_mask)
        all_nodes_mask[target_nodes] = True
        g = torch.Generator().manual_seed(seed + 77)
        for hop in range(hops):
            neighborhoods = ru.get_neighborhoods(previous_nodes, adj)
            prev_nodes_mask.zero_(); batch_nodes_mask.zero_()
            prev_nodes_mask[previous_nodes] = True
            batch_nodes_mask[neighborhoods.view(-1)] = True
            neighbor_nodes_mask = batch_nodes_mask & ~prev_nodes_mask
            batch_nodes = node_map.values[batch_nodes_mask]
            neighbor_nodes = node_map.values[neighbor_nodes_mask]
            node_map.update(batch_nodes)
            local_neighborhoods = node_map.map(neighborhoods)
            logits = torch.randn(neighbor_nodes.shape[0], 1, generator=g) * 2
            torch.manual_seed(1000 * seed + hop)                  # seeds the Gumbel draw at utils.py:40-41
            sampled, log_prob, stats = ru.sample_neighborhoods_from_probs(logits, neighbor_nodes, k)
            torch.manual_seed(1000 * seed + hop)                  # re-draw the identical noise to store it
            fi = torch.finfo(torch.float32)
            n = neighbor_nodes.shape[0]
            noise = np.zeros(0, np.float32)
            if k < n:
                from torch.distributions import Gumbel
                noise = Gumbel(torch.tensor(0.), torch.tensor(1.)).sample((n,)).numpy()
            all_nodes_mask[sampled] = True
            batch_next = torch.cat([target_nodes, sampled], dim=0)
            k_hop_edges = ru.slice_adjacency(adj, rows=batch_next, cols=previous_nodes)
            p = f"hop{hop}_"
            out.update({p + "prev": previous_nodes.numpy(), p + "neighborhoods": neighborhoods.numpy(),
                        p + "batch_nodes": batch_nodes.numpy(), p + "neighbor_nodes": neighbor_nodes.numpy(),
                        p + "local_neighborhoods": local_neighborhoods.numpy(), p + "logits": logits.numpy(),
                        p + "gumbel": noise, p + "sampled": sampled.numpy(), p + "log_prob": log_prob.numpy(),
                        p + "stats": np.array([float(stats[s]) for s in ("min_prob", "max_prob", "mean_entropy", "std_entropy")]
                                              if stats else [], np.float64),
                        p + "block_edges": k_hop_edges.numpy()})
            previous_nodes = batch_next.clone()
        all_nodes = node_map.values[all_nodes_mask]
        node_map.update(all_nodes)
        out["all_nodes"] = all_nodes.numpy()
        out["local_target_ids"] = node_map.map(target_nodes).numpy()
        path = os.path.join(HERE, f"hoploop_{name}_s{seed}.npz")
        np.savez_compressed(path, **out)
        print("wrote", path, os.path.getsize(path), "bytes")
    # TensorMap docstring vector (utils.py:104-108)
    nodes = torch.tensor([22, 32, 42, 52])
    tm = ru.TensorMap(size=nodes.max() + 1)
    tm.update(nodes)
    np.savez(os.path.join(HERE, "tensormap_docstring.npz"), keys=np.array([52, 42, 32, 22, 22]),
             mapped=tm.map(torch.tensor([52, 42, 32, 22, 22])).numpy())


EVAL_CASES = [("tiny", 0, 32, 8, 2), ("tiny", 2, 50, 4, 3), ("small", 1, 256, 64, 2)]


def main_eval():
    """eval_*.npz: the reference's OWN ``evaluate`` (eval.py:11-165, imported live) run full-batch and mini-batch on seeded
    synthetic graphs with seeded models; what it handed to / got from ``gcn_c`` is recorded per batch (the blocks the
    evaluation hop loop built, the logits) next to the (accuracy, f1) it returned.  The models are the oracle's GCN restatement
    (PyG is absent here): the fixture pins the evaluation LOOP -- deterministic top-k selection, evaluation-direction block
    slice, relabelling, batching, scores -- not GCNConv."""
    import argparse
    from oracle import reference_port as rp
    mod, ru = ref_import.load_reference_eval()
    for name, seed, B, k, hops in EVAL_CASES:
        d = make_synth(name, seed=seed)
        st = rp.OracleState(d, sampling_hops=hops, num_samples=k, seed=seed + 5, dtype=torch.float32)
        st.gcn_c.eval(); st.gcn_gf.eval()
        args = argparse.Namespace(sampling_hops=hops, use_indicators=True, num_samples=k)
        adj = ref_import.reference_adjacency(d.edge_index, d.num_nodes)
        mask = d.test_mask
        out = {"name": name, "seed": seed, "B": B, "k": k, "hops": hops, "mask": mask.numpy()}
        for key, net in (("gcn_c", st.gcn_c), ("gcn_gf", st.gcn_gf)):
            for n, t in net.state_dict().items():
                out[f"w_{key}.{n}"] = t.numpy()
        for full in (True, False):
            node_map = ru.TensorMap(size=d.num_nodes)
            loader = torch.utils.data.DataLoader(torch.utils.data.TensorDataset(mask.nonzero().squeeze(1)), batch_size=B)
            rc, rg = ref_import.RecordingModule(st.gcn_c), ref_import.RecordingModule(st.gcn_gf)
            acc, f1 = mod.evaluate(rc, rg, d, args, adj, node_map, hops + 1, torch.device("cpu"), mask=mask,
                                   eval_on_cpu=True, loader=loader, full_batch=full)
            tag = "full_" if full else "mini_"
            out[tag + "accuracy"], out[tag + "f1"] = acc, f1
            if full:
                out["full_logits"] = rc.calls[0]["logits"].numpy()
            else:
                out["mini_batches"] = len(rc.calls)
                for b, c in enumerate(rc.calls):
                    out[f"mini_b{b}_logits"] = c["logits"].numpy()
                    for h, e in enumerate(c["edge_index"]):
                        out[f"mini_b{b}_edges{h}"] = e.numpy()            # local ids, evaluation direction (eval.py:140-142,150)
        path = os.path.join(HERE, f"eval_{name}_s{seed}.npz")
        np.savez_compressed(path, **out)
        print("wrote", path, os.path.getsize(path), "bytes")


TRAIN_CASES = {                     # name -> (graph, seed, batch, k, hops, data overrides, argument overrides)
    "tb":        ("tiny", 0, 32, 8, 2, {}, {}),
    "reinforce": ("tiny", 1, 50, 4, 3, {}, {"reinforce_baseline": True}),
    "random":    ("tiny", 2, 32, 8, 2, {}, {"random_sampling": True}),
    "reg_logz":  ("tiny", 3, 40, 6, 2, {}, {"reg_param": 0.1, "log_z_init": 0.7, "loss_coef": 100.0}),
    "multilabel": ("tiny", 4, 32, 8, 2, {"multilabel": True}, {}),
}


def main_train():
    """train_*.npz: the reference's OWN ``train(args)`` (main.py:57-340, executed live through
    oracle/ref_import.py::load_reference_train) for one epoch on seeded synthetic graphs: every batch's loss_c / loss_gfn /
    log_z / sum of log-probs as train() logged them, the weights of gcn_c / gcn_gf / gcn_z after the epoch, the test score.
    GCN modules: the oracle's restatement (PyG is absent); global RNG seeded right before the call; one CPU thread."""
    import json
    torch.set_num_threads(1)
    for case, (name, seed, B, k, hops, dover, over) in TRAIN_CASES.items():
        d = make_synth(name, seed=seed, **dover)
        test_f1, logs, nets = ref_import.run_reference_train(d, weight_seed=seed + 100, rng_seed=4242 + seed, batch_size=B,
                                                             num_samples=k, sampling_hops=hops, **over)
        out = {"case": case, "name": name, "seed": seed, "B": B, "k": k, "hops": hops,
               "data_overrides": json.dumps(dover), "arg_overrides": json.dumps(over), "test_f1": test_f1,
               "loss_c": np.array([l["batch_loss_c"] for l in logs], np.float64),
               "loss_gfn": np.array([float(l["batch_loss_gfn"]) for l in logs], np.float64),
               "log_z": np.array([float(l["log_z"].detach()) for l in logs], np.float64),
               "neg_log_probs": np.array([float(l["-log_probs"].detach()) for l in logs], np.float64)}
        for key, net in zip(("gcn_c", "gcn_gf", "gcn_z"), nets):
            for n, p in net.named_parameters():
                out[f"w_{key}.{n}"] = p.detach().numpy()
        path = os.path.join(HERE, f"train_{case}.npz")
        np.savez_compressed(path, **out)
        print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    if not ref_import.reference_available():
        sys.exit("make_golden.py: set GRAPES_REFERENCE_ROOT to a checkout of the reference GRAPES project")
    main()
    main_eval()
    main_train()
