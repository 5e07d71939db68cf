"""CPU ORACLE -- TEST INFRASTRUCTURE ONLY.  Never imported by the product path.

A restatement, in numpy / scipy / CPU torch, of the GRAPES per-batch
sample -> aggregate -> train path of the reference (dfdazac/grapes):

    main.py:134-140,161-291      the batch / hop loop of ``train()``
    modules/utils.py:13-120      sample_neighborhoods_from_probs, get_neighborhoods,
                                 slice_adjacency, TensorMap
    modules/gcn.py:9-42          GCN (two GCNConv layers, tensor or per-layer list of edges)

The arithmetic of ``GCNConv`` / ``gcn_norm`` lives in a third-party dependency
that is NOT vendored in the reference tree and NOT installed here:
``torch_geometric`` pinned ``pyg=2.5.2`` (environment.yml:83).  Its published
algorithm (defaults improved=False, cached=False, add_self_loops=True,
normalize=True, bias=True, flow=source_to_target) is restated in
:func:`gcn_norm` / :func:`gcn_conv` below; the parity anchor for it is the
reference's own call sites (gcn.py:18,21,32,36) plus a dense
``D^-1/2 (A+I) D^-1/2 X W^T + b`` cross-check (tests/test_oracle.py).

Pinning status (SURVEY.md section 8c):
  * integer path (get_neighborhoods, slice_adjacency, TensorMap, mask dedup) and
    sample_neighborhoods_from_probs: PINNED against the reference's own
    ``modules/utils.py`` imported live (oracle/ref_import.py,
    tests/test_oracle.py::test_oracle_matches_live_reference) and against the committed fixtures in
    tests/golden/ produced by tests/golden/make_golden.py from that import, and
    against the only known-answer vector the reference holds (TensorMap
    docstring, utils.py:104-108).
  * evaluation (``reference_evaluate``, eval.py:11-165, full-batch and mini-batch): PINNED against the reference's
    own ``evaluate`` imported live from the reference's eval.py (oracle/ref_import.py::load_reference_eval;
    tests/test_oracle.py::test_oracle_evaluate_matches_live_reference_eval: scores equal, logits of every ``gcn_c`` call
    equal bit for bit) and against the committed tests/golden/eval_*.npz produced by that function (evaluation blocks
    bit-exact, logits, scores).  The models inside are this file's GCN restatement, so this pins the evaluation LOOP
    (deterministic top-k, evaluation-direction slice, relabelling, batching, scores), not GCNConv.
  * the batch loop as a whole (``reference_step``, main.py:161-291: hop loop, both losses, autograd backward, both Adam
    optimisers): PINNED against the reference's own ``train(args)`` executed live from the reference's main.py
    (oracle/ref_import.py::load_reference_train runs the file's import statements and its ``train`` FunctionDef verbatim;
    wandb / tap / the dataset loader are stand-ins; the GCN class is the reference's own modules/gcn.py over this file's
    one-layer GCNConv restatement) --
    tests/test_oracle.py::test_oracle_step_matches_live_reference_train: trajectory balance, REINFORCE, random sampling,
    reg_param / log_z_init / loss_coef, multi-label; every batch's loss_c / loss_gfn / log_z / sum of log-probs and sampler
    statistics equal bit for bit, the weights after the epoch to 1e-7, the test score equal -- and against the committed
    tests/golden/train_*.npz produced by that function.
  * the arithmetic INSIDE GCNConv / gcn_norm: "parity unpinned" by the reference (it has no tests and PyG cannot be
    installed here); pinned only by the dense closed form and a hand-computed 4-node example.  Every live comparison
    above runs the reference's loop on THIS restatement of GCNConv.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
reference legs may import this module.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Sequence, Tuple, Union

import numpy as np
import scipy.sparse as sp
import torch
import torch.nn as nn
import torch.nn.functional as F_


# --------------------------------------------------------------------------- #
# graph helpers  (modules/utils.py:74-120, main.py:134-136)
# --------------------------------------------------------------------------- #
def build_adjacency(edge_index: torch.Tensor, num_nodes: int) -> sp.csr_matrix:
    """main.py:134-136 -- ``csr_matrix((ones bool, edge_index), (N, N))``.
    Duplicate pairs collapse (bool sum), self-loops stay, columns end up sorted."""
    ei = edge_index.cpu().numpy() if isinstance(edge_index, torch.Tensor) else np.asarray(edge_index)
    adj = sp.csr_matrix((np.ones(ei.shape[1], dtype=bool), (ei[0], ei[1])),
                        shape=(num_nodes, num_nodes))
    adj.sum_duplicates()
    adj.sort_indices()
    return adj


def _np(idx) -> np.ndarray:
    return idx.cpu().numpy() if isinstance(idx, torch.Tensor) else np.asarray(idx)


def get_neighborhoods(nodes: torch.Tensor, adjacency: sp.csr_matrix) -> torch.Tensor:
    """utils.py:74-82.  Row gather of the CSR; COO ``[nodes[row], col]``, row-major by
    position in ``nodes``, neighbour ids ascending inside a row."""
    coo = adjacency[_np(nodes)].tocoo()
    return torch.stack([nodes[torch.from_numpy(coo.row.astype(np.int64))],
                        torch.from_numpy(coo.col.astype(np.int64))], dim=0)


def slice_adjacency(adjacency: sp.csr_matrix, rows: torch.Tensor, cols: torch.Tensor) -> torch.Tensor:
    """utils.py:85-95.  Block ``A[rows][:, cols]`` as an edge index in GLOBAL ids:
    [0] = rows (sources), [1] = cols (destinations)."""
    block = adjacency[_np(rows)][:, _np(cols)].tocoo()
    return torch.stack([rows[torch.from_numpy(block.row.astype(np.int64))],
                        cols[torch.from_numpy(block.col.astype(np.int64))]], dim=0)


class TensorMap:
    """utils.py:98-120.  global -> local map; never cleared (stale entries are never read)."""

    def __init__(self, size):
        self.map_tensor = torch.empty(int(size), dtype=torch.long)
        self.values = torch.arange(int(size))

    def update(self, keys: torch.Tensor):
        self.map_tensor[keys] = self.values[:len(keys)]

    def map(self, keys):
        return self.map_tensor[keys]


# --------------------------------------------------------------------------- #
# sampler  (modules/utils.py:13-71)
# --------------------------------------------------------------------------- #
def draw_gumbel_like_reference(n: int, generator: Optional[torch.Generator] = None) -> torch.Tensor:
    """What ``Gumbel(0,1).sample((n,))`` evaluates (utils.py:40-41, torch
    distributions/gumbel.py): u ~ U(tiny, 1-eps) via torch.rand, g = -log(-log(u))."""
    fi = torch.finfo(torch.float32)
    u = torch.rand(n, generator=generator) * ((1 - fi.eps) - fi.tiny) + fi.tiny
    return -torch.log(-torch.log(u))


def perturbed_keys(logits: torch.Tensor, gumbel_noise: torch.Tensor) -> torch.Tensor:
    """utils.py:37,42 -- ``b.probs.log() + gumbel`` (log(sigmoid(l)), NOT logsigmoid)."""
    return torch.sigmoid(logits).log() + gumbel_noise


def stable_topk_indices(keys: torch.Tensor, k: int) -> torch.Tensor:
    """top-k with the tie-break the CUDA path commits to: among equal keys the LOWEST
    index wins (torch.topk leaves ties unspecified; utils.py:44 uses sorted=False so only
    the SET matters).  NaN keys rank lowest."""
    kk = torch.nan_to_num(keys.detach().double(), nan=-np.inf)
    order = torch.sort(kk, descending=True, stable=True).indices
    return order[:k]


def sample_neighborhoods_from_probs(logits: torch.Tensor, neighbor_nodes: torch.Tensor,
                                    num_samples: int = -1,
                                    gumbel_noise: Optional[torch.Tensor] = None,
                                    stable_ties: bool = True,
                                    ) -> Tuple[torch.Tensor, torch.Tensor, Dict[str, torch.Tensor]]:
    """utils.py:13-71 with the noise injectable.  Returns (sampled ids ascending,
    log_prob [c] (carries grad), stats dict)."""
    k = num_samples
    n = neighbor_nodes.shape[0]
    if k >= n:                                                     # utils.py:31-33
        return neighbor_nodes, F_.logsigmoid(logits.squeeze(-1)), {}
    assert k < n
    assert k > 0
    l = logits.squeeze(-1) if logits.dim() > 1 else logits
    probs = torch.sigmoid(l)                                       # Bernoulli(logits).probs
    if gumbel_noise is None:
        gumbel_noise = draw_gumbel_like_reference(n)
    keys = probs.log() + gumbel_noise.to(probs.dtype)              # utils.py:42
    if stable_ties:
        samples = stable_topk_indices(keys, k)
    else:
        samples = torch.topk(keys, k=k, dim=0, sorted=False)[1]    # utils.py:44
    entropy = -(probs * probs.log2() + (1 - probs) * (1 - probs).log2())   # utils.py:47
    min_prob = probs.min(-1)[0]
    max_prob = probs.max(-1)[0]
    entropy = torch.where(torch.isnan(entropy), torch.zeros_like(entropy), entropy)  # :52-54
    std_entropy, mean_entropy = torch.std_mean(entropy)            # unbiased, :56
    mask = torch.zeros_like(l, dtype=torch.float)
    mask[samples] = 1
    sampled = neighbor_nodes[mask.bool().cpu()]                    # ascending ids, :60
    stats = {"min_prob": min_prob, "max_prob": max_prob,
             "mean_entropy": mean_entropy, "std_entropy": std_entropy}
    # Bernoulli(logits).log_prob(mask) == -binary_cross_entropy_with_logits(l, mask)  (:71)
    log_prob = -F_.binary_cross_entropy_with_logits(l, mask.to(l.dtype), reduction="none")
    return sampled, log_prob, stats


# --------------------------------------------------------------------------- #
# GCNConv / GCN  (PyG 2.5.2 restated; modules/gcn.py:9-42)
# --------------------------------------------------------------------------- #
def gcn_norm(edge_index: torch.Tensor, num_nodes: int, dtype=torch.float32
             ) -> Tuple[torch.Tensor, torch.Tensor]:
    """PyG ``gcn_norm`` with add_remaining_self_loops (SURVEY.md section 3.2 steps 1-3):
    drop src==dst edges, append one (i,i) per node, deg = in-degree over dst incl. the
    loop, w = deg^-1/2[src] * deg^-1/2[dst]."""
    row, col = edge_index[0], edge_index[1]
    keep = row != col
    loop = torch.arange(num_nodes, dtype=row.dtype, device=row.device)
    row = torch.cat([row[keep], loop])
    col = torch.cat([col[keep], loop])
    w = torch.ones(row.numel(), dtype=dtype, device=row.device)
    deg = torch.zeros(num_nodes, dtype=dtype, device=row.device).scatter_add_(0, col, w)
    dis = deg.pow(-0.5)
    dis = dis.masked_fill(dis == float("inf"), 0)
    return torch.stack([row, col]), dis[row] * w * dis[col]


def gcn_conv(x: torch.Tensor, edge_index: torch.Tensor, weight: torch.Tensor,
             bias: Optional[torch.Tensor]) -> torch.Tensor:
    """PyG ``GCNConv.forward`` (SURVEY.md section 3.2 steps 4-5): H = X W^T,
    out[dst] += w_e H[src], out += bias.  ``weight`` is [out, in]."""
    n = x.shape[0]
    ei, w = gcn_norm(edge_index, n, dtype=x.dtype)
    h = x @ weight.t()
    out = torch.zeros(n, weight.shape[0], dtype=x.dtype, device=x.device)
    out = out.index_add(0, ei[1], h[ei[0]] * w.unsqueeze(1))
    if bias is not None:
        out = out + bias
    return out


def glorot_(w: torch.Tensor, generator: Optional[torch.Generator] = None) -> torch.Tensor:
    """PyG ``Linear(weight_initializer='glorot')``: U(-a, a), a = sqrt(6 / (fan_in + fan_out))."""
    a = (6.0 / (w.shape[0] + w.shape[1])) ** 0.5
    with torch.no_grad():
        w.copy_((torch.rand(w.shape, generator=generator, dtype=torch.float32) * 2 - 1) * a)
    return w


class _Lin(nn.Module):
    def __init__(self, i, o):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(o, i))


class OracleGCNConv(nn.Module):
    """Parameter names follow PyG so a reference state_dict loads:
    ``lin.weight`` [out, in] and ``bias`` [out]."""

    def __init__(self, in_channels: int, out_channels: int, generator=None):
        super().__init__()
        self.lin = _Lin(in_channels, out_channels)
        self.bias = nn.Parameter(torch.zeros(out_channels))
        glorot_(self.lin.weight, generator)

    def forward(self, x, edge_index):
        return gcn_conv(x, edge_index, self.lin.weight, self.bias)


class OracleGCN(nn.Module):
    """modules/gcn.py:9-42 (dims, layer wiring, the per-layer edge list quirk, tuple return)."""

    def __init__(self, in_features: int, hidden_dims: List[int], dropout: float = 0., generator=None):
        super().__init__()
        self.dropout = dropout
        dims = [in_features] + hidden_dims
        layers = []
        for i in range(len(hidden_dims) - 1):
            layers.append(OracleGCNConv(dims[i], dims[i + 1], generator))
        layers.append(OracleGCNConv(dims[-2], dims[-1], generator))
        self.gcn_layers = nn.ModuleList(layers)

    def forward(self, x, edge_index: Union[torch.Tensor, List[torch.Tensor]]):
        layerwise = type(edge_index) == list
        for i, layer in enumerate(self.gcn_layers[:-1], start=1):
            edges = edge_index[-i] if layerwise else edge_index
            x = torch.relu(layer(x, edges))
            x = F_.dropout(x, p=self.dropout, training=self.training)
        edges = edge_index[0] if layerwise else edge_index
        logits = self.gcn_layers[-1](x, edges)
        logits = F_.dropout(logits, p=self.dropout, training=self.training)
        return logits, 0.0


# --------------------------------------------------------------------------- #
# one batch of train()   (main.py:161-291)
# --------------------------------------------------------------------------- #
class OracleState:
    """The objects ``train()`` creates before its loop (main.py:102-140)."""

    def __init__(self, data, *, sampling_hops=2, num_samples=16, use_indicators=True,
                 hidden_dim=256, lr_gc=1e-3, lr_gf=1e-4, loss_coef=1e4, log_z_init=0.,
                 reg_param=0., dropout=0., random_sampling=False, reinforce_baseline=False,
                 seed: int = 0, dtype=torch.float32, adjacency: Optional[sp.csr_matrix] = None,
                 embed_nodes: bool = False):
        self.data = data
        self.hops, self.k = sampling_hops, num_samples
        self.use_indicators = use_indicators
        self.loss_coef, self.log_z_init, self.reg_param = loss_coef, log_z_init, reg_param
        self.random_sampling, self.reinforce_baseline = random_sampling, reinforce_baseline
        self.num_indicators = sampling_hops + 1 if use_indicators else 0
        N, Fdim = data.num_nodes, data.num_features
        g = torch.Generator().manual_seed(seed)
        C = data.num_classes
        self.gcn_c = OracleGCN(Fdim, [hidden_dim, C], dropout, g).to(dtype)
        self.gcn_gf = OracleGCN(Fdim + self.num_indicators, [hidden_dim, 1], generator=g).to(dtype)
        self.gcn_z = OracleGCN(Fdim, [hidden_dim, 1], generator=g).to(dtype)
        # main.py:89-100,116: learned node features are an nn.Parameter table inside optimizer_c (the caller passes the
        # nn.init.normal_ draw as data.x so the oracle and the device engine start from the same table)
        self.embed_nodes = bool(embed_nodes)
        self.x = data.x.to(dtype)
        embedding_params = []
        if self.embed_nodes:
            self.x = nn.Parameter(self.x.clone(), requires_grad=True)
            embedding_params.append(self.x)
        self.opt_c = torch.optim.Adam(list(self.gcn_c.parameters()) + embedding_params, lr=lr_gc)
        self.opt_gf = torch.optim.Adam(list(self.gcn_gf.parameters()) + list(self.gcn_z.parameters()), lr=lr_gf)
        self.loss_fn = nn.CrossEntropyLoss() if data.y.dim() == 1 else nn.BCEWithLogitsLoss()
        self.adjacency = adjacency if adjacency is not None else build_adjacency(data.edge_index, N)
        self.node_map = TensorMap(N)
        self.prev_nodes_mask = torch.zeros(N, dtype=torch.bool)
        self.batch_nodes_mask = torch.zeros(N, dtype=torch.bool)
        self.indicator_features = torch.zeros((N, self.num_indicators), dtype=dtype)
        self.dtype = dtype


def reference_step(st: OracleState, target_nodes: torch.Tensor,
                   gumbel_noise: Optional[Sequence[Optional[torch.Tensor]]] = None,
                   apply_optim: bool = True, stable_ties: bool = True) -> dict:
    """Functional restatement of main.py:161-291 for ONE batch.  ``gumbel_noise[h]`` (length
    c_h) replaces the draw at utils.py:40-41 when given.  Returns every intermediate the
    parity tests compare."""
    data, adjacency, node_map = st.data, st.adjacency, st.node_map
    rec: dict = {"hops": []}
    previous_nodes = target_nodes.clone()
    all_nodes_mask = torch.zeros_like(st.prev_nodes_mask)
    all_nodes_mask[target_nodes] = True
    ind = st.indicator_features
    ind.zero_()
    if st.use_indicators:
        ind[target_nodes, -1] = 1.0
    global_edge_indices, log_probs, all_stats = [], [], []
    log_z = torch.tensor([0.0], dtype=st.dtype)
    for hop in range(st.hops):
        neighborhoods = get_neighborhoods(previous_nodes, adjacency)           # main.py:180
        st.prev_nodes_mask.zero_(); st.batch_nodes_mask.zero_()
        st.prev_nodes_mask[previous_nodes] = True
        st.batch_nodes_mask[neighborhoods.view(-1)] = True
        neighbor_mask = st.batch_nodes_mask & ~st.prev_nodes_mask
        batch_nodes = node_map.values[st.batch_nodes_mask]                      # ascending
        neighbor_nodes = node_map.values[neighbor_mask]
        if st.use_indicators:
            ind[neighbor_nodes, hop] = 1.0                                      # :191
        node_map.update(batch_nodes)
        local_nb = node_map.map(neighborhoods)                                  # :195
        if st.use_indicators:
            x = torch.cat([st.x[batch_nodes], ind[batch_nodes]], dim=1)         # :198-202
        else:
            x = st.x[batch_nodes]
        if st.random_sampling:
            node_logits_all = 100 * torch.ones((x.shape[0], 1), dtype=st.dtype)  # :207
        else:
            node_logits_all, _ = st.gcn_gf(x, local_nb)                         # :210
        nb_local = node_map.map(neighbor_nodes)
        node_logits = node_logits_all[nb_local]                                 # :213
        noise = None if gumbel_noise is None else gumbel_noise[hop]
        c = neighbor_nodes.shape[0]
        if noise is None and st.k < c:
            noise = draw_gumbel_like_reference(c)
        sampled, log_prob, stats = sample_neighborhoods_from_probs(
            node_logits, neighbor_nodes, st.k, gumbel_noise=noise, stable_ties=stable_ties)
        all_nodes_mask[sampled] = True
        if hop == 0 and not st.random_sampling:                                 # :223-228
            pred_z = st.gcn_z(st.x[batch_nodes], local_nb)[0].squeeze()
            log_z = pred_z.mean() - st.log_z_init
        log_probs.append(log_prob)
        all_stats.append(stats)
        batch_nodes_next = torch.cat([target_nodes, sampled], dim=0)            # :236-238
        k_hop_edges = slice_adjacency(adjacency, rows=batch_nodes_next, cols=previous_nodes)  # :241
        global_edge_indices.append(k_hop_edges)
        rec["hops"].append(dict(
            prev=previous_nodes.clone(), neighborhoods=neighborhoods, local_neighborhoods=local_nb,
            batch_nodes=batch_nodes.clone(), neighbor_nodes=neighbor_nodes.clone(), nb_local=nb_local,
            x=x.detach().clone(), logits_all=node_logits_all.detach().clone().squeeze(-1),
            logits=node_logits.detach().clone().squeeze(-1), noise=noise,
            keys=None if (noise is None or st.k >= c) else perturbed_keys(node_logits.detach().squeeze(-1), noise),
            sampled=sampled.clone(), log_prob=log_prob.detach().clone(), stats=stats,
            block_edges=k_hop_edges.clone()))
        previous_nodes = batch_nodes_next.clone()

    all_nodes = node_map.values[all_nodes_mask]                                 # :252
    node_map.update(all_nodes)
    edge_indices = [node_map.map(e) for e in global_edge_indices]
    xc = st.x[all_nodes]
    logits, _ = st.gcn_c(xc, edge_indices)                                      # :257
    local_target_ids = node_map.map(target_nodes)
    y = data.y[target_nodes]
    if data.y.dim() != 1:
        y = y.to(st.dtype)
    loss_c = st.loss_fn(logits[local_target_ids], y) + st.reg_param * torch.sum(torch.var(logits, dim=1))
    st.opt_c.zero_grad()
    loss_c.backward()
    grads_c = {n: p.grad.detach().clone() for n, p in st.gcn_c.named_parameters()}
    if getattr(st, "embed_nodes", False):
        rec["grad_x"] = st.x.grad.detach().clone()          # dense [N, F]; rows outside all_nodes are zero
    if apply_optim:
        st.opt_c.step()
    rec.update(all_nodes=all_nodes.clone(), edge_indices=[e.clone() for e in edge_indices],
               logits_c=logits.detach().clone(), local_target_ids=local_target_ids.clone(),
               loss_c=loss_c.detach().clone(), grads_c=grads_c)
    loss_gfn = torch.zeros((), dtype=st.dtype)
    tot_log_prob = torch.sum(torch.cat(log_probs, dim=0))
    if not st.random_sampling:                                                  # :272-291
        st.opt_gf.zero_grad()
        cost_gfn = loss_c.detach()
        if st.reinforce_baseline:
            loss_gfn = -tot_log_prob * cost_gfn                                 # :279
        else:
            loss_gfn = (log_z + tot_log_prob + st.loss_coef * cost_gfn) ** 2    # :282
        loss_gfn = loss_gfn.sum()
        loss_gfn.backward()
        rec["grads_gf"] = {n: (None if p.grad is None else p.grad.detach().clone())
                           for n, p in st.gcn_gf.named_parameters()}
        rec["grads_z"] = {n: (None if p.grad is None else p.grad.detach().clone())
                          for n, p in st.gcn_z.named_parameters()}
        if apply_optim:
            st.opt_gf.step()
    rec.update(loss_gfn=loss_gfn.detach().clone(), log_z=log_z.detach().clone().reshape(()),
               tot_log_prob=tot_log_prob.detach().clone())
    return rec


# =============================================================================================
# evaluation (eval.py:11-165)
# =============================================================================================
@torch.inference_mode()
def reference_evaluate(st: OracleState, mask: torch.Tensor, full_batch: bool = True,
                       batch_size: int = 256, stable_ties: bool = True) -> dict:
    """Restatement of ``evaluate`` (eval.py:12-165) on the oracle's models.

    full_batch (eval.py:47-70): one whole-graph forward ``gcn_c(x, edge_index)``; accuracy / micro-F1
    (single label: both are the fraction of correct predictions) or the TP/FP/FN F1 for multi-label.
    mini-batch (eval.py:71-163): the hop loop with deterministic ``topk(Bernoulli(logits).probs)`` (:126-127)
    and ``slice_adjacency(rows=previous_nodes, cols=batch_nodes)`` (:140-142); batches are consecutive slices of
    ``mask.nonzero()`` like the un-shuffled DataLoader of main.py:127-132.  ``stable_ties`` breaks ties of equal
    probabilities towards the lower candidate index (torch.topk leaves ties unspecified)."""
    data, adjacency, node_map = st.data, st.adjacency, st.node_map
    out: dict = {}
    if full_batch:
        logits_total, _ = st.gcn_c(st.x, data.edge_index)                       # eval.py:50
        out["logits"] = logits_total
        if data.y[mask].dim() == 1:
            predictions = torch.argmax(logits_total, dim=1)[mask]
            out["predictions"] = predictions
            out["accuracy"] = out["f1"] = float((predictions == data.y[mask]).double().mean())
        else:
            y_pred = logits_total[mask] > 0
            y_true = data.y[mask] > 0.5
            tp = int((y_true & y_pred).sum()); fp = int((~y_true & y_pred).sum()); fn = int((y_true & ~y_pred).sum())
            try:
                precision, recall = tp / (tp + fp), tp / (tp + fn)
                out["accuracy"] = out["f1"] = 2 * (precision * recall) / (precision + recall)
            except ZeroDivisionError:
                out["accuracy"] = out["f1"] = 0.
        return out

    idx = mask.nonzero().squeeze(1)
    prev_nodes_mask = torch.zeros(data.num_nodes, dtype=torch.bool)
    batch_nodes_mask = torch.zeros(data.num_nodes, dtype=torch.bool)
    indicator_features = torch.zeros((data.num_nodes, st.num_indicators), dtype=st.dtype)
    all_predictions, per_batch = [], []
    for target_nodes in torch.split(idx, batch_size):
        previous_nodes = target_nodes.clone()
        all_nodes_mask = torch.zeros_like(prev_nodes_mask)
        all_nodes_mask[target_nodes] = True
        indicator_features.zero_()
        if st.use_indicators:
            indicator_features[target_nodes, -1] = 1.0
        global_edge_indices, hops = [], []
        for hop in range(st.hops):
            neighborhoods = get_neighborhoods(previous_nodes, adjacency)        # eval.py:94
            prev_nodes_mask.zero_(); batch_nodes_mask.zero_()
            prev_nodes_mask[previous_nodes] = True
            batch_nodes_mask[neighborhoods.view(-1)] = True
            neighbor_nodes_mask = batch_nodes_mask & ~prev_nodes_mask
            batch_nodes = node_map.values[batch_nodes_mask]
            neighbor_nodes = node_map.values[neighbor_nodes_mask]
            if st.use_indicators:
                indicator_features[neighbor_nodes, hop] = 1.0
            node_map.update(batch_nodes)
            local_neighborhoods = node_map.map(neighborhoods)
            if st.use_indicators:
                x = torch.cat([st.x[batch_nodes], indicator_features[batch_nodes]], dim=1)
            else:
                x = st.x[batch_nodes]
            if neighbor_nodes.numel() > 0:
                node_logits, _ = st.gcn_gf(x, local_neighborhoods)              # eval.py:121
                node_logits = node_logits[node_map.map(neighbor_nodes)]
                probs = torch.sigmoid(node_logits.squeeze(-1))                  # Bernoulli(logits).probs
                k = min(neighbor_nodes.size(0), st.k)
                samples = stable_topk_indices(probs, k) if stable_ties else torch.topk(probs, k, sorted=False)[1]
                sample_mask = torch.zeros_like(probs)
                sample_mask[samples] = 1
                sampled = neighbor_nodes[sample_mask.bool()]
            else:
                sampled = neighbor_nodes
            all_nodes_mask[sampled] = True
            batch_nodes = torch.cat([target_nodes, sampled], dim=0)
            k_hop_edges = slice_adjacency(adjacency, rows=previous_nodes, cols=batch_nodes)   # eval.py:140-142
            global_edge_indices.append(k_hop_edges)
            hops.append({"neighbor_nodes": neighbor_nodes.clone(), "sampled": sampled.clone(),
                         "block_edges": k_hop_edges.clone()})
            previous_nodes = batch_nodes.clone()
        all_nodes = node_map.values[all_nodes_mask]
        node_map.update(all_nodes)
        edge_indices = [node_map.map(e) for e in global_edge_indices]
        logits_total, _ = st.gcn_c(st.x[all_nodes], edge_indices)
        predictions = torch.argmax(logits_total, dim=1)[node_map.map(target_nodes)]
        all_predictions.append(predictions)
        per_batch.append({"hops": hops, "all_nodes": all_nodes.clone(), "logits": logits_total.clone()})
    all_predictions = torch.cat(all_predictions)
    out["predictions"] = all_predictions
    out["batches"] = per_batch
    out["accuracy"] = out["f1"] = float((all_predictions == data.y[mask]).double().mean())
    return out


def full_graph_logits_cpu(gcn: "OracleGCN", x: torch.Tensor, adjacency: sp.csr_matrix) -> torch.Tensor:
    """eval.py:50 on the host at BASELINE sizes: ``gcn_c(x, edge_index)`` over every stored entry of ``adjacency`` in PyG's
    order (lin, then propagate, SURVEY.md section 3.2 steps 1-5), with the propagate written as ONE sparse-CSR x dense
    product per layer (torch / MKL threads) instead of :func:`gcn_conv`'s ``h[src]`` gather, which would materialise an
    [E, 256] array (127 GB on the products-shaped graph).  Same arithmetic: out[dst] = sum_e w_e h[src_e] + b with
    w_e = deg^-1/2[src] deg^-1/2[dst] over the stored edges minus self-loops plus one loop per node."""
    n = adjacency.shape[0]
    A = adjacency.astype(np.float32).tocsr(copy=True)
    A.setdiag(0)
    A.eliminate_zeros()
    AT = (A.T + sp.identity(n, dtype=np.float32, format="csr")).tocsr()      # rows = destinations, cols = sources
    deg = np.asarray(AT.sum(axis=1)).reshape(-1)                              # in-degree + 1
    dis = (1.0 / np.sqrt(deg)).astype(np.float32)
    AT = sp.diags(dis) @ AT @ sp.diags(dis)
    AT = AT.tocsr()
    a_hat = torch.sparse_csr_tensor(torch.from_numpy(AT.indptr.astype(np.int64)), torch.from_numpy(AT.indices.astype(np.int64)),
                                    torch.from_numpy(AT.data.astype(np.float32)).to(x.dtype), size=(n, n))
    h = x
    layers = list(gcn.gcn_layers)
    for i, layer in enumerate(layers):
        h = a_hat @ (h @ layer.lin.weight.t()) + layer.bias
        if i + 1 < len(layers):
            h = torch.relu(h)
    return h
