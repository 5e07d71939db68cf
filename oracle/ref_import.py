"""TEST INFRASTRUCTURE ONLY.  Imports the reference's own ``modules/utils.py`` from the
checkout of the reference GRAPES project that ``GRAPES_REFERENCE_ROOT`` names (it is not
part of this repository) so the restatement in oracle/reference_port.py can be validated
against it and golden vectors can be generated from it.  Without it the live comparisons
skip; the committed golden vectors hold the reference's outputs only for the cases
tests/golden/make_golden.py records.  Nothing under tests -m gpu, smoke() or bench.py may
use this.

The reference pins scipy 1.13.1 (environment.yml:95); on scipy 1.18 indexing a CSR matrix
with a ``torch.Tensor`` raises, so :class:`TensorIndexCSR` converts tensor indices to numpy
first -- an index-type shim, not a semantic change (SURVEY.md section 0).
"""
from __future__ import annotations

import importlib.util
import os
import sys

import numpy as np
import scipy.sparse as sp
import torch

REFERENCE_ROOT = os.environ.get("GRAPES_REFERENCE_ROOT", "")


def reference_available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(REFERENCE_ROOT, "modules", "utils.py"))


def load_reference_utils():
    """Import the reference's modules/utils.py (under ``REFERENCE_ROOT``) as a stand-alone module (it only needs
    logging/os/numpy/psutil/scipy/torch, utils.py:1-10)."""
    path = os.path.join(REFERENCE_ROOT, "modules", "utils.py")
    spec = importlib.util.spec_from_file_location("grapes_reference_utils", path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules["grapes_reference_utils"] = mod
    spec.loader.exec_module(mod)
    return mod


def _conv(i):
    if isinstance(i, torch.Tensor):
        return i.cpu().numpy()
    if isinstance(i, tuple):
        return tuple(_conv(j) for j in i)
    return i


class TensorIndexCSR:
    """Wraps a scipy CSR so ``adj[tensor]`` / ``adj[:, tensor]`` work like they did on scipy 1.13."""

    def __init__(self, m: sp.csr_matrix):
        self.m = m

    def __getitem__(self, idx):
        return TensorIndexCSR(self.m[_conv(idx)])

    def tocoo(self):
        return self.m.tocoo()

    @property
    def shape(self):
        return self.m.shape


def reference_adjacency(edge_index: torch.Tensor, num_nodes: int) -> TensorIndexCSR:
    """main.py:134-136 verbatim call (bool ones, edge_index as (row, col))."""
    ei = edge_index.numpy()
    adj = sp.csr_matrix((np.ones(ei.shape[1], dtype=bool), ei), shape=(num_nodes, num_nodes))
    return TensorIndexCSR(adj)


def load_reference_eval():
    """Import the reference's eval.py (``evaluate``, eval.py:11-165) as a stand-alone module.  It imports
    ``torch_geometric`` for ONE type annotation (eval.py:4,14: absent here) and ``modules.utils`` (the reference's own,
    loaded by :func:`load_reference_utils`); both names are bound for the duration of the import only.  Everything the
    function then executes is the reference's own code."""
    import types
    ru = load_reference_utils()
    path = os.path.join(REFERENCE_ROOT, "eval.py")
    tg = types.ModuleType("torch_geometric")
    tg.data = types.ModuleType("torch_geometric.data")
    tg.data.Data = object
    pkg = types.ModuleType("modules")
    pkg.utils = ru
    names = {"torch_geometric": tg, "torch_geometric.data": tg.data, "modules": pkg, "modules.utils": ru}
    saved = {k: sys.modules.get(k) for k in names}
    sys.modules.update(names)
    try:
        spec = importlib.util.spec_from_file_location("grapes_reference_eval", path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return mod, ru


def load_reference_gcn(conv_factory):
    """Import the reference's modules/gcn.py with ``torch_geometric.nn.GCNConv`` bound to ``conv_factory`` (PyG is absent;
    the other convolutions it imports are never instantiated on this path).  The returned module's ``GCN`` is the
    reference's own class -- layer list, which edge list feeds which layer, relu / dropout placement, ``(logits,
    memory_alloc)`` return (gcn.py:9-42) -- over the oracle's restatement of the one GCNConv layer."""
    import types
    path = os.path.join(REFERENCE_ROOT, "modules", "gcn.py")
    tg = types.ModuleType("torch_geometric")
    tg.nn = types.ModuleType("torch_geometric.nn")
    tg.nn.GCNConv = conv_factory
    for other in ("GATConv", "GCN2Conv", "Linear", "PNAConv"):
        setattr(tg.nn, other, object)
    names = {"torch_geometric": tg, "torch_geometric.nn": tg.nn}
    saved = {k: sys.modules.get(k) for k in names}
    sys.modules.update(names)
    try:
        spec = importlib.util.spec_from_file_location("grapes_reference_gcn", path)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return mod


class RecordingModule(torch.nn.Module):
    """Wraps a model handed to the reference's ``evaluate`` and keeps what it was called with and what it returned (the
    reference returns only (accuracy, f1); the per-batch blocks and logits are read off its ``gcn_c`` calls)."""

    def __init__(self, inner):
        super().__init__()
        self.inner = inner
        self.calls = []

    def forward(self, x, edge_index):
        out = self.inner(x, edge_index)
        ei = [e.clone() for e in edge_index] if isinstance(edge_index, list) else edge_index.clone()
        self.calls.append({"x": x.clone(), "edge_index": ei, "logits": out[0].clone()})
        return out


class _SparseShim:
    """``sp`` as main.py sees it: ``csr_matrix`` returns the CSR wrapped in :class:`TensorIndexCSR` (tensor indices on
    scipy >= 1.14) and accepts a torch ``edge_index`` as the (row, col) pair like scipy 1.13 did (main.py:134-136)."""

    @staticmethod
    def csr_matrix(arg1, *a, **k):
        if isinstance(arg1, tuple) and len(arg1) == 2 and isinstance(arg1[1], torch.Tensor):
            arg1 = (arg1[0], arg1[1].cpu().numpy())
        return TensorIndexCSR(sp.csr_matrix(arg1, *a, **k))


class WandbStub:
    """Stands in for ``wandb`` (not installed): ``init`` is a no-op, ``log`` keeps every dict train() logs."""

    def __init__(self):
        self.logged = []

    def init(self, **kw):
        return None

    def log(self, d):
        self.logged.append(dict(d))


def load_reference_train(get_data, gcn_factory, utils_overrides=None):
    """The reference's own ``train(args)`` (main.py:57-340) as a callable.  main.py trains at import time (main.py:342-364),
    so only its import statements, the ``device`` assignment and the ``train`` FunctionDef are executed, verbatim from the AST
    of the reference's main.py.  Bound while its imports run (none of them installed here or usable offline):
      wandb -> :class:`WandbStub` (returned);  tap.Tap -> object;  modules.data.get_data -> ``get_data`` (synthetic data);
      modules.gcn.GCN -> ``gcn_factory`` (the oracle's GCN restatement: PyG is absent);  modules.utils, eval -> the
      reference's own modules;  sp.csr_matrix -> :class:`_SparseShim` (index-type shim only).
    Every statement of the batch loop that then runs is the reference's."""
    import ast
    import types
    ev, ru = load_reference_eval()
    if utils_overrides:                       # e.g. this repo's host-side drop-ins (TensorMap, get_logger) inside the real loop
        ru2 = types.ModuleType("modules.utils")
        ru2.__dict__.update({k: v for k, v in ru.__dict__.items() if not k.startswith("__")})
        ru2.__dict__.update(utils_overrides)
        ru = ru2
    src = open(os.path.join(REFERENCE_ROOT, "main.py")).read()
    tree = ast.parse(src)
    keep = []
    for node in tree.body:
        if isinstance(node, (ast.Import, ast.ImportFrom)):
            keep.append(node)
        elif isinstance(node, ast.Assign) and len(node.targets) == 1 and getattr(node.targets[0], "id", "") == "device":
            keep.append(node)
        elif isinstance(node, ast.FunctionDef) and node.name == "train":
            keep.append(node)
    assert any(isinstance(n, ast.FunctionDef) for n in keep), "main.py: def train not found"
    wb = WandbStub()
    wandb_mod = types.ModuleType("wandb")
    wandb_mod.init, wandb_mod.log = wb.init, wb.log
    tap_mod = types.ModuleType("tap")
    tap_mod.Tap = object
    pkg = types.ModuleType("modules")
    data_mod = types.ModuleType("modules.data")
    data_mod.get_data = get_data
    gcn_mod = types.ModuleType("modules.gcn")
    gcn_mod.GCN = gcn_factory
    pkg.utils, pkg.data, pkg.gcn = ru, data_mod, gcn_mod
    names = {"wandb": wandb_mod, "tap": tap_mod, "modules": pkg, "modules.utils": ru, "modules.data": data_mod,
             "modules.gcn": gcn_mod, "eval": ev}
    saved = {k: sys.modules.get(k) for k in names}
    sys.modules.update(names)
    ns = {"__name__": "grapes_reference_main", "Arguments": object}
    try:
        exec(compile(ast.Module(body=keep, type_ignores=[]), os.path.join(REFERENCE_ROOT, "main.py"), "exec"), ns)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    ns["sp"] = _SparseShim
    return ns["train"], wb


def run_reference_train(data, *, weight_seed: int, rng_seed: int, batch_size: int = 0, num_samples: int = 0,
                        sampling_hops: int = 0, max_epochs: int = 1, args_obj=None, utils_overrides=None, **over):
    """Runs the reference's own ``train(args)`` (see :func:`load_reference_train`) on ``data`` with the reference's own ``GCN``
    class over the oracle's GCNConv layer (:func:`load_reference_gcn`), the layers initialised from ``torch.Generator().manual_seed(weight_seed)`` in the order main.py creates them (gcn_c, gcn_gf, gcn_z,
    main.py:107-112 -- the order OracleState uses) and the global RNG seeded with ``rng_seed`` right before the call (Gumbel
    noise, utils.py:40-41).  Returns (test_f1, the per-batch dicts train() logged, [gcn_c, gcn_gf, gcn_z])."""
    import argparse
    from . import reference_port as rp
    gen = torch.Generator().manual_seed(weight_seed)
    made = []
    # the reference's OWN GCN class (modules/gcn.py:9-42) over the oracle's GCNConv layer
    ref_gcn = load_reference_gcn(lambda in_channels, out_channels: rp.OracleGCNConv(in_channels, out_channels, gen))

    def factory(in_features, hidden_dims, dropout=0.):
        m = ref_gcn.GCN(in_features, hidden_dims=hidden_dims, dropout=dropout)
        made.append(m)
        return m

    train, wb = load_reference_train(lambda **kw: (data, data.num_features, data.num_classes), factory, utils_overrides)

    class Args(argparse.Namespace):
        def as_dict(self):
            return dict(vars(self))

    args = Args(dataset="synthetic", sampling_hops=sampling_hops, num_samples=num_samples, use_indicators=True, lr_gf=1e-4,
                lr_gc=1e-3, loss_coef=1e4, log_z_init=0., reg_param=0., dropout=0., model_type="gcn", hidden_dim=256,
                embed_nodes=False, node_emb_dim=64, max_epochs=max_epochs, batch_size=batch_size, eval_frequency=5,
                eval_on_cpu=True, eval_full_batch=True, random_sampling=False, runs=1, split_id=0, seed=0, notes=None,
                log_wandb=False, config_file=None, reinforce_baseline=False)
    for k, v in over.items():
        assert hasattr(args, k), k
        setattr(args, k, v)
    if args_obj is not None:                 # e.g. grapes_b200.args.Arguments: the drop-in for main.py's Tap class
        args = args_obj
    torch.manual_seed(rng_seed)
    test_f1, *_ = train(args)
    logs = [l for l in wb.logged if "batch_loss_c" in l]
    stats = [l for l in wb.logged if "batch_loss_c" not in l and "test_f1" not in l and "epoch" not in l]
    for l, s in zip(logs, stats):
        l["stats"] = s
    return float(test_f1), logs, made
