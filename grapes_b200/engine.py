"""Device-resident GRAPES training step (the batch body of ``train()``,
/root/reference/main.py:161-291) as ONE stream of hand-written sm_100a kernels behind the C ABI.

Differences in *mechanism* (never in results) from the reference loop:
  * the graph, features and labels stay in HBM; nothing is gathered on the host or shipped per hop
    (the reference does 5 H2D copies + 1 D2H sync per hop, SURVEY.md section 3.1);
  * every data-dependent size (m, n, c, |sampled|, |block|, |all_nodes|) lives in device memory,
    buffers are capacity-bounded, so the whole step enqueues without a host sync and can be
    captured into a CUDA graph and replayed;
  * GCNConv aggregation is done at the narrower width (A_hat (X W) == (A_hat X) W);
  * the GFlowNet / REINFORCE gradient is linear in the scalar 2*(log_z + sum log_prob + coef*loss_c)
    (resp. -loss_c), so each hop's gradient DIRECTION is accumulated right after that hop's
    selection while its aggregated features are still hot in L2, and scaled once at the end;
    no autograd graph is kept across hops.
"""
from __future__ import annotations

import contextlib
import ctypes
import math
from typing import Dict, List, Optional, Sequence

import torch

from ._lib import lib, ptr, GrapesError
from .graph import DeviceGraph

SCAL = dict(loss_c=0, tot_log_prob=1, log_z_mean=2, log_z=3, loss_gfn=4, g_gf=5, g_z=6, sum_dl=7, flags=15)
STAT_NAMES = ("min_prob", "max_prob", "mean_entropy", "std_entropy")          # utils.py:62-69, per hop
NOISE_PHILOX, NOISE_GUMBEL, NOISE_UNIFORM, NOISE_KEYS, NOISE_TOPK_PROBS = 0, 1, 2, 3, 4
OVF_NAMES = {1: "rows>cap_P", 2: "edges>cap_m", 4: "nodes>cap_n", 8: "block>cap_blk", 16: "hub worklist",
             32: "a peer rank never published its gradients"}


def _round_up(a: int, b: int) -> int:
    return (a + b - 1) // b * b


class _Net:
    """Offsets of one 2-layer GCN (hidden D, in K, out O) inside the flat parameter buffer.
    Parameter names/shapes follow PyG GCNConv: lin.weight [out, in], bias [out] (SURVEY.md section 3.2)."""

    def __init__(self, base: int, K: int, D: int, O: int):
        self.K, self.D, self.O = K, D, O
        self.W1 = base
        self.b1 = self.W1 + D * K
        self.W2 = self.b1 + D
        self.b2 = self.W2 + O * D
        self.end = self.b2 + O
        self.base = base

    @property
    def size(self):
        return self.end - self.base

    def views(self, flat: torch.Tensor) -> Dict[str, torch.Tensor]:
        return {
            "gcn_layers.0.bias": flat[self.b1:self.b1 + self.D],
            "gcn_layers.0.lin.weight": flat[self.W1:self.W1 + self.D * self.K].view(self.D, self.K),
            "gcn_layers.1.bias": flat[self.b2:self.b2 + self.O],
            "gcn_layers.1.lin.weight": flat[self.W2:self.W2 + self.O * self.D].view(self.O, self.D),
        }


def glorot_(w: torch.Tensor, generator=None):
    """PyG Linear(weight_initializer='glorot'): U(-a, a), a = sqrt(6/(fan_in+fan_out)); bias zeros."""
    a = math.sqrt(6.0 / (w.shape[0] + w.shape[1]))
    cpu = (torch.rand(w.shape, generator=generator, dtype=torch.float32) * 2 - 1) * a
    w.copy_(cpu.to(w.device))


class _Hop:
    """Workspace of ONE hop.  Every array a later consumer reads (the hop's backward on the side stream, the
    induced-block slice, the recorder of the tests) is per hop, so nothing is overwritten inside a step and the
    branches of the step graph only synchronise where data really flows."""
    CNT = dict(P=0, m=1, n=2, c=3, nnz=4, s=5, blk=6)


class GrapesEngine:
    # largest cap_A = B + H * k whose classifier takes the "prep" form (one grapes_classifier_prep launch and the
    # row-parallel loss); above it the step relabels with grapes_relabel, builds the CSRs with grapes_build_csr and takes
    # the target-row loss.  It may be lowered (the two forms compute the same step) but never raised:
    # grapes_classifier_prep refuses cap_A > SMALL_N (4096, csrc/frontier.cu).
    PREP_MAX_ROWS = 4096

    def __init__(self, graph: DeviceGraph, x: torch.Tensor, y: torch.Tensor, *, num_classes: int,
                 batch_size: int, num_samples: int, sampling_hops: int, use_indicators: bool = True,
                 hidden_dim: int = 256, lr_gc: float = 1e-3, lr_gf: float = 1e-4, loss_coef: float = 1e4,
                 log_z_init: float = 0., reg_param: float = 0., random_sampling: bool = False,
                 reinforce_baseline: bool = False, seed: int = 0, cap_edges: Optional[int] = None,
                 cap_nodes: Optional[int] = None, cap_block: Optional[int] = None,
                 use_tensor_cores: bool = True, multi_stream: bool = True, embed_nodes: bool = False,
                 dropout: float = 0.):
        dropout = float(dropout)
        if not 0. <= dropout <= 1.:
            raise ValueError(f"dropout probability has to be between 0 and 1, but got {dropout}")
        from .dist import ShardedEmbedding, ShardedFeatures
        # a feature table sharded across the data-parallel ranks: both feature gathers read each row from its owner
        # (grapes_aggregate_peer); nothing else of the step changes.  A learned table sharded with its Adam moments
        # (ShardedEmbedding) is also updated shard by shard: each rank walks only its own rows.
        self.features = x if isinstance(x, ShardedFeatures) else None
        self.embed_shards = x if (embed_nodes and isinstance(x, ShardedEmbedding)) else None
        if self.features is not None:
            if embed_nodes and self.embed_shards is None:
                raise GrapesError("learned node features (embed_nodes) with a sharded feature table: the table optimiser "
                                  "is not sharded; replicate the table")
            if x.N != graph.num_nodes:
                raise GrapesError(f"sharded feature table of {x.N} rows for a graph of {graph.num_nodes} nodes")
        self.g = graph
        self.L = lib()
        dev = graph.device
        self.device = dev
        if self.features is None:
            assert x.is_cuda and x.dtype in (torch.float32, torch.bfloat16) and x.is_contiguous()
        # bf16 feature table (papers100M-shaped config): rows are gathered as stored and widened to fp32 in the aggregation
        self.x_bf16 = x.dtype == torch.bfloat16
        assert sampling_hops <= 7, "indicator bits are packed in 8 columns"
        self.x, self.y = (None if self.features is not None else x), y.contiguous()
        # main.py:89-100,116: `x` is a learned table (nn.Parameter inside optimizer_c); it is updated IN PLACE by every
        # optimiser step (dense Adam from the sparse classifier gradient, grapes_adam_embed)
        self.embed_nodes = bool(embed_nodes)
        if self.embed_nodes:
            assert x.dtype == torch.float32 and (x.F if self.features is not None else x.shape[1]) % 4 == 0, \
                "learned node features: fp32, width a multiple of 4"
        self.multilabel = (y.dim() == 2)
        if self.multilabel:
            self.y = self.y.to(torch.float32)
        else:
            self.y = self.y.to(torch.int64)
        N, F = graph.num_nodes, int(x.shape[1]) if self.features is None else x.F
        # TMA row copies need 16-byte rows: a table whose width is not a multiple of 4 floats (Reddit 602, Cora 1433) is
        # re-pitched once to ldx = round_up(F, 4); self.x stays the [N, F] view, the kernels get (F, ldx)
        self.ldx = F if self.features is None else x.ldx
        if self.features is None and x.dtype == torch.float32 and F % 4 != 0 and not embed_nodes:
            self.ldx = _round_up(F, 4)
            xp = torch.zeros((N, self.ldx), dtype=torch.float32, device=x.device)
            xp[:, :F].copy_(x)
            self.x = xp[:, :F]
        self.N, self.F, self.C, self.D = N, F, int(num_classes), int(hidden_dim)
        self.B, self.k, self.H = int(batch_size), int(num_samples), int(sampling_hops)
        self.use_ind = bool(use_indicators)
        self.num_ind = self.H + 1 if self.use_ind else 0
        self.Fp = F + self.num_ind
        self.ldY = _round_up(self.Fp, 4)
        # tcgen05 path: hidden dim a multiple of 128.  Any K: the forward promotes its tensor-core accumulator to an fp32
        # master every 256 columns (the tensor core adds with truncation; long chains drift past the 1e-5 bar) and the
        # backward walks Y in chunks of 128 columns.
        self.use_tc = bool(use_tensor_cores) and (self.D % 128 == 0) and self.D <= 512
        self.use_tc_bwd = self.use_tc and self.D // 128 <= 2    # backward accumulators: halves x (hi | lo) x 128 columns of TMEM
        # Fp <= 1024: the aggregation writes Y once as fp32 and the tcgen05 kernels split it into (hi, lo) themselves
        # (half the Y bytes written and read; the default forward k_l1_fwd_ts needs the raw fp32 Y: it splits it on the way into
        # tensor memory; products-shape: aggregation 73.8 -> 60.8,
        # forward 120 -> 136, backward 155 -> 149 us per step, step 0.512 -> 0.508 ms)
        self.y_single = self.use_tc and self.Fp <= 1024    # Cora-shape (K = 1436): the (hi, lo) pair is 2 % faster
        if self.use_tc_bwd:
            self.ldY = _round_up(self.Fp + 1, 4)           # room for the column of ones (bias column)
        self.ldW = _round_up(self.Fp, 4)
        self.lr_gc, self.lr_gf = float(lr_gc), float(lr_gf)
        self.loss_coef, self.log_z_init, self.reg_param = float(loss_coef), float(log_z_init), float(reg_param)
        self.random_sampling, self.reinforce = bool(random_sampling), bool(reinforce_baseline)
        W = graph.num_words
        self.W = W
        H = self.H

        # ---- streams: main = the caller's current stream; side A carries every hop's backward and the gcn_z
        # chain, side B the induced-block slices.  Each stream has its own library context (scan / split-K scratch).
        self.multi_stream = bool(multi_stream)
        if self.multi_stream:
            self.side_a, self.side_b = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
            self.side_p = torch.cuda.Stream(device=dev)          # front end of the NEXT batch (cross-step prefetch)
            self.ctx_a, self.ctx_b, self.ctx_p = graph.new_ctx(), graph.new_ctx(16 << 20), graph.new_ctx(16 << 20)
            # the backward / gcn_z branch is off the critical path: its persistent tcgen05 kernels get a share of the SMs
            # so the hop chain's small kernels are not queued behind them (measured, DESIGN.md section 9)
            # products / arxiv shape (K ~ 100): 96 of 148 SMs -> 0.549 -> 0.533 / 0.251 -> 0.236 ms/step; with long K
            # (Reddit 602, Cora 1433 columns) the backward is heavy enough to become the critical path when limited
            if (F + self.H + 1) <= 256:
                self.L.grapes_ctx_set_sm_limit(self.ctx_a, 96)
        else:
            self.side_a = self.side_b = self.side_p = None
            self.ctx_a = self.ctx_b = self.ctx_p = graph.ctx

        # ---- capacities -------------------------------------------------------------------
        self.cap_P = self.B + self.k
        deg = graph.indptr[1:] - graph.indptr[:-1]
        max_deg = int(deg.max().item()) if graph.nnz > 0 else 0
        if cap_edges is None:
            cap_edges = min(graph.nnz, self.cap_P * max(max_deg, 1), 1 << 26)
        self.cap_m = max(int(cap_edges), 1)
        if cap_nodes is None:
            cap_nodes = min(N, self.cap_m + self.cap_P)
        self.cap_n = max(int(cap_nodes), 1)
        self.cap_A = self.B + self.H * self.k
        if cap_block is None:
            cap_block = min(self.cap_m, self.cap_P * self.cap_P)
        self.cap_blk = max(int(cap_block), 1)
        if max(self.cap_m, self.cap_n) > graph.max_frontier:
            raise GrapesError("frontier capacity exceeds the graph context's max_frontier")

        i32 = dict(dtype=torch.int32, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        z = torch.zeros
        e = torch.empty
        cap_m, cap_n, cap_P = self.cap_m, self.cap_n, self.cap_P
        D, C = self.D, self.C

        # ---- parameters (flat), gradients, Adam state -------------------------------------
        self.net_c = _Net(0, F, D, C)
        self.net_gf = _Net(self.net_c.end, self.Fp, D, 1)
        self.net_z = _Net(self.net_gf.end, F, D, 1)
        n_par = self.net_z.end
        self.n_par = n_par

        self.pref_all = z(W + 1, **i32)
        self.ukeys = e(cap_n, **i32)
        self.sel_work = z(int(self.L.cdll.grapes_select_work_floats(graph.ctx, cap_n)), **f32)   # zero once: the library keeps its histogram clean
        self.overflow = z(1, **i32)
        self.rng_state = torch.tensor([seed & 0x7fffffffffffffff, 0], dtype=torch.int64, device=dev)
        # inverted dropout of gcn_c (modules/gcn.py:33,37): keep with probability 1 - p, as an integer threshold on 24 random
        # bits (llrint, so a host mirror reproduces the masks exactly); kept entries are scaled by 1 / (1 - p).  The masks
        # come from their own counter pair {seed, step}, advanced once per training step inside the step, so the sampler's
        # Philox stream (rng_state) is the same with and without dropout.
        self.dropout = dropout
        self.drop_threshold = int(round((1. - dropout) * (1 << 24)))
        self.drop_scale = 1. / (1. - dropout) if dropout < 1. else 0.
        self.drop_state = torch.tensor([seed & 0x7fffffffffffffff, 0], dtype=torch.int64, device=dev)
        # ---- two step states (see _alloc_step_state); self.<buffer> always refers to the ACTIVE one ----
        base_names = set(self.__dict__)
        self._states = []
        for _ in range(2):
            self._alloc_step_state()
            self._states.append({k: v for k, v in self.__dict__.items() if k not in base_names and k != "_states"})
        self.par = 0
        self._activate(0)
        self._front_ready = [False, False]       # hop-0 front end of the state already enqueued (prefetched)
        self._pref_key = None                    # (data_ptr, numel) of the targets the prefetched front end was built from
        self._prefetch_next = False              # this step enqueues the other state's front end next to its classifier tail
        need_Y = not self.random_sampling
        # sampler-net scratch
        if need_Y:
            if self.use_tc:
                self.Wgf_hi, self.Wgf_lo = z((D, self.ldW), **f32), z((D, self.ldW), **f32)
                self.Wz_hi, self.Wz_lo = z((D, self.ldW), **f32), z((D, self.ldW), **f32)
                self.zpart, self.zpart_z = z((2 * (D // 128), cap_n), **f32), z((2 * (D // 128), cap_n), **f32)   # two partial rows per 128-unit half
                if self.use_tc_bwd:
                    self.mask_z = z(((cap_n + 127) // 128 * 4, D), **i32)
            else:
                self.z_gf, self.z_z = e(cap_n, **f32), e(cap_n, **f32)
            self.zlogits, self.dz_z = e(cap_n, **f32), e(cap_n, **f32)
            self.dpre = e((1 if self.use_tc_bwd else cap_n, D), **f32)
        self.const100 = torch.full((cap_n,), 100.0, **f32)
        # classifier workspace
        A = self.cap_A
        self.all_nodes = e(A, **i32)
        self.target_local = e(self.B, **i32)
        self.tgt_of_row = e(A, **i32)
        self.cl_src = [e(self.cap_blk, **i32) for _ in range(2)]      # [0]: layer-1 block (last hop), [1]: layer-2 block (hop 0)
        self.cl_dst = [e(self.cap_blk, **i32) for _ in range(2)]
        self.cl_in_off = [z(A + 1, **i32) for _ in range(2)]
        self.cl_in_src = [e(self.cap_blk, **i32) for _ in range(2)]
        self.cl_dinv = [e(A, **f32) for _ in range(2)]
        self.cl_out_off = z(A + 1, **i32)
        self.cl_out_dst = e(self.cap_blk, **i32)
        self.cl_tmp = e(self.cap_blk, **i32)
        self.Yc = z((A, _round_up(F, 4)), **f32)
        self.out1 = e((A, D), **f32)
        self.Zc = e((A, C), **f32)
        self.logits_c = z((A, C), **f32)
        self.dlogits = z((A, C), **f32)
        self.dZ = e((A, C), **f32)
        self.dpre1 = e((A, D), **f32)
        if self.embed_nodes:
            # d loss_c / d x[all_nodes] = A_hat_1^T (dpre1 W1): needs the layer-1 block keyed by SOURCE as well
            self.cl_out_off0 = z(A + 1, **i32)
            self.cl_out_dst0 = e(self.cap_blk, **i32)
            self.dYc = z((A, _round_up(F, 4)), **f32)
            self.dXc = z((A, _round_up(F, 4)), **f32)
            if self.embed_shards is None:                 # a sharded table keeps the moments of its rows itself
                self.emb_exp_avg, self.emb_exp_avg_sq = torch.zeros_like(x), torch.zeros_like(x)

        self.params = z(n_par, **f32)
        self.grads = z(n_par, **f32)
        self.exp_avg, self.exp_avg_sq = z(n_par, **f32), z(n_par, **f32)
        self.adam_steps = z(2, **f32)        # [0] optimizer_c, [1] optimizer_gf
        gen = torch.Generator().manual_seed(seed)
        for net in (self.net_c, self.net_gf, self.net_z):
            v = net.views(self.params)
            glorot_(v["gcn_layers.0.lin.weight"], gen)
            glorot_(v["gcn_layers.1.lin.weight"], gen)
        self._graphs: Dict[tuple, torch.cuda.CUDAGraph] = {}
        # data parallelism (enable_data_parallel): the step owns the gradient exchange and the optimiser launch
        self.peer = None                         # PeerGradExchange when the exchange runs over NVLink peer memory
        self.dp_group = None                     # process group of the NCCL exchange
        self.dp_world, self.dp_rank = 1, 0
        self.epoch_spin_limit = 0                # tries of grapes_embed_epoch_wait (0: the step tail's bound)
        self.tail_state = torch.zeros(int(self.L.cdll.grapes_peer_state_words()), dtype=torch.int32, device=dev)
        self._graph_launches: Dict[tuple, int] = {}
        self.launches_per_graph = 0
        self.record: Optional[dict] = None
        # timing experiments only (scripts/ablate.py): leave out parts of the step to see what the rest costs
        self.ablate = set()
        # where the gcn_z chain sits on the backward branch: behind the LAST hop's backward it overlaps the classifier tail
        # (small kernels) instead of hop 1's aggregation + GEMM: products 0.533 -> 0.511 ms/step; neutral with long K
        self.z_at = "last" if (F + self.H + 1) <= 256 else "hop0"

    def _alloc_step_state(self):
        """Every buffer that belongs to ONE step in flight (bitmap / scalar pool, id lists, device-side sizes, per-hop
        workspaces).  Allocated twice: the engine keeps two step states so the weight-independent front end of the NEXT
        batch (expand .. aggregate of hop 0) can be enqueued next to the classifier tail of the current one."""
        dev, H, W, N, F, D = self.device, self.H, self.W, self.N, self.F, self.D
        n_par = self.n_par
        cap_m, cap_n, cap_P = self.cap_m, self.cap_n, self.cap_P
        i32 = dict(dtype=torch.int32, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        z = torch.zeros
        e = torch.empty
        need_Y = not self.random_sampling
        # ---- ONE pool that is cleared by ONE memset at the start of every step:
        #   bitmaps (int32 words): all_nodes | indicator rows | prev rows of hop 0..H-1 | batch rows of hop 0..H-1 | prev rows H
        #   floats: scalars | per-hop stats | gradient direction of the sampler nets
        #   (+ with a learned table: the union of the ranks' rows of a data-parallel step, grapes_embed_merge_adam)
        n_bm = 1 + max(self.num_ind, 1) + 2 * H + 1
        n_fl = 16 + 4 * H + n_par
        n_un = 1 if self.embed_nodes else 0
        self.step_pool = z((n_bm + n_un) * W + n_fl, **i32)
        bm = self.step_pool[:n_bm * W].view(n_bm, W)
        if self.embed_nodes:
            self.bm_union = self.step_pool[n_bm * W:(n_bm + 1) * W]
        self.bm_all = bm[0]
        self.bm_ind = bm[1:1 + max(self.num_ind, 1)]
        self.bm_prev = [bm[1 + max(self.num_ind, 1) + h] for h in range(H)] + [bm[n_bm - 1]]   # [H]: rows of the last block (evaluation)
        self.bm_batch = [bm[1 + max(self.num_ind, 1) + H + h] for h in range(H)]
        fl = self.step_pool[(n_bm + n_un) * W:].view(torch.float32)
        self.zero_pool = fl
        self.scal = fl[:16]
        self.stats = fl[16:16 + 4 * H].view(H, 4)
        self.scal_stats = fl[:16 + 4 * H]    # one contiguous read-back: losses, overflow bits, per-hop sampler statistics
        self.gdir = fl[16 + 4 * H:]          # gradient DIRECTION of (log_z, sum log_prob) w.r.t. gf / z params
        self.pref_batch, self.pref_nb = z(W + 1, **i32), z(W + 1, **i32)

        # ---- id lists and device-side sizes ------------------------------------------------
        self.targets = z(self.B, **i32)
        self.prev_pool = z((H + 1, cap_P), **i32)            # prev[h] = rows expanded at hop h; prev[H] = last block's rows
        self.prev = [self.prev_pool[h] for h in range(H + 1)]
        self.counts = z(16 * (H + 2), **i32)                 # [0:16] globals, then one 16-int block per hop (+ final)
        self.cnt_scratch = z(max(cap_n, self.cap_A), **i32)
        self.tmp_val = e(cap_m, **i32)
        self.log_prob = z((H, cap_n), **f32)

        # ---- per-hop workspaces ------------------------------------------------------------
        self.hops: List[_Hop] = []
        for h in range(H):
            hw = _Hop()
            hw.row_off = z(cap_P + 1, **i32)
            hw.e_row, hw.e_col = e(cap_m, **i32), e(cap_m, **i32)
            hw.e_src, hw.e_dst = e(cap_m, **i32), e(cap_m, **i32)
            hw.batch_nodes, hw.nb_nodes, hw.nb_local = e(cap_n, **i32), e(cap_n, **i32), e(cap_n, **i32)
            hw.nb_index = e(cap_n, **i32)
            hw.ind_bits = z(cap_n, **i32)
            hw.in_off, hw.in_src, hw.dinv = z(cap_n + 1, **i32), e(cap_m, **i32), e(cap_n, **f32)
            hw.logits_all, hw.dl_all, hw.dz = z(cap_n, **f32), z(cap_n, **f32), e(cap_n, **f32)
            hw.Y = hw.Y_lo = hw.mask_gf = None
            if need_Y:
                # tensor-core path: (Y, Y_lo) is the 3xTF32 (hi, lo) pair written by the aggregation; else plain fp32 Y
                hw.Y = z((cap_n, self.ldY), **f32)
                if self.use_tc and not self.y_single:
                    hw.Y_lo = z((cap_n, self.ldY), **f32)
                if self.use_tc_bwd:
                    hw.mask_gf = z(((cap_n + 127) // 128 * 4, D), **i32)
            hw.blk_src, hw.blk_dst = e(self.cap_blk, **i32), e(self.cap_blk, **i32)
            self.hops.append(hw)
        # expansion of the last block's rows (T u S_{H-1})
        self.fin_row_off = z(cap_P + 1, **i32)
        self.fin_e_row, self.fin_e_col = e(cap_m, **i32), e(cap_m, **i32)
        self.bsz = self.B                   # current batch size (<= capacity B); the last batch of an epoch is partial

    def _activate(self, p: int):
        self.__dict__.update(self._states[p])
        self.par = p

    # ------------------------------------------------------------------ helpers
    _CNT = dict(B=0, A=1, cl_nnz=2, U=6)

    def _cnt(self, name: str, idx: int = 0) -> int:
        """device address of a global size (B, A, cl_nnz[0..3], U: union rows of a data-parallel table step)"""
        return self.counts.data_ptr() + 4 * (self._CNT[name] + idx)

    def _hc(self, h: int, name: str) -> int:
        """device address of a per-hop size (P, m, n, c, nnz, s, blk); h == H is the last block's row list"""
        return self.counts.data_ptr() + 4 * (16 * (h + 1) + _Hop.CNT[name])

    def _par(self, off: int) -> int:
        return self.params.data_ptr() + 4 * off

    def _dir(self, off: int) -> int:
        return self.gdir.data_ptr() + 4 * off

    def _grd(self, off: int) -> int:
        return self.grads.data_ptr() + 4 * off

    def _scal(self, name: str) -> int:
        return self.scal.data_ptr() + 4 * SCAL[name]

    def _drop_tag(self, site: int) -> int:
        """Philox counter word of a dropout site (0: hidden layer, 1: logits) on this rank: data-parallel ranks draw
        independent masks, and rank 0 of any world draws what one GPU draws"""
        return 1 + site + 2 * self.dp_rank

    def state_dicts(self) -> Dict[str, Dict[str, torch.Tensor]]:
        return {"gcn_c": self.net_c.views(self.params), "gcn_gf": self.net_gf.views(self.params),
                "gcn_z": self.net_z.views(self.params)}

    def grad_dicts(self) -> Dict[str, Dict[str, torch.Tensor]]:
        return {"gcn_c": self.net_c.views(self.grads), "gcn_gf": self.net_gf.views(self.grads),
                "gcn_z": self.net_z.views(self.grads)}

    def load_state_dicts(self, gcn_c=None, gcn_gf=None, gcn_z=None):
        for net, sd in ((self.net_c, gcn_c), (self.net_gf, gcn_gf), (self.net_z, gcn_z)):
            if sd is None:
                continue
            v = net.views(self.params)
            for name, t in v.items():
                t.copy_(sd[name].detach().to(self.device, torch.float32))

    # ------------------------------------------------------------------ the step
    def _enqueue(self, gumbel_noise: Optional[Sequence[Optional[torch.Tensor]]], apply_optim: bool,
                 noise_mode: int = NOISE_GUMBEL):
        L, g = self.L, self.g
        main = torch.cuda.current_stream()
        multi = self.multi_stream and self.side_a is not None
        ctx, st = g.ctx, main.cuda_stream
        ctx_a, ctx_b = self.ctx_a, self.ctx_b
        sA, sB, sP = (self.side_a, self.side_b, self.side_p) if multi else (main, main, main)
        stA, stB, stP = sA.cuda_stream, sB.cuda_stream, sP.cuda_stream
        on = (lambda s: torch.cuda.stream(s)) if multi else (lambda s: contextlib.nullcontext())

        forked = set()

        def fork(side):                     # `side` continues from everything enqueued on main so far
            if multi:
                side.wait_stream(main)
                forked.add(side)

        def join(side):                     # only streams that took part in this step (graph capture forbids others)
            if multi and side in forked:
                main.wait_stream(side)
                forked.discard(side)

        B, k, H, F, Fp, D, C, W = self.bsz, self.k, self.H, self.F, self.Fp, self.D, self.C, self.W
        cap_P, cap_m, cap_n = self.cap_P, self.cap_m, self.cap_n
        ovf = ptr(self.overflow)
        rec = self.record
        indptr, indices, X = ptr(g.indptr), ptr(g.indices), ptr(self.x)
        need_Y = not self.random_sampling
        tc = self.use_tc
        gf, nz = self.net_gf, self.net_z

        self._enqueue_epoch_wait(ctx, st)
        # ---- per-batch reset + hop-0 front end: already enqueued next to the previous step's classifier tail when this
        # state was prefetched (step(..., next_targets=...)), else inline ----
        if self._front_ready[self.par]:
            self._front_ready[self.par] = False
        else:
            self._enqueue_front0(ctx, st)

        self._enqueue_prefetch(fork, on, sP, stP)

        for h in range(H):
            hw = self.hops[h]
            rows, P_dev = ptr(self.prev[h]), self._hc(h, "P")
            m_dev, n_dev, c_dev = self._hc(h, "m"), self._hc(h, "n"), self._hc(h, "c")
            if h > 0:
                # get_neighborhoods + mask dedup (main.py:180-190)
                L.grapes_expand_frontier(ctx, indptr, indices, rows, P_dev, cap_P, ptr(hw.row_off), m_dev, cap_m,
                                         ptr(hw.e_row), ptr(hw.e_col), ptr(self.bm_prev[h]), ptr(self.bm_batch[h]), ovf, st)
                # slice_adjacency(rows = T u S_{h-1}, cols = prev_{h-1}) (main.py:241-244): same row expansion; side B
                pw = self.hops[h - 1]
                fork(sB)
                with on(sB):
                    L.grapes_slice_block(ctx_b, rows, ptr(hw.e_row), ptr(hw.e_col), m_dev, cap_m,
                                         ptr(self.bm_prev[h - 1]), ptr(pw.blk_src), ptr(pw.blk_dst), self.cap_blk,
                                         self._hc(h - 1, "blk"), ovf, stB)
                self._enqueue_hop_graph(h, ctx, st)
            if need_Y:
                if tc:
                    if h == 0:
                        self._split_weights(ctx, st)
                    L.grapes_sampler_l1_fwd_tc(ctx, ptr(hw.Y), ptr(hw.Y_lo), self.ldY, n_dev, cap_n, Fp,
                                               ptr(self.Wgf_hi), ptr(self.Wgf_lo), self.ldW, D, self._par(gf.b1),
                                               self._par(gf.W2), ptr(self.zpart), ptr(hw.mask_gf), st)
                    z_ptr, z_parts, z_stride = ptr(self.zpart), 2 * (D // 128), cap_n
                else:
                    L.grapes_sampler_l1_fwd(ctx, ptr(hw.Y), self.ldY, n_dev, cap_n, Fp, self._par(gf.W1), Fp, D,
                                            self._par(gf.b1), self._par(gf.W2), ptr(self.z_gf), st)
                    z_ptr, z_parts, z_stride = ptr(self.z_gf), 1, 0
            noise = None if gumbel_noise is None else gumbel_noise[h]
            mode = noise_mode if noise is not None else NOISE_PHILOX
            lp = self.log_prob.data_ptr() + 4 * cap_n * h
            # layer 2 of gcn_gf at width 1 -> logits (main.py:210-213), then sample_neighborhoods_from_probs
            # (utils.py:13-71): keys, Gumbel-top-k, log-probs, stats, d(sum log_prob)/d logits
            if need_Y:
                agg = (z_ptr, z_parts, z_stride, n_dev, cap_n, ptr(hw.in_off), ptr(hw.in_src), ptr(hw.dinv),
                       self._par(gf.b2))
            else:
                agg = (ptr(self.const100), 1, 0, n_dev, cap_n, None, None, None, None)        # main.py:207
            L.grapes_select_hop(ctx, *agg, ptr(hw.nb_index), ptr(hw.nb_local), ptr(hw.nb_nodes), c_dev, k, mode,
                                ptr(noise), ptr(self.rng_state), ptr(self.sel_work), ptr(self.ukeys),
                                ptr(hw.logits_all) if need_Y else None,
                                ptr(rec["keys"][h]) if rec is not None else None,
                                ptr(self.prev[h + 1]), B, self._hc(h, "s"), self._hc(h + 1, "P"), None, lp,
                                self._scal("tot_log_prob"), self.stats.data_ptr() + 16 * h,
                                ptr(hw.dl_all) if need_Y else None,
                                self._dir(gf.b2) if need_Y else None, ptr(self.bm_all), st)
            if need_Y and "nobwd" not in self.ablate:
                # ---- side A: d(sum log_prob)/d(theta_gf), direction accumulated now, scaled by g at the end ----
                fork(sA)
                with on(sA):
                    self._enqueue_hop_backward(h, ctx_a, stA)
                    if h == H - 1 and self.z_at != "hop0":
                        self._enqueue_gcn_z(ctx_a, stA)

        # ---- last block: slice_adjacency(rows = T u S_{H-1}, cols = prev_{H-1}) ----
        rows, P_dev, m_dev = ptr(self.prev[H]), self._hc(H, "P"), self._hc(H, "m")
        L.grapes_expand_frontier(ctx, indptr, indices, rows, P_dev, cap_P, ptr(self.fin_row_off), m_dev, cap_m,
                                 ptr(self.fin_e_row), ptr(self.fin_e_col), None, None, ovf, st)
        lw = self.hops[H - 1]
        join(sB)                                                                  # earlier blocks + frees ctx_b's scratch order
        L.grapes_slice_block(ctx, rows, ptr(self.fin_e_row), ptr(self.fin_e_col), m_dev, cap_m,
                             ptr(self.bm_prev[H - 1]), ptr(lw.blk_src), ptr(lw.blk_dst), self.cap_blk,
                             self._hc(H - 1, "blk"), ovf, st)

        if "nocls" in self.ablate:
            join(sA)
            join(sP)
            return
        self._enqueue_classifier_forward(ctx, st, training=True)
        L.tag = "[cls]"
        nc = self.net_c
        ldYc = self.Yc.shape[1]
        A_dev, cap_A = self._cnt("A"), self.cap_A
        # loss + d loss / d logits + d loss / d b2 (column sums) in one launch (main.py:260-261)
        loss_args = (ctx, ptr(self.logits_c), C, C, A_dev, cap_A, ptr(self.target_local),
                     ptr(self.tgt_of_row) if self.cap_A <= self.PREP_MAX_ROWS else None, ptr(self.targets), B,
                     None if self.multilabel else ptr(self.y), ptr(self.y) if self.multilabel else None, self.reg_param,
                     ptr(self.dlogits), self._scal("loss_c"), self._grd(nc.b2))
        if self.dropout > 0:
            # on dropout(logits) (modules/gcn.py:37); the last launch advances drop_state (every reader has run)
            L.grapes_classifier_loss_dropout(*loss_args, ptr(self.drop_state), self._drop_tag(1), self.drop_threshold,
                                             self.drop_scale, st)
        else:
            L.grapes_classifier_loss(*loss_args, st)
        # backward of the classifier (loss_c.backward(), main.py:267); the two weight-gradient products that nothing
        # else waits for run on side B next to the chain dZ -> dpre1 -> dW1
        L.grapes_aggregate(ctx, ptr(self.dlogits), C, C, None, A_dev, cap_A, ptr(self.cl_out_off),
                           ptr(self.cl_out_dst), ptr(self.cl_dinv[1]), None, 0, None, 0, ptr(self.dZ), C, None, None, -1, st)
        fork(sB)
        with on(sB):
            L.grapes_gemm_tn(ctx_b, ptr(self.dZ), C, ptr(self.out1), D, A_dev, cap_A, C, D, 1.0, 0, self._grd(nc.W2), stB)
        if self.dropout > 0:
            # out1 holds dropout(relu(pre1)): zero wherever the unit is inactive or dropped, so the gate is relu' * keep
            L.grapes_gemm_gated_scaled(ctx, ptr(self.dZ), C, self._par(nc.W2), D, ptr(self.dpre1), D, A_dev, cap_A, D, C,
                                       ptr(self.out1), D, self.drop_scale, st)
        else:
            L.grapes_gemm(ctx, 1, ptr(self.dZ), C, self._par(nc.W2), D, ptr(self.dpre1), D, A_dev, cap_A, D, C, None, 0,
                          ptr(self.out1), D, st)
        fork(sB)
        with on(sB):
            L.grapes_colsum(ctx_b, ptr(self.dpre1), A_dev, cap_A, D, D, 1.0, 0, self._grd(nc.b1), stB)
        L.grapes_gemm_tn(ctx, ptr(self.dpre1), D, ptr(self.Yc), ldYc, A_dev, cap_A, D, F, 1.0, 0, self._grd(nc.W1),
                         st)
        if self.embed_nodes:
            # d loss_c / d x[all_nodes] (main.py:267 with embeddings in optimizer_c): dYc = dpre1 W1, dX = A_hat_1^T dYc
            L.grapes_gemm(ctx, 1, ptr(self.dpre1), D, self._par(nc.W1), F, ptr(self.dYc), ldYc, A_dev, cap_A, F, D,
                          None, 0, None, 0, st)
            L.grapes_aggregate(ctx, ptr(self.dYc), F, ldYc, None, A_dev, cap_A, ptr(self.cl_out_off0),
                               ptr(self.cl_out_dst0), ptr(self.cl_dinv[0]), None, 0, None, 0, ptr(self.dXc), ldYc,
                               None, None, -1, st)
        L.tag = ""
        # ---- GFlowNet / REINFORCE loss (main.py:271-291): loss, gradient scale, scaled directions in one launch ----
        join(sB)
        join(sA)
        join(sP)
        if apply_optim:
            self._enqueue_tail(st)
        elif not self.random_sampling:
            n_z = 0 if self.reinforce else nz.size
            L.grapes_gfn_finalize_scale(ctx, ptr(self.scal), self.loss_coef, self.log_z_init, int(self.reinforce), 1,
                                        self._dir(gf.base), gf.size, self._grd(gf.base),
                                        self._dir(nz.base), n_z, self._grd(nz.base), st)

    def _enqueue_classifier_forward(self, ctx, st, training: bool):
        """all_nodes + relabel of the per-hop blocks + gcn_norm structure of the classifier's two layers, then
        logits = gcn_c(x[all_nodes], [block_0 .. block_{H-1}]) (main.py:252-257, eval.py:147-151).  ``training``: the
        hidden layer is dropped (modules/gcn.py:33); the logits are dropped by the training step's loss launch."""
        L = self.L
        H, F, D, C, B = self.H, self.F, self.D, self.C, self.bsz
        ovf = ptr(self.overflow)
        # ---- classifier on the sampled subgraph (main.py:252-269) ----
        L.tag = "[cls]"
        L.grapes_rank_nodes(ctx, ptr(self.bm_all), None, ptr(self.pref_all), None, ptr(self.all_nodes), None, None,
                            None, None, None, 0, 0, self.cap_A, self._cnt("A"), None, ovf, st)
        # GCN.forward with a per-layer list: hidden layer <- edge_indices[-1], last layer <- edge_indices[0] (gcn.py:30-36)
        b0, b1 = self.hops[H - 1], self.hops[0]
        if self.cap_A <= self.PREP_MAX_ROWS:
            L.grapes_classifier_prep(ctx, ptr(self.bm_all), ptr(self.pref_all), self._cnt("A"), self.cap_A,
                                     ptr(self.targets), self._cnt("B"), B, ptr(self.target_local),
                                     ptr(b0.blk_src), ptr(b0.blk_dst), self._hc(H - 1, "blk"),
                                     ptr(b1.blk_src), ptr(b1.blk_dst), self._hc(0, "blk"), self.cap_blk,
                                     ptr(self.cl_src[0]), ptr(self.cl_dst[0]), ptr(self.cl_src[1]), ptr(self.cl_dst[1]),
                                     ptr(self.cl_in_off[0]), ptr(self.cl_in_src[0]), ptr(self.cl_dinv[0]),
                                     ptr(self.cl_in_off[1]), ptr(self.cl_in_src[1]), ptr(self.cl_dinv[1]),
                                     ptr(self.cl_out_off), ptr(self.cl_out_dst), ptr(self.cl_tmp),
                                     self._cnt("cl_nnz"), ptr(self.tgt_of_row), st)
        else:
            L.grapes_relabel(ctx, ptr(self.targets), self._cnt("B"), B, ptr(self.bm_all), ptr(self.pref_all),
                             ptr(self.target_local), st)
            for slot, hop in ((0, H - 1), (1, 0)):
                bw = self.hops[hop]
                L.grapes_relabel(ctx, ptr(bw.blk_src), self._hc(hop, "blk"), self.cap_blk, ptr(self.bm_all),
                                 ptr(self.pref_all), ptr(self.cl_src[slot]), st)
                L.grapes_relabel(ctx, ptr(bw.blk_dst), self._hc(hop, "blk"), self.cap_blk, ptr(self.bm_all),
                                 ptr(self.pref_all), ptr(self.cl_dst[slot]), st)
                L.grapes_build_csr(ctx, ptr(self.cl_dst[slot]), ptr(self.cl_src[slot]), self._hc(hop, "blk"),
                                   self.cap_blk, self._cnt("A"), self.cap_A, ptr(self.cnt_scratch), 0,
                                   ptr(self.cl_in_off[slot]), ptr(self.cl_in_src[slot]), ptr(self.cl_tmp),
                                   ptr(self.cl_dinv[slot]), self._cnt("cl_nnz", slot), ovf, st)
            L.grapes_build_csr(ctx, ptr(self.cl_src[1]), ptr(self.cl_dst[1]), self._hc(0, "blk"), self.cap_blk,
                               self._cnt("A"), self.cap_A, ptr(self.cnt_scratch), 0, ptr(self.cl_out_off),
                               ptr(self.cl_out_dst), ptr(self.cl_tmp), None, self._cnt("cl_nnz", 2), ovf, st)
        nc = self.net_c
        ldYc = self.Yc.shape[1]
        A_dev, cap_A = self._cnt("A"), self.cap_A
        if self.embed_nodes:
            L.grapes_build_csr(ctx, ptr(self.cl_src[0]), ptr(self.cl_dst[0]), self._hc(H - 1, "blk"), self.cap_blk,
                               A_dev, cap_A, ptr(self.cnt_scratch), 0, ptr(self.cl_out_off0), ptr(self.cl_out_dst0),
                               ptr(self.cl_tmp), None, self._cnt("cl_nnz", 3), ovf, st)
        self._aggregate_x(ctx, ptr(self.all_nodes), A_dev, cap_A, ptr(self.cl_in_off[0]), ptr(self.cl_in_src[0]),
                          ptr(self.cl_dinv[0]), None, 0, ptr(self.Yc), ldYc, None, None, -1, st)
        if training and self.dropout > 0:
            L.grapes_gemm_bias_relu_dropout(ctx, ptr(self.Yc), ldYc, self._par(nc.W1), F, ptr(self.out1), D, A_dev, cap_A,
                                            D, F, self._par(nc.b1), ptr(self.drop_state), self._drop_tag(0),
                                            self.drop_threshold, self.drop_scale, st)
        else:
            L.grapes_gemm(ctx, 3, ptr(self.Yc), ldYc, self._par(nc.W1), F, ptr(self.out1), D, A_dev, cap_A, D, F,
                          self._par(nc.b1), 1, None, 0, st)
        L.grapes_gemm(ctx, 3, ptr(self.out1), D, self._par(nc.W2), D, ptr(self.Zc), C, A_dev, cap_A, C, D, None, 0,
                      None, 0, st)
        L.grapes_aggregate(ctx, ptr(self.Zc), C, C, None, A_dev, cap_A, ptr(self.cl_in_off[1]),
                           ptr(self.cl_in_src[1]), ptr(self.cl_dinv[1]), None, 0, self._par(nc.b2), 0,
                           ptr(self.logits_c), C, None, None, -1, st)
        L.tag = ""

    def _enqueue_eval(self, pred_ptr):
        """The mini-batch evaluator's batch body (/root/reference/eval.py:84-153) on the training step's kernels, forward
        only: per hop the sampler GCN's logits, DETERMINISTIC top-k on the probabilities (eval.py:126-130,
        GRAPES_NOISE_NONE_TOPK_PROBS) and -- unlike training -- the block ``A[rows = previous_nodes][:, cols = T u sampled]``
        (eval.py:140-142), which is a filter of the hop's OWN row expansion; then the classifier forward and the argmax of
        the target rows.  One stream, no host synchronisation, graph-capturable."""
        L, g = self.L, self.g
        ctx, st = g.ctx, torch.cuda.current_stream().cuda_stream
        if self.random_sampling:
            raise GrapesError("mini-batch evaluation runs the sampler net (eval.py:121): build the engine with random_sampling=False")
        B, k, H, Fp, D = self.bsz, self.k, self.H, self.Fp, self.D
        cap_P, cap_m, cap_n = self.cap_P, self.cap_m, self.cap_n
        ovf = ptr(self.overflow)
        gf = self.net_gf
        self._front_ready = [False, False]
        self._enqueue_epoch_wait(ctx, st)
        self._enqueue_front0(ctx, st)
        for h in range(H):
            hw = self.hops[h]
            rows, P_dev = ptr(self.prev[h]), self._hc(h, "P")
            m_dev, n_dev, c_dev = self._hc(h, "m"), self._hc(h, "n"), self._hc(h, "c")
            if h > 0:
                L.grapes_expand_frontier(ctx, ptr(g.indptr), ptr(g.indices), rows, P_dev, cap_P, ptr(hw.row_off), m_dev,
                                         cap_m, ptr(hw.e_row), ptr(hw.e_col), ptr(self.bm_prev[h]), ptr(self.bm_batch[h]),
                                         ovf, st)
                self._enqueue_hop_graph(h, ctx, st)
            if self.use_tc:
                if h == 0:
                    self._split_weights(ctx, st)
                L.grapes_sampler_l1_fwd_tc(ctx, ptr(hw.Y), ptr(hw.Y_lo), self.ldY, n_dev, cap_n, Fp, ptr(self.Wgf_hi),
                                           ptr(self.Wgf_lo), self.ldW, D, self._par(gf.b1), self._par(gf.W2),
                                           ptr(self.zpart), ptr(hw.mask_gf), st)
                z_ptr, z_parts, z_stride = ptr(self.zpart), 2 * (D // 128), cap_n
            else:
                L.grapes_sampler_l1_fwd(ctx, ptr(hw.Y), self.ldY, n_dev, cap_n, Fp, self._par(gf.W1), Fp, D,
                                        self._par(gf.b1), self._par(gf.W2), ptr(self.z_gf), st)
                z_ptr, z_parts, z_stride = ptr(self.z_gf), 1, 0
            L.grapes_select_hop(ctx, z_ptr, z_parts, z_stride, n_dev, cap_n, ptr(hw.in_off), ptr(hw.in_src), ptr(hw.dinv),
                                self._par(gf.b2), ptr(hw.nb_index), ptr(hw.nb_local), ptr(hw.nb_nodes), c_dev, k,
                                NOISE_TOPK_PROBS, None, ptr(self.rng_state), ptr(self.sel_work), ptr(self.ukeys),
                                ptr(hw.logits_all), None, ptr(self.prev[h + 1]), B, self._hc(h, "s"), self._hc(h + 1, "P"),
                                None, None, None, None, None, None, ptr(self.bm_all), st)
            # eval.py:140-142: rows = previous_nodes (the hop's expansion), cols = cat(targets, sampled)
            L.grapes_bitmap_set(ctx, ptr(self.prev[h + 1]), self._hc(h + 1, "P"), cap_P, ptr(self.bm_prev[h + 1]), st)
            L.grapes_slice_block(ctx, rows, ptr(hw.e_row), ptr(hw.e_col), m_dev, cap_m, ptr(self.bm_prev[h + 1]),
                                 ptr(hw.blk_src), ptr(hw.blk_dst), self.cap_blk, self._hc(h, "blk"), ovf, st)
        self._enqueue_classifier_forward(ctx, st, training=False)          # evaluation never drops
        # predictions = argmax(logits)[node_map.map(target_nodes)]   (eval.py:152-153)
        L.grapes_argmax_rows(ctx, ptr(self.logits_c), self.C, self.C, ptr(self.target_local), self._cnt("B"), self.B,
                             pred_ptr, st)

    def predict(self, target_nodes: torch.Tensor, out: torch.Tensor, use_graph: bool = True):
        """Class predictions of one evaluation batch (eval.py:84-153) written to ``out[:len(target_nodes)]`` (int32, device).
        Enqueues only; the caller synchronises once after the last batch."""
        assert out.dtype == torch.int32 and out.is_cuda and out.is_contiguous()
        self.set_targets(target_nodes)
        self._pref_key = None
        if not use_graph:
            self._enqueue_eval(out.data_ptr())
            return
        # the output address is baked into the captured launch: predictions land in a fixed buffer, then one copy
        if not hasattr(self, "_pred_buf"):
            self._pred_buf = torch.zeros(self.B, dtype=torch.int32, device=self.device)
        key = ("eval", self.bsz, self.par)
        gr = self._graphs.get(key)
        if gr is None:
            self._enqueue_eval(self._pred_buf.data_ptr())            # warm-up outside capture (deterministic: no RNG)
            torch.cuda.synchronize()
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                self._enqueue_eval(self._pred_buf.data_ptr())
            self._graphs[key] = gr
        gr.replay()
        out[:self.bsz].copy_(self._pred_buf[:self.bsz])

    def _enqueue_prefetch(self, fork, on, sP, stP):
        # ---- cross-step prefetch: the hop chain and the classifier tail of THIS batch are chains of small, latency-bound
        # kernels -> the reset and the weight-independent hop-0 front end of the NEXT batch run next to them on the other
        # step state (own stream, own scan scratch; joined before the optimiser step) ----
        if not self._prefetch_next:
            return
        cur = self.par
        fork(sP)
        self._activate(1 - cur)
        try:
            with on(sP):
                self._enqueue_front0(self.ctx_p, stP)
        finally:
            self._activate(cur)
        self._front_ready[1 - cur] = True

    def _enqueue_hop_graph(self, h: int, ctx, st):
        """After the row expansion of hop h: mask dedup + id lists + indicator bits (main.py:183-195), local relabel,
        gcn_norm structure of the hop graph (dst-sorted CSR, deg^-1/2) and Y = A_hat [x | indicators] (feature gather
        fused, main.py:198-204 + GCNConv aggregation).  None of it depends on the weights."""
        L = self.L
        hw = self.hops[h]
        cap_m, cap_n = self.cap_m, self.cap_n
        rows = ptr(self.prev[h])
        m_dev, n_dev, c_dev = self._hc(h, "m"), self._hc(h, "n"), self._hc(h, "c")
        ovf = ptr(self.overflow)
        L.grapes_rank_nodes(ctx, ptr(self.bm_batch[h]), ptr(self.bm_prev[h]), ptr(self.pref_batch),
                            ptr(self.pref_nb), ptr(hw.batch_nodes), ptr(hw.nb_nodes), ptr(hw.nb_local),
                            ptr(hw.nb_index), ptr(hw.ind_bits) if self.use_ind else None,
                            ptr(self.bm_ind) if self.use_ind else None, self.num_ind, h, cap_n,
                            n_dev, c_dev, ovf, st)
        L.grapes_edges_to_local(ctx, rows, ptr(hw.e_row), ptr(hw.e_col), m_dev, cap_m, ptr(self.bm_batch[h]),
                                ptr(self.pref_batch), cap_n, ptr(hw.e_src), ptr(hw.e_dst), ptr(self.cnt_scratch), st)
        L.grapes_build_csr(ctx, ptr(hw.e_dst), ptr(hw.e_src), m_dev, cap_m, n_dev, cap_n, ptr(self.cnt_scratch),
                           1, ptr(hw.in_off), ptr(hw.in_src), ptr(self.tmp_val), ptr(hw.dinv),
                           self._hc(h, "nnz"), ovf, st)
        if not self.random_sampling:
            tc = self.use_tc
            self._aggregate_x(ctx, ptr(hw.batch_nodes), n_dev, cap_n, ptr(hw.in_off), ptr(hw.in_src), ptr(hw.dinv),
                              ptr(hw.ind_bits) if self.use_ind else None, self.num_ind,
                              None if (tc and not self.y_single) else ptr(hw.Y), self.ldY,
                              ptr(hw.Y) if (tc and not self.y_single) else None, ptr(hw.Y_lo),
                              self.Fp if self.use_tc_bwd else -1, st)

    def _aggregate_x(self, ctx, nodes, n_dev, cap_n, in_off, in_src, dinv, ind_bits, num_ind, out, ldo, out_hi, out_lo,
                     ones_col, st):
        """The two reads of the feature table (hop aggregation, classifier layer 1): Y = A_hat x[nodes] (| indicators),
        one launch over the replicated table, or over the shards of a sharded one (bit-identical)."""
        L, fs = self.L, self.features
        if fs is not None:
            L.grapes_aggregate_peer(ctx, fs.ptrs, fs.bounds_c, fs.world, int(self.x_bf16), self.F, self.ldx, nodes, n_dev,
                                    cap_n, in_off, in_src, dinv, ind_bits, num_ind, None, 0, out, ldo, out_hi, out_lo,
                                    ones_col, st)
        else:
            (L.grapes_aggregate_bf16 if self.x_bf16 else L.grapes_aggregate)(
                ctx, ptr(self.x), self.F, self.ldx, nodes, n_dev, cap_n, in_off, in_src, dinv, ind_bits, num_ind, None, 0,
                out, ldo, out_hi, out_lo, ones_col, st)

    def _sharded_dp(self) -> bool:
        """The learned table is sharded across the ranks of this engine's data-parallel group."""
        return self.embed_shards is not None and self.dp_world > 1

    def _enqueue_epoch_wait(self, ctx, st):
        """Sharded learned table under data parallelism: before the first read of the table, wait until every rank has
        applied as many table steps to its shard as this one (grapes_embed_epoch_wait; csrc/peer_comm.cu)."""
        if not self._sharded_dp():
            return
        es, pe = self.embed_shards, self.peer
        self.L.grapes_embed_epoch_wait(ctx, ptr(es.epoch), es.world, ptr(pe.state) if pe is not None else None,
                                       ptr(self.overflow), self.epoch_spin_limit, st)

    def _enqueue_front0(self, ctx, st):
        """Per-batch reset (main.py:161-176: one memset + one kernel) and the whole hop-0 front end of the ACTIVE step
        state on stream `st`: everything of a batch that can be computed before the previous batch's optimiser step."""
        L, g = self.L, self.g
        hw = self.hops[0]
        L.grapes_zero(ctx, ptr(self.step_pool), 4 * self.step_pool.numel(), st)
        L.grapes_step_reset(ctx, ptr(self.targets), self._cnt("B"), self.bsz, ptr(self.prev_pool), self.cap_P, self.H + 1,
                            self._hc(0, "P"), ptr(self.bm_all),
                            self.bm_ind.data_ptr() + 4 * self.W * (self.num_ind - 1) if self.use_ind else None, st)
        L.grapes_expand_frontier(ctx, ptr(g.indptr), ptr(g.indices), ptr(self.prev[0]), self._hc(0, "P"), self.cap_P,
                                 ptr(hw.row_off), self._hc(0, "m"), self.cap_m, ptr(hw.e_row), ptr(hw.e_col),
                                 ptr(self.bm_prev[0]), ptr(self.bm_batch[0]), ptr(self.overflow), st)
        self._enqueue_hop_graph(0, ctx, st)

    def _enqueue_hop_backward(self, h: int, ctx, st):
        """Side stream A.  Gradient direction of sum(log_prob_h) w.r.t. gcn_gf (main.py:271-287 via
        d log_prob_i / d logit_i = mask_i - sigmoid(logit_i)); at hop 0 also gcn_z forward (log_z,
        main.py:223-228) and its gradient direction.  Reads only this hop's workspace."""
        L = self.L
        hw = self.hops[h]
        F, Fp, D, cap_n, cap_P = self.F, self.Fp, self.D, self.cap_n, self.cap_P
        gf, nz = self.net_gf, self.net_z
        n_dev, P_dev = self._hc(h, "n"), self._hc(h, "P")
        L.grapes_aggregate_scalar_T(ctx, ptr(hw.dl_all), n_dev, cap_n, P_dev, cap_P, ptr(hw.row_off), ptr(hw.e_src),
                                    ptr(hw.e_dst), ptr(hw.dinv), ptr(self.bm_prev[h]), ptr(hw.batch_nodes),
                                    ptr(self.g.indptr), ptr(hw.dz), st)
        if self.use_tc_bwd:
            L.grapes_sampler_l1_bwd_tc(ctx, ptr(hw.Y), ptr(hw.Y_lo), self.ldY, Fp + 1, n_dev, cap_n, Fp, Fp,
                                       ptr(hw.mask_gf), self._par(gf.W1), Fp, D, self._par(gf.b1), self._par(gf.W2),
                                       ptr(hw.dz), 1.0, self._dir(gf.W1), self._dir(gf.b1), self._dir(gf.W2), st)
        else:
            L.grapes_sampler_l1_bwd(ctx, ptr(hw.Y), self.ldY, n_dev, cap_n, Fp, self._par(gf.W1), Fp, D,
                                    self._par(gf.b1), self._par(gf.W2), ptr(hw.dz), ptr(self.dpre), 1.0, 1,
                                    self._dir(gf.W1), Fp, self._dir(gf.b1), self._dir(gf.W2), st)
        if h == 0 and self.z_at == "hop0":
            self._enqueue_gcn_z(ctx, st)

    def _enqueue_gcn_z(self, ctx, st):
        """Side stream A.  gcn_z on the hop-0 frontier: log_z (main.py:223-228) and its gradient direction.  Needs only
        the hop-0 workspace, so it can sit anywhere on the branch; `z_at` = "last" puts it behind the last hop's backward,
        where it overlaps the classifier tail (small kernels) instead of hop 1's aggregation and GEMM."""
        L = self.L
        h = 0
        hw = self.hops[0]
        F, Fp, D, cap_n, cap_P = self.F, self.Fp, self.D, self.cap_n, self.cap_P
        nz = self.net_z
        n_dev, P_dev = self._hc(0, "n"), self._hc(0, "P")
        # log_z = mean(gcn_z(x[batch_nodes], edges)) - log_z_init   (main.py:223-228)
        if self.use_tc:
            L.grapes_sampler_l1_fwd_tc(ctx, ptr(hw.Y), ptr(hw.Y_lo), self.ldY, n_dev, cap_n, F, ptr(self.Wz_hi),
                                       ptr(self.Wz_lo), self.ldW, D, self._par(nz.b1), self._par(nz.W2),
                                       ptr(self.zpart_z), ptr(self.mask_z) if self.use_tc_bwd else None, st)
            L.grapes_aggregate_scalar(ctx, ptr(self.zpart_z), 2 * (D // 128), cap_n, n_dev, cap_n, ptr(hw.in_off),
                                      ptr(hw.in_src), ptr(hw.dinv), self._par(nz.b2), ptr(self.zlogits), None, st)
        else:
            L.grapes_sampler_l1_fwd(ctx, ptr(hw.Y), self.ldY, n_dev, cap_n, F, self._par(nz.W1), F, D,
                                    self._par(nz.b1), self._par(nz.W2), ptr(self.z_z), st)
            L.grapes_aggregate_scalar(ctx, ptr(self.z_z), 1, 0, n_dev, cap_n, ptr(hw.in_off), ptr(hw.in_src),
                                      ptr(hw.dinv), self._par(nz.b2), ptr(self.zlogits), None, st)
        L.grapes_vec_sum(ctx, ptr(self.zlogits), n_dev, cap_n, 1.0, 1, 0, self._scal("log_z_mean"), st)
        if self.reinforce:
            return                                             # gcn_z has no gradient under REINFORCE (main.py:279)
        L.grapes_fill_inv_count(ctx, ptr(self.zlogits), n_dev, cap_n, st)
        L.grapes_aggregate_scalar_T(ctx, ptr(self.zlogits), n_dev, cap_n, P_dev, cap_P, ptr(hw.row_off),
                                    ptr(hw.e_src), ptr(hw.e_dst), ptr(hw.dinv), ptr(self.bm_prev[h]),
                                    ptr(hw.batch_nodes), ptr(self.g.indptr), ptr(self.dz_z), st)
        if self.use_tc_bwd:
            L.grapes_sampler_l1_bwd_tc(ctx, ptr(hw.Y), ptr(hw.Y_lo), self.ldY, Fp + 1, n_dev, cap_n, F, Fp,
                                       ptr(self.mask_z), self._par(nz.W1), F, D, self._par(nz.b1), self._par(nz.W2),
                                       ptr(self.dz_z), 1.0, self._dir(nz.W1), self._dir(nz.b1), self._dir(nz.W2), st)
        else:
            L.grapes_sampler_l1_bwd(ctx, ptr(hw.Y), self.ldY, n_dev, cap_n, F, self._par(nz.W1), F, D,
                                    self._par(nz.b1), self._par(nz.W2), ptr(self.dz_z), ptr(self.dpre), 1.0, 1,
                                    self._dir(nz.W1), F, self._dir(nz.b1), self._dir(nz.W2), st)
        L.grapes_fill_f32(ctx, self._dir(nz.b2), 1.0, 1, st)

    def _split_weights(self, ctx, st):
        """3xTF32 operand split of the (per-step changing) layer-1 weights of gcn_gf / gcn_z."""
        L = self.L
        gf, nz = self.net_gf, self.net_z
        L.grapes_split_tf32(ctx, self._par(gf.W1), self.Fp, self.D, self.Fp, ptr(self.Wgf_hi), ptr(self.Wgf_lo),
                            self.ldW, st)
        L.grapes_split_tf32(ctx, self._par(nz.W1), self.F, self.D, self.F, ptr(self.Wz_hi), ptr(self.Wz_lo),
                            self.ldW, st)

    def enable_data_parallel(self, group=None, exchange: str = "peer"):
        """Data-parallel mode (BASELINE.json north_star; the reference is single-process): this rank's ``step`` runs its
        own batch, exchanges the flat gradient (mean over the ranks of ``group``) and applies both Adam updates, so every
        rank holds bit-identical parameters after every step.  ``exchange``:
          "peer"  one launch over NVLink peer memory (``grapes_step_tail``: gradient scale + push all-reduce + Adam),
                  captured with the rest of the step -- the N-rank step is ONE graph launch;
          "nccl"  ``ncclAllReduce(AVG)`` on the flat buffer between the scale and the Adam launch (captured into the step
                  graph as well when the step is replayed from a graph).
        With learned node features (``embed_nodes``) the table is replicated like ``x``: rank 0's table is broadcast once
        here (the moments start at zero), every step ships its row-sparse table gradient (at most cap_A rows) to every
        rank -- inside the peer tail, or by one ``all_gather`` -- and every rank applies the same dense Adam to the mean
        of the ranks' gradients (``grapes_embed_merge_adam``), so the tables stay bit-identical.  A learned table
        sharded across ``group`` (``x`` a :class:`grapes_b200.dist.ShardedEmbedding`) is not broadcast (every rank
        filled its rows from the same draw); each rank applies that Adam to its own rows only and posts a table epoch
        (``grapes_embed_merge_adam_rows`` + ``grapes_embed_epoch_post``), and every read of the table waits for the
        peers' posts."""
        import torch.distributed as dist
        if exchange not in ("peer", "nccl"):
            raise ValueError("exchange must be 'peer' or 'nccl'")
        group = group or dist.group.WORLD
        self.dp_world, self.dp_rank = dist.get_world_size(group), dist.get_rank(group)
        self.peer, self.dp_group = None, None
        if self.embed_nodes and self.dp_world > 8:
            raise GrapesError("learned node features are exchanged among at most 8 ranks (one NVLink box)")
        es = self.embed_shards
        if es is not None and self.dp_world > 1 and (es.group is None or es.world != self.dp_world or
                                                     es.rank != self.dp_rank):
            raise GrapesError("the sharded learned table must be sharded across the data-parallel group itself")
        embed_floats = 0
        if self.embed_nodes and self.dp_world > 1:
            self.emb_slot = int(self.L.cdll.grapes_embed_slot_floats(self.cap_A, self.F))
            embed_floats = int(self.L.cdll.grapes_embed_peer_buffer_floats(self.cap_A, self.F, self.dp_world))
            # union of the ranks' rows: at most world * cap_A distinct ids
            self.cap_U = min(self.N, self.dp_world * self.cap_A)
            self.pref_union = torch.zeros(self.W + 1, dtype=torch.int32, device=self.device)
            self.union_ids = torch.zeros(self.cap_U, dtype=torch.int32, device=self.device)
            self.mean_rows = torch.zeros((self.cap_U, self.F), dtype=torch.float32, device=self.device)
            if es is None:
                dist.broadcast(self.x, src=dist.get_global_rank(group, 0), group=group)
                self.emb_exp_avg.zero_()
                self.emb_exp_avg_sq.zero_()
            else:
                es.exp_avg.zero_()
                es.exp_avg_sq.zero_()
        if self.dp_world > 1:
            if exchange == "peer":
                # symmetric (peer-mapped) buffers need P2P access between every pair of GPUs of the group.  Every rank tries,
                # the ranks agree (MIN over a success flag), and if any of them could not map its peers ALL of them take the
                # NCCL exchange -- a rank-local decision would deadlock the first step.
                from .dist import PeerGradExchange, ranks_agree
                ok, why = True, ""
                try:
                    self.peer = PeerGradExchange(self.n_par, self.device, group, embed_floats=embed_floats)
                except Exception as exc:                      # noqa: BLE001 -- reported below, never silent
                    ok, why, self.peer = False, f"{type(exc).__name__}: {exc}", None
                if not ranks_agree(ok, self.device, group):
                    import warnings
                    warnings.warn("grapes_b200: peer-memory gradient exchange unavailable on this box"
                                  + (f" ({why})" if why else " (another rank could not map its peers)")
                                  + "; every rank uses the NCCL exchange instead")
                    self.peer, exchange = None, "nccl"
            if exchange == "nccl":
                self.dp_group = group
                # the first collectives of a communicator set up its channels: not inside a captured or timed step
                warm = torch.zeros_like(self.grads)
                for _ in range(24):
                    dist.all_reduce(warm, op=dist.ReduceOp.AVG, group=group)
                if self.embed_nodes:
                    # fixed-size payload of this rank (one slot) and the world slots it is gathered into
                    self.emb_payload = torch.zeros(self.emb_slot, dtype=torch.float32, device=self.device)
                    self.emb_gathered = torch.zeros(self.dp_world * self.emb_slot, dtype=torch.float32, device=self.device)
                    for _ in range(24):
                        dist.all_gather_into_tensor(self.emb_gathered, self.emb_payload, group=group)
                torch.cuda.synchronize(self.device)
        self._graphs.clear()

    def enable_peer_exchange(self, group=None):
        self.enable_data_parallel(group, "peer")

    def _enqueue_tail(self, st):
        """The tail of the step (main.py:271-291 after both backward passes): loss_gfn and the scale of the sampler nets'
        gradient directions, the data-parallel gradient exchange, optimizer_c.step() and optimizer_gf.step() -- one
        launch (``grapes_step_tail``); with the NCCL exchange: scale, all-reduce, Adam."""
        L, ctx = self.L, self.g.ctx
        nc, gf, nz = self.net_c, self.net_gf, self.net_z
        scale = not self.random_sampling
        n_z = 0 if self.reinforce else nz.size                       # gcn_z has no grad under REINFORCE (main.py:279)
        n1 = (gf.size + n_z) if scale else 0
        embed_dp = self.embed_nodes and self.dp_world > 1
        if self.embed_nodes and not embed_dp and self.embed_shards is not None:
            # emulated ranks (one process): every shard's walk over its own rows, in rank order
            if self.embed_shards.shards is None:
                raise GrapesError("a learned table sharded across a process group needs enable_data_parallel(group)")
            for sh in self.embed_shards.shards:
                L.grapes_adam_embed_rows(ctx, ptr(sh.table.rows), ptr(sh.exp_avg), ptr(sh.exp_avg_sq), self.N, sh.lo,
                                         sh.hi - sh.lo, self.F, ptr(self.bm_all), ptr(self.pref_all), ptr(self.dXc),
                                         self.dXc.shape[1], self.lr_gc, 0.9, 0.999, 1e-8, ptr(self.adam_steps), st)
        elif self.embed_nodes and not embed_dp:
            L.grapes_adam_embed(ctx, ptr(self.x), ptr(self.emb_exp_avg), ptr(self.emb_exp_avg_sq), self.N, self.F,
                                ptr(self.bm_all), ptr(self.pref_all), ptr(self.dXc), self.dXc.shape[1], self.lr_gc,
                                0.9, 0.999, 1e-8, ptr(self.adam_steps), st)
        if self.dp_group is not None:
            import torch.distributed as dist
            if scale:
                L.grapes_gfn_finalize_scale(ctx, ptr(self.scal), self.loss_coef, self.log_z_init, int(self.reinforce), 1,
                                            self._dir(gf.base), gf.size, self._grd(gf.base),
                                            self._dir(nz.base), n_z, self._grd(nz.base), st)
            dist.all_reduce(self.grads, op=dist.ReduceOp.AVG, group=self.dp_group)
            L.grapes_adam_step2(ctx, ptr(self.params), ptr(self.grads), ptr(self.exp_avg), ptr(self.exp_avg_sq),
                                nc.base, nc.size, self.lr_gc, gf.base, n1, self.lr_gf, 0.9, 0.999, 1e-8,
                                ptr(self.adam_steps), st)
            if embed_dp:
                # this rank's slot (A | all_nodes | dXc rows): three device copies, then one all-gather of the fixed slot
                pi, A = self.emb_payload.view(torch.int32), self.cap_A
                rows_at = 4 + _round_up(A, 4)
                pi[0:1].copy_(self.counts[self._CNT["A"]:self._CNT["A"] + 1])
                pi[4:4 + A].copy_(self.all_nodes)
                self.emb_payload[rows_at:rows_at + A * self.F].view(A, self.F).copy_(self.dXc[:, :self.F])
                dist.all_gather_into_tensor(self.emb_gathered, self.emb_payload, group=self.dp_group)
                self._enqueue_embed_merge(ptr(self.emb_gathered), None, st)
            return
        pe = self.peer
        if embed_dp:
            L.grapes_step_tail_embed(ctx, ptr(self.scal), int(scale), self.loss_coef, self.log_z_init, int(self.reinforce),
                                     1, ptr(self.gdir), gf.base, gf.size if scale else 0, nz.base, n_z if scale else 0,
                                     pe.peer_ptrs, pe.embed_ptrs, pe.rank, pe.world, self.n_par, ptr(self.params),
                                     ptr(self.grads), ptr(self.exp_avg), ptr(self.exp_avg_sq), nc.base, nc.size,
                                     self.lr_gc, gf.base, n1, self.lr_gf, 0.9, 0.999, 1e-8, ptr(self.adam_steps),
                                     ptr(pe.state), ptr(self.overflow), self._cnt("A"), ptr(self.all_nodes),
                                     ptr(self.dXc), self.dXc.shape[1], self.F, self.cap_A, st)
            # same stream, before the next tail: the parity argument of csrc/peer_comm.cu needs it there
            self._enqueue_embed_merge(ptr(pe.ebuf), ptr(pe.state), st)
            return
        L.grapes_step_tail(ctx, ptr(self.scal), int(scale), self.loss_coef, self.log_z_init, int(self.reinforce), 1,
                           ptr(self.gdir), gf.base, gf.size if scale else 0, nz.base, n_z if scale else 0,
                           pe.peer_ptrs if pe is not None else None, pe.rank if pe is not None else 0,
                           pe.world if pe is not None else 1, self.n_par, ptr(self.params), ptr(self.grads),
                           ptr(self.exp_avg), ptr(self.exp_avg_sq), nc.base, nc.size, self.lr_gc, gf.base, n1, self.lr_gf,
                           0.9, 0.999, 1e-8, ptr(self.adam_steps), ptr(pe.state if pe is not None else self.tail_state),
                           ptr(self.overflow), st)

    def _enqueue_embed_merge(self, slots, state, st):
        """optimizer_c's step of the table on the mean of the ranks' row-sparse gradients (after the parameter Adam, so
        the step count it reads already includes this step).  A sharded table: the walk covers this rank's rows only,
        then this rank posts its table epoch."""
        es = self.embed_shards
        if es is not None:
            self.L.grapes_embed_merge_adam_rows(
                self.g.ctx, slots, self.dp_world, self.cap_A, self.F, state, ptr(self.bm_union), ptr(self.pref_union),
                ptr(self.union_ids), self.cap_U, self._cnt("U"), ptr(self.mean_rows), ptr(es.table.rows),
                ptr(es.exp_avg), ptr(es.exp_avg_sq), self.N, es.lo, es.hi - es.lo, self.lr_gc, 0.9, 0.999, 1e-8,
                ptr(self.adam_steps), ptr(self.overflow), st)
            self.L.grapes_embed_epoch_post(self.g.ctx, es.epoch_ptrs, es.rank, es.world, state, st)
            return
        self.L.grapes_embed_merge_adam(self.g.ctx, slots, self.dp_world, self.cap_A, self.F, state, ptr(self.bm_union),
                                       ptr(self.pref_union), ptr(self.union_ids), self.cap_U, self._cnt("U"),
                                       ptr(self.mean_rows), ptr(self.x), ptr(self.emb_exp_avg), ptr(self.emb_exp_avg_sq),
                                       self.N, self.lr_gc, 0.9, 0.999, 1e-8, ptr(self.adam_steps), ptr(self.overflow), st)

    # ------------------------------------------------------------------ public API
    def set_targets(self, target_nodes: torch.Tensor, state: Optional[int] = None):
        """Writes the batch's target ids into a step state (default: the active one).  ``target_nodes`` may live on the
        device or in pinned host memory (int32: one cudaMemcpyAsync straight into the state's list, no staging)."""
        t = target_nodes
        b = int(t.numel())
        if b > self.B or b < 1:
            raise GrapesError(f"engine built for batch_size<={self.B}, got {b} targets")
        p = self.par if state is None else state
        stt = self._states[p]
        if stt["bsz"] != b or not stt.get("_b_written", False):
            stt["counts"][self._CNT["B"]] = b
            stt["bsz"] = b
            stt["_b_written"] = True
            if p == self.par:
                self.bsz = b
        stt["targets"][:b].copy_(t if t.dtype == torch.int32 else t.to(torch.int32), non_blocking=True)

    def step(self, target_nodes: Optional[torch.Tensor] = None, gumbel_noise=None, apply_optim: bool = True,
             use_graph: bool = False, record: bool = False, noise_mode: int = NOISE_GUMBEL,
             next_targets: Optional[torch.Tensor] = None):
        """One batch of main.py:161-291.  ``next_targets`` (optional) names the batch of the NEXT call: its reset and
        hop-0 front end (weight independent) are enqueued next to this step's classifier tail on the second step state,
        and the next call -- which must pass the same tensor as ``target_nodes`` -- starts at the sampler GEMM of hop 0.
        Results are bit-identical with and without it (tests/test_gpu_engine.py::test_prefetch_matches_plain_steps)."""
        if target_nodes is not None:
            key = (target_nodes.data_ptr(), int(target_nodes.numel()))
            if self._front_ready[1 - self.par] and self._pref_key == key:
                self._activate(1 - self.par)                 # front end already there
            else:
                self._front_ready = [False, False]           # a prefetched front end for other targets is dropped
                self.set_targets(target_nodes)
        self._pref_key = None
        self._prefetch_next = False
        if self.embed_nodes:
            next_targets = None          # the hop-0 front end reads x, which this step's optimiser updates: no prefetch
        if next_targets is not None and not record and gumbel_noise is None:
            self.set_targets(next_targets, state=1 - self.par)
            self._pref_key = (next_targets.data_ptr(), int(next_targets.numel()))
            self._prefetch_next = True
        if use_graph:
            assert gumbel_noise is None and not record
            ready = self._front_ready[self.par]
            key = (apply_optim, self.bsz, self.par, ready, self._prefetch_next,
                   self._states[1 - self.par]["bsz"] if self._prefetch_next else 0)
            gr = self._graphs.get(key)
            if gr is None:
                if not ready:
                    # warm the allocator / lazy init outside capture (a state whose front end is prefetched cannot be
                    # re-run: its reset already happened; every kernel has been launched by an earlier variant then)
                    flags, pf = list(self._front_ready), self._prefetch_next
                    rng = self.rng_state.clone()             # the warm-up must not consume the Philox stream
                    drop = self.drop_state.clone()           # ... nor a dropout step
                    self._prefetch_next = False
                    self._enqueue(None, False)
                    torch.cuda.synchronize()
                    self.rng_state.copy_(rng)
                    self.drop_state.copy_(drop)
                    self._front_ready, self._prefetch_next = flags, pf
                gr = torch.cuda.CUDAGraph()
                n0 = self.L.grapes_kernel_launches()
                flags = list(self._front_ready)
                with torch.cuda.graph(gr):
                    self._enqueue(None, apply_optim)
                self._front_ready = flags
                self._graph_launches[key] = int(self.L.grapes_kernel_launches() - n0)
                self._graphs[key] = gr
            self.launches_per_graph = self._graph_launches[key]
            gr.replay()
            self._front_ready[self.par] = False
            if self._prefetch_next:
                self._front_ready[1 - self.par] = True
            return None
        if record:
            self.record = {"keys": [torch.zeros(self.cap_n, dtype=torch.float32, device=self.device)
                                    for _ in range(self.H)]}
        try:
            self._enqueue(gumbel_noise, apply_optim, noise_mode)
        finally:
            rec, self.record = self.record, None
        if record:
            return self._record_all(rec)
        return None

    @staticmethod
    def raise_on_flags(v: int):
        """GRAPES_OVF_* bits of a step (``scalars()['flags']`` / the ``overflow`` word) -> GrapesError"""
        v = int(v)
        if v:
            names = [n for b, n in OVF_NAMES.items() if v & b]
            if v & 32:
                raise GrapesError("data-parallel exchange failed (" + ", ".join(names) + "): the step was not applied")
            raise GrapesError("frontier capacity exceeded (" + ", ".join(names) + "): raise cap_edges / cap_nodes")

    def check_overflow(self):
        self.raise_on_flags(int(self.overflow.item()))

    def sampler_stats(self) -> List[Dict[str, float]]:
        """per-hop statistics of the last step's sampler (utils.py:62-69; what main.py:304-308 logs); syncs"""
        s = self.stats.cpu()
        return [{k: float(s[h, i]) for i, k in enumerate(STAT_NAMES)} for h in range(self.H)]

    def scalars(self) -> Dict[str, float]:
        s = self.scal.cpu()
        return {k: float(s[i]) for k, i in SCAL.items()}

    def count(self, name: str, idx: int = 0) -> int:
        return int(self.counts[self._CNT[name] + idx].item())

    def hop_sizes(self) -> List[Dict[str, int]]:
        """device-side sizes of the last step, one dict per hop (syncs)"""
        c = self.counts.cpu().tolist()
        return [{k: c[16 * (h + 1) + i] for k, i in _Hop.CNT.items()} for h in range(self.H)]

    # ------------------------------------------------------------------ recording (tests only; syncs)
    def _record_all(self, rec: dict) -> dict:
        torch.cuda.synchronize()
        H = self.H
        sizes = self.hop_sizes()
        out = {"hops": []}
        for h in range(H):
            hw, sz = self.hops[h], sizes[h]
            P, m, n, c, s, e = sz["P"], sz["m"], sz["n"], sz["c"], sz["s"], sz["blk"]
            Y = None if self.random_sampling else (hw.Y[:n] + hw.Y_lo[:n] if hw.Y_lo is not None else hw.Y[:n].clone())
            r = dict(P=P, m=m, n=n, c=c, s=s,
                     prev=self.prev[h][:P].clone(), e_row=hw.e_row[:m].clone(), e_col=hw.e_col[:m].clone(),
                     e_src=hw.e_src[:m].clone(), e_dst=hw.e_dst[:m].clone(),
                     batch_nodes=hw.batch_nodes[:n].clone(), neighbor_nodes=hw.nb_nodes[:c].clone(),
                     nb_local=hw.nb_local[:c].clone(), ind_bits=hw.ind_bits[:n].clone(),
                     in_off=hw.in_off[:n + 1].clone(), in_src=hw.in_src[:sz["nnz"]].clone(),
                     dinv=hw.dinv[:n].clone(), Y=Y, logits_all=hw.logits_all[:n].clone(),
                     sampled=self.prev[h + 1][self.bsz:self.bsz + s].clone(), log_prob=self.log_prob[h, :c].clone(),
                     keys=rec["keys"][h][:c].clone(), stats=self.stats[h].clone(),
                     dl_all=hw.dl_all[:n].clone(), dz=hw.dz[:n].clone(),
                     block_edges=torch.stack([hw.blk_src[:e], hw.blk_dst[:e]]).clone())
            out["hops"].append(r)
        A = self.count("A")
        out["all_nodes"] = self.all_nodes[:A].clone()
        out["target_local"] = self.target_local[:self.bsz].clone()
        out["logits_c"] = self.logits_c[:A].clone()          # after dropout (modules/gcn.py:37)
        if self.dropout > 0:
            # the step's masks, evaluated by the kernels' keep function at the step value the step used
            seed, step = (int(v) for v in self.drop_state.tolist())
            step -= 1
            keep = []
            for site, width in ((0, self.D), (1, self.C)):
                k = torch.zeros((A, width), dtype=torch.uint8, device=self.device)
                if A > 0:
                    self.L.grapes_dropout_mask(self.g.ctx, seed, step, self._drop_tag(site), self.drop_threshold,
                                               self._cnt("A"), A, width, ptr(k), torch.cuda.current_stream().cuda_stream)
                keep.append(k.bool())
            out["dropout_keep"], out["dropout_step"] = tuple(keep), step
            out["hidden_c"] = self.out1[:A].clone()              # dropout(relu(layer 1))
        out["scalars"] = self.scalars()
        out["grads"] = {k: {n: t.clone() for n, t in v.items()} for k, v in self.grad_dicts().items()}
        if self.embed_nodes:
            out["grad_x_rows"] = self.dXc[:A, :self.F].clone()       # d loss_c / d x[all_nodes]
            if self.dp_world > 1:                                     # the rows the data-parallel table step applied
                U = self.count("U")
                out["embed_union"] = self.union_ids[:U].clone()
                out["embed_mean_rows"] = self.mean_rows[:U].clone()
        out["cl_edges"] = []
        for slot, hop in ((0, H - 1), (1, 0)):
            e = sizes[hop]["blk"]
            out["cl_edges"].append(torch.stack([self.cl_src[slot][:e], self.cl_dst[slot][:e]]).clone())
        return out
