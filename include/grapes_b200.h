/*
 * grapes_b200 -- C ABI of the B200-native GRAPES sampling-and-aggregation hot path.
 *
 * The reference (dfdazac/grapes) has no FFI of its own: its hot path is a set of Python callables
 * (main.py:15-17 imports GCN, TensorMap, get_neighborhoods, sample_neighborhoods_from_probs,
 * slice_adjacency).  Every entry point below cites the reference code it replaces
 * (file:line under /root/reference); INTEGRATION.md shows the ctypes binding a maintainer adds.
 *
 * Conventions
 *   - every function returns GRAPES_OK (0) or a GRAPES_ERR_* code; grapes_last_error() has the text.
 *     No C++ exceptions cross the ABI.
 *   - all pointers except `ctx`, `overflow`-style outputs documented otherwise are DEVICE pointers
 *     owned by the caller (torch's caching allocator in the Python host).  The library retains
 *     nothing past a call; its only own state is the ctx workspace.
 *   - node ids are int32 on the device, CSR `indptr` is int64 (papers100M-shape: nnz = 3.2e9).
 *   - sizes that depend on the data (`*_dev`) live in device memory so a whole training step can be
 *     enqueued -- and CUDA-graph captured -- without a host round-trip.  `cap_*` are the host-side
 *     capacities of the caller's buffers; when data outgrows a capacity the kernel clamps, stays
 *     memory-safe and ORs a GRAPES_OVF_* bit into `*overflow` (device int).
 *   - `stream` is a cudaStream_t; kernels are enqueued there, never synchronised, and are safe to
 *     capture.  One ctx per (process, device), not re-entrant.
 */
#ifndef GRAPES_B200_H
#define GRAPES_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GRAPES_OK 0
#define GRAPES_ERR_ARG 1
#define GRAPES_ERR_CUDA 2
#define GRAPES_ERR_NOMEM 3

#define GRAPES_OVF_ROWS 1   /* more rows than cap_P            */
#define GRAPES_OVF_EDGES 2  /* frontier edges exceed cap_m     */
#define GRAPES_OVF_NODES 4  /* frontier nodes exceed cap_n     */
#define GRAPES_OVF_BLOCK 8  /* induced block exceeds cap_out   */
#define GRAPES_OVF_HUB 16   /* hub-row worklist exceeded       */
#define GRAPES_OVF_PEER_TIMEOUT 32 /* a peer rank never published its gradients (grapes_allreduce_adam_peer) */

/* noise modes of grapes_select_topk */
#define GRAPES_NOISE_PHILOX 0          /* draw u on the device (Philox4x32-10), g = -log(-log u)          */
#define GRAPES_NOISE_GUMBEL 1          /* noise[i] = Gumbel(0,1) sample (what utils.py:40-41 draws)       */
#define GRAPES_NOISE_UNIFORM 2         /* noise[i] = u in (tiny, 1-eps)                                   */
#define GRAPES_NOISE_KEYS 3            /* noise[i] = perturbed log-prob itself (utils.py:42)              */
#define GRAPES_NOISE_NONE_TOPK_PROBS 4 /* key = sigmoid(logit): deterministic top-k (eval.py:126-127)     */

/* layout of the float `scal` block of grapes_gfn_finalize */
#define GRAPES_SCAL_LOSS_C 0
#define GRAPES_SCAL_TOT_LOG_PROB 1
#define GRAPES_SCAL_LOG_Z_MEAN 2
#define GRAPES_SCAL_LOG_Z 3
#define GRAPES_SCAL_LOSS_GFN 4
#define GRAPES_SCAL_G_GF 5
#define GRAPES_SCAL_G_Z 6
#define GRAPES_SCAL_SUM_DL 7
#define GRAPES_SCAL_FLAGS 15   /* GRAPES_OVF_* bits seen by the step's tail launch, as an integer-valued float */
#define GRAPES_SCAL_COUNT 16

typedef struct grapes_ctx grapes_ctx;

/* ---- context ------------------------------------------------------------------------------- */
/* Workspace for one graph of `num_nodes` nodes on CUDA device `device`; `max_frontier` bounds the
 * number of frontier nodes/edges any later call is given (sizes the scan scratch);
 * `partials_bytes` sizes the split-K partial buffer of the weight-gradient GEMMs.                 */
int grapes_ctx_create(int device, int64_t num_nodes, int64_t max_frontier, int64_t partials_bytes, grapes_ctx** out);
/* Grid-size budget of this context: every launch through `ctx` sizes its grid for `sms` SMs instead of the whole GPU
 * (<= 0 restores the device's count).  Used for the contexts of side streams whose kernels are off the critical path
 * (the sampler backward): persistent tcgen05 kernels that take every SM would stall the critical path's small kernels. */
int grapes_ctx_set_sm_limit(grapes_ctx* ctx, int sms);
int grapes_ctx_destroy(grapes_ctx* ctx);
const char* grapes_last_error(void);
int grapes_abi_version(void);
/* sha1 over the library's sources + this header at build time: the host loader compares it with the tree it parses its
 * prototypes from and refuses (or rebuilds) a binary that does not match                                                */
const char* grapes_build_id(void);
/* programmatic dependent launch between consecutive kernels of a stream: bit mask over the library's source files
 * (1 frontier, 2 gcn, 4 gemm_tc, 8 loss_optim, 16 select) whose kernels may start before their predecessor ends;
 * 0 = plain stream order */
int grapes_set_pdl(int mask);
/* number of kernels this library has launched (or recorded into a capturing stream) so far      */
int64_t grapes_kernel_launches(void);
int grapes_zero(grapes_ctx* ctx, void* ptr, int64_t bytes, void* stream);

/* ---- CSR construction (main.py:134-136: sp.csr_matrix((ones bool, edge_index), shape=(N, N))) ---------------- */
/* bytes of caller-owned device scratch grapes_csr_from_edges needs for this (N, E)                               */
int64_t grapes_csr_workspace_bytes(int64_t num_nodes, int64_t num_edges);
/* edge list (src[e], dst[e]), int64 like the reference's edge_index rows -> scipy's canonical CSR of the bool
 * matrix: indptr int64 [N+1], indices int32 (capacity E; rows ascending, duplicate edges collapsed, self-loops
 * kept), *nnz_dev = stored entries.  *err_dev = 1 when an id is outside [0, N) (scipy raises ValueError; such edges
 * are skipped here and the caller raises).  No ctx: the graph's context is created from the result.  Counting sort by
 * row + per-row sort/unique in registers / shared memory; enqueued on `stream`, no host synchronisation.           */
/* how the edges are grouped by row: 0 (default) = chosen by shape, 1 = ONE random scatter (4x the algorithmic DRAM
 * traffic when short rows spread over a table larger than L2), 2 = bucket partition + L2-windowed scatter            */
int grapes_csr_set_direct_scatter(int mode);
int grapes_csr_from_edges(const int64_t* src, const int64_t* dst, int64_t num_edges, int64_t num_nodes, int64_t* indptr,
                          int* indices, int64_t* nnz_dev, int* err_dev, void* workspace, int64_t workspace_bytes,
                          void* stream);

/* ---- whole-graph gcn_norm structure with int64 offsets (replaces PyG gcn_norm at modules/gcn.py:18,21 for full-batch
 * evaluation of graphs of any edge count): in_off int64 [N+1], in_src int32 [nnz'] (the in-neighbours of each destination,
 * sources ascending, stored self-loops dropped, duplicates of an edge list kept and counted), dinv fp32 [N] =
 * (indeg + 1)^-1/2.  Equal, bit for bit, to sorting the (destination, source) keys.  Sequence, all on `stream`, no host
 * synchronisation inside:
 *   begin -> add_*(pass 0) over the whole input -> offsets (in_off, dinv, *nnz_dev = nnz') -> add_*(pass 1) over the
 *   same input in the same chunks or others -> finish (per-row sorts).
 * The input is the graph's CSR (rows [r0, r1) of indptr / indices; row = source, index = destination) or chunks of an
 * int64 edge list (src[e] -> dst[e], e.g. the rows of a slice of edge_index), read in place.  in_src needs nnz' entries,
 * which the caller reads back after `offsets`.  *err_dev |= 1: an id outside [0, N) (the edge is skipped; the caller
 * raises), |= 2: a node with 2^31 - 1 or more in-edges.
 * Device scratch beyond the outputs: the caller's workspace, grapes_graph_norm_workspace_bytes(N) = 4 N bytes + 8 bytes
 * per 8192 nodes + 1 KB of alignment, and nothing else (no chunk copies: the input is read where it lies).            */
int64_t grapes_graph_norm_workspace_bytes(int64_t num_nodes);
int grapes_graph_norm_begin(int64_t num_nodes, void* workspace, int64_t workspace_bytes, int* err_dev, void* stream);
int grapes_graph_norm_add_csr(int pass, int64_t num_nodes, const int64_t* indptr, const int* indices, int64_t r0, int64_t r1,
                              int64_t* in_off, int* in_src, void* workspace, int* err_dev, void* stream);
int grapes_graph_norm_add_edges(int pass, int64_t num_nodes, const int64_t* src, const int64_t* dst, int64_t num_edges,
                                int64_t* in_off, int* in_src, void* workspace, int* err_dev, void* stream);
int grapes_graph_norm_offsets(int64_t num_nodes, void* workspace, int64_t* in_off, float* dinv, int64_t* nnz_dev,
                              void* stream);
int grapes_graph_norm_finish(int64_t num_nodes, const int64_t* in_off, int* in_src, void* workspace, void* stream);
/* ---- one destination window [lo, hi) of that structure (the row partition of the data-parallel full-batch evaluation).
 * window_bounds: from the full in_off of `offsets`, bounds_dev[0 .. world] (int64, on the device) = the least i with
 * (in_off[i] + i) * world >= k * (in_off[N] + N): the rows cut into `world` contiguous windows balanced by the prefix of
 * indeg + 1, each within one row's indeg + 1 of the mean; windows are empty when N < world.  Deterministic: every rank
 * computes the same bounds.
 * Sequence for the window of one rank: begin -> add_*(pass 0) over the WHOLE input (dinv and the bounds need every
 * degree) -> offsets into a full [N+1] in_off -> window_bounds -> the caller forms win_off[j] = in_off[lo + j] - in_off[lo]
 * (j <= hi - lo) and may free the full in_off -> window_add_* over the whole input (only edges into [lo, hi) are
 * scattered, to in_src[win_off[c - lo] + k]) -> finish(hi - lo, win_off, in_src, workspace) (the per-row sorts of the
 * window; skip it for an empty window).  The window equals rows [lo, hi) of the whole structure bit for bit.
 * Peak device scratch beyond the outputs (win_off, the window's in_src, dinv [N]): the workspace (~4 N bytes) plus the
 * full in_off (8 (N + 1) bytes), which is needed only until win_off is formed.                                        */
int grapes_graph_norm_window_bounds(int64_t num_nodes, const int64_t* in_off, int world, int64_t* bounds_dev,
                                    void* stream);
int grapes_graph_norm_window_add_csr(int64_t num_nodes, const int64_t* indptr, const int* indices, int64_t r0, int64_t r1,
                                     int64_t lo, int64_t hi, const int64_t* win_off, int* in_src, void* workspace,
                                     void* stream);
int grapes_graph_norm_window_add_edges(int64_t num_nodes, const int64_t* src, const int64_t* dst, int64_t num_edges,
                                       int64_t lo, int64_t hi, const int64_t* win_off, int* in_src, void* workspace,
                                       void* stream);

/* ---- frontier expansion / dedup / relabel  (utils.py:74-82, main.py:183-195, utils.py:98-120) */
/* rows[P] -> row_off[P+1] = exclusive scan of CSR degrees, *m_dev = total.  Sets the bit of every
 * row in bm_rows (prev_nodes_mask, main.py:185) and of rows with degree > 0 in bm_batch.          */
int grapes_row_offsets(grapes_ctx* ctx, const int64_t* indptr, const int* rows, const int* P_dev, int cap_P,
                       int* row_off, int* m_dev, int cap_m, uint32_t* bm_rows, uint32_t* bm_batch, int* overflow,
                       void* stream);
/* get_neighborhoods (utils.py:74-82): e_row[e] = position in rows, e_col[e] = neighbour id, row-major
 * by position, ascending neighbour inside a row.  Marks the neighbours in bm_batch (main.py:186).   */
int grapes_expand_rows(grapes_ctx* ctx, const int64_t* indptr, const int* indices, const int* rows,
                       const int* P_dev, int cap_P, const int* row_off, const int* m_dev, int cap_m, int* e_row,
                       int* e_col, uint32_t* bm_batch, void* stream);
/* grapes_row_offsets + grapes_expand_rows in ONE launch (every CTA rebuilds the row offsets in shared memory)     */
int grapes_expand_frontier(grapes_ctx* ctx, const int64_t* indptr, const int* indices, const int* rows,
                           const int* P_dev, int cap_P, int* row_off, int* m_dev, int cap_m, int* e_row, int* e_col,
                           uint32_t* bm_rows, uint32_t* bm_batch, int* overflow, void* stream);
/* mask -> ascending id lists + local numbering (main.py:187-195).  pref_* = per-word exclusive
 * popcount prefix (local id of v = pref[v>>5] + popc(bm[v>>5] & ((1<<(v&31))-1)) = TensorMap.map).
 * nb_* describe batch & ~prev (neighbor_nodes; nb_index[j] = position of batch node j in it or -1, optional);
 * bm_ind[hop] receives that mask and ind_bits[j]
 * the indicator columns of batch node j (indicator_features, main.py:167-168,191,199-202).        */
int grapes_rank_nodes(grapes_ctx* ctx, const uint32_t* bm_batch, const uint32_t* bm_prev, int* pref_batch,
                      int* pref_nb, int* batch_nodes, int* nb_nodes, int* nb_local, int* nb_index, uint32_t* ind_bits,
                      uint32_t* bm_ind, int ind_rows, int hop, int cap_n, int* n_dev, int* c_dev, int* overflow,
                      void* stream);
/* node_map.map(neighborhoods) (main.py:195): local (src, dst) of every expanded edge.  cnt_hist
 * (optional, all-zero on entry) receives the in-degree histogram grapes_build_csr(hist_done=1) needs.
 * cap_n = capacity of every node-indexed buffer downstream (cnt_hist, in_off, dinv, Y ...): when the frontier holds
 * more nodes than that (GRAPES_OVF_NODES, raised by grapes_rank_nodes) an edge touching a node past the capacity is
 * written as the dropped self-edge (0, 0), so an overflowing step is flagged AND memory-safe.                       */
int grapes_edges_to_local(grapes_ctx* ctx, const int* rows, const int* e_row, const int* e_col, const int* m_dev,
                          int cap_m, const uint32_t* bm, const int* pref, int cap_n, int* e_src, int* e_dst,
                          int* cnt_hist, void* stream);
/* TensorMap.map on an id list (main.py:213,253-254,259).                                          */
int grapes_relabel(grapes_ctx* ctx, const int* ids, const int* count_dev, int cap, const uint32_t* bm,
                   const int* pref, int* out, void* stream);
/* slice_adjacency (utils.py:85-95) on an already expanded row set: keeps edges whose neighbour is
 * in bm_cols; GLOBAL ids out, [src = row id, dst = col id], reference ordering.                    */
int grapes_slice_block(grapes_ctx* ctx, const int* rows, const int* e_row, const int* e_col, const int* m_dev,
                       int cap_m, const uint32_t* bm_cols, int* out_src, int* out_dst, int cap_out, int* count_dev,
                       int* overflow, void* stream);
/* main.py:252-259 + gcn.py:30-36 for a sampled subgraph of <= 4096 nodes, in one launch: local ids of the targets,
 * relabel of the layer-1 block (blk0 = edge_indices[-1]) and the layer-2 block (blk1 = edge_indices[0]), their
 * dst-sorted CSRs with deg^-1/2, and the src-sorted CSR of blk1 (classifier backward).  nnz_dev3[3] counts.
 * tgt_of_row[cap_A] (optional) = index of the target sitting at that local row, or -1.                        */
int grapes_classifier_prep(grapes_ctx* ctx, const uint32_t* bm_all, const int* pref_all, const int* A_dev, int cap_A,
                           const int* targets, const int* B_dev, int cap_B, int* target_local, const int* blk0_src,
                           const int* blk0_dst, const int* E0_dev, const int* blk1_src, const int* blk1_dst,
                           const int* E1_dev, int cap_blk, int* cl_src0, int* cl_dst0, int* cl_src1, int* cl_dst1,
                           int* in_off0, int* in_src0, float* dinv0, int* in_off1, int* in_src1, float* dinv1,
                           int* out_off1, int* out_dst1, int* tmp, int* nnz_dev3, int* tgt_of_row, void* stream);
int grapes_bitmap_set(grapes_ctx* ctx, const int* ids, const int* count_dev, int cap, uint32_t* bm, void* stream);
int grapes_bitmap_clear_words(grapes_ctx* ctx, const int* ids, const int* count_dev, int cap, uint32_t* bm,
                              void* stream);
/* dst[off..off+n) = src; *total_dev = off + n   (batch_nodes = cat([targets, sampled]), main.py:236) */
int grapes_append_list(grapes_ctx* ctx, const int* src, const int* count_dev, int cap, int* dst, int dst_offset,
                       int* total_dev, void* stream);
/* per-batch reset (main.py:161-168): targets -> head of `nlists` row lists `list_stride` ints apart, their bits
 * set in bm_a / bm_b (all_nodes_mask, last indicator row; either may be NULL), *P0_dev = batch size.       */
int grapes_step_reset(grapes_ctx* ctx, const int* targets, const int* B_dev, int cap_B, int* lists,
                      int64_t list_stride, int nlists, int* P0_dev, uint32_t* bm_a, uint32_t* bm_b, void* stream);
int grapes_ids_i64_to_i32(grapes_ctx* ctx, const int64_t* in, int n, int* out, int* count_dev, void* stream);
int grapes_ids_i32_to_i64(grapes_ctx* ctx, const int* in, const int* count_dev, int cap, int64_t* out, void* stream);

/* ---- gcn_norm + aggregation (PyG 2.5.2 GCNConv / gcn_norm; call sites gcn.py:18,21,32,36) ----- */
/* Edge list (key, val) -> CSR keyed by `key` with key==val edges dropped (add_remaining_self_loops),
 * values ascending inside a row.  dinv (optional) = (count + 1)^-1/2 = deg^-1/2 incl. the self-loop.
 * cnt_scratch[cap_n] must be all-zero on entry and is all-zero again on exit; hist_done=1 means it already
 * holds the per-key counts (grapes_edges_to_local's cnt_hist).                                          */
int grapes_build_csr(grapes_ctx* ctx, const int* key, const int* val, const int* E_dev, int cap_E, const int* n_dev,
                     int cap_n, int* cnt_scratch, int hist_done, int* off, int* sorted_val, int* tmp_val, float* dinv,
                     int* nnz_dev, int* overflow, void* stream);
/* out[j,:F] = dinv[j]^2 X[g(j)] + sum_s dinv[s] dinv[j] X[g(s)] (+bias)(relu); g = nodes[] or identity.
 * Indicator columns [F, F+num_ind) from ind_bits; [F+num_ind, ldo) zero-filled.  out_hi/out_lo
 * (optional, same ldo) receive the 3xTF32 operand split tf32(v), tf32(v - tf32(v)) for the tcgen05 GEMM;
 * ones_col >= 0 puts a column of ones there (bias column of the tensor-core backward), -1 = none.        * TMA-staged form (feature rows copied by cp.async.bulk into shared memory): 16-byte aligned X / outputs, ldx % 4 == 0 and
 * ldx >= round_up(F, 4) -- F itself may be any width (Reddit 602, Cora 1433: pad the row PITCH, the pad values are never
 * stored); other layouts take the register-staged kernels.  Bitwise identical results either way.                       */
int grapes_aggregate(grapes_ctx* ctx, const float* X, int F, int ldx, const int* nodes, const int* n_dev, int cap_n,
                     const int* in_off, const int* in_src, const float* dinv, const uint32_t* ind_bits, int num_ind,
                     const float* bias, int relu, float* out, int ldo, float* out_hi, float* out_lo, int ones_col,
                     void* stream);
/* 0 (default) = aggregation form chosen by shape; 1 = the register-staged kernels only, the bit-exact reference of the
 * TMA-staged form (csrc/gcn.cu aggregate_impl).  Any other value is GRAPES_ERR_ARG.                                */
int grapes_agg_variant(int v);
/* the same with the feature table stored as bf16 (papers100M-shaped config: 128 bf16 features, BASELINE.json configs[4]);
 * rows are widened to fp32 as they are read, arithmetic and outputs stay fp32.  ldx in elements.                */
int grapes_aggregate_bf16(grapes_ctx* ctx, const void* X_bf16, int F, int ldx, const int* nodes, const int* n_dev,
                          int cap_n, const int* in_off, const int* in_src, const float* dinv, const uint32_t* ind_bits,
                          int num_ind, const float* bias, int relu, float* out, int ldo, float* out_hi, float* out_lo,
                          int ones_col, void* stream);
/* Whole-graph aggregation over one row slab of the int64 structure above (grapes_graph_norm_*), for graphs past 2^31
 * entries.  slab_dev = {R, r0} on the device, R <= cap_r:
 *   out[j, :F] = dinv[r0+j]^2 X[r0+j] + sum_{s in in(r0+j)} dinv[s] dinv[r0+j] X[s]  (+ bias),  j < R;  out[j, F:ldo) = 0.
 * in_off is read at r0 + j, sources / dinv / X rows are graph ids.  X is fp32 or bf16 (x_bf16 = 1, widened on read); fp32
 * arithmetic in the summation order of grapes_aggregate, so on a graph below 2^31 the rows are bit-identical to those of
 * grapes_aggregate / grapes_aggregate_bf16 on the int32 structure.  TMA-staged where that kernel takes the layout,
 * register-staged otherwise and under grapes_agg_variant(1).                                                           */
int grapes_aggregate_rows64(grapes_ctx* ctx, const void* X, int x_bf16, int F, int ldx, const int* slab_dev, int cap_r,
                            const int64_t* in_off, const int* in_src, const float* dinv, const float* bias, float* out,
                            int ldo, void* stream);
/* The same slab aggregation, fp32, over an operand whose rows are partitioned between `world` <= 8 owners (layer 2 of the
 * data-parallel full-batch evaluation): row s of Z is z_rows[o][(s - bounds[o]) * ldz ...] for the owner o with
 * bounds[o] <= s < bounds[o + 1].  z_rows: HOST array of `world` device pointers -- peer-mapped buffers of the ranks (own
 * at its rank's index) or any allocations this device can read; bounds: HOST array of world + 1 row bounds, bounds[0] = 0.
 * in_off is read at r0 + j (for a window structure pass its local offsets shifted back by the window's first row).  The
 * summation order is grapes_aggregate_rows64's, so the rows are bit-identical to it over the unpartitioned Z.
 * Register-staged; out[j, F:ldo) = 0.  grapes_aggregate_rows64_peer_x with x_bf16 = 0.                               */
int grapes_aggregate_rows64_peer(grapes_ctx* ctx, const void* const* z_rows, const int64_t* bounds, int world, int F,
                                 int ldz, const int* slab_dev, int cap_r, const int64_t* in_off, const int* in_src,
                                 const float* dinv, const float* bias, float* out, int ldo, void* stream);
/* grapes_aggregate_rows64 over a table whose rows are partitioned between `world` <= 8 owners, fp32 or bf16 (x_bf16 = 1,
 * widened on read): row s is x_rows[o] + (s - bounds[o]) * ldx elements for the owner o with bounds[o] <= s <
 * bounds[o + 1].  x_rows / bounds as for grapes_aggregate_rows64_peer (empty windows allowed, their base may be NULL).
 * Bit-identical to grapes_aggregate_rows64 over the unpartitioned table; register-staged.                            */
int grapes_aggregate_rows64_peer_x(grapes_ctx* ctx, const void* const* x_rows, const int64_t* bounds, int world,
                                   int x_bf16, int F, int ldx, const int* slab_dev, int cap_r, const int64_t* in_off,
                                   const int* in_src, const float* dinv, const float* bias, float* out, int ldo,
                                   void* stream);
/* grapes_aggregate / grapes_aggregate_bf16 (x_bf16 = 1) over a feature table sharded by rows between `world` <= 8 owners:
 * the feature row of node g = nodes[j] (or j when nodes is NULL) is x_rows[o] + (g - bounds[o]) * ldx elements for the
 * owner o with bounds[o] <= g < bounds[o + 1] -- this rank's shard or a peer's over NVLink.  x_rows: HOST array of `world`
 * device pointers; bounds: HOST array of world + 1 non-decreasing bounds, bounds[0] = 0, bounds[world] < 2^31.  Indicator
 * columns, bias / relu, out or out_hi / out_lo, ones_col and the zero pad as grapes_aggregate; the summation order is
 * theirs, so the rows are bit-identical to them over the unpartitioned table.  Register-staged, one launch.          */
int grapes_aggregate_peer(grapes_ctx* ctx, const void* const* x_rows, const int64_t* bounds, int world, int x_bf16, int F,
                          int ldx, const int* nodes, const int* n_dev, int cap_n, const int* in_off, const int* in_src,
                          const float* dinv, const uint32_t* ind_bits, int num_ind, const float* bias, int relu,
                          float* out, int ldo, float* out_hi, float* out_lo, int ones_col, void* stream);
/* z may be given as `nparts` partial vectors `part_stride` floats apart (summed on the fly)           */
int grapes_aggregate_scalar(grapes_ctx* ctx, const float* z, int nparts, int part_stride, const int* n_dev, int cap_n, const int* in_off,
                            const int* in_src, const float* dinv, const float* bias, float* out, float* zero_out,
                            void* stream);
/* transposed scalar aggregation on the hop graph (backward of the above) from the row-major edge list of the expansion
 * (rows[P] of the graph's CSR -> row_off, e_src, e_dst in local ids): writes dz[j] for every j < *n_dev,
 *   dz[j] = dinv[j]^2 dl[j] + sum over edges j -> d of the hop graph, d != j, of dinv[j] dinv[d] dl[d].
 * bm_prev (the expanded rows' bitmap), batch_nodes (local -> graph id) and indptr (the CSR the rows were expanded from)
 * given together: one launch; all three NULL: two launches.  Same bits either way; no atomics.                       */
int grapes_aggregate_scalar_T(grapes_ctx* ctx, const float* dl, const int* n_dev, int cap_n, const int* P_dev,
                              int cap_P, const int* row_off, const int* e_src, const int* e_dst, const float* dinv,
                              const uint32_t* bm_prev, const int* batch_nodes, const int64_t* indptr, float* dz,
                              void* stream);
/* v[j] = 1/n: gradient of log_z = mean(gcn_z logits) w.r.t. those logits (main.py:227-228)          */
int grapes_fill_inv_count(grapes_ctx* ctx, float* v, const int* n_dev, int cap_n, void* stream);
int grapes_vec_sum(grapes_ctx* ctx, const float* v, const int* n_dev, int cap_n, float scale, int divide_by_n,
                   int accumulate, float* out, void* stream);

/* ---- dense transforms (GCNConv.lin; fp32) ---------------------------------------------------- */
/* C[M x N] = A . B (+bias)(relu)(gated by relu_gate > 0).  layout bit0: A is [M x K] K-contiguous
 * (else [K x M]); bit1: B is [N x K] K-contiguous (else [K x N]).  M may be a device count.          */
int grapes_gemm(grapes_ctx* ctx, int layout, const float* A, int lda, const float* B, int ldb, float* C, int ldc,
                const int* M_dev, int M_cap, int N, int K, const float* bias, int relu, const float* relu_gate,
                int ldg, void* stream);
/* Dropout of the classifier's hidden layer, h = dropout(relu(A_hat_1 (x W1^T) + b1)) (modules/gcn.py:33).  Masks: the keep
 * bit of entry (row, col) of a site of width w is a pure function of (seed, step, tag, row * w + col) -- Philox4x32-10 with
 * counter (i / 4, tag, step), key = seed, keep iff the low 24 bits of word i % 4 are < threshold -- where
 * drop_state = {seed, step} (device, 2 x uint64), tag = 1 + site + 2 * rank (site 0: hidden, 1: logits) and
 * threshold = llrint((1 - p) * 2^24); kept entries are multiplied by scale = 1 / (1 - p) (0 when p == 1).
 * H[M x N] = dropout(relu(A W^T + b)): A [M x K] and W [N x K] K-contiguous (grapes_gemm layout 3).                    */
int grapes_gemm_bias_relu_dropout(grapes_ctx* ctx, const float* A, int lda, const float* W, int ldw, float* H, int ldh,
                                  const int* M_dev, int M_cap, int N, int K, const float* bias,
                                  unsigned long long* drop_state, uint32_t tag, uint32_t threshold, float scale,
                                  void* stream);
/* its backward (modules/gcn.py:33): C = (gate > 0) ? scale * (A B) : 0, A [M x K] K-contiguous, B [K x N] (layout 1); with
 * gate = the dropped activations H this is d pre = (dZ W2) (.) relu' (.) keep * scale                                  */
int grapes_gemm_gated_scaled(grapes_ctx* ctx, const float* A, int lda, const float* B, int ldb, float* C, int ldc,
                             const int* M_dev, int M_cap, int N, int K, const float* gate, int ldg, float scale,
                             void* stream);
/* out[M x N] (+)= scale * A[R x M]^T B[R x N]  (weight gradients; deterministic split over rows)     */
int grapes_gemm_tn(grapes_ctx* ctx, const float* A, int lda, const float* B, int ldb, const int* R_dev, int R_cap,
                   int M, int N, float scale, int accumulate, float* out, void* stream);
int grapes_colsum(grapes_ctx* ctx, const float* Mx, const int* R_dev, int R_cap, int ld, int C, float scale,
                  int accumulate, float* out, void* stream);
/* sampler nets (hidden D, out_dim 1; main.py:112-114): z = relu(Y W1^T + b1) . w2, hidden never stored */
int grapes_sampler_l1_fwd(grapes_ctx* ctx, const float* Y, int ldy, const int* n_dev, int cap_n, int K,
                          const float* W1, int ldw, int D, const float* b1, const float* w2, float* z, void* stream);
int grapes_sampler_l1_bwd(grapes_ctx* ctx, const float* Y, int ldy, const int* n_dev, int cap_n, int K,
                          const float* W1, int ldw, int D, const float* b1, const float* w2, const float* dz,
                          float* dpre_scratch, float scale, int accumulate, float* gW1, int ldgw, float* gb1,
                          float* gw2, void* stream);

/* tcgen05 path of the same layer (sm_100a tensor cores, 3xTF32 split operands, TMA + TMEM).  (Y, Y_lo) is the
 * (hi, lo) pair grapes_aggregate's out_hi/out_lo wrote; Y_lo == NULL means Y is plain fp32 and is split inside the
 * kernels (no hi/lo copies in HBM, one more pipeline step).  Weights are pre-split with grapes_split_tf32;
 * zpart[2 * D/128][cap_n] partial row dots (two per 128-column half: sum them); maskT[(rows/32)][D] relu mask bits (optional).                            */
int grapes_split_tf32(grapes_ctx* ctx, const float* src, int ld_src, int R, int K, float* hi, float* lo, int ld_dst,
                      void* stream);
/* measurement knob of the tcgen05 kernels (bit 1: stream the weight tiles instead of keeping them resident; bit 2: the
 * forward with both operands in shared memory, k_l1_fwd_tc, instead of the default k_l1_fwd_ts whose A operand lives in
 * tensor memory; bit 3: the backward with both operands in shared memory, k_l1_bwd_tc, instead of the default k_l1_bwd_ts;
 * bit 4: timeline stamps for scripts/trace_*_ts.py)                                                                    */
int grapes_tc_debug(int flags);
/* debugging aid (scripts/trace_fwd_ts.py): device address of the ctx's split-K partial buffer, where grapes_tc_debug bit 4
 * makes k_l1_fwd_ts park the globaltimer stamps of CTA 0's MMA issuer / epilogue / converter warps                  */
int64_t grapes_debug_partials(grapes_ctx* ctx);
int64_t grapes_debug_partials_bytes(grapes_ctx* ctx);   /* k_l1_bwd_ts parks its stamps in the last KB */
int grapes_sampler_l1_fwd_tc(grapes_ctx* ctx, const float* Y, const float* Y_lo, int ldy, const int* n_dev, int cap_n,
                             int K, const float* W_hi, const float* W_lo, int ldw, int D, const float* b1,
                             const float* w2, float* zpart, uint32_t* maskT, void* stream);

/* dense layer with bias + relu on the tensor cores (same kernel, hidden activations written out): H[n x D] = relu(Y W^T + b),
 * the hidden layer of the full-graph evaluation forward gcn_c(x, edge_index) (eval.py:50).  ldh % 4 == 0, H 16-byte aligned.  */
int grapes_gemm_bias_relu_tc(grapes_ctx* ctx, const float* Y, int ldy, const int* n_dev, int cap_n, int K, const float* W_hi,
                             const float* W_lo, int ldw, int D, const float* b, float* H, int ldh, void* stream);

/* backward on tensor cores: S = mask^T (dz * Y) from the relu mask bits; Y must hold a column of ones at
 * `ones_col` (K <= ones_col < ncols <= ldy).  Accumulates scale * d(sum dz.z)/d(W1,b1,w2).               */
int grapes_sampler_l1_bwd_tc(grapes_ctx* ctx, const float* Y, const float* Y_lo, int ldy, int ncols, const int* n_dev,
                             int cap_n, int K, int ones_col, const uint32_t* maskT, const float* W1, int ldw, int D,
                             const float* b1, const float* w2, const float* dz, float scale, float* gW1, float* gb1,
                             float* gw2, void* stream);

/* ---- selection (utils.py:13-71; eval.py:126-130) --------------------------------------------- */
/* floats of scratch (`work`, 16-byte aligned, ZEROED ONCE by the caller: every launch leaves its counters clean) the
 * two calls below need for cap_c candidates                                                              */
int64_t grapes_select_work_floats(grapes_ctx* ctx, int cap_c);
/* debugging aid: globaltimer stamps (ns) of block 0 at the phase boundaries of the last fused selection launch that used
 * `work` (start, keys done, histogram merged, barrier 1, members listed, barrier 2, outputs done, last block done);
 * HOST array of 8, synchronises                                                                                      */
int grapes_debug_select_fused_stamps(grapes_ctx* ctx, const float* work, int cap_c, int64_t* out8);
/* One hop of the sampler head: layer-2 aggregation of the sampler GCN at width 1 -> logits (main.py:210-213;
 * arguments as grapes_aggregate_scalar, in_off == NULL: z already holds the logits), then
 * sample_neighborhoods_from_probs (utils.py:13-71) on the candidate rows: Gumbel-top-k, Bernoulli log-prob of the
 * mask, statistics, d(sum log_prob)/d logit.  nb_index[j] = candidate index of frontier row j or -1.       */
int grapes_select_hop(grapes_ctx* ctx, const float* z, int nparts, int part_stride, const int* n_dev, int cap_n,
                      const int* in_off, const int* in_src, const float* dinv, const float* bias,
                      const int* nb_index, const int* nb_local, const int* nb_nodes, const int* c_dev, int k,
                      int noise_mode, const float* noise, unsigned long long* rng_state, float* work,
                      uint32_t* ukeys_scratch, float* logits_all, float* keys_out, int* sampled_out,
                      int sampled_offset, int* s_dev, int* total_dev, uint8_t* mask_out, float* log_prob,
                      float* tot_log_prob, float* stats, float* dl_all, float* sum_dl, uint32_t* bm_mark,
                      void* stream);
/* the same on per-candidate logits (logits_all[i] = logit of candidate i; nb_local must be NULL)          */
int grapes_select_topk(grapes_ctx* ctx, const float* logits_all, const int* nb_local, const int* nb_nodes,
                       const int* c_dev, int cap_c, int k, int noise_mode, const float* noise,
                       unsigned long long* rng_state, uint32_t* ukeys_scratch, float* work, float* keys_out,
                       int* sampled_out, int sampled_offset, int* s_dev, int* total_dev, uint8_t* mask_out,
                       float* log_prob, float* tot_log_prob, float* stats, float* dl_all, float* sum_dl,
                       uint32_t* bm_mark, void* stream);

/* ---- losses + optimiser (main.py:117-123,260-291) -------------------------------------------- */
int grapes_classifier_loss(grapes_ctx* ctx, const float* logits, int ldl, int C, const int* A_dev, int A_cap,
                           const int* row_ids, const int* tgt_of_row /* optional inverse of row_ids (-1: not a target):
                           enables the row-parallel 2-launch form */, const int* targets, int B, const int64_t* labels_i64,
                           const float* labels_f32, float reg_param, float* dlogits, float* loss_out,
                           float* colsum_out /* optional: column sums of dlogits = d loss / d last bias */,
                           void* stream);
/* the same loss on dropout(logits) (modules/gcn.py:37; masks as grapes_gemm_bias_relu_dropout, site width C): `logits`
 * holds the pre-dropout logits and receives the dropped ones in place; dlogits = d loss / d (pre-dropout logits), i.e.
 * the gradient at the dropped logits times keep * scale; colsum_out its column sums.  Its last launch advances
 * drop_state's step word by one: call it once per training step, after every other reader of the step's masks.   */
int grapes_classifier_loss_dropout(grapes_ctx* ctx, float* logits, int ldl, int C, const int* A_dev, int A_cap,
                                   const int* row_ids, const int* tgt_of_row, const int* targets, int B,
                                   const int64_t* labels_i64, const float* labels_f32, float reg_param, float* dlogits,
                                   float* loss_out, float* colsum_out, unsigned long long* drop_state, uint32_t tag,
                                   uint32_t threshold, float scale, void* stream);
/* keep[r * width + c] (0 / 1) = keep bit of entry (r, c) of a dropout site at (seed, step), r < *rows_dev
 * (modules/gcn.py:33,37): the masks a training step drew, for inspection and replay                               */
int grapes_dropout_mask(grapes_ctx* ctx, int64_t seed, int64_t step, uint32_t tag, uint32_t threshold,
                        const int* rows_dev, int cap_rows, int width, uint8_t* keep, void* stream);
/* out[i] = argmax_c logits[row_ids[i], c], i < *B_dev: predictions of the target rows (eval.py:152-153); ties -> lowest c */
int grapes_argmax_rows(grapes_ctx* ctx, const float* logits, int ldl, int C, const int* row_ids, const int* B_dev,
                       int cap_B, int* out, void* stream);
int grapes_gfn_finalize(grapes_ctx* ctx, float* scal, float loss_coef, float log_z_init, int reinforce,
                        int have_log_z, void* stream);
/* grapes_gfn_finalize + both grapes_scale_by_device_scalar calls (gcn_gf, gcn_z ranges) in one launch            */
int grapes_gfn_finalize_scale(grapes_ctx* ctx, float* scal, float loss_coef, float log_z_init, int reinforce,
                              int have_log_z, const float* dir_gf, int n_gf, float* grad_gf, const float* dir_z,
                              int n_z, float* grad_z, void* stream);
int grapes_scale_by_device_scalar(grapes_ctx* ctx, const float* dir, const float* g_dev, int n, float* grad,
                                  void* stream);
int grapes_adam_step(grapes_ctx* ctx, float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int n,
                     float lr, float beta1, float beta2, float eps, float* step_dev, int increment_step, void* stream);
/* two Adam parameter groups (optimizer_c at off0, optimizer_gf at off1 of the flat buffers; main.py:117-118) in one
 * launch; steps_dev[2] are the per-group step counts, incremented by the kernel itself                        */
int grapes_adam_step2(grapes_ctx* ctx, float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                      int off0, int n0, float lr0, int off1, int n1, float lr1, float beta1, float beta2, float eps,
                      float* steps_dev, void* stream);
/* Learned node features (main.py:89-100,116: embeddings = nn.Parameter [N, node_emb_dim] inside optimizer_c): dense
 * torch.optim.Adam update of the whole table from a SPARSE gradient -- grad_rows[r, :F] (pitch ldg) is the gradient of
 * the node whose bit has rank r in bm_rows / pref_rows (the batch's all_nodes bitmap), every other row has gradient 0
 * (its moments still decay and it still moves, as in the reference).  step_dev = optimizer_c's step count BEFORE this
 * update; call it before grapes_adam_step2, which increments the count.                                           */
int grapes_adam_embed(grapes_ctx* ctx, float* table, float* exp_avg, float* exp_avg_sq, int64_t num_nodes, int F,
                      const uint32_t* bm_rows, const int* pref_rows, const float* grad_rows, int ldg, float lr,
                      float beta1, float beta2, float eps, const float* step_dev, void* stream);
/* grapes_adam_embed over the rows [row0, row0 + rows) of a table of num_nodes rows (0 <= row0 <= row0 + rows <= num_nodes):
 * table, exp_avg and exp_avg_sq point at row row0 (one rank's shard of a table sharded by rows, pitch F), while bm_rows /
 * pref_rows / grad_rows are those of the whole table (bit row0 + i).  Per element the arithmetic of grapes_adam_embed, so
 * a shard's rows equal the same rows of the whole-table walk bit for bit.  rows == 0: no launch.                     */
int grapes_adam_embed_rows(grapes_ctx* ctx, float* table, float* exp_avg, float* exp_avg_sq, int64_t num_nodes,
                           int64_t row0, int64_t rows, int F, const uint32_t* bm_rows, const int* pref_rows,
                           const float* grad_rows, int ldg, float lr, float beta1, float beta2, float eps,
                           const float* step_dev, void* stream);
int grapes_fill_f32(grapes_ctx* ctx, float* p, float value, int n, void* stream);

/* ---- step tail: gradient scale + data-parallel exchange + both Adam groups in ONE launch -------------------------- */
/* floats of symmetric buffer each rank must provide for an n-float gradient exchanged among `world` ranks
 * (2 parities x world slots + flag words), and the uint32 words of device state of one exchange endpoint        */
int64_t grapes_peer_buffer_floats(int n, int world);
int grapes_peer_state_words(void);
/* Mean all-reduce over NVLink peer memory + grapes_adam_step2's arithmetic, one launch, no per-step host argument
 * (capturable into the step's CUDA graph; main.py:268,289 on the mean of the per-rank gradients -- the reference itself
 * is single-process).  Every rank WRITES its gradient into its slot of every rank's buffer, signals, waits (bounded) for
 * all peers' signals, then sums its own buffer's slots in rank order: identical bits on every rank.  peer_bufs: HOST array
 * of `world` peer-mapped device pointers (own buffer at index `rank`), zeroed once; state: grapes_peer_state_words()
 * device uint32, zeroed once.  grads_mean_out must be `grads` (the mean replaces it in place).  A peer that never arrives
 * raises GRAPES_OVF_PEER_TIMEOUT in *err_flag and the step is a NO-OP on this rank (parameters, moments, step counts
 * untouched); the failure is sticky: every later call is a no-op too.                                                  */
int grapes_allreduce_adam_peer(grapes_ctx* ctx, void* const* peer_bufs, int rank, int world, const float* grads, int n,
                               float* params, float* grads_mean_out, float* exp_avg, float* exp_avg_sq, int off0,
                               int n0, float lr0, int off1, int n1, float lr1, float beta1, float beta2, float eps,
                               float* steps_dev, unsigned int* state, int* err_flag, void* stream);
/* The whole tail of a training step (main.py:271-291) in one launch: grapes_gfn_finalize_scale's arithmetic when
 * do_scale != 0 (`dir` is indexed like the flat parameter buffer; ranges [gf_off, gf_off + n_gf), [z_off, z_off + n_z)),
 * the exchange above when peer_bufs != NULL and world > 1, then both Adam groups.  `grads` [n] holds the classifier
 * gradient on entry and the step's (mean) gradient of every parameter on exit.  scal[GRAPES_SCAL_FLAGS] receives the
 * bits of *err_flag (GRAPES_OVF_*) as an integer-valued float, so the 64-byte loss read-back of a step also carries its
 * overflow / peer-failure verdict.  state: grapes_peer_state_words() device uint32 (needed with or without peers).      */
int grapes_step_tail(grapes_ctx* ctx, float* scal, int do_scale, float loss_coef, float log_z_init, int reinforce,
                     int have_log_z, const float* dir, int gf_off, int n_gf, int z_off, int n_z, void* const* peer_bufs,
                     int rank, int world, int n, float* params, float* grads, float* exp_avg, float* exp_avg_sq, int off0,
                     int n0, float lr0, int off1, int n1, float lr1, float beta1, float beta2, float eps, float* steps_dev,
                     unsigned int* state, int* err_flag, void* stream);

/* ---- data parallelism with learned node features (main.py:89-100,116: the table inside optimizer_c) ---------------
 * The table is replicated like x; its gradient is row-sparse (the step's all_nodes rows, at most cap_rows = B + H*k),
 * so every rank ships only (A, all_nodes[:A], d loss_c / d x[all_nodes[:A], :F]).  One slot holds that payload:
 * [A, 3 pad | cap_rows ids rounded up to 4 | cap_rows x F floats]; the second symmetric buffer of the peer exchange is
 * 2 parities x world slots.                                                                                         */
int64_t grapes_embed_slot_floats(int cap_rows, int F);
int64_t grapes_embed_peer_buffer_floats(int cap_rows, int F, int world);
/* grapes_step_tail with peers (world <= 8) that also pushes this step's table payload -- A = *count_dev rows, ids[:A]
 * ascending, rows[:A, :F] at pitch ldg (16-byte aligned) -- into slot[rank] of parity (step & 1) of every rank's
 * second buffer (embed_bufs: HOST array of `world` peer-mapped pointers, grapes_embed_peer_buffer_floats each).  The
 * step's one flag covers both payloads; on a failed exchange nothing is pushed.  Follow it, on the same stream and before
 * the next tail, with grapes_embed_merge_adam(state = the same state): its read of this step's slots must finish before
 * any peer can push two steps later.                                                                                  */
int grapes_step_tail_embed(grapes_ctx* ctx, float* scal, int do_scale, float loss_coef, float log_z_init, int reinforce,
                           int have_log_z, const float* dir, int gf_off, int n_gf, int z_off, int n_z,
                           void* const* peer_bufs, void* const* embed_bufs, int rank, int world, int n, float* params,
                           float* grads, float* exp_avg, float* exp_avg_sq, int off0, int n0, float lr0, int off1, int n1,
                           float lr1, float beta1, float beta2, float eps, float* steps_dev, unsigned int* state,
                           int* err_flag, const int* count_dev, const int* ids, const float* rows, int ldg, int F,
                           int cap_rows, void* stream);
/* optimizer_c's step of the table on the mean over ranks of the row-sparse gradients, g(v) = (1/world) sum_r G_r(v)
 * added in rank order (identical bits on every rank): union bitmap of the world id lists (bm_union: num_words uint32,
 * zero on entry), its popcount-prefix rank (pref_union: num_words + 1; union_ids[:*union_count], cap_union >= the union
 * size), the mean rows (mean_rows [cap_union, F]), then grapes_adam_embed's dense table walk with step_dev = optimizer_c's
 * count AFTER this step's parameter Adam (the bias correction uses *step_dev as is).  state != NULL: `slots` is this
 * rank's second peer buffer and the exchange's go word picks the parity; a failed exchange makes all of it a no-op
 * (table, moments untouched).  state == NULL: `slots` holds the world slots contiguously (an all-gather).             */
int grapes_embed_merge_adam(grapes_ctx* ctx, const float* slots, int world, int cap_rows, int F,
                            const unsigned int* state, uint32_t* bm_union, int* pref_union, int* union_ids, int cap_union,
                            int* union_count, float* mean_rows, float* table, float* exp_avg, float* exp_avg_sq,
                            int64_t num_nodes, float lr, float beta1, float beta2, float eps, const float* step_dev,
                            int* overflow, void* stream);
/* grapes_embed_merge_adam whose table walk covers only the rows [row0, row0 + rows) (this rank's shard of a table
 * sharded by rows; table / exp_avg / exp_avg_sq point at row row0, pitch F).  Union, rank and mean rows are unchanged;
 * the go word of `state` is honoured as there.  Follow it on the same stream with grapes_embed_epoch_post.         */
int grapes_embed_merge_adam_rows(grapes_ctx* ctx, const float* slots, int world, int cap_rows, int F,
                                 const unsigned int* state, uint32_t* bm_union, int* pref_union, int* union_ids,
                                 int cap_union, int* union_count, float* mean_rows, float* table, float* exp_avg,
                                 float* exp_avg_sq, int64_t num_nodes, int64_t row0, int64_t rows, float lr, float beta1,
                                 float beta2, float eps, const float* step_dev, int* overflow, void* stream);
/* Table epoch of a learned table sharded by rows (ordering argument: csrc/peer_comm.cu).  Every rank owns one symmetric
 * buffer of grapes_embed_epoch_words(world) uint32, zeroed once: word[r] = table steps rank r has applied, then this
 * rank's own count.  post: after this rank's shard walk, count += 1 and a system-scope release of it into word[rank] of
 * every rank's buffer (epoch_bufs: HOST array of `world` peer-mapped pointers); no-op when state != NULL and the step's
 * go word carries GO_FAIL.  wait (epoch = this rank's own buffer): before any read of the table, a bounded acquire spin
 * until every word[p] has reached the own count.  spin_limit tries (0: the step tail's bound, a few seconds); on timeout
 * GRAPES_OVF_PEER_TIMEOUT is ORed into *err_flag and, state != NULL, the exchange's sticky failure is set, so that
 * step's tail and merge are no-ops.  Both launches read everything from device memory (graph-capturable).          */
int grapes_embed_epoch_words(int world);
int grapes_embed_epoch_post(grapes_ctx* ctx, void* const* epoch_bufs, int rank, int world, const unsigned int* state,
                            void* stream);
int grapes_embed_epoch_wait(grapes_ctx* ctx, const unsigned int* epoch, int world, unsigned int* state, int* err_flag,
                            uint32_t spin_limit, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GRAPES_B200_H */
