// Classifier loss (+ its gradient w.r.t. the logits), the GFlowNet / REINFORCE loss wiring and Adam,
// as device-resident kernels so a whole GRAPES step can be replayed as one CUDA graph.
//   CrossEntropyLoss / BCEWithLogitsLoss + reg_param * sum(var(logits, dim=1))   main.py:120-123,260-261
//   trajectory-balance / REINFORCE loss                                          main.py:271-282
//   torch.optim.Adam (defaults betas=(0.9,0.999), eps=1e-8, no weight decay)     main.py:117-118
#define GRAPES_PDL_GROUP 8
#include "common.cuh"

#define LOSS_THREADS 1024

__device__ __forceinline__ float block_sum_1024(float v, float* s) {
    v = warp_sum(v);
    if (lane_id() == 0) s[threadIdx.x >> 5] = v;
    __syncthreads();
    float r = (threadIdx.x < (blockDim.x >> 5)) ? s[threadIdx.x] : 0.f;
    if (threadIdx.x < 32) { r = warp_sum(r); if (threadIdx.x == 0) s[0] = r; }
    __syncthreads();
    r = s[0];
    __syncthreads();
    return r;
}

// logits [A x C] (ld = ldl).  Target rows: row_ids[B] (local ids of the target nodes, main.py:259).
// labels: int64 class ids per GLOBAL node (multiclass) or float [N x C] (multilabel), indexed by targets[B].
// dlogits must be zeroed by the caller (grapes_classifier_loss does it).
// Stage 1 (one warp per target row): per-row loss term -> row_loss[r], gradient rows.  Stage 2 (one block): fixed-order
// sum of the B terms (+ the reg_param * sum_rows var(logits) term and its gradient) -> *loss_out.
// CE_LSE_NOTE: the cross-entropy terms keep log-sum-exp relative to the row maximum, p = exp((l - mx) - ls) and
// loss = (mx - l_y) + ls with ls = log sum exp(l - mx).  Forming lse = mx + ls first rounds it to the ulp of |mx|
// (3e-5 at |mx| ~ 500, 5e-4 at 5000), an error every probability of the row would inherit.
__global__ void __launch_bounds__(256) k_loss_rows(const float* __restrict__ logits, int ldl, int C,
                                                   const int* __restrict__ row_ids, const int* __restrict__ targets,
                                                   int B, const int64_t* __restrict__ labels_i64,
                                                   const float* __restrict__ labels_f32, float* __restrict__ dlogits,
                                                   float* __restrict__ row_loss) {
    pdl_begin();
    const int lane = lane_id();
    const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= B) return;
    const int row = row_ids[r];
    const float* lr = logits + (size_t)row * ldl;
    if (labels_i64) {
        const float invB = 1.0f / (float)B;
        const int y = (int)labels_i64[targets[r]];
        float mx = -INFINITY;
        for (int c = lane; c < C; c += 32) mx = fmaxf(mx, lr[c]);
        mx = warp_max(mx);
        float se = 0.f;
        for (int c = lane; c < C; c += 32) se += expf(lr[c] - mx);
        se = warp_sum(se);
        const float ls = logf(se);                       // log-sum-exp - mx (see CE_LSE_NOTE)
        for (int c = lane; c < C; c += 32) {
            const float pr = expf((lr[c] - mx) - ls);
            dlogits[(size_t)row * ldl + c] = (pr - (c == y ? 1.f : 0.f)) * invB;
        }
        if (lane == 0) row_loss[r] = ((mx - lr[y]) + ls) * invB;
    } else {
        const float inv = 1.0f / ((float)B * (float)C);
        const float* yr = labels_f32 + (size_t)targets[r] * C;
        float a = 0.f;
        for (int c = lane; c < C; c += 32) {
            const float l = lr[c], y = yr[c];
            a += (1.0f - y) * l + fmaxf(-l, 0.f) + log1pf(expf(-fabsf(l)));
            dlogits[(size_t)row * ldl + c] = (1.0f / (1.0f + expf(-l)) - y) * inv;
        }
        a = warp_sum(a);
        if (lane == 0) row_loss[r] = a * inv;
    }
}

__global__ void __launch_bounds__(LOSS_THREADS) k_loss_final(const float* __restrict__ logits, int ldl, int C,
                                                             const int* __restrict__ A_dev, int A_cap, int B,
                                                             const float* __restrict__ row_loss, float reg_param,
                                                             float* __restrict__ dlogits, float* loss_out) {
    pdl_begin();
    __shared__ float s[32];
    const int A = min(*A_dev, A_cap);
    const int lane = lane_id(), warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    float part = 0.f;
    for (int r = threadIdx.x; r < B; r += blockDim.x) part += row_loss[r];
    float loss = block_sum_1024(part, s);
    if (reg_param != 0.f && C > 1) {                     // reg_param * sum_rows var(logits, dim=1), unbiased
        float rp = 0.f;
        const float invc1 = 1.0f / (float)(C - 1);
        for (int row = warp; row < A; row += nwarps) {
            const float* lr = logits + (size_t)row * ldl;
            float sm = 0.f;
            for (int c = lane; c < C; c += 32) sm += lr[c];
            const float mean = warp_sum(sm) / (float)C;
            float sq = 0.f;
            for (int c = lane; c < C; c += 32) {
                const float d = lr[c] - mean;
                sq = fmaf(d, d, sq);
                dlogits[(size_t)row * ldl + c] += reg_param * 2.0f * d * invc1;
            }
            sq = warp_sum(sq);
            if (lane == 0) rp += sq * invc1;
        }
        loss += reg_param * block_sum_1024(rp, s);
    }
    if (threadIdx.x == 0) *loss_out = loss;
}

// ---------------------------------------------------------------------------------------
// Row-parallel classifier loss (main.py:260-261).  k_loss_rows2: one warp per row of the sampled subgraph; a target
// row (tgt_of_row[row] = r >= 0) gets its CrossEntropy / BCE term and gradient, every row the
// reg_param * var(logits) term, other rows zeros -- so dlogits needs no memset.  Each block also leaves the column
// sums of its rows in colpart[block][C].  k_loss_final2 (one CTA) adds the A row terms and the per-block column
// sums (= gradient of the last layer's bias) in a fixed order.
// ---------------------------------------------------------------------------------------
#define LR2_WARPS 8
__global__ void __launch_bounds__(LR2_WARPS * 32) k_loss_rows2(
    const float* __restrict__ logits, int ldl, int C, const int* __restrict__ A_dev, int A_cap,
    const int* __restrict__ tgt_of_row, const int* __restrict__ targets, int B,
    const int64_t* __restrict__ labels_i64, const float* __restrict__ labels_f32, float reg_param,
    float* __restrict__ dlogits, float* __restrict__ row_loss, float* __restrict__ colpart) {
    pdl_begin();
    extern __shared__ float s_cols[];                    // [LR2_WARPS][C]
    const int A = min(*A_dev, A_cap);
    const int lane = lane_id(), warp = threadIdx.x >> 5;
    const int row = blockIdx.x * LR2_WARPS + warp;
    float* mycols = s_cols + warp * C;
    for (int c = lane; c < C; c += 32) mycols[c] = 0.f;
    if (row < A) {
        const float* lr = logits + (size_t)row * ldl;
        float* dr = dlogits + (size_t)row * ldl;
        const int r = tgt_of_row[row];
        float loss = 0.f;
        if (r >= 0 && labels_i64) {
            const float invB = 1.0f / (float)B;
            const int y = (int)labels_i64[targets[r]];
            float mx = -INFINITY;
            for (int c = lane; c < C; c += 32) mx = fmaxf(mx, lr[c]);
            mx = warp_max(mx);
            float se = 0.f;
            for (int c = lane; c < C; c += 32) se += expf(lr[c] - mx);
            se = warp_sum(se);
            const float ls = logf(se);                   // log-sum-exp - mx (see CE_LSE_NOTE)
            for (int c = lane; c < C; c += 32) mycols[c] = (expf((lr[c] - mx) - ls) - (c == y ? 1.f : 0.f)) * invB;
            loss = ((mx - lr[y]) + ls) * invB;
        } else if (r >= 0) {
            const float inv = 1.0f / ((float)B * (float)C);
            const float* yr = labels_f32 + (size_t)targets[r] * C;
            float a = 0.f;
            for (int c = lane; c < C; c += 32) {
                const float l = lr[c], y = yr[c];
                a += (1.0f - y) * l + fmaxf(-l, 0.f) + log1pf(expf(-fabsf(l)));
                mycols[c] = (1.0f / (1.0f + expf(-l)) - y) * inv;
            }
            loss = warp_sum(a) * inv;
        }
        if (reg_param != 0.f && C > 1) {                 // reg_param * var(logits[row], unbiased)
            const float invc1 = 1.0f / (float)(C - 1);
            float sm = 0.f;
            for (int c = lane; c < C; c += 32) sm += lr[c];
            const float mean = warp_sum(sm) / (float)C;
            float sq = 0.f;
            for (int c = lane; c < C; c += 32) {
                const float d = lr[c] - mean;
                sq = fmaf(d, d, sq);
                mycols[c] += reg_param * 2.0f * d * invc1;
            }
            loss += reg_param * warp_sum(sq) * invc1;
        }
        __syncwarp();
        for (int c = lane; c < C; c += 32) dr[c] = mycols[c];
        if (lane == 0) row_loss[row] = loss;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float a = 0.f;
#pragma unroll
        for (int w = 0; w < LR2_WARPS; ++w) a += s_cols[w * C + c];
        colpart[(size_t)blockIdx.x * C + c] = a;
    }
}

__device__ __forceinline__ void loss_final2_body(const int* __restrict__ A_dev, int A_cap, int C,
                                                 const float* __restrict__ row_loss, const float* __restrict__ colpart,
                                                 int nblocks, float* loss_out, float* __restrict__ colsum_out) {
    __shared__ float s[32];
    __shared__ float s_col[LOSS_THREADS];
    const int A = min(*A_dev, A_cap);
    float part = 0.f;
    for (int r = threadIdx.x; r < A; r += LOSS_THREADS) part += row_loss[r];
    const float loss = block_sum_1024(part, s);
    if (threadIdx.x == 0) *loss_out = loss;
    if (!colsum_out) return;
    const int used = (A + LR2_WARPS - 1) / LR2_WARPS;    // blocks that own rows; the rest wrote zeros
    const int nb = min(nblocks, used);
    const int groups = max(1, LOSS_THREADS / C);
    const int g = threadIdx.x / C, c = threadIdx.x % C;
    float a = 0.f;
    if (g < groups)
        for (int b0 = g; b0 < nb; b0 += 8 * groups) {
            float v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) { const int b = b0 + u * groups; v[u] = (b < nb) ? colpart[(size_t)b * C + c] : 0.f; }
#pragma unroll
            for (int u = 0; u < 8; ++u) a += v[u];
        }
    s_col[threadIdx.x] = a;
    __syncthreads();
    if ((int)threadIdx.x < C) {
        float t = 0.f;
        for (int gg = 0; gg < groups; ++gg) t += s_col[gg * C + threadIdx.x];
        colsum_out[threadIdx.x] = t;
    }
}

__global__ void __launch_bounds__(LOSS_THREADS) k_loss_final2(const int* __restrict__ A_dev, int A_cap, int C,
                                                              const float* __restrict__ row_loss,
                                                              const float* __restrict__ colpart, int nblocks,
                                                              float* loss_out, float* __restrict__ colsum_out) {
    pdl_begin();
    loss_final2_body(A_dev, A_cap, C, row_loss, colpart, nblocks, loss_out, colsum_out);
}

// ---------------------------------------------------------------------------------------
// Dropout forms of the classifier loss (modules/gcn.py:37: logits = dropout(A_hat_2 (h W2^T) + b2), the loss on the
// dropped logits).  `logits` holds the pre-dropout values the +b2 aggregation wrote; the dropped logits are written back
// in place and the gradient leaves as d logits_pre = d logits (.) keep * s, the input of dZ and of the b2 column sums.
// The keep bit of (row, c) is entry row * C + c of the logits site.  The loss-final kernel is the last reader of the
// step's drop_state and advances its step word.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(LR2_WARPS * 32) k_loss_rows2_dropout(
    float* __restrict__ logits, int ldl, int C, const int* __restrict__ A_dev, int A_cap,
    const int* __restrict__ tgt_of_row, const int* __restrict__ targets, int B,
    const int64_t* __restrict__ labels_i64, const float* __restrict__ labels_f32, float reg_param,
    float* __restrict__ dlogits, float* __restrict__ row_loss, float* __restrict__ colpart, DropParams dp) {
    pdl_begin();
    extern __shared__ float s_cols[];                    // [LR2_WARPS][C]
    const int A = min(*A_dev, A_cap);
    const int lane = lane_id(), warp = threadIdx.x >> 5;
    const int row = blockIdx.x * LR2_WARPS + warp;
    float* mycols = s_cols + warp * C;
    for (int c = lane; c < C; c += 32) mycols[c] = 0.f;
    if (row < A) {
        float* lr = logits + (size_t)row * ldl;
        float* dr = dlogits + (size_t)row * ldl;
        const unsigned long long seed = dp.state[0], step = dp.state[1];
        uint32_t keep = 0u;                              // bit j: column lane + 32 j (C <= LOSS_THREADS)
        for (int c = lane, j = 0; c < C; c += 32, ++j) {
            const bool k = dropout_keep(seed, step, dp.tag, dp.threshold, (unsigned long long)row * C + c);
            keep |= k ? (1u << j) : 0u;
            lr[c] = k ? lr[c] * dp.scale : 0.f;
        }
        __syncwarp();
        const int r = tgt_of_row[row];
        float loss = 0.f;
        if (r >= 0 && labels_i64) {
            const float invB = 1.0f / (float)B;
            const int y = (int)labels_i64[targets[r]];
            float mx = -INFINITY;
            for (int c = lane; c < C; c += 32) mx = fmaxf(mx, lr[c]);
            mx = warp_max(mx);
            float se = 0.f;
            for (int c = lane; c < C; c += 32) se += expf(lr[c] - mx);
            se = warp_sum(se);
            const float ls = logf(se);                   // log-sum-exp - mx (see CE_LSE_NOTE)
            for (int c = lane; c < C; c += 32) mycols[c] = (expf((lr[c] - mx) - ls) - (c == y ? 1.f : 0.f)) * invB;
            loss = ((mx - lr[y]) + ls) * invB;
        } else if (r >= 0) {
            const float inv = 1.0f / ((float)B * (float)C);
            const float* yr = labels_f32 + (size_t)targets[r] * C;
            float a = 0.f;
            for (int c = lane; c < C; c += 32) {
                const float l = lr[c], y = yr[c];
                a += (1.0f - y) * l + fmaxf(-l, 0.f) + log1pf(expf(-fabsf(l)));
                mycols[c] = (1.0f / (1.0f + expf(-l)) - y) * inv;
            }
            loss = warp_sum(a) * inv;
        }
        if (reg_param != 0.f && C > 1) {                 // reg_param * var(logits[row], unbiased)
            const float invc1 = 1.0f / (float)(C - 1);
            float sm = 0.f;
            for (int c = lane; c < C; c += 32) sm += lr[c];
            const float mean = warp_sum(sm) / (float)C;
            float sq = 0.f;
            for (int c = lane; c < C; c += 32) {
                const float d = lr[c] - mean;
                sq = fmaf(d, d, sq);
                mycols[c] += reg_param * 2.0f * d * invc1;
            }
            loss += reg_param * warp_sum(sq) * invc1;
        }
        __syncwarp();
        for (int c = lane, j = 0; c < C; c += 32, ++j) {
            const float g = ((keep >> j) & 1u) ? mycols[c] * dp.scale : 0.f;
            mycols[c] = g;
            dr[c] = g;
        }
        if (lane == 0) row_loss[row] = loss;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float a = 0.f;
#pragma unroll
        for (int w = 0; w < LR2_WARPS; ++w) a += s_cols[w * C + c];
        colpart[(size_t)blockIdx.x * C + c] = a;
    }
}

__global__ void __launch_bounds__(LOSS_THREADS) k_loss_final2_dropout(const int* __restrict__ A_dev, int A_cap, int C,
                                                                      const float* __restrict__ row_loss,
                                                                      const float* __restrict__ colpart, int nblocks,
                                                                      float* loss_out, float* __restrict__ colsum_out,
                                                                      DropParams dp) {
    pdl_begin();
    if (threadIdx.x == 0) dp.state[1] += 1ull;         // every reader of this step's masks has completed
    loss_final2_body(A_dev, A_cap, C, row_loss, colpart, nblocks, loss_out, colsum_out);
}

// dropped value of logits[row, c] (the k_loss_rows form reads the pre-dropout logits; k_loss_final_dropout writes them)
__device__ __forceinline__ float dropped_logit(const float* lr, int c, unsigned long long i, unsigned long long seed,
                                               unsigned long long step, const DropParams& dp) {
    return dropout_keep(seed, step, dp.tag, dp.threshold, i) ? lr[c] * dp.scale : 0.f;
}

__global__ void __launch_bounds__(256) k_loss_rows_dropout(const float* __restrict__ logits, int ldl, int C,
                                                           const int* __restrict__ row_ids,
                                                           const int* __restrict__ targets, int B,
                                                           const int64_t* __restrict__ labels_i64,
                                                           const float* __restrict__ labels_f32,
                                                           float* __restrict__ dlogits, float* __restrict__ row_loss,
                                                           DropParams dp) {
    pdl_begin();
    const int lane = lane_id();
    const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= B) return;
    const int row = row_ids[r];
    const float* lr = logits + (size_t)row * ldl;
    const unsigned long long seed = dp.state[0], step = dp.state[1], i0 = (unsigned long long)row * C;
    if (labels_i64) {
        const float invB = 1.0f / (float)B;
        const int y = (int)labels_i64[targets[r]];
        float mx = -INFINITY;
        for (int c = lane; c < C; c += 32) mx = fmaxf(mx, dropped_logit(lr, c, i0 + c, seed, step, dp));
        mx = warp_max(mx);
        float se = 0.f;
        for (int c = lane; c < C; c += 32) se += expf(dropped_logit(lr, c, i0 + c, seed, step, dp) - mx);
        se = warp_sum(se);
        const float ls = logf(se);                       // log-sum-exp - mx (see CE_LSE_NOTE)
        for (int c = lane; c < C; c += 32) {
            const float pr = expf((dropped_logit(lr, c, i0 + c, seed, step, dp) - mx) - ls);
            dlogits[(size_t)row * ldl + c] = (pr - (c == y ? 1.f : 0.f)) * invB;
        }
        if (lane == 0) row_loss[r] = ((mx - dropped_logit(lr, y, i0 + y, seed, step, dp)) + ls) * invB;
    } else {
        const float inv = 1.0f / ((float)B * (float)C);
        const float* yr = labels_f32 + (size_t)targets[r] * C;
        float a = 0.f;
        for (int c = lane; c < C; c += 32) {
            const float l = dropped_logit(lr, c, i0 + c, seed, step, dp), y = yr[c];
            a += (1.0f - y) * l + fmaxf(-l, 0.f) + log1pf(expf(-fabsf(l)));
            dlogits[(size_t)row * ldl + c] = (1.0f / (1.0f + expf(-l)) - y) * inv;
        }
        a = warp_sum(a);
        if (lane == 0) row_loss[r] = a * inv;
    }
}

// one CTA: drops every row of the logits in place, adds the reg_param term on the dropped logits, masks the whole
// gradient, then advances the step word
__global__ void __launch_bounds__(LOSS_THREADS) k_loss_final_dropout(float* __restrict__ logits, int ldl, int C,
                                                                     const int* __restrict__ A_dev, int A_cap, int B,
                                                                     const float* __restrict__ row_loss,
                                                                     float reg_param, float* __restrict__ dlogits,
                                                                     float* loss_out, DropParams dp) {
    pdl_begin();
    __shared__ float s[32];
    const int A = min(*A_dev, A_cap);
    const int lane = lane_id(), warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const unsigned long long seed = dp.state[0], step = dp.state[1];
    float part = 0.f;
    for (int r = threadIdx.x; r < B; r += blockDim.x) part += row_loss[r];
    float loss = block_sum_1024(part, s);
    const bool reg = reg_param != 0.f && C > 1;
    float rp = 0.f;
    for (int row = warp; row < A; row += nwarps) {
        float* lr = logits + (size_t)row * ldl;
        float* dr = dlogits + (size_t)row * ldl;
        const unsigned long long i0 = (unsigned long long)row * C;
        for (int c = lane; c < C; c += 32) lr[c] = dropped_logit(lr, c, i0 + c, seed, step, dp);
        if (reg) {                                       // reg_param * sum_rows var(logits, dim=1), unbiased
            const float invc1 = 1.0f / (float)(C - 1);
            float sm = 0.f;
            for (int c = lane; c < C; c += 32) sm += lr[c];
            const float mean = warp_sum(sm) / (float)C;
            float sq = 0.f;
            for (int c = lane; c < C; c += 32) {
                const float d = lr[c] - mean;
                sq = fmaf(d, d, sq);
                dr[c] += reg_param * 2.0f * d * invc1;
            }
            sq = warp_sum(sq);
            if (lane == 0) rp += sq * invc1;
        }
        for (int c = lane; c < C; c += 32)
            dr[c] = dropout_keep(seed, step, dp.tag, dp.threshold, i0 + c) ? dr[c] * dp.scale : 0.f;
    }
    if (reg) loss += reg_param * block_sum_1024(rp, s);
    __syncthreads();
    if (threadIdx.x == 0) {
        *loss_out = loss;
        dp.state[1] = step + 1ull;
    }
}

// keep[r * width + c] = keep bit of entry (r, c) of a dropout site, r < *rows_dev (the step's masks, for inspection)
__global__ void __launch_bounds__(256) k_dropout_mask(unsigned long long seed, unsigned long long step, uint32_t tag,
                                                      uint32_t threshold, const int* __restrict__ rows_dev, int cap_rows,
                                                      int width, uint8_t* __restrict__ keep) {
    pdl_begin();
    const long long n = (long long)min(*rows_dev, cap_rows) * width;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        keep[i] = dropout_keep(seed, step, tag, threshold, (unsigned long long)i) ? 1 : 0;
}

// scal layout (float): see GRAPES_SCAL_* in the header.
//   TB       : loss_gfn = (log_z + tot + coef*loss_c)^2 ; d/dtheta = 2(...) * (dlog_z + dtot)      main.py:282
//   REINFORCE: loss_gfn = -tot * loss_c                 ; d/dtheta = -loss_c * dtot               main.py:279
__global__ void k_gfn_finalize(float* scal, float loss_coef, float log_z_init, int reinforce, int have_log_z) {
    pdl_begin();
    const float loss_c = scal[GRAPES_SCAL_LOSS_C];
    const float tot = scal[GRAPES_SCAL_TOT_LOG_PROB];
    const float log_z = have_log_z ? scal[GRAPES_SCAL_LOG_Z_MEAN] - log_z_init : 0.f;
    scal[GRAPES_SCAL_LOG_Z] = log_z;
    if (reinforce) {
        scal[GRAPES_SCAL_LOSS_GFN] = -tot * loss_c;
        scal[GRAPES_SCAL_G_GF] = -loss_c;
        scal[GRAPES_SCAL_G_Z] = 0.f;
    } else {
        const float r = log_z + tot + loss_coef * loss_c;
        scal[GRAPES_SCAL_LOSS_GFN] = r * r;
        scal[GRAPES_SCAL_G_GF] = 2.0f * r;
        scal[GRAPES_SCAL_G_Z] = 2.0f * r;
    }
}

// grad[i] = (*g) * dir[i]
__global__ void __launch_bounds__(256) k_scale_by_dev(const float* __restrict__ dir, const float* __restrict__ g, int n,
                                                      float* __restrict__ grad) {
    pdl_begin();
    const float gg = *g;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) grad[i] = gg * dir[i];
}

// torch.optim.Adam single-tensor math on a flat buffer; `step` (device, float) is the count BEFORE this update.
__global__ void __launch_bounds__(256) k_adam(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                              float* __restrict__ v, int n, float lr, float beta1, float beta2,
                                              float eps, const float* __restrict__ step) {
    pdl_begin();
    __shared__ float s_step_size, s_bc2_sqrt;
    if (threadIdx.x == 0) {
        const double t = (double)(*step) + 1.0;
        const double bc1 = 1.0 - pow((double)beta1, t), bc2 = 1.0 - pow((double)beta2, t);
        s_step_size = (float)((double)lr / bc1);
        s_bc2_sqrt = (float)sqrt(bc2);
    }
    __syncthreads();
    const float step_size = s_step_size, bc2s = s_bc2_sqrt;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float gi = g[i];
        const float mi = m[i] + (gi - m[i]) * (1.0f - beta1);          // exp_avg.lerp_(grad, 1-beta1)
        const float vi = v[i] * beta2 + (1.0f - beta2) * gi * gi;      // mul_(beta2).addcmul_(g, g, 1-beta2)
        m[i] = mi; v[i] = vi;
        const float denom = sqrtf(vi) / bc2s + eps;
        p[i] = p[i] - step_size * (mi / denom);
    }
}
__global__ void k_step_inc(float* step) {
    pdl_begin(); *step += 1.0f; }
// finalize + scale in one launch: every block recomputes the scalar from the (read-only) inputs of `scal`, block 0
// publishes the derived scalars; grad = g * direction for the gcn_gf and gcn_z parameter ranges.
__global__ void __launch_bounds__(256) k_gfn_finalize_scale(float* scal, float loss_coef, float log_z_init, int reinforce,
                                                            int have_log_z, const float* __restrict__ dir_gf, int n_gf,
                                                            float* __restrict__ grad_gf,
                                                            const float* __restrict__ dir_z, int n_z,
                                                            float* __restrict__ grad_z) {
    pdl_begin();
    const float loss_c = scal[GRAPES_SCAL_LOSS_C];
    const float tot = scal[GRAPES_SCAL_TOT_LOG_PROB];
    const float log_z = have_log_z ? scal[GRAPES_SCAL_LOG_Z_MEAN] - log_z_init : 0.f;
    float loss_gfn, g_gf, g_z;
    if (reinforce) { loss_gfn = -tot * loss_c; g_gf = -loss_c; g_z = 0.f; }
    else { const float r = log_z + tot + loss_coef * loss_c; loss_gfn = r * r; g_gf = 2.0f * r; g_z = 2.0f * r; }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        scal[GRAPES_SCAL_LOG_Z] = log_z;
        scal[GRAPES_SCAL_LOSS_GFN] = loss_gfn;
        scal[GRAPES_SCAL_G_GF] = g_gf;
        scal[GRAPES_SCAL_G_Z] = g_z;
    }
    const int tot_n = n_gf + n_z;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < tot_n; i += gridDim.x * blockDim.x) {
        if (i < n_gf) grad_gf[i] = g_gf * dir_gf[i];
        else grad_z[i - n_gf] = g_z * dir_z[i - n_gf];
    }
}

// Learned node features (main.py:89-100,116: an nn.Parameter table [N, F] inside optimizer_c).  torch.optim.Adam is DENSE:
// every row's moments decay and every row whose moments are non-zero keeps moving, not only the rows of this batch.  The
// gradient is sparse -- d loss_c / d x is non-zero only on the batch's all_nodes rows -- so it is read through the
// all_nodes bitmap (local row = rank of the bit) instead of being scattered into a dense [N, F] buffer first.  Rows that
// were never touched (m = v = 0, no gradient) are left alone: their update is exactly 0.  The bias correction uses
// t = *step + t_add: t_add = 1 when `step` is optimizer_c's count BEFORE this update (grapes_adam_embed: the parameter
// Adam launched afterwards increments it), 0 when that launch already ran (grapes_embed_merge_adam).  go != NULL: the
// go word of a data-parallel exchange; a failed exchange (GO_FAIL) makes the launch a no-op.  The walk covers the N
// rows [row0, row0 + N) of the table: x, m and v point at row row0 (a shard of a table sharded by rows), while the
// gradient bitmap and its rank are those of the whole table, tested at row0 + the local row.
__global__ void __launch_bounds__(256) k_adam_embed(float* __restrict__ x, float* __restrict__ m, float* __restrict__ v,
                                                    int row0, int64_t N, int F4, const uint32_t* __restrict__ bm,
                                                    const int* __restrict__ pref, const float* __restrict__ grows,
                                                    int ldg4, float lr, float beta1, float beta2, float eps,
                                                    const float* __restrict__ step, const unsigned int* go, float t_add) {
    pdl_begin();
    if (go && (*(volatile const unsigned int*)go & GO_FAIL)) return;
    __shared__ float s_step_size, s_bc2_sqrt;
    if (threadIdx.x == 0) {
        const double t = (double)(*step) + (double)t_add;
        const double bc1 = 1.0 - pow((double)beta1, t), bc2 = 1.0 - pow((double)beta2, t);
        s_step_size = (float)((double)lr / bc1);
        s_bc2_sqrt = (float)sqrt(bc2);
    }
    __syncthreads();
    const float step_size = s_step_size, bc2s = s_bc2_sqrt;
    const int64_t total = N * (int64_t)F4;
    float4* x4 = reinterpret_cast<float4*>(x);
    float4* m4 = reinterpret_cast<float4*>(m);
    float4* v4 = reinterpret_cast<float4*>(v);
    const float4* g4 = reinterpret_cast<const float4*>(grows);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int local = (int)(i / F4), c = (int)(i - (int64_t)local * F4), node = row0 + local;
        const bool hit = bitmap_test(bm, node);
        float4 mi = m4[i], vi = v4[i];
        if (!hit && mi.x == 0.f && mi.y == 0.f && mi.z == 0.f && mi.w == 0.f && vi.x == 0.f && vi.y == 0.f &&
            vi.z == 0.f && vi.w == 0.f)
            continue;
        float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
        if (hit) g = g4[(size_t)bitmap_rank(bm, pref, node) * ldg4 + c];
        float4 p = x4[i];
#define GRAPES_ADAM1(f)                                                                       \
        mi.f = mi.f + (g.f - mi.f) * (1.0f - beta1);                                          \
        vi.f = vi.f * beta2 + (1.0f - beta2) * g.f * g.f;                                     \
        p.f = p.f - step_size * (mi.f / (sqrtf(vi.f) / bc2s + eps));
        GRAPES_ADAM1(x) GRAPES_ADAM1(y) GRAPES_ADAM1(z) GRAPES_ADAM1(w)
#undef GRAPES_ADAM1
        m4[i] = mi; v4[i] = vi; x4[i] = p;
    }
}

// ---- data-parallel learned table: merge of the ranks' row-sparse gradients (grapes_embed_merge_adam) ----
// world slots of grapes_embed_slot_floats floats, each [A, 3 pad | ids, cap rounded up to 4 | rows, cap x F]
// (peer_comm.cu).  state != NULL: `slots` is this rank's second symmetric buffer (both parities) and the go word of the
// step's exchange picks the parity, or makes every launch a no-op when the peers did not arrive.
#define EMBED_MAX_WORLD 8

__device__ __forceinline__ const float* embed_slots(const float* slots, long long slot, int world,
                                                    const unsigned int* state, bool* skip) {
    *skip = false;
    if (!state) return slots;
    const unsigned int go = *(volatile const unsigned int*)(state + PS_GO);
    *skip = (go & GO_FAIL) != 0u;
    return slots + (size_t)(go & 1u) * world * slot;
}

__global__ void __launch_bounds__(256) k_embed_union(const float* slots, long long slot, int world, int cap,
                                                     const unsigned int* state, uint32_t* bm) {
    pdl_begin();
    bool skip;
    const float* base = embed_slots(slots, slot, world, state, &skip);
    if (skip) return;
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
    for (int r = 0; r < world; ++r) {
        const int* s = reinterpret_cast<const int*>(base + (size_t)r * slot);
        const int A = min(__ldcg(s), cap);
        for (int i = gtid; i < A; i += gsz) bitmap_set(bm, __ldcg(s + 4 + i));
    }
}

// one warp per union row v: lane r < world finds v in slot r's ascending id list (binary search), then the lanes walk
// the row's float4 columns and add the ranks' rows in rank order (identical bits on every rank), times 1 / world
__global__ void __launch_bounds__(256) k_embed_mean_rows(const float* slots, long long slot, int world, int cap, int F4,
                                                         const unsigned int* state, const int* __restrict__ ids,
                                                         const int* __restrict__ U_dev, int cap_U, float* __restrict__ mean,
                                                         float inv_w) {
    pdl_begin();
    bool skip;
    const float* base = embed_slots(slots, slot, world, state, &skip);
    if (skip) return;
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    const int U = min(*U_dev, cap_U);
    const int cap4 = (cap + 3) & ~3;
    for (int row = warp; row < U; row += nwarps) {
        const int v = ids[row];
        int pos = -1;
        if (lane < world) {
            const int* s = reinterpret_cast<const int*>(base + (size_t)lane * slot);
            const int A = min(__ldcg(s), cap);
            int lo = 0, hi = A;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (__ldcg(s + 4 + mid) < v) lo = mid + 1; else hi = mid;
            }
            if (lo < A && __ldcg(s + 4 + lo) == v) pos = lo;
        }
        int p[EMBED_MAX_WORLD];
#pragma unroll
        for (int r = 0; r < EMBED_MAX_WORLD; ++r) p[r] = __shfl_sync(0xffffffffu, pos, r);
        for (int c = lane; c < F4; c += 32) {
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int r = 0; r < EMBED_MAX_WORLD; ++r) {
                if (r < world && p[r] >= 0) {
                    const float4* rows = reinterpret_cast<const float4*>(base + (size_t)r * slot + 4 + cap4);
                    const float4 g = __ldcg(rows + (size_t)p[r] * F4 + c);
                    acc.x += g.x; acc.y += g.y; acc.z += g.z; acc.w += g.w;
                }
            }
            acc.x *= inv_w; acc.y *= inv_w; acc.z *= inv_w; acc.w *= inv_w;
            reinterpret_cast<float4*>(mean)[(size_t)row * F4 + c] = acc;
        }
    }
}

// Two Adam parameter groups (optimizer_c, optimizer_gf: main.py:117-118) in one launch.  Every block reads the step
// counts before anyone changes them; the last block to finish increments both (threadfence + ticket), so no
// separate increment launch is needed.
__global__ void __launch_bounds__(256) k_adam2(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                               float* __restrict__ v, int off0, int n0, float lr0, int off1, int n1,
                                               float lr1, float beta1, float beta2, float eps, float* steps,
                                               unsigned int* ticket) {
    pdl_begin();
    __shared__ float s_step_size[2], s_bc2_sqrt[2];
    __shared__ int s_last;
    if (threadIdx.x < 2) {
        const double t = (double)steps[threadIdx.x] + 1.0;
        const double bc1 = 1.0 - pow((double)beta1, t), bc2 = 1.0 - pow((double)beta2, t);
        s_step_size[threadIdx.x] = (float)((double)(threadIdx.x ? lr1 : lr0) / bc1);
        s_bc2_sqrt[threadIdx.x] = (float)sqrt(bc2);
    }
    __syncthreads();
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < n0 + n1; t += gridDim.x * blockDim.x) {
        const int grp = t < n0 ? 0 : 1;
        const int i = grp ? off1 + (t - n0) : off0 + t;
        const float gi = g[i];
        const float mi = adam_exp_avg(m[i], gi, beta1);
        const float vi = adam_exp_avg_sq(v[i], gi, beta2);
        m[i] = mi; v[i] = vi;
        const float denom = sqrtf(vi) / s_bc2_sqrt[grp] + eps;
        p[i] = p[i] - s_step_size[grp] * (mi / denom);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1) ? 1 : 0;
    }
    __syncthreads();
    if (s_last && threadIdx.x == 0) {
        if (n0 > 0) steps[0] += 1.0f;
        if (n1 > 0) steps[1] += 1.0f;
        *ticket = 0u;
    }
}

// predictions = argmax(logits, dim=1)[row_ids]  (eval.py:152-153); ties go to the lowest class index, NaN never wins
__global__ void __launch_bounds__(256) k_argmax_rows(const float* __restrict__ logits, int ldl, int C,
                                                     const int* __restrict__ row_ids, const int* __restrict__ B_dev,
                                                     int cap_B, int* __restrict__ out) {
    pdl_begin();
    const int B = min(*B_dev, cap_B);
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < B; i += warps) {
        const float* row = logits + (size_t)row_ids[i] * ldl;
        float best = -INFINITY;
        int arg = 0x7fffffff;
        for (int c = lane; c < C; c += 32) {
            const float v = row[c];
            if (v > best || (v == best && c < arg)) { best = v; arg = c; }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ob = __shfl_xor_sync(GRAPES_FULL_MASK, best, o);
            const int oa = __shfl_xor_sync(GRAPES_FULL_MASK, arg, o);
            if (ob > best || (ob == best && oa < arg)) { best = ob; arg = oa; }
        }
        if (lane == 0) out[i] = (arg == 0x7fffffff) ? 0 : arg;
    }
}

__global__ void __launch_bounds__(256) k_fill_f32(float* p, float v, int n) {
    pdl_begin();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) p[i] = v;
}

static inline int grid_for(const grapes_ctx* ctx, long long work, int threads, int per_sm = 8) {
    long long b = (work + threads - 1) / threads;
    long long cap = (long long)ctx->sm_count * per_sm;
    if (b < 1) b = 1;
    return (int)(b < cap ? b : cap);
}

extern "C" {

int grapes_classifier_loss(grapes_ctx* ctx, const float* logits, int ldl, int C, const int* A_dev, int A_cap,
                           const int* row_ids, const int* tgt_of_row, const int* targets, int B, const int64_t* labels_i64,
                           const float* labels_f32, float reg_param, float* dlogits, float* loss_out,
                           float* colsum_out, void* stream) {
    GRAPES_REQUIRE(ctx && logits && A_dev && row_ids && targets && dlogits && loss_out, "null argument");
    GRAPES_REQUIRE((labels_i64 != nullptr) != (labels_f32 != nullptr), "exactly one label array");
    GRAPES_REQUIRE(B > 0 && C > 0, "bad shape");
    cudaStream_t s = (cudaStream_t)stream;
    if (tgt_of_row && C <= LOSS_THREADS) {
        const int nblocks = grapes_div_up(A_cap, LR2_WARPS);
        GRAPES_REQUIRE(((size_t)A_cap + (size_t)nblocks * C) * sizeof(float) <= ctx->partials_bytes, "partial buffer too small");
        float* row_loss = ctx->partials;
        float* colpart = ctx->partials + A_cap;
        pdl((k_loss_rows2), nblocks, LR2_WARPS * 32, LR2_WARPS * C * sizeof(float), s)(
            logits, ldl, C, A_dev, A_cap, tgt_of_row, targets, B, labels_i64, labels_f32, reg_param, dlogits, row_loss,
            colpart);
        grapes_count_launches(1);
        pdl((k_loss_final2), 1, LOSS_THREADS, 0, s)(A_dev, A_cap, C, row_loss, colpart, nblocks, loss_out, colsum_out);
        grapes_count_launches(1);
        GRAPES_LAUNCH_OK();
        return GRAPES_OK;
    }
    GRAPES_CUDA_OK(cudaMemsetAsync(dlogits, 0, sizeof(float) * (size_t)A_cap * ldl, s));
    GRAPES_REQUIRE((size_t)B * sizeof(float) <= ctx->partials_bytes, "partial buffer too small");
    pdl((k_loss_rows), grapes_div_up((long long)B * 32, 256), 256, 0, s)(logits, ldl, C, row_ids, targets, B, labels_i64,
                                                                      labels_f32, dlogits, ctx->partials);
    grapes_count_launches(1);
    pdl((k_loss_final), 1, LOSS_THREADS, 0, s)(logits, ldl, C, A_dev, A_cap, B, ctx->partials, reg_param, dlogits,
                                            loss_out);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    if (colsum_out) return grapes_colsum(ctx, dlogits, A_dev, A_cap, ldl, C, 1.0f, 0, colsum_out, stream);
    return GRAPES_OK;
}

int grapes_classifier_loss_dropout(grapes_ctx* ctx, float* logits, int ldl, int C, const int* A_dev, int A_cap,
                                   const int* row_ids, const int* tgt_of_row, const int* targets, int B,
                                   const int64_t* labels_i64, const float* labels_f32, float reg_param, float* dlogits,
                                   float* loss_out, float* colsum_out, unsigned long long* drop_state, uint32_t tag,
                                   uint32_t threshold, float scale, void* stream) {
    GRAPES_REQUIRE(ctx && logits && A_dev && row_ids && targets && dlogits && loss_out && drop_state, "null argument");
    GRAPES_REQUIRE((labels_i64 != nullptr) != (labels_f32 != nullptr), "exactly one label array");
    GRAPES_REQUIRE(B > 0 && C > 0, "bad shape");
    GRAPES_REQUIRE(tag >= 1u && threshold <= (1u << 24), "bad dropout parameters");
    cudaStream_t s = (cudaStream_t)stream;
    const DropParams dp = {drop_state, tag, threshold, scale};
    if (tgt_of_row && C <= LOSS_THREADS) {
        const int nblocks = grapes_div_up(A_cap, LR2_WARPS);
        GRAPES_REQUIRE(((size_t)A_cap + (size_t)nblocks * C) * sizeof(float) <= ctx->partials_bytes, "partial buffer too small");
        float* row_loss = ctx->partials;
        float* colpart = ctx->partials + A_cap;
        pdl((k_loss_rows2_dropout), nblocks, LR2_WARPS * 32, LR2_WARPS * C * sizeof(float), s)(
            logits, ldl, C, A_dev, A_cap, tgt_of_row, targets, B, labels_i64, labels_f32, reg_param, dlogits, row_loss,
            colpart, dp);
        grapes_count_launches(1);
        pdl((k_loss_final2_dropout), 1, LOSS_THREADS, 0, s)(A_dev, A_cap, C, row_loss, colpart, nblocks, loss_out,
                                                            colsum_out, dp);
        grapes_count_launches(1);
        GRAPES_LAUNCH_OK();
        return GRAPES_OK;
    }
    GRAPES_CUDA_OK(cudaMemsetAsync(dlogits, 0, sizeof(float) * (size_t)A_cap * ldl, s));
    GRAPES_REQUIRE((size_t)B * sizeof(float) <= ctx->partials_bytes, "partial buffer too small");
    pdl((k_loss_rows_dropout), grapes_div_up((long long)B * 32, 256), 256, 0, s)(logits, ldl, C, row_ids, targets, B,
                                                                              labels_i64, labels_f32, dlogits,
                                                                              ctx->partials, dp);
    grapes_count_launches(1);
    pdl((k_loss_final_dropout), 1, LOSS_THREADS, 0, s)(logits, ldl, C, A_dev, A_cap, B, ctx->partials, reg_param,
                                                       dlogits, loss_out, dp);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    if (colsum_out) return grapes_colsum(ctx, dlogits, A_dev, A_cap, ldl, C, 1.0f, 0, colsum_out, stream);
    return GRAPES_OK;
}

int grapes_dropout_mask(grapes_ctx* ctx, int64_t seed, int64_t step, uint32_t tag, uint32_t threshold,
                        const int* rows_dev, int cap_rows, int width, uint8_t* keep, void* stream) {
    GRAPES_REQUIRE(ctx && rows_dev && keep, "null argument");
    GRAPES_REQUIRE(cap_rows >= 0 && width > 0, "bad shape");
    pdl((k_dropout_mask), grid_for(ctx, (long long)cap_rows * width, 256), 256, 0, (cudaStream_t)stream)(
        (unsigned long long)seed, (unsigned long long)step, tag, threshold, rows_dev, cap_rows, width, keep);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_gfn_finalize(grapes_ctx* ctx, float* scal, float loss_coef, float log_z_init, int reinforce, int have_log_z,
                        void* stream) {
    GRAPES_REQUIRE(ctx && scal, "null argument");
    pdl((k_gfn_finalize), 1, 1, 0, (cudaStream_t)stream)(scal, loss_coef, log_z_init, reinforce, have_log_z);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_scale_by_device_scalar(grapes_ctx* ctx, const float* dir, const float* g_dev, int n, float* grad,
                                  void* stream) {
    GRAPES_REQUIRE(ctx && dir && g_dev && grad, "null argument");
    pdl((k_scale_by_dev), grid_for(ctx, n, 256), 256, 0, (cudaStream_t)stream)(dir, g_dev, n, grad);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_adam_step(grapes_ctx* ctx, float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int n,
                     float lr, float beta1, float beta2, float eps, float* step_dev, int increment_step,
                     void* stream) {
    GRAPES_REQUIRE(ctx && params && grads && exp_avg && exp_avg_sq && step_dev, "null argument");
    cudaStream_t s = (cudaStream_t)stream;
    pdl((k_adam), grid_for(ctx, n, 256), 256, 0, s)(params, grads, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps,
                                                 step_dev);
    grapes_count_launches(1);
    if (increment_step) pdl((k_step_inc), 1, 1, 0, s)(step_dev);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_gfn_finalize_scale(grapes_ctx* ctx, float* scal, float loss_coef, float log_z_init, int reinforce,
                              int have_log_z, const float* dir_gf, int n_gf, float* grad_gf, const float* dir_z,
                              int n_z, float* grad_z, void* stream) {
    GRAPES_REQUIRE(ctx && scal && dir_gf && grad_gf && (n_z == 0 || (dir_z && grad_z)), "null argument");
    pdl((k_gfn_finalize_scale), grid_for(ctx, n_gf + n_z, 256), 256, 0, (cudaStream_t)stream)(
        scal, loss_coef, log_z_init, reinforce, have_log_z, dir_gf, n_gf, grad_gf, dir_z, n_z, grad_z);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_adam_step2(grapes_ctx* ctx, float* params, const float* grads, float* exp_avg, float* exp_avg_sq,
                      int off0, int n0, float lr0, int off1, int n1, float lr1, float beta1, float beta2, float eps,
                      float* steps_dev, void* stream) {
    GRAPES_REQUIRE(ctx && params && grads && exp_avg && exp_avg_sq && steps_dev, "null argument");
    GRAPES_REQUIRE(n0 >= 0 && n1 >= 0 && n0 + n1 > 0, "empty parameter groups");
    pdl((k_adam2), grid_for(ctx, n0 + n1, 256), 256, 0, (cudaStream_t)stream)(params, grads, exp_avg, exp_avg_sq, off0, n0,
                                                                           lr0, off1, n1, lr1, beta1, beta2, eps,
                                                                           steps_dev, ctx->scan_counters + 2);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

// the walk of k_adam_embed over rows [row0, row0 + rows) (0 rows: no launch); go: see k_adam_embed
static void launch_adam_embed(grapes_ctx* ctx, float* table, float* exp_avg, float* exp_avg_sq, int64_t row0,
                              int64_t rows, int F, const uint32_t* bm, const int* pref, const float* grad_rows, int ldg,
                              float lr, float beta1, float beta2, float eps, const float* step_dev, const unsigned int* go,
                              float t_add, cudaStream_t s) {
    if (rows == 0) return;
    const long long total = (long long)rows * (F / 4);
    long long blocks = (total + 255) / 256;
    const long long cap = (long long)ctx->sm_count * 8;
    if (blocks > cap) blocks = cap;
    pdl((k_adam_embed), (int)blocks, 256, 0, s)(table, exp_avg, exp_avg_sq, (int)row0, rows, F / 4, bm, pref, grad_rows,
                                               ldg / 4, lr, beta1, beta2, eps, step_dev, go, t_add);
    grapes_count_launches(1);
}

int grapes_adam_embed(grapes_ctx* ctx, float* table, float* exp_avg, float* exp_avg_sq, int64_t num_nodes, int F,
                      const uint32_t* bm_rows, const int* pref_rows, const float* grad_rows, int ldg, float lr,
                      float beta1, float beta2, float eps, const float* step_dev, void* stream) {
    GRAPES_REQUIRE(ctx && table && exp_avg && exp_avg_sq && bm_rows && pref_rows && grad_rows && step_dev, "null argument");
    GRAPES_REQUIRE(F > 0 && F % 4 == 0 && ldg % 4 == 0 && ldg >= F, "embedding width and gradient pitch must be multiples of 4");
    GRAPES_REQUIRE(num_nodes == ctx->num_nodes, "table rows != graph nodes");
    launch_adam_embed(ctx, table, exp_avg, exp_avg_sq, 0, num_nodes, F, bm_rows, pref_rows, grad_rows, ldg, lr, beta1,
                      beta2, eps, step_dev, nullptr, 1.0f, (cudaStream_t)stream);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_adam_embed_rows(grapes_ctx* ctx, float* table, float* exp_avg, float* exp_avg_sq, int64_t num_nodes,
                           int64_t row0, int64_t rows, int F, const uint32_t* bm_rows, const int* pref_rows,
                           const float* grad_rows, int ldg, float lr, float beta1, float beta2, float eps,
                           const float* step_dev, void* stream) {
    GRAPES_REQUIRE(ctx && bm_rows && pref_rows && grad_rows && step_dev, "null argument");
    GRAPES_REQUIRE(rows == 0 || (table && exp_avg && exp_avg_sq), "null shard");
    GRAPES_REQUIRE(F > 0 && F % 4 == 0 && ldg % 4 == 0 && ldg >= F, "embedding width and gradient pitch must be multiples of 4");
    GRAPES_REQUIRE(0 <= row0 && rows >= 0 && row0 + rows <= num_nodes, "row range outside the table");
    GRAPES_REQUIRE(num_nodes <= ctx->num_nodes, "table rows > graph nodes");
    launch_adam_embed(ctx, table, exp_avg, exp_avg_sq, row0, rows, F, bm_rows, pref_rows, grad_rows, ldg, lr, beta1,
                      beta2, eps, step_dev, nullptr, 1.0f, (cudaStream_t)stream);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

// union, rank and mean rows of the world slots, then the table walk over [row0, row0 + rows)
static int embed_merge_adam(grapes_ctx* ctx, const float* slots, int world, int cap_rows, int F,
                            const unsigned int* state, uint32_t* bm_union, int* pref_union, int* union_ids, int cap_union,
                            int* union_count, float* mean_rows, float* table, float* exp_avg, float* exp_avg_sq,
                            int64_t row0, int64_t rows, float lr, float beta1, float beta2, float eps,
                            const float* step_dev, int* overflow, void* stream) {
    cudaStream_t s = (cudaStream_t)stream;
    const long long slot = grapes_embed_slot_floats(cap_rows, F);
    pdl((k_embed_union), grid_for(ctx, (long long)cap_rows, 256), 256, 0, s)(slots, slot, world, cap_rows, state, bm_union);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    // popcount-prefix rank of the union bitmap: ascending union ids and the local row of every id
    const int rc = grapes_rank_nodes(ctx, bm_union, nullptr, pref_union, nullptr, union_ids, nullptr, nullptr, nullptr,
                                     nullptr, nullptr, 0, 0, cap_union, union_count, nullptr, overflow, stream);
    if (rc != GRAPES_OK) return rc;
    pdl((k_embed_mean_rows), grid_for(ctx, (long long)cap_union * 32, 256), 256, 0, s)(
        slots, slot, world, cap_rows, F / 4, state, union_ids, union_count, cap_union, mean_rows, 1.0f / (float)world);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    launch_adam_embed(ctx, table, exp_avg, exp_avg_sq, row0, rows, F, bm_union, pref_union, mean_rows, F, lr, beta1,
                      beta2, eps, step_dev, state ? state + PS_GO : nullptr, 0.0f, s);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_embed_merge_adam(grapes_ctx* ctx, const float* slots, int world, int cap_rows, int F,
                            const unsigned int* state, uint32_t* bm_union, int* pref_union, int* union_ids, int cap_union,
                            int* union_count, float* mean_rows, float* table, float* exp_avg, float* exp_avg_sq,
                            int64_t num_nodes, float lr, float beta1, float beta2, float eps, const float* step_dev,
                            int* overflow, void* stream) {
    GRAPES_REQUIRE(ctx && slots && bm_union && pref_union && union_ids && union_count && mean_rows && table && exp_avg &&
                       exp_avg_sq && step_dev && overflow, "null argument");
    GRAPES_REQUIRE(world >= 1 && world <= EMBED_MAX_WORLD, "1 <= world <= 8");
    GRAPES_REQUIRE(F > 0 && F % 4 == 0 && cap_rows > 0 && cap_union > 0, "table width must be a multiple of 4");
    GRAPES_REQUIRE(num_nodes == ctx->num_nodes, "table rows != graph nodes");
    return embed_merge_adam(ctx, slots, world, cap_rows, F, state, bm_union, pref_union, union_ids, cap_union,
                            union_count, mean_rows, table, exp_avg, exp_avg_sq, 0, num_nodes, lr, beta1, beta2, eps,
                            step_dev, overflow, stream);
}

int grapes_embed_merge_adam_rows(grapes_ctx* ctx, const float* slots, int world, int cap_rows, int F,
                                 const unsigned int* state, uint32_t* bm_union, int* pref_union, int* union_ids,
                                 int cap_union, int* union_count, float* mean_rows, float* table, float* exp_avg,
                                 float* exp_avg_sq, int64_t num_nodes, int64_t row0, int64_t rows, float lr, float beta1,
                                 float beta2, float eps, const float* step_dev, int* overflow, void* stream) {
    GRAPES_REQUIRE(ctx && slots && bm_union && pref_union && union_ids && union_count && mean_rows && step_dev &&
                       overflow, "null argument");
    GRAPES_REQUIRE(rows == 0 || (table && exp_avg && exp_avg_sq), "null shard");
    GRAPES_REQUIRE(world >= 1 && world <= EMBED_MAX_WORLD, "1 <= world <= 8");
    GRAPES_REQUIRE(F > 0 && F % 4 == 0 && cap_rows > 0 && cap_union > 0, "table width must be a multiple of 4");
    GRAPES_REQUIRE(0 <= row0 && rows >= 0 && row0 + rows <= num_nodes, "row range outside the table");
    GRAPES_REQUIRE(num_nodes <= ctx->num_nodes, "table rows > graph nodes");
    return embed_merge_adam(ctx, slots, world, cap_rows, F, state, bm_union, pref_union, union_ids, cap_union,
                            union_count, mean_rows, table, exp_avg, exp_avg_sq, row0, rows, lr, beta1, beta2, eps,
                            step_dev, overflow, stream);
}

int grapes_argmax_rows(grapes_ctx* ctx, const float* logits, int ldl, int C, const int* row_ids, const int* B_dev,
                       int cap_B, int* out, void* stream) {
    GRAPES_REQUIRE(ctx && logits && row_ids && B_dev && out, "null argument");
    GRAPES_REQUIRE(C > 0 && ldl >= C && cap_B > 0, "bad shape");
    pdl((k_argmax_rows), grid_for(ctx, (long long)cap_B * 32, 256), 256, 0, (cudaStream_t)stream)(logits, ldl, C, row_ids,
                                                                                                B_dev, cap_B, out);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_fill_f32(grapes_ctx* ctx, float* p, float value, int n, void* stream) {
    GRAPES_REQUIRE(ctx && p, "null argument");
    pdl((k_fill_f32), grid_for(ctx, n, 256), 256, 0, (cudaStream_t)stream)(p, value, n);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

}  // extern "C"
