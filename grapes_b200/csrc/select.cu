// Per-hop node selection: Gumbel-top-k over the candidate frontier + Bernoulli log-probability of
// the chosen mask + sampler statistics.  Replaces sample_neighborhoods_from_probs
// (/root/reference/modules/utils.py:13-71) and the deterministic top-k of the mini-batch evaluator
// (/root/reference/eval.py:126-130), without the per-hop D2H of the mask (utils.py:60).
//
// One kernel, k_select_fused, does the whole hop on every SM: layer-2 aggregation of the sampler net -> logits
// (main.py:210-213), the perturbed keys (utils.py:37-42) as order-preserving uint32, a 2048-bucket histogram of a
// monotone coarse image of the keys, the exact k-th largest key, and the selected items in ascending order with their
// log-probability / gradient and the entropy statistics.
// Ties at the threshold go to the LOWEST candidate index (torch.topk leaves ties unspecified; the oracle uses
// the same rule).  Integer counting only -> the selected set does not depend on scheduling.
#define GRAPES_PDL_GROUP 16
#include "common.cuh"

#define SEL_BUCKETS 2048
#define SEL_STAT_FLOATS 8            // per-block partials: min p, max p, sum e, sum e^2, sum lp, sum dl

__device__ __forceinline__ uint32_t float_to_ordered(float f) {
    if (f != f) return 0u;                                   // NaN ranks lowest
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ordered_to_float(uint32_t u) {
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}
__device__ __forceinline__ unsigned long long composite(uint32_t ukey, int idx) {
    return ((unsigned long long)ukey << 32) | (unsigned long long)(0xffffffffu - (uint32_t)idx);
}

__device__ __forceinline__ float sigmoidf_(float l) { return 1.0f / (1.0f + expf(-l)); }
// Bernoulli(logits=l).log_prob(y) = -BCEWithLogits(l, y)  (utils.py:71)
__device__ __forceinline__ float bern_log_prob(float l, float y) {
    return -((1.0f - y) * l + fmaxf(-l, 0.f) + log1pf(expf(-fabsf(l))));
}
__device__ __forceinline__ float entropy_bits(float p) {
    const float e = -(p * log2f(p) + (1.0f - p) * log2f(1.0f - p));
    return (e != e) ? 0.f : e;                                // NaN entropy -> 0 (utils.py:52-54)
}

template <typename T, typename Op, int WARPS>
__device__ __forceinline__ T block_reduce(T v, T* smem, Op op, T identity) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = op(v, __shfl_xor_sync(GRAPES_FULL_MASK, v, o));
    if (lane_id() == 0) smem[threadIdx.x >> 5] = v;
    __syncthreads();
    T r = (threadIdx.x < WARPS) ? smem[threadIdx.x] : identity;
    if (threadIdx.x < 32) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) r = op(r, __shfl_xor_sync(GRAPES_FULL_MASK, r, o));
        if (threadIdx.x == 0) smem[0] = r;
    }
    __syncthreads();
    r = smem[0];
    __syncthreads();
    return r;
}
struct OpAdd { __device__ float operator()(float a, float b) const { return a + b; } };
struct OpMin { __device__ float operator()(float a, float b) const { return fminf(a, b); } };
struct OpMax { __device__ float operator()(float a, float b) const { return fmaxf(a, b); } };

// ---------------------------------------------------------------------------------------
// k_select_fused: the whole sampler head of a hop in ONE launch on every SM:
//   phase A  (all blocks; block b owns a contiguous range of frontier rows, hence of candidates)  layer-2 aggregation
//            -> logits, probabilities, noise, perturbed keys, log-prob / gradient of the UNSELECTED outcome, statistic
//            partials; bucket histogram of the keys: shared memory per block, merged into ONE global histogram.
//   barrier 1
//   phase B  every block reads the global histogram and finds the threshold bucket (redundantly, 2048 bins); items of
//            buckets above it are counted (def_count[b]); the few members of the threshold bucket go to a global list.
//   barrier 2
//   phase C  every block ranks the member list exactly on the composite (key desc, index asc) -> the k-th largest
//            composite; selected = composite >= threshold.  Output position of a selected item = selected items of
//            lower blocks (definite counts + selected members below the block's first candidate) + rank inside the
//            block (ballot scan): ascending candidate order, as the reference's mask indexing yields (utils.py:60).
//            Selected items get their log-prob / gradient fixed; per-block deltas.
//   ticket   the last block to finish combines the statistic partials and deltas in block order (deterministic) and
//            cleans the scratch for the next launch.
// The barriers are software (arrive counter + bounded spin): the grid is at most one block per SM, so every block becomes
// resident without the all-at-once admission of a cooperative launch (early blocks start while late ones still wait for
// an SM held by a side-stream kernel).  Integer counting only -> the selected set does not depend on scheduling.
// Crowded threshold bucket (massive ties): block 0 runs an MSB-first radix select on the 64-bit composites.
// ---------------------------------------------------------------------------------------
#define SF_THREADS 512
#define SF_WARPS (SF_THREADS / 32)
#define SF_MEMBER_CAP 2048
// int words of scratch behind the float part of `work`
#define SF_I_BAR1 0
#define SF_I_BAR2 1
#define SF_I_TICKET 2
#define SF_I_MCOUNT 3
#define SF_I_THR_READY 4
#define SF_I_ERR 5
#define SF_I_THR_LO 6
#define SF_I_THR_HI 7
#define SF_I_HIST 8                                   // [SEL_BUCKETS]
#define SF_I_DEF (SF_I_HIST + SEL_BUCKETS)            // [max blocks]: definite count per block
#define SF_MAX_BLOCKS 256
#define SF_I_FIRST (SF_I_DEF + SF_MAX_BLOCKS)         // [max blocks]: first candidate index per block
#define SF_I_MEMBER (SF_I_FIRST + SF_MAX_BLOCKS)      // [2 * SF_MEMBER_CAP]: member composites (64-bit)
#define SF_I_STAMP (SF_I_MEMBER + 2 * SF_MEMBER_CAP)   // [16] 64-bit phase time stamps of block 0 (globaltimer ns)
#define SF_I_TOTAL (SF_I_STAMP + 32)
#define SF_DELTA_FLOATS 2                             // per block: lp_delta, dl_delta

__device__ __forceinline__ int key_bucket_m(uint32_t ukey, int mode) {
    if (ukey == 0u) return 0;                                // NaN
    const float v = ordered_to_float(ukey);
    // probabilities (deterministic top-k of the evaluator) live in [0, 1]; perturbed log-probabilities in about [-20, 10]
    const float x = (mode == GRAPES_NOISE_NONE_TOPK_PROBS) ? v * (float)(SEL_BUCKETS - 1) : (v + 32.0f) * 32.0f;
    return (int)fminf(fmaxf(x, 0.f), (float)(SEL_BUCKETS - 1));
}

__device__ __forceinline__ void sf_stamp(int* iw, int slot) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        reinterpret_cast<unsigned long long*>(iw + SF_I_STAMP)[slot] = t;
    }
}
__device__ __forceinline__ int ld_acquire_gpu_i32(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// all threads of the block call it; returns false when the bounded spin ran out (never hangs the GPU)
__device__ __forceinline__ bool sf_grid_barrier(int* counter, int nblocks, int* err) {
    __shared__ int s_ok;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(counter, 1);
        unsigned it = 0;
        int ok = 1;
        while (ld_acquire_gpu_i32(counter) < nblocks) {
            if (++it > 8000000u) { ok = 0; atomicOr(err, 1); break; }     // seconds, never a hang
        }
        s_ok = ok;
    }
    __syncthreads();
    return s_ok != 0;
}

__global__ void __launch_bounds__(SF_THREADS, 1) k_select_fused(
    const float* __restrict__ z, int nparts, int part_stride, const int* __restrict__ n_dev, int cap_n,
    const int* __restrict__ in_off, const int* __restrict__ in_src, const float* __restrict__ dinv,
    const float* __restrict__ bias, const int* __restrict__ nb_index, const int* __restrict__ nb_local,
    const int* __restrict__ nb_nodes, const int* __restrict__ c_dev, int k, int mode, const float* __restrict__ noise,
    unsigned long long* rng_state, float* __restrict__ logits_all, float* lg_c, uint32_t* ukeys,
    float* __restrict__ keys_out, int* __restrict__ sampled_out, int sampled_offset, int* __restrict__ s_dev,
    int* __restrict__ total_dev, uint8_t* __restrict__ mask_out, float* log_prob, float* tot_log_prob,
    float* __restrict__ stats, float* dl_all, float* sum_dl, uint32_t* bm_mark, float* stat_part, float* delta_part,
    int* iw) {
    pdl_begin();
    __shared__ int s_hist[SEL_BUCKETS];
    __shared__ float s_red[SF_WARPS];
    __shared__ long long s_scan[SF_WARPS + 2];
    __shared__ int s_coarse[64];
    __shared__ unsigned long long s_member[SF_MEMBER_CAP];
    __shared__ int s_cb, s_above_c, s_bucket, s_above, s_first, s_wcnt[SF_WARPS], s_last;
    __shared__ unsigned long long s_thr;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nb = gridDim.x, b = blockIdx.x;
    const int n = min(*n_dev, cap_n);
    const int c = min(*c_dev, cap_n);
    const bool take_all = (k >= c);                                   // utils.py:31-33: no noise is drawn
    // block b owns rows [r0, r1): a multiple of the block size per block, so rounds line up with warps
    const int per = ((n + nb - 1) / nb + SF_THREADS - 1) / SF_THREADS * SF_THREADS;
    const int r0 = min(n, b * per), r1 = min(n, r0 + per);
    unsigned long long seed = 0ull, offset = 0ull;
    if (mode == GRAPES_NOISE_PHILOX) { seed = rng_state[0]; offset = rng_state[1]; }
    const float bs = bias ? bias[0] : 0.f;
    int* hist_g = iw + SF_I_HIST;

    // ---------------- phase A ----------------
    sf_stamp(iw, 0);
    for (int q = tid; q < SEL_BUCKETS; q += SF_THREADS) s_hist[q] = 0;
    if (tid == 0) s_first = 0x7fffffff;
    __syncthreads();
    float pmin = INFINITY, pmax = -INFINITY, esum = 0.f, esq = 0.f, lpsum = 0.f, dlsum = 0.f;
    // candidate index, ordered key and logit of this thread's rows of the first two rounds stay in registers for the
    // phases behind the barriers (<= 1024 rows per block: frontiers up to ~150 k rows); later rounds re-read them
    int ci0 = -1, ci1 = -1;
    uint32_t cu0 = 0u, cu1 = 0u;
    float cl0 = 0.f, cl1 = 0.f;
    for (int j = r0 + tid; j < r1; j += SF_THREADS) {
        const int rd = (j - r0) / SF_THREADS;
        float logit;
        if (in_off) {
            const float dj = dinv[j];
            float zj = z[j];
            for (int t = 1; t < nparts; ++t) zj += z[(size_t)t * part_stride + j];
            float a = dj * dj * zj;
            const int end = in_off[j + 1];
            for (int p = in_off[j]; p < end; ++p) {
                const int sl = in_src[p];
                float zs = z[sl];
                for (int t = 1; t < nparts; ++t) zs += z[(size_t)t * part_stride + sl];
                a = fmaf(dinv[sl] * dj, zs, a);
            }
            logit = a + bs;
        } else {
            logit = z[j];
        }
        if (logits_all) logits_all[j] = logit;
        const int i = nb_index ? nb_index[j] : j;
        if (i < 0) {
            if (dl_all) dl_all[j] = 0.f;
            continue;
        }
        if (i < s_first) atomicMin(&s_first, i);
        lg_c[i] = logit;
        const float p = sigmoidf_(logit);
        const float y = take_all ? 1.f : 0.f;
        const float lp = bern_log_prob(logit, y);
        const float d = y - p;
        if (log_prob) log_prob[i] = lp;
        if (dl_all) dl_all[j] = d;
        if (mask_out) mask_out[i] = take_all ? 1 : 0;
        lpsum += lp; dlsum += d;
        if (take_all) {                                               // everything is kept, in candidate order
            const int g = nb_nodes ? nb_nodes[i] : i;
            if (sampled_out) sampled_out[sampled_offset + i] = g;
            if (bm_mark && nb_nodes) bitmap_set(bm_mark, g);
            continue;
        }
        float key;
        if (mode == GRAPES_NOISE_KEYS) key = noise[i];
        else if (mode == GRAPES_NOISE_NONE_TOPK_PROBS) key = p;               // eval.py:126
        else {
            float g;
            if (mode == GRAPES_NOISE_GUMBEL) g = noise[i];
            else {
                float u = (mode == GRAPES_NOISE_UNIFORM) ? noise[i] : philox_uniform(seed, offset, i);
                if (mode == GRAPES_NOISE_PHILOX) u = u * ((1.0f - 1.1920929e-07f) - 1.17549435e-38f) + 1.17549435e-38f;
                g = -logf(-logf(u));
            }
            key = logf(p) + g;                                                // utils.py:42
        }
        const uint32_t uk = float_to_ordered(key);
        ukeys[i] = uk;
        if (rd == 0) { ci0 = i; cu0 = uk; cl0 = logit; } else if (rd == 1) { ci1 = i; cu1 = uk; cl1 = logit; }
        if (keys_out) keys_out[i] = key;
        atomicAdd(&s_hist[key_bucket_m(uk, mode)], 1);
        pmin = fminf(pmin, p); pmax = fmaxf(pmax, p);
        const float e = entropy_bits(p);
        esum += e; esq = fmaf(e, e, esq);
    }
    pmin = block_reduce<float, OpMin, SF_WARPS>(pmin, s_red, OpMin(), INFINITY);
    pmax = block_reduce<float, OpMax, SF_WARPS>(pmax, s_red, OpMax(), -INFINITY);
    esum = block_reduce<float, OpAdd, SF_WARPS>(esum, s_red, OpAdd(), 0.f);
    esq = block_reduce<float, OpAdd, SF_WARPS>(esq, s_red, OpAdd(), 0.f);
    lpsum = block_reduce<float, OpAdd, SF_WARPS>(lpsum, s_red, OpAdd(), 0.f);
    dlsum = block_reduce<float, OpAdd, SF_WARPS>(dlsum, s_red, OpAdd(), 0.f);
    if (tid == 0) {
        float* sp = stat_part + (size_t)b * SEL_STAT_FLOATS;
        sp[0] = pmin; sp[1] = pmax; sp[2] = esum; sp[3] = esq; sp[4] = lpsum; sp[5] = dlsum; sp[6] = 0.f; sp[7] = 0.f;
        delta_part[b * SF_DELTA_FLOATS] = 0.f; delta_part[b * SF_DELTA_FLOATS + 1] = 0.f;
    }
    bool alive = true;
    float lp_delta = 0.f, dl_delta = 0.f;
    sf_stamp(iw, 1);
    if (!take_all) {
        for (int q = tid; q < SEL_BUCKETS; q += SF_THREADS) {
            const int h = s_hist[q];
            if (h) atomicAdd(&hist_g[q], h);
        }
        sf_stamp(iw, 2);
        alive = sf_grid_barrier(iw + SF_I_BAR1, nb, iw + SF_I_ERR);
        sf_stamp(iw, 3);
        // ---------------- phase B: threshold bucket (coarse level of 64 x 32 buckets, then inside the coarse bin) ----
        for (int q = tid; q < SEL_BUCKETS; q += SF_THREADS) s_hist[q] = __ldcg(&hist_g[q]);
        __syncthreads();
        for (int cbn = warp; cbn < 64; cbn += SF_WARPS) {
            const int t = warp_sum(s_hist[cbn * 32 + lane]);
            if (lane == 0) s_coarse[cbn] = t;
        }
        __syncthreads();
        if (warp == 0) {                             // lane l owns coarse bins 63-2l, 62-2l (descending)
            const int t0 = s_coarse[63 - 2 * lane], t1 = s_coarse[62 - 2 * lane];
            const int incl = warp_scan_incl(t0 + t1), excl = incl - (t0 + t1);
            if (excl < k && excl + t0 >= k) { s_cb = 63 - 2 * lane; s_above_c = excl; }
            else if (excl + t0 < k && incl >= k) { s_cb = 62 - 2 * lane; s_above_c = excl + t0; }
        }
        __syncthreads();
        if (warp == 0) {                             // lane l owns bucket 31-l of the coarse bin (descending)
            const int t = s_hist[s_cb * 32 + 31 - lane];
            const int incl = warp_scan_incl(t), excl = incl - t;
            const int krem = k - s_above_c;
            if (excl < krem && incl >= krem) { s_bucket = s_cb * 32 + 31 - lane; s_above = s_above_c + excl; }
        }
        __syncthreads();
        const int bucket = s_bucket, above = s_above;
        const int M = s_hist[bucket];                // members of the threshold bucket, GPU-wide
        const bool crowded = M > SF_MEMBER_CAP;
        // definite items of this block + members into the global list
        int my_def = 0;
        for (int j = r0 + tid; j < r1; j += SF_THREADS) {
            const int rd = (j - r0) / SF_THREADS;
            const int i = rd == 0 ? ci0 : rd == 1 ? ci1 : (nb_index ? nb_index[j] : j);
            if (i < 0) continue;
            const uint32_t u = rd == 0 ? cu0 : rd == 1 ? cu1 : ukeys[i];
            const int bk = key_bucket_m(u, mode);
            if (bk > bucket) ++my_def;
            else if (bk == bucket && !crowded) {
                const int pos = atomicAdd(iw + SF_I_MCOUNT, 1);
                if (pos < SF_MEMBER_CAP) reinterpret_cast<unsigned long long*>(iw + SF_I_MEMBER)[pos] = composite(u, i);
            }
        }
        long long tot_def;
        block_scan_excl<long long>((long long)my_def, s_scan, &tot_def);
        if (tid == 0) { iw[SF_I_DEF + b] = (int)tot_def; iw[SF_I_FIRST + b] = s_first; }
        sf_stamp(iw, 4);
        alive = sf_grid_barrier(iw + SF_I_BAR2, nb, iw + SF_I_ERR) && alive;
        sf_stamp(iw, 5);
        // ---------------- phase C: exact threshold, positions, fix-ups ----------------
        unsigned long long thr_comp;
        if (!crowded) {
            for (int t = tid; t < M; t += SF_THREADS)
                s_member[t] = __ldcg(reinterpret_cast<const unsigned long long*>(iw + SF_I_MEMBER) + t);
            __syncthreads();
            const int want = k - above - 1;          // members that must rank above the threshold member
            for (int t = tid; t < M; t += SF_THREADS) {
                const unsigned long long mine = s_member[t];
                int r = 0;
                for (int o = 0; o < M; ++o) r += (s_member[o] > mine);
                if (r == want) s_thr = mine;
            }
            __syncthreads();
            thr_comp = s_thr;
        } else {
            // massive ties: block 0 finds the k-th largest composite by an MSB-first radix select over all candidates
            if (b == 0) {
                unsigned long long prefix = 0ull;
                int krem = k;
                for (int shift = 56; shift >= 0; shift -= 8) {
                    for (int q = tid; q < 256; q += SF_THREADS) s_hist[q] = 0;
                    __syncthreads();
                    const unsigned long long himask = (shift == 56) ? 0ull : (~0ull << (shift + 8));
                    for (int i = tid; i < c; i += SF_THREADS) {
                        const unsigned long long cm = composite(__ldcg(&ukeys[i]), i);
                        if ((cm & himask) == prefix) atomicAdd(&s_hist[(int)((cm >> shift) & 255ull)], 1);
                    }
                    __syncthreads();
                    if (tid == 0) {
                        int cum = 0;
                        for (int bin = 255; bin >= 0; --bin) {
                            const int hc = s_hist[bin];
                            if (cum + hc >= krem) { s_thr = prefix | ((unsigned long long)bin << shift); s_cb = krem - cum; break; }
                            cum += hc;
                        }
                    }
                    __syncthreads();
                    prefix = s_thr; krem = s_cb;
                    __syncthreads();
                }
                if (tid == 0) {
                    iw[SF_I_THR_LO] = (int)(uint32_t)(prefix & 0xffffffffull);
                    iw[SF_I_THR_HI] = (int)(uint32_t)(prefix >> 32);
                    __threadfence();
                    atomicExch(iw + SF_I_THR_READY, 1);
                }
            }
            if (tid == 0) {
                unsigned it = 0;
                while (ld_acquire_gpu_i32(iw + SF_I_THR_READY) == 0) {
                    if (++it > 8000000u) { atomicOr(iw + SF_I_ERR, 2); break; }
                }
                s_thr = ((unsigned long long)(uint32_t)__ldcg(iw + SF_I_THR_HI) << 32) |
                        (unsigned long long)(uint32_t)__ldcg(iw + SF_I_THR_LO);
            }
            __syncthreads();
            thr_comp = s_thr;
        }
        // selected items of lower blocks: their definite counts + members at or above the threshold that lie below
        // this block's first candidate.  In the crowded case "definite" is not enough (selected members are not in the
        // list): lower blocks' totals are then counted from the keys directly.
        int carry = 0;
        if (!crowded) {
            int part = 0;
            for (int q = tid; q < b; q += SF_THREADS) part += __ldcg(iw + SF_I_DEF + q);
            const unsigned long long first = (unsigned long long)(uint32_t)s_first;
            for (int t = tid; t < M; t += SF_THREADS) {
                const unsigned long long m = s_member[t];
                const unsigned long long idx = 0xffffffffull - (m & 0xffffffffull);
                part += (m >= thr_comp && idx < first);
            }
            long long tot;
            block_scan_excl<long long>((long long)part, s_scan, &tot);
            carry = (int)tot;
        } else {
            int part = 0;
            const int first = min(s_first, c);
            for (int i = tid; i < first; i += SF_THREADS) part += (composite(__ldcg(&ukeys[i]), i) >= thr_comp);
            long long tot;
            block_scan_excl<long long>((long long)part, s_scan, &tot);
            carry = (int)tot;
        }
        for (int base = r0; base < r1; base += SF_THREADS) {
            const int j = base + tid;
            const int rd = (base - r0) / SF_THREADS;
            int i = -1;
            if (j < r1) i = rd == 0 ? ci0 : rd == 1 ? ci1 : (nb_index ? nb_index[j] : j);
            bool sel = false;
            if (i >= 0) sel = composite(rd == 0 ? cu0 : rd == 1 ? cu1 : ukeys[i], i) >= thr_comp;
            const uint32_t bal = __ballot_sync(GRAPES_FULL_MASK, sel);
            if (lane == 0) s_wcnt[warp] = __popc(bal);
            __syncthreads();
            int before = 0, round_total = 0;
#pragma unroll
            for (int w = 0; w < SF_WARPS; ++w) { const int v = s_wcnt[w]; if (w < warp) before += v; round_total += v; }
            if (sel) {
                const int pos = carry + before + __popc(bal & ((1u << lane) - 1u));
                const int g = nb_nodes ? nb_nodes[i] : i;
                if (sampled_out) sampled_out[sampled_offset + pos] = g;
                if (bm_mark && nb_nodes) bitmap_set(bm_mark, g);
                const float l = rd == 0 ? cl0 : rd == 1 ? cl1 : lg_c[i];
                const float lp1 = bern_log_prob(l, 1.f), lp0 = bern_log_prob(l, 0.f);
                if (log_prob) log_prob[i] = lp1;
                if (dl_all) dl_all[j] = 1.f - sigmoidf_(l);      // j == nb_local[i]
                if (mask_out) mask_out[i] = 1;
                lp_delta += lp1 - lp0;
                dl_delta += 1.f;
            }
            carry += round_total;
            __syncthreads();
        }
        lp_delta = block_reduce<float, OpAdd, SF_WARPS>(lp_delta, s_red, OpAdd(), 0.f);
        dl_delta = block_reduce<float, OpAdd, SF_WARPS>(dl_delta, s_red, OpAdd(), 0.f);
        if (tid == 0) { delta_part[b * SF_DELTA_FLOATS] = lp_delta; delta_part[b * SF_DELTA_FLOATS + 1] = dl_delta; }
    }
    (void)alive;
    sf_stamp(iw, 6);
    // ---------------- ticket: the last block combines the partials in block order and cleans the scratch ----------------
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        s_last = (atomicAdd(iw + SF_I_TICKET, 1) == nb - 1) ? 1 : 0;
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    for (int q = tid; q < SEL_BUCKETS; q += SF_THREADS) hist_g[q] = 0;
    // every block's partials in ONE round of parallel loads (s_hist is free now: 8 floats per block), then a fixed-order
    // combine by warp 0
    float* s_part = reinterpret_cast<float*>(s_hist);
    for (int q = tid; q < nb * SEL_STAT_FLOATS; q += SF_THREADS) {
        float v = __ldcg(stat_part + q);
        const int bq = q / SEL_STAT_FLOATS, f = q % SEL_STAT_FLOATS;
        if (f == 6) v = __ldcg(delta_part + bq * SF_DELTA_FLOATS);
        if (f == 7) v = __ldcg(delta_part + bq * SF_DELTA_FLOATS + 1);
        s_part[q] = v;
    }
    __syncthreads();
    if (tid < 32) {
        float mn = INFINITY, mx = -INFINITY;
        double es = 0.0, eq = 0.0, lp = 0.0, dl = 0.0;
        for (int bq = tid; bq < nb; bq += 32) {
            const float* p = s_part + bq * SEL_STAT_FLOATS;
            mn = fminf(mn, p[0]); mx = fmaxf(mx, p[1]);
            es += (double)p[2]; eq += (double)p[3];
            lp += (double)p[4] + (double)p[6];
            dl += (double)p[5] + (double)p[7];
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            mn = fminf(mn, __shfl_xor_sync(GRAPES_FULL_MASK, mn, o));
            mx = fmaxf(mx, __shfl_xor_sync(GRAPES_FULL_MASK, mx, o));
            es += __shfl_xor_sync(GRAPES_FULL_MASK, es, o);
            eq += __shfl_xor_sync(GRAPES_FULL_MASK, eq, o);
            lp += __shfl_xor_sync(GRAPES_FULL_MASK, lp, o);
            dl += __shfl_xor_sync(GRAPES_FULL_MASK, dl, o);
        }
        if (tid == 0) {
            const int s = take_all ? c : k;
            if (s_dev) *s_dev = s;
            if (total_dev) *total_dev = sampled_offset + s;
            if (tot_log_prob) *tot_log_prob += (float)lp;
            if (sum_dl) *sum_dl += (float)dl;
            if (stats) {
                if (take_all) { stats[0] = stats[1] = stats[2] = stats[3] = 0.f; }   // reference returns {}
                else {
                    const double mean = (c > 0) ? es / (double)c : 0.0;
                    const double var = (c > 1) ? fmax(0.0, (eq - (double)c * mean * mean) / (double)(c - 1)) : 0.0;
                    stats[0] = mn; stats[1] = mx; stats[2] = (float)mean; stats[3] = (float)sqrt(var);   // unbiased (utils.py:56)
                }
            }
            if (mode == GRAPES_NOISE_PHILOX && !take_all) rng_state[1] += 1ull;
            iw[SF_I_BAR1] = 0; iw[SF_I_BAR2] = 0; iw[SF_I_TICKET] = 0; iw[SF_I_MCOUNT] = 0; iw[SF_I_THR_READY] = 0;
            unsigned long long tend;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tend));
            reinterpret_cast<unsigned long long*>(iw + SF_I_STAMP)[7] = tend;
        }
    }
}

// floats of scratch grapes_select_* needs in `work` (zeroed ONCE by the caller; every launch leaves the integer part clean):
// per-block statistics | per-block deltas | candidate logits | integer words (barrier counters, global histogram,
// per-block counts, member list)
#define SEL_LG_OFFSET ((int64_t)(SEL_STAT_FLOATS + SF_DELTA_FLOATS) * SF_MAX_BLOCKS)
static inline int64_t sel_int_offset(int cap_c) { return (SEL_LG_OFFSET + (int64_t)cap_c + 16 + 3) / 4 * 4; }

extern "C" {

int64_t grapes_select_work_floats(grapes_ctx* ctx, int cap_c) {
    if (!ctx) return 0;
    return sel_int_offset(cap_c) + SF_I_TOTAL + 16;
}

// debugging aid: phase time stamps (ns) of the last fused selection launch that used `work` (synchronises)
int grapes_debug_select_fused_stamps(grapes_ctx* ctx, const float* work, int cap_c, int64_t* out8) {
    if (!ctx || !work || !out8) return GRAPES_ERR_ARG;
    const int* iw = reinterpret_cast<const int*>(work + sel_int_offset(cap_c));
    if (cudaMemcpy(out8, iw + SF_I_STAMP, 8 * sizeof(int64_t), cudaMemcpyDeviceToHost) != cudaSuccess) return GRAPES_ERR_CUDA;
    return GRAPES_OK;
}

// Sampler-net layer 2 + keys for one hop (main.py:210-213 + utils.py:37-42), then the selection (utils.py:43-71).
//   z / nparts / part_stride, in_off / in_src / dinv / bias: as grapes_aggregate_scalar; in_off == NULL means
//   `z` already holds the per-row logits.  nb_index[j] = candidate index of frontier row j or -1 (NULL: every row is
//   candidate j).  work: grapes_select_work_floats(cap_n) floats, 16-byte aligned.
int grapes_select_hop(grapes_ctx* ctx, const float* z, int nparts, int part_stride, const int* n_dev, int cap_n,
                      const int* in_off, const int* in_src, const float* dinv, const float* bias,
                      const int* nb_index, const int* nb_local, const int* nb_nodes, const int* c_dev, int k,
                      int noise_mode, const float* noise, unsigned long long* rng_state, float* work,
                      uint32_t* ukeys_scratch, float* logits_all, float* keys_out, int* sampled_out,
                      int sampled_offset, int* s_dev, int* total_dev, uint8_t* mask_out, float* log_prob,
                      float* tot_log_prob, float* stats, float* dl_all, float* sum_dl, uint32_t* bm_mark,
                      void* stream) {
    GRAPES_REQUIRE(ctx && z && n_dev && c_dev && work && ukeys_scratch, "null argument");
    GRAPES_REQUIRE(!in_off || (in_src && dinv), "aggregated mode needs in_src and dinv");
    GRAPES_REQUIRE(nparts >= 1, "nparts >= 1");
    GRAPES_REQUIRE(k > 0, "num_samples must be positive (utils.py:35)");
    GRAPES_REQUIRE(noise_mode >= 0 && noise_mode <= GRAPES_NOISE_NONE_TOPK_PROBS, "bad noise mode");
    GRAPES_REQUIRE(!(noise_mode == GRAPES_NOISE_GUMBEL || noise_mode == GRAPES_NOISE_UNIFORM ||
                     noise_mode == GRAPES_NOISE_KEYS) || noise, "noise array required");
    GRAPES_REQUIRE(noise_mode != GRAPES_NOISE_PHILOX || rng_state, "rng_state required");
    GRAPES_REQUIRE((((size_t)work) & 15) == 0, "work must be 16-byte aligned");
    GRAPES_REQUIRE(!(nb_index && dl_all) || nb_local, "a frontier (nb_index) needs nb_local for the gradient scatter");
    // one block per SM at most: every block must become resident for the two grid barriers
    const int nb = grapes_min_i(grapes_min_i(ctx->sm_count, SF_MAX_BLOCKS), grapes_max_i(1, grapes_div_up(cap_n, SF_THREADS)));
    float* stat_part = work;
    float* delta_part = work + (int64_t)SEL_STAT_FLOATS * SF_MAX_BLOCKS;
    float* lg_c = work + SEL_LG_OFFSET;
    int* iw = reinterpret_cast<int*>(work + sel_int_offset(cap_n));
    pdl((k_select_fused), nb, SF_THREADS, 0, (cudaStream_t)stream)(
        z, nparts, part_stride, n_dev, cap_n, in_off, in_src, dinv, bias, nb_index, nb_local, nb_nodes, c_dev, k,
        noise_mode, noise, rng_state, logits_all, lg_c, ukeys_scratch, keys_out, sampled_out, sampled_offset, s_dev,
        total_dev, mask_out, log_prob, tot_log_prob, stats, dl_all, sum_dl, bm_mark, stat_part, delta_part, iw);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

// sample_neighborhoods_from_probs on given logits (utils.py:13-71): logits_all[i] is candidate i's logit.
// Thin form of grapes_select_hop for callers that already hold the logits.
int grapes_select_topk(grapes_ctx* ctx, const float* logits_all, const int* nb_local, const int* nb_nodes,
                       const int* c_dev, int cap_c, int k, int noise_mode, const float* noise,
                       unsigned long long* rng_state, uint32_t* ukeys_scratch, float* work, float* keys_out,
                       int* sampled_out, int sampled_offset, int* s_dev, int* total_dev, uint8_t* mask_out,
                       float* log_prob, float* tot_log_prob, float* stats, float* dl_all, float* sum_dl,
                       uint32_t* bm_mark, void* stream) {
    GRAPES_REQUIRE(nb_local == nullptr, "grapes_select_topk takes per-candidate logits; use grapes_select_hop for a frontier");
    return grapes_select_hop(ctx, logits_all, 1, 0, c_dev, cap_c, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                             nb_nodes, c_dev, k, noise_mode, noise, rng_state, work, ukeys_scratch, nullptr, keys_out,
                             sampled_out, sampled_offset, s_dev, total_dev, mask_out, log_prob, tot_log_prob, stats,
                             dl_all, sum_dl, bm_mark, stream);
}

}  // extern "C"
