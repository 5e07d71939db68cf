// Frontier expansion, bitmap dedup, rank relabel, induced-block extraction and the
// dst-sorted (deterministic) CSR build used by the aggregation kernels.
//
// Replaces, on the device, the scipy/torch CPU code of the reference:
//   get_neighborhoods           /root/reference/modules/utils.py:74-82
//   mask dedup + id lists       /root/reference/main.py:183-191
//   TensorMap.update / .map     /root/reference/modules/utils.py:98-120
//   slice_adjacency             /root/reference/modules/utils.py:85-95
// All outputs are bit-exact with those (ordering contracts in DESIGN.md section 3).
#define GRAPES_PDL_GROUP 1
#include "common.cuh"

// ---------------------------------------------------------------------------------------
// k_row_offsets: one block.  rows[P] -> row_off[P+1] (exclusive scan of CSR degrees), m.
// Marks bm_rows (every row) and bm_batch (rows with degree > 0: a row with no neighbours never
// shows up in `neighborhoods`, main.py:186, so it is not a batch node).
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) k_row_offsets(const int64_t* __restrict__ indptr,
                                                      const int* __restrict__ rows,
                                                      const int* __restrict__ P_dev, int cap_P,
                                                      int* __restrict__ row_off, int* __restrict__ m_out,
                                                      int cap_m, uint32_t* bm_rows, uint32_t* bm_batch,
                                                      int* overflow) {
    pdl_begin();
    __shared__ long long s_scan[34];
    int P = *P_dev;
    if (P > cap_P) { P = cap_P; if (threadIdx.x == 0) atomicOr(overflow, GRAPES_OVF_ROWS); }
    long long carry = 0;
    for (int base = 0; base < P; base += blockDim.x) {
        const int i = base + threadIdx.x;
        long long deg = 0;
        if (i < P) {
            const int r = rows[i];
            deg = indptr[r + 1] - indptr[r];
            if (bm_rows) bitmap_set(bm_rows, r);
            if (bm_batch && deg > 0) bitmap_set(bm_batch, r);
        }
        long long total;
        const long long excl = block_scan_excl<long long>(deg, s_scan, &total);
        if (i < P) row_off[i] = (int)min(carry + excl, (long long)cap_m);
        carry += total;
    }
    if (threadIdx.x == 0) {
        if (carry > cap_m) { atomicOr(overflow, GRAPES_OVF_EDGES); carry = cap_m; }
        row_off[P] = (int)carry;
        *m_out = (int)carry;
    }
}

// ---------------------------------------------------------------------------------------
// k_expand: edge-balanced CSR row gather.  Slot e of the concatenated neighbour lists belongs
// to row i = upper_bound(row_off, e) - 1; adjacent threads read adjacent `indices` entries.
// Emits (e_row = position in rows, e_col = neighbour global id) and marks bm_batch.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_expand(const int64_t* __restrict__ indptr,
                                                const int* __restrict__ indices,
                                                const int* __restrict__ rows, const int* __restrict__ P_dev,
                                                int cap_P, const int* __restrict__ row_off,
                                                const int* __restrict__ m_dev,
                                                int* __restrict__ e_row, int* __restrict__ e_col,
                                                uint32_t* bm_batch) {
    pdl_begin();
    const int P = min(*P_dev, cap_P);
    const int m = *m_dev;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < m; e += gridDim.x * blockDim.x) {
        int lo = 0, hi = P;                       // largest i with row_off[i] <= e
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (__ldg(&row_off[mid]) <= e) lo = mid; else hi = mid;
        }
        const int r = rows[lo];
        const int v = indices[indptr[r] + (e - row_off[lo])];
        e_row[e] = lo;
        e_col[e] = v;
        if (bm_batch) bitmap_set(bm_batch, v);
    }
}

// ---------------------------------------------------------------------------------------
// k_expand_fused: k_row_offsets + k_expand in one launch for row lists that fit shared memory (P <= EXF_MAX_P).
// Every CTA recomputes the exclusive scan of the P CSR degrees into shared memory (P is ~1k: a few L2 hits per
// thread), CTA 0 also publishes row_off / m and marks the row bitmaps; then the CTAs split the m edge slots and
// locate each slot's row by binary search in SHARED memory.  Same outputs as the two kernels.
// ---------------------------------------------------------------------------------------
#define EXF_THREADS 512
#define EXF_MAX_P 8192
__global__ void __launch_bounds__(EXF_THREADS) k_expand_fused(
    const int64_t* __restrict__ indptr, const int* __restrict__ indices, const int* __restrict__ rows,
    const int* __restrict__ P_dev, int cap_P, int* __restrict__ row_off, int* __restrict__ m_out, int cap_m,
    int* __restrict__ e_row, int* __restrict__ e_col, uint32_t* bm_rows, uint32_t* bm_batch, int* overflow) {
    pdl_begin();
    extern __shared__ int s_off[];                       // [P + 1]
    __shared__ long long s_scan[EXF_THREADS / 32 + 2];
    __shared__ long long s_carry;
    int P = *P_dev;
    if (P > cap_P) { P = cap_P; if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(overflow, GRAPES_OVF_ROWS); }
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < P; base += EXF_THREADS) {
        const int i = base + threadIdx.x;
        long long deg = 0;
        if (i < P) {
            const int r = rows[i];
            deg = indptr[r + 1] - indptr[r];
            if (blockIdx.x == 0) {
                if (bm_rows) bitmap_set(bm_rows, r);
                if (bm_batch && deg > 0) bitmap_set(bm_batch, r);
            }
        }
        long long total;
        const long long excl = block_scan_excl<long long>(deg, s_scan, &total);
        const long long carry = s_carry;
        if (i < P) s_off[i] = (int)min(carry + excl, (long long)cap_m);
        __syncthreads();
        if (threadIdx.x == 0) s_carry = carry + total;
        __syncthreads();
    }
    long long mm = s_carry;
    if (mm > cap_m) { mm = cap_m; if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(overflow, GRAPES_OVF_EDGES); }
    const int m = (int)mm;
    if (threadIdx.x == 0) s_off[P] = m;
    __syncthreads();
    if (blockIdx.x == 0) {
        for (int i = threadIdx.x; i <= P; i += EXF_THREADS) row_off[i] = s_off[i];
        if (threadIdx.x == 0) *m_out = m;
    }
    for (int e = blockIdx.x * EXF_THREADS + threadIdx.x; e < m; e += gridDim.x * EXF_THREADS) {
        int lo = 0, hi = P;                              // largest i with s_off[i] <= e
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (s_off[mid] <= e) lo = mid; else hi = mid;
        }
        const int r = rows[lo];
        const int v = indices[indptr[r] + (e - s_off[lo])];
        e_row[e] = lo;
        e_col[e] = v;
        if (bm_batch) bitmap_set(bm_batch, v);
    }
}

// ---------------------------------------------------------------------------------------
// k_rank_scan: single-pass scan over the node bitmap.  For every word: exclusive popcount
// prefix (pref_batch; pref_nb for batch & ~prev).  Enumerates the set bits in ascending id
// order, which IS the reference's local numbering (mask -> nonzero, main.py:189-195):
//   batch_nodes[j] = v, nb_nodes[q] = v, nb_local[q] = j, nb_index[j] = q (-1 if v is not a neighbour),
//   ind_bits[j] = indicator columns of v.
// bm_ind row `hop` receives batch & ~prev (indicator[neighbor_nodes, hop] = 1, main.py:191).
// ---------------------------------------------------------------------------------------
#define RANK_THREADS 256
#define RANK_WPT 4
#define RANK_TILE (RANK_THREADS * RANK_WPT)

__global__ void __launch_bounds__(RANK_THREADS) k_rank_scan(
    const uint32_t* __restrict__ bm_batch, const uint32_t* __restrict__ bm_prev, int W,
    int* __restrict__ pref_batch, int* __restrict__ pref_nb, int* __restrict__ batch_nodes,
    int* __restrict__ nb_nodes, int* __restrict__ nb_local, int* __restrict__ nb_index,
    uint32_t* __restrict__ ind_bits, uint32_t* bm_ind, int ind_rows, int hop, int cap_n, int* __restrict__ n_out,
    int* __restrict__ c_out, int* overflow, unsigned long long* status, unsigned int* counters) {
    pdl_begin();
    __shared__ unsigned long long s_scan[RANK_THREADS / 32 + 2];
    __shared__ int s_tile;
    __shared__ unsigned long long s_excl;
    __shared__ int s_last;
    if (threadIdx.x == 0) s_tile = lb_take_ticket(counters);
    __syncthreads();
    const int tile = s_tile;
    const int w0 = tile * RANK_TILE + threadIdx.x * RANK_WPT;
    uint32_t b[RANK_WPT], p[RANK_WPT];
    unsigned long long mine = 0ull;
#pragma unroll
    for (int i = 0; i < RANK_WPT; ++i) {
        const int w = w0 + i;
        b[i] = (w < W) ? bm_batch[w] : 0u;
        p[i] = (w < W && bm_prev) ? bm_prev[w] : 0u;
        mine += ((unsigned long long)__popc(b[i]) << 31) | (unsigned long long)__popc(b[i] & ~p[i]);
    }
    // indicator rows of the words that hold batch nodes: loaded now, consumed after the scan (latency hidden)
    uint32_t iw[RANK_WPT][8];
    if (ind_bits) {
#pragma unroll
        for (int i = 0; i < RANK_WPT; ++i) {
            const int w = w0 + i;
#pragma unroll
            for (int h = 0; h < 8; ++h) {
                iw[i][h] = 0u;
                if (b[i] && ((h < ind_rows - 1 && h < hop) || h == ind_rows - 1)) iw[i][h] = bm_ind[(size_t)h * W + w];
            }
        }
    }
    unsigned long long total;
    const unsigned long long excl_in_tile = block_scan_excl<unsigned long long>(mine, s_scan, &total);
    const bool nonempty = tile * RANK_TILE < W;
    if (threadIdx.x < 32) {
        unsigned long long ex = 0ull;
        if (nonempty) ex = lb_exclusive(status, tile, total);
        if (threadIdx.x == 0) { s_excl = ex; s_last = lb_finish(counters) ? 1 : 0; }
    }
    __syncthreads();
    if (nonempty) {
        const unsigned long long pre = s_excl + excl_in_tile;
        int rb = (int)(pre >> 31), rn = (int)(pre & 0x7fffffffull);
#pragma unroll
        for (int i = 0; i < RANK_WPT; ++i) {
            const int w = w0 + i;
            if (w >= W) break;
            pref_batch[w] = rb;
            if (pref_nb) pref_nb[w] = rn;
            uint32_t bits = b[i];
            const uint32_t nbits = bits & ~p[i];
            if (bm_ind) bm_ind[(size_t)hop * W + w] = nbits;
            uint32_t ind_w[8];
            if (ind_bits && bits) {
#pragma unroll
                for (int h = 0; h < 8; ++h) {
                    ind_w[h] = iw[i][h];
                    if (h == hop && h < ind_rows - 1) ind_w[h] = nbits;
                }
            }
            while (bits) {
                const int t = __ffs(bits) - 1;
                bits &= bits - 1u;
                const int v = (w << 5) + t;
                const int j = rb++;
                if (j < cap_n) {
                    batch_nodes[j] = v;
                    if (ind_bits) {
                        uint32_t ib = 0u;
#pragma unroll
                        for (int h = 0; h < 8; ++h) ib |= ((ind_w[h] >> t) & 1u) << h;
                        ind_bits[j] = ib;
                    }
                }
                if ((nbits >> t) & 1u) {
                    const int q = rn++;
                    if (q < cap_n && nb_nodes) { nb_nodes[q] = v; nb_local[q] = min(j, cap_n - 1); }   // (clamped only when GRAPES_OVF_NODES is raised)
                    if (nb_index && j < cap_n) nb_index[j] = q < cap_n ? q : -1;
                } else if (nb_index && j < cap_n) nb_index[j] = -1;
            }
        }
        if ((W - 1) / RANK_TILE == tile && threadIdx.x == RANK_THREADS - 1) {
            // last thread of the last non-empty tile holds the grand totals
            const unsigned long long tot = s_excl + total;
            int n = (int)(tot >> 31), c = (int)(tot & 0x7fffffffull);
            if (n > cap_n) { atomicOr(overflow, GRAPES_OVF_NODES); n = cap_n; if (c > cap_n) c = cap_n; }
            *n_out = n;
            if (c_out) *c_out = c;
        }
    }
    if (s_last) lb_cleanup(status, counters);
}

// ---------------------------------------------------------------------------------------
// k_edge_local: global (row position, neighbour id) -> local (src, dst) ids = TensorMap.map of
// `neighborhoods` (main.py:195).
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_edge_local(const int* __restrict__ rows,
                                                    const int* __restrict__ e_row,
                                                    const int* __restrict__ e_col,
                                                    const int* __restrict__ m_dev,
                                                    const uint32_t* __restrict__ bm,
                                                    const int* __restrict__ pref, int cap_n,
                                                    int* __restrict__ e_src, int* __restrict__ e_dst, int* cnt_hist) {
    pdl_begin();
    const int m = *m_dev;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < m; e += gridDim.x * blockDim.x) {
        int s = bitmap_rank(bm, pref, rows[e_row[e]]);
        int d = bitmap_rank(bm, pref, e_col[e]);
        // frontier larger than the caller's node capacity (GRAPES_OVF_NODES is already raised by the rank pass): an edge
        // that touches a node past the capacity becomes a dropped self-edge, so every later index stays inside cap_n
        if (s >= cap_n || d >= cap_n) s = d = 0;
        e_src[e] = s;
        e_dst[e] = d;
        if (cnt_hist && s != d) atomicAdd(&cnt_hist[d], 1);       // in-degree histogram of the CSR build, fused
    }
}

// k_relabel: out[i] = rank(ids[i])  (TensorMap.map on an arbitrary id list, main.py:213,253-254,259)
__global__ void __launch_bounds__(256) k_relabel(const int* __restrict__ ids, const int* __restrict__ cnt_dev,
                                                 int cap, const uint32_t* __restrict__ bm,
                                                 const int* __restrict__ pref, int* __restrict__ out) {
    pdl_begin();
    const int n = min(*cnt_dev, cap);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        out[i] = bitmap_rank(bm, pref, ids[i]);
}

// ---------------------------------------------------------------------------------------
// CSR build from a (key, val) edge list with self-loop edges (key == val) dropped -- what
// add_remaining_self_loops does before it appends its own loops (SURVEY.md section 3.2 step 1).
//   k_hist: cnt[key]++           k_scan_i32: off = exclusive scan(cnt) (+ dinv = (cnt+1)^-1/2)
//   k_fill: slot claim            k_sort_rows / k_sort_hub: ascending val inside each row, so
// the summation order of every aggregation is fixed (run-to-run deterministic, no fp atomics).
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_hist(const int* __restrict__ key, const int* __restrict__ val,
                                              const int* __restrict__ E_dev, int cap_E, int* cnt) {
    pdl_begin();
    const int E = min(*E_dev, cap_E);
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < E; e += gridDim.x * blockDim.x) {
        const int k = key[e];
        if (k != val[e]) atomicAdd(&cnt[k], 1);
    }
}

#define SCAN_THREADS 256
#define SCAN_IPT 4
#define SCAN_TILE (SCAN_THREADS * SCAN_IPT)

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_i32(const int* __restrict__ in,
                                                           const int* __restrict__ n_dev, int cap_n,
                                                           int* __restrict__ out, float* __restrict__ dinv,
                                                           int* __restrict__ total_out,
                                                           unsigned long long* status, unsigned int* counters) {
    pdl_begin();
    __shared__ unsigned long long s_scan[SCAN_THREADS / 32 + 2];
    __shared__ int s_tile;
    __shared__ unsigned long long s_excl;
    __shared__ int s_last;
    if (threadIdx.x == 0) s_tile = lb_take_ticket(counters);
    __syncthreads();
    const int tile = s_tile;
    const int n = min(*n_dev, cap_n);
    const int i0 = tile * SCAN_TILE + threadIdx.x * SCAN_IPT;
    int v[SCAN_IPT];
    unsigned long long mine = 0ull;
#pragma unroll
    for (int i = 0; i < SCAN_IPT; ++i) {
        v[i] = (i0 + i < n) ? in[i0 + i] : 0;
        mine += (unsigned long long)v[i];
    }
    unsigned long long total;
    const unsigned long long excl_in_tile = block_scan_excl<unsigned long long>(mine, s_scan, &total);
    const bool nonempty = (tile * SCAN_TILE < n) || (tile == 0);
    if (threadIdx.x < 32) {
        unsigned long long ex = 0ull;
        if (nonempty) ex = lb_exclusive(status, tile, total);
        if (threadIdx.x == 0) { s_excl = ex; s_last = lb_finish(counters) ? 1 : 0; }
    }
    __syncthreads();
    if (nonempty) {
        int run = (int)(s_excl + excl_in_tile);
#pragma unroll
        for (int i = 0; i < SCAN_IPT; ++i) {
            const int idx = i0 + i;
            if (idx < n) {
                out[idx] = run;
                if (dinv) dinv[idx] = 1.0f / sqrtf((float)(v[i] + 1));
                run += v[i];
            }
        }
        const int last_tile = (n == 0) ? 0 : (n - 1) / SCAN_TILE;
        if (tile == last_tile && threadIdx.x == SCAN_THREADS - 1) {
            const int tot = (int)(s_excl + total);
            out[n] = tot;
            if (total_out) *total_out = tot;
        }
    }
    if (s_last) lb_cleanup(status, counters);
}

// claim slots from the back of each row; leaves cnt[] all-zero again
__global__ void __launch_bounds__(256) k_fill(const int* __restrict__ key, const int* __restrict__ val,
                                              const int* __restrict__ E_dev, int cap_E,
                                              const int* __restrict__ off, int* cnt, int* __restrict__ out_val) {
    pdl_begin();
    const int E = min(*E_dev, cap_E);
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < E; e += gridDim.x * blockDim.x) {
        const int k = key[e], v = val[e];
        if (k != v) {
            const int pos = off[k] + atomicSub(&cnt[k], 1) - 1;
            out_val[pos] = v;
        }
    }
}

// One warp per row: rows of <= 32 values are rank-sorted in registers (shuffles), longer rows by a rank sort
// through `tmp` (O(len^2 / 32) per warp; in-degrees are bounded by the number of expanded rows).
__global__ void __launch_bounds__(256) k_sort_rows(const int* __restrict__ off, const int* __restrict__ n_dev,
                                                   int cap_n, int* vals, int* tmp) {
    pdl_begin();
    const int n = min(*n_dev, cap_n);
    const int lane = lane_id();
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int j0 = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * 32; j0 < n; j0 += warps * 32) {
        // each lane inspects one row of a 32-row group; rows needing work are then handled by the whole warp
        const int jr = j0 + lane;
        const int len_l = (jr < n) ? off[jr + 1] - off[jr] : 0;
        unsigned todo = __ballot_sync(GRAPES_FULL_MASK, len_l >= 2);
        while (todo) {
            const int t = __ffs(todo) - 1;
            todo &= todo - 1u;
            const int j = j0 + t;
            const int beg = off[j], len = off[j + 1] - beg;
            if (len <= 32) {
                const int x = (lane < len) ? vals[beg + lane] : 0x7fffffff;
                int r = 0;
                for (int u = 0; u < len; ++u) {
                    const int y = __shfl_sync(GRAPES_FULL_MASK, x, u);
                    r += (y < x) || (y == x && u < lane);
                }
                __syncwarp();
                if (lane < len) vals[beg + r] = x;
            } else {
                for (int i = lane; i < len; i += 32) {
                    const int x = vals[beg + i];
                    int r = 0;
                    for (int u = 0; u < len; ++u) { const int y = vals[beg + u]; r += (y < x) || (y == x && u < i); }
                    tmp[beg + r] = x;
                }
                __syncwarp();
                for (int i = lane; i < len; i += 32) vals[beg + i] = tmp[beg + i];
            }
            __syncwarp();
        }
    }
}

// ---------------------------------------------------------------------------------------
// k_build_csr_small: the whole build (hist -> scan -> fill -> per-row sort -> deg^-1/2) in ONE 1024-thread CTA for
// graphs with at most SMALL_N nodes (the classifier's sampled blocks: <= B + hops*k nodes, main.py:252-257).
// ---------------------------------------------------------------------------------------
#define SMALL_N 4096
struct CsrSmallSmem {
    int cnt[SMALL_N];
    int off[SMALL_N + 1];
    int scan[34];
    int hub[64];
    int nhub;
};

// whole-CTA (1024 threads) CSR build of <= SMALL_N rows; key/val may have been written earlier by this CTA (no
// read-only-cache loads).  Ends with all threads past the last shared-memory use except `sm` contents.
__device__ void csr_small_build(const int* key, const int* val, int E, int n, int* off, int* out_val, int* tmp,
                                float* dinv, int* nnz_out, CsrSmallSmem& sm) {
    const int tid = threadIdx.x;
    for (int i = tid; i < n; i += 1024) sm.cnt[i] = 0;
    if (tid == 0) sm.nhub = 0;
    __syncthreads();
    for (int e = tid; e < E; e += 1024) {
        const int k = key[e];
        if (k != val[e]) atomicAdd(&sm.cnt[k], 1);
    }
    __syncthreads();
    int carry = 0;
    for (int base = 0; base < n; base += 1024) {
        const int i = base + tid;
        const int c = (i < n) ? sm.cnt[i] : 0;
        int total;
        const int ex = block_scan_excl<int>(c, sm.scan, &total);
        if (i < n) {
            sm.off[i] = carry + ex;
            off[i] = carry + ex;
            if (dinv) dinv[i] = 1.0f / sqrtf((float)(c + 1));
        }
        carry += total;
    }
    if (tid == 0) { sm.off[n] = carry; off[n] = carry; if (nnz_out) *nnz_out = carry; }
    __syncthreads();
    for (int e = tid; e < E; e += 1024) {
        const int k = key[e], v = val[e];
        if (k != v) out_val[sm.off[k] + atomicSub(&sm.cnt[k], 1) - 1] = v;
    }
    __syncthreads();
    for (int j = tid; j < n; j += 1024) {
        const int beg = sm.off[j], len = sm.off[j + 1] - beg;
        if (len < 2) continue;
        if (len > 64) {
            const int slot = atomicAdd(&sm.nhub, 1);
            if (slot < 64) { sm.hub[slot] = j; continue; }        // > 64 hub rows: fall through to the slow exact path
        }
        int* a = out_val + beg;
        for (int i = 1; i < len; ++i) {
            const int x = a[i];
            int k = i - 1;
            while (k >= 0 && a[k] > x) { a[k + 1] = a[k]; --k; }
            a[k + 1] = x;
        }
    }
    __syncthreads();
    const int nh = min(sm.nhub, 64);
    for (int h = 0; h < nh; ++h) {                                // whole-block rank sort of each hub row
        const int j = sm.hub[h];
        const int beg = sm.off[j], len = sm.off[j + 1] - beg;
        const int* a = out_val + beg;
        for (int i = tid; i < len; i += 1024) {
            const int x = a[i];
            int r = 0;
            for (int t = 0; t < len; ++t) { const int y = a[t]; r += (y < x) || (y == x && t < i); }
            tmp[beg + r] = x;
        }
        __syncthreads();
        for (int i = tid; i < len; i += 1024) out_val[beg + i] = tmp[beg + i];
        __syncthreads();
    }
}

__global__ void __launch_bounds__(1024) k_build_csr_small(const int* key, const int* val, const int* __restrict__ E_dev,
                                                          int cap_E, const int* __restrict__ n_dev, int cap_n, int* off,
                                                          int* out_val, int* tmp, float* dinv, int* nnz_out) {
    pdl_begin();
    __shared__ CsrSmallSmem sm;
    const int E = min(*E_dev, cap_E);
    const int n = min(min(*n_dev, cap_n), SMALL_N);
    csr_small_build(key, val, E, n, off, out_val, tmp, dinv, nnz_out, sm);
}

// ---------------------------------------------------------------------------------------
// k_cls_prep: everything between "all_nodes is ranked" and "the classifier can run" in ONE CTA (main.py:252-257):
// local ids of the targets (main.py:259), relabel of the two induced blocks GCN.forward consumes (layer 1 <-
// edge_indices[-1], layer 2 <- edge_indices[0]; gcn.py:30-36), their dst-sorted CSRs + deg^-1/2 (gcn_norm) and the
// src-sorted CSR of the layer-2 block for the backward.  The sampled subgraph has <= SMALL_N nodes.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) k_cls_prep(
    const uint32_t* __restrict__ bm, const int* __restrict__ pref, const int* __restrict__ A_dev, int cap_A,
    const int* __restrict__ targets, const int* __restrict__ B_dev, int cap_B, int* target_local,
    const int* __restrict__ blk0_src, const int* __restrict__ blk0_dst, const int* __restrict__ E0_dev,
    const int* __restrict__ blk1_src, const int* __restrict__ blk1_dst, const int* __restrict__ E1_dev, int cap_blk,
    int* cl_src0, int* cl_dst0, int* cl_src1, int* cl_dst1, int* in_off0, int* in_src0, float* dinv0, int* in_off1,
    int* in_src1, float* dinv1, int* out_off1, int* out_dst1, int* tmp, int* nnz_out3, int* tgt_of_row) {
    pdl_begin();
    __shared__ CsrSmallSmem sm;
    const int tid = threadIdx.x;
    const int A = min(min(*A_dev, cap_A), SMALL_N);
    const int B = min(*B_dev, cap_B);
    const int E0 = min(*E0_dev, cap_blk), E1 = min(*E1_dev, cap_blk);
    if (tgt_of_row) {
        for (int i = tid; i < A; i += 1024) tgt_of_row[i] = -1;
        __syncthreads();
    }
    for (int i = tid; i < B; i += 1024) {
        const int loc = bitmap_rank(bm, pref, targets[i]);
        target_local[i] = loc;
        if (tgt_of_row) tgt_of_row[loc] = i;
    }
    for (int e = tid; e < E0; e += 1024) {
        cl_src0[e] = bitmap_rank(bm, pref, blk0_src[e]);
        cl_dst0[e] = bitmap_rank(bm, pref, blk0_dst[e]);
    }
    for (int e = tid; e < E1; e += 1024) {
        cl_src1[e] = bitmap_rank(bm, pref, blk1_src[e]);
        cl_dst1[e] = bitmap_rank(bm, pref, blk1_dst[e]);
    }
    __syncthreads();                                              // this CTA's global writes are visible to itself
    csr_small_build(cl_dst0, cl_src0, E0, A, in_off0, in_src0, tmp, dinv0, nnz_out3 + 0, sm);
    __syncthreads();
    csr_small_build(cl_dst1, cl_src1, E1, A, in_off1, in_src1, tmp, dinv1, nnz_out3 + 1, sm);
    __syncthreads();
    csr_small_build(cl_src1, cl_dst1, E1, A, out_off1, out_dst1, tmp, nullptr, nnz_out3 + 2, sm);
}

// ---------------------------------------------------------------------------------------
// k_filter_compact: ordered stream compaction of the expanded edge list by membership of the
// neighbour in a column bitmap == slice_adjacency(adjacency, rows, cols) (utils.py:85-95):
// row-major by position in rows, ascending neighbour id inside a row, GLOBAL ids out.
// ---------------------------------------------------------------------------------------
#define FC_THREADS 256
#define FC_IPT 4
#define FC_TILE (FC_THREADS * FC_IPT)

__global__ void __launch_bounds__(FC_THREADS) k_filter_compact(
    const int* __restrict__ rows, const int* __restrict__ e_row, const int* __restrict__ e_col,
    const int* __restrict__ m_dev, int cap_m, const uint32_t* __restrict__ bm_cols,
    int* __restrict__ out_src, int* __restrict__ out_dst, int cap_out, int* __restrict__ count_out,
    int* overflow, unsigned long long* status, unsigned int* counters) {
    pdl_begin();
    __shared__ unsigned long long s_scan[FC_THREADS / 32 + 2];
    __shared__ int s_tile;
    __shared__ unsigned long long s_excl;
    __shared__ int s_last;
    if (threadIdx.x == 0) s_tile = lb_take_ticket(counters);
    __syncthreads();
    const int tile = s_tile;
    const int m = min(*m_dev, cap_m);
    const int i0 = tile * FC_TILE + threadIdx.x * FC_IPT;
    int col[FC_IPT];
    bool keep[FC_IPT];
    unsigned long long mine = 0ull;
#pragma unroll
    for (int i = 0; i < FC_IPT; ++i) {
        const int e = i0 + i;
        keep[i] = false;
        col[i] = 0;
        if (e < m) { col[i] = e_col[e]; keep[i] = bitmap_test(bm_cols, col[i]); }
        mine += keep[i] ? 1ull : 0ull;
    }
    unsigned long long total;
    const unsigned long long excl_in_tile = block_scan_excl<unsigned long long>(mine, s_scan, &total);
    const bool nonempty = (tile * FC_TILE < m) || (tile == 0);
    if (threadIdx.x < 32) {
        unsigned long long ex = 0ull;
        if (nonempty) ex = lb_exclusive(status, tile, total);
        if (threadIdx.x == 0) { s_excl = ex; s_last = lb_finish(counters) ? 1 : 0; }
    }
    __syncthreads();
    if (nonempty) {
        int run = (int)(s_excl + excl_in_tile);
#pragma unroll
        for (int i = 0; i < FC_IPT; ++i) {
            if (keep[i]) {
                if (run < cap_out) { out_src[run] = rows[e_row[i0 + i]]; out_dst[run] = col[i]; }
                ++run;
            }
        }
        const int last_tile = (m == 0) ? 0 : (m - 1) / FC_TILE;
        if (tile == last_tile && threadIdx.x == FC_THREADS - 1) {
            int tot = (int)(s_excl + total);
            if (tot > cap_out) { atomicOr(overflow, GRAPES_OVF_BLOCK); tot = cap_out; }
            *count_out = tot;
        }
    }
    if (s_last) lb_cleanup(status, counters);
}

// ---------------------------------------------------------------------------------------
// small list <-> bitmap utilities
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_bitmap_set_list(const int* __restrict__ ids, const int* __restrict__ cnt_dev,
                                                         int cap, uint32_t* bm) {
    pdl_begin();
    const int n = min(*cnt_dev, cap);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) bitmap_set(bm, ids[i]);
}
__global__ void __launch_bounds__(256) k_bitmap_clear_list(const int* __restrict__ ids, const int* __restrict__ cnt_dev,
                                                           int cap, uint32_t* bm) {
    pdl_begin();
    const int n = min(*cnt_dev, cap);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) bm[ids[i] >> 5] = 0u;
}
// dst[off .. off+n) = src[0..n); *total = off + n   (next-hop assembly, main.py:236-238)
__global__ void __launch_bounds__(256) k_append_list(const int* __restrict__ src, const int* __restrict__ cnt_dev,
                                                     int cap, int* __restrict__ dst, int off, int* total) {
    pdl_begin();
    const int n = min(*cnt_dev, cap);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) dst[off + i] = src[i];
    if (blockIdx.x == 0 && threadIdx.x == 0 && total) *total = off + n;
}
// k_step_reset: per-batch reset of the id lists (main.py:161-168): copies the targets to the head of every hop's
// row list (batch_nodes = cat([targets, sampled]), main.py:236), marks them in up to two bitmaps and publishes P0.
__global__ void __launch_bounds__(256) k_step_reset(const int* __restrict__ targets, const int* __restrict__ B_dev,
                                                    int cap_B, int* __restrict__ lists, long long list_stride,
                                                    int nlists, int* __restrict__ P0_dev, uint32_t* bm_a,
                                                    uint32_t* bm_b) {
    pdl_begin();
    const int n = min(*B_dev, cap_B);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int t = targets[i];
        for (int l = 0; l < nlists; ++l) lists[(long long)l * list_stride + i] = t;
        if (bm_a) bitmap_set(bm_a, t);
        if (bm_b) bitmap_set(bm_b, t);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0 && P0_dev) *P0_dev = n;
}
__global__ void __launch_bounds__(256) k_i64_to_i32(const int64_t* __restrict__ in, int* __restrict__ out, int n,
                                                    int* count_out) {
    pdl_begin();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = (int)in[i];
    if (count_out && blockIdx.x == 0 && threadIdx.x == 0) *count_out = n;
}
__global__ void __launch_bounds__(256) k_i32_to_i64(const int* __restrict__ in, const int* __restrict__ cnt_dev,
                                                    int cap, int64_t* __restrict__ out) {
    pdl_begin();
    const int n = cnt_dev ? min(*cnt_dev, cap) : cap;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = (int64_t)in[i];
}

// =======================================================================================
// C ABI
// =======================================================================================
static inline int grid_for(const grapes_ctx* ctx, long long work, int threads, int per_sm = 8) {
    long long b = (work + threads - 1) / threads;
    long long cap = (long long)ctx->sm_count * per_sm;
    if (b < 1) b = 1;
    return (int)(b < cap ? b : cap);
}

extern "C" {

int grapes_row_offsets(grapes_ctx* ctx, const int64_t* indptr, const int* rows, const int* P_dev, int cap_P,
                       int* row_off, int* m_dev, int cap_m, uint32_t* bm_rows, uint32_t* bm_batch,
                       int* overflow, void* stream) {
    GRAPES_REQUIRE(ctx && indptr && rows && P_dev && row_off && m_dev && overflow, "null argument");
    pdl((k_row_offsets), 1, 1024, 0, (cudaStream_t)stream)(indptr, rows, P_dev, cap_P, row_off, m_dev, cap_m,
                                                          bm_rows, bm_batch, overflow);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_expand_rows(grapes_ctx* ctx, const int64_t* indptr, const int* indices, const int* rows,
                       const int* P_dev, int cap_P, const int* row_off, const int* m_dev, int cap_m,
                       int* e_row, int* e_col, uint32_t* bm_batch, void* stream) {
    GRAPES_REQUIRE(ctx && indptr && indices && rows && P_dev && row_off && m_dev && e_row && e_col, "null argument");
    pdl((k_expand), grid_for(ctx, cap_m, 256), 256, 0, (cudaStream_t)stream)(indptr, indices, rows, P_dev, cap_P,
                                                                          row_off, m_dev, e_row, e_col, bm_batch);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

/* grapes_row_offsets + grapes_expand_rows in one launch (row lists of <= 8192 rows; larger lists take the two calls) */
int grapes_expand_frontier(grapes_ctx* ctx, const int64_t* indptr, const int* indices, const int* rows,
                           const int* P_dev, int cap_P, int* row_off, int* m_dev, int cap_m, int* e_row, int* e_col,
                           uint32_t* bm_rows, uint32_t* bm_batch, int* overflow, void* stream) {
    GRAPES_REQUIRE(ctx && indptr && indices && rows && P_dev && row_off && m_dev && e_row && e_col && overflow, "null argument");
    if (cap_P > EXF_MAX_P) {
        int rc = grapes_row_offsets(ctx, indptr, rows, P_dev, cap_P, row_off, m_dev, cap_m, bm_rows, bm_batch, overflow, stream);
        if (rc != GRAPES_OK) return rc;
        return grapes_expand_rows(ctx, indptr, indices, rows, P_dev, cap_P, row_off, m_dev, cap_m, e_row, e_col, bm_batch, stream);
    }
    const int smem = (cap_P + 1) * (int)sizeof(int);
    int blocks = grapes_div_up(cap_m, EXF_THREADS * 2);
    if (blocks > ctx->sm_count * 2) blocks = ctx->sm_count * 2;
    if (blocks < 1) blocks = 1;
    pdl((k_expand_fused), blocks, EXF_THREADS, smem, (cudaStream_t)stream)(indptr, indices, rows, P_dev, cap_P, row_off, m_dev,
                                                                        cap_m, e_row, e_col, bm_rows, bm_batch, overflow);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_rank_nodes(grapes_ctx* ctx, const uint32_t* bm_batch, const uint32_t* bm_prev, int* pref_batch,
                      int* pref_nb, int* batch_nodes, int* nb_nodes, int* nb_local, int* nb_index,
                      uint32_t* ind_bits, uint32_t* bm_ind, int ind_rows, int hop, int cap_n, int* n_dev, int* c_dev,
                      int* overflow, void* stream) {
    GRAPES_REQUIRE(ctx && bm_batch && pref_batch && batch_nodes && n_dev && overflow, "null argument");
    GRAPES_REQUIRE(ind_rows >= 0 && ind_rows <= 8, "at most 8 indicator columns (sampling_hops <= 7)");
    GRAPES_REQUIRE(!ind_bits || bm_ind, "ind_bits needs bm_ind");
    GRAPES_REQUIRE(!nb_nodes || (nb_local && pref_nb && c_dev), "nb_nodes needs nb_local, pref_nb, c_dev");
    const int tiles = grapes_div_up(ctx->num_words, RANK_TILE);
    GRAPES_REQUIRE(tiles <= ctx->scan_cap_tiles, "scan scratch too small");
    pdl((k_rank_scan), tiles, RANK_THREADS, 0, (cudaStream_t)stream)(
        bm_batch, bm_prev, ctx->num_words, pref_batch, pref_nb, batch_nodes, nb_nodes, nb_local, nb_index, ind_bits,
        bm_ind, ind_rows, hop, cap_n, n_dev, c_dev, overflow, ctx->scan_status, ctx->scan_counters);
        grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_edges_to_local(grapes_ctx* ctx, const int* rows, const int* e_row, const int* e_col, const int* m_dev,
                          int cap_m, const uint32_t* bm, const int* pref, int cap_n, int* e_src, int* e_dst,
                          int* cnt_hist, void* stream) {
    GRAPES_REQUIRE(ctx && rows && e_row && e_col && m_dev && bm && pref && e_src && e_dst, "null argument");
    GRAPES_REQUIRE(cap_n > 0, "cap_n: capacity of the node-indexed buffers (cnt_hist, in_off, dinv, ...)");
    pdl((k_edge_local), grid_for(ctx, cap_m, 256), 256, 0, (cudaStream_t)stream)(rows, e_row, e_col, m_dev, bm, pref,
                                                                              cap_n, e_src, e_dst, cnt_hist);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_relabel(grapes_ctx* ctx, const int* ids, const int* count_dev, int cap, const uint32_t* bm,
                   const int* pref, int* out, void* stream) {
    GRAPES_REQUIRE(ctx && ids && count_dev && bm && pref && out, "null argument");
    pdl((k_relabel), grid_for(ctx, cap, 256), 256, 0, (cudaStream_t)stream)(ids, count_dev, cap, bm, pref, out);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_build_csr(grapes_ctx* ctx, const int* key, const int* val, const int* E_dev, int cap_E,
                     const int* n_dev, int cap_n, int* cnt_scratch, int hist_done, int* off, int* sorted_val,
                     int* tmp_val, float* dinv, int* nnz_dev, int* overflow, void* stream) {
    GRAPES_REQUIRE(ctx && key && val && E_dev && n_dev && cnt_scratch && off && sorted_val && tmp_val && overflow,
                   "null argument");
    cudaStream_t s = (cudaStream_t)stream;
    if (!hist_done && cap_n <= SMALL_N) {
        pdl((k_build_csr_small), 1, 1024, 0, s)(key, val, E_dev, cap_E, n_dev, cap_n, off, sorted_val, tmp_val, dinv,
                                             nnz_dev);
        grapes_count_launches(1);
        GRAPES_LAUNCH_OK();
        return GRAPES_OK;
    }
    const int tiles = grapes_div_up(cap_n, SCAN_TILE);
    GRAPES_REQUIRE(tiles <= ctx->scan_cap_tiles, "scan scratch too small for cap_n");
    if (!hist_done) {
        // cnt_scratch is all-zero on entry by contract (zero-initialised by the caller; k_fill returns it to zero)
        pdl((k_hist), grid_for(ctx, cap_E, 256), 256, 0, s)(key, val, E_dev, cap_E, cnt_scratch);
        grapes_count_launches(1);
    }
    pdl((k_scan_i32), grapes_max_i(tiles, 1), SCAN_THREADS, 0, s)(cnt_scratch, n_dev, cap_n, off, dinv, nnz_dev,
                                                              ctx->scan_status, ctx->scan_counters);
    grapes_count_launches(1);
    pdl((k_fill), grid_for(ctx, cap_E, 256), 256, 0, s)(key, val, E_dev, cap_E, off, cnt_scratch, sorted_val);
    grapes_count_launches(1);
    pdl((k_sort_rows), grid_for(ctx, cap_n, 256), 256, 0, s)(off, n_dev, cap_n, sorted_val, tmp_val);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_classifier_prep(grapes_ctx* ctx, const uint32_t* bm_all, const int* pref_all, const int* A_dev, int cap_A,
                           const int* targets, const int* B_dev, int cap_B, int* target_local, const int* blk0_src,
                           const int* blk0_dst, const int* E0_dev, const int* blk1_src, const int* blk1_dst,
                           const int* E1_dev, int cap_blk, int* cl_src0, int* cl_dst0, int* cl_src1, int* cl_dst1,
                           int* in_off0, int* in_src0, float* dinv0, int* in_off1, int* in_src1, float* dinv1,
                           int* out_off1, int* out_dst1, int* tmp, int* nnz_dev3, int* tgt_of_row, void* stream) {
    GRAPES_REQUIRE(ctx && bm_all && pref_all && A_dev && targets && B_dev && target_local && blk0_src && blk0_dst &&
                       E0_dev && blk1_src && blk1_dst && E1_dev && cl_src0 && cl_dst0 && cl_src1 && cl_dst1 && in_off0 &&
                       in_src0 && dinv0 && in_off1 && in_src1 && dinv1 && out_off1 && out_dst1 && tmp && nnz_dev3,
                   "null argument");
    GRAPES_REQUIRE(cap_A <= SMALL_N, "sampled subgraph too large for the single-CTA preparation");
    pdl((k_cls_prep), 1, 1024, 0, (cudaStream_t)stream)(bm_all, pref_all, A_dev, cap_A, targets, B_dev, cap_B, target_local,
                                                      blk0_src, blk0_dst, E0_dev, blk1_src, blk1_dst, E1_dev, cap_blk,
                                                      cl_src0, cl_dst0, cl_src1, cl_dst1, in_off0, in_src0, dinv0,
                                                      in_off1, in_src1, dinv1, out_off1, out_dst1, tmp, nnz_dev3,
                                                      tgt_of_row);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_slice_block(grapes_ctx* ctx, const int* rows, const int* e_row, const int* e_col, const int* m_dev,
                       int cap_m, const uint32_t* bm_cols, int* out_src, int* out_dst, int cap_out,
                       int* count_dev, int* overflow, void* stream) {
    GRAPES_REQUIRE(ctx && rows && e_row && e_col && m_dev && bm_cols && out_src && out_dst && count_dev && overflow,
                   "null argument");
    const int tiles = grapes_max_i(grapes_div_up(cap_m, FC_TILE), 1);
    GRAPES_REQUIRE(tiles <= ctx->scan_cap_tiles, "scan scratch too small for cap_m");
    pdl((k_filter_compact), tiles, FC_THREADS, 0, (cudaStream_t)stream)(rows, e_row, e_col, m_dev, cap_m, bm_cols,
                                                                     out_src, out_dst, cap_out, count_dev, overflow,
                                                                     ctx->scan_status, ctx->scan_counters);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_bitmap_set(grapes_ctx* ctx, const int* ids, const int* count_dev, int cap, uint32_t* bm, void* stream) {
    GRAPES_REQUIRE(ctx && ids && count_dev && bm, "null argument");
    pdl((k_bitmap_set_list), grid_for(ctx, cap, 256), 256, 0, (cudaStream_t)stream)(ids, count_dev, cap, bm);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_bitmap_clear_words(grapes_ctx* ctx, const int* ids, const int* count_dev, int cap, uint32_t* bm,
                              void* stream) {
    GRAPES_REQUIRE(ctx && ids && count_dev && bm, "null argument");
    pdl((k_bitmap_clear_list), grid_for(ctx, cap, 256), 256, 0, (cudaStream_t)stream)(ids, count_dev, cap, bm);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_append_list(grapes_ctx* ctx, const int* src, const int* count_dev, int cap, int* dst, int dst_offset,
                       int* total_dev, void* stream) {
    GRAPES_REQUIRE(ctx && src && count_dev && dst, "null argument");
    pdl((k_append_list), grid_for(ctx, cap, 256), 256, 0, (cudaStream_t)stream)(src, count_dev, cap, dst, dst_offset,
                                                                             total_dev);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_step_reset(grapes_ctx* ctx, const int* targets, const int* B_dev, int cap_B, int* lists,
                      int64_t list_stride, int nlists, int* P0_dev, uint32_t* bm_a, uint32_t* bm_b, void* stream) {
    GRAPES_REQUIRE(ctx && targets && B_dev && lists && nlists >= 1, "null argument");
    pdl((k_step_reset), grid_for(ctx, cap_B, 256), 256, 0, (cudaStream_t)stream)(targets, B_dev, cap_B, lists,
                                                                              (long long)list_stride, nlists, P0_dev,
                                                                              bm_a, bm_b);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_ids_i64_to_i32(grapes_ctx* ctx, const int64_t* in, int n, int* out, int* count_dev, void* stream) {
    GRAPES_REQUIRE(ctx && out && (in || n == 0), "null argument");
    pdl((k_i64_to_i32), grid_for(ctx, n, 256), 256, 0, (cudaStream_t)stream)(in, out, n, count_dev);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_ids_i32_to_i64(grapes_ctx* ctx, const int* in, const int* count_dev, int cap, int64_t* out, void* stream) {
    GRAPES_REQUIRE(ctx && out && (in || cap == 0), "null argument");
    pdl((k_i32_to_i64), grid_for(ctx, cap, 256), 256, 0, (cudaStream_t)stream)(in, count_dev, cap, out);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

}  // extern "C"
