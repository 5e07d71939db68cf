// CSR construction on the device: edge_index [2, E] -> (indptr int64, indices int32), rows sorted, duplicate edges collapsed,
// self-loops kept -- the canonical form scipy gives /root/reference/main.py:134-136
// (`sp.csr_matrix((np.ones(E, bool), edge_index), shape=(N, N))`, then row slicing in modules/utils.py:78,89-91).
//
// HBM-bound integer work, one pass per phase, no global sort: a counting sort by row (degree histogram -> 64-bit scan ->
// scatter) groups the edges, then every row segment is sorted and deduplicated where it lies -- a warp in registers for
// rows of <= 128 entries (1, 2 or 4 per lane), a warp in shared memory up to 256, a CTA in shared memory up to 32768,
// a CTA in global memory for longer hub rows (all use the same ascending-only bitonic network, so tails never need
// padding) -- and a second scan + copy
// closes the gaps the duplicates left.  The scatter order inside a row depends on atomics, the result does not.
//
// Phases (E = edges in, N = nodes):                                algorithmic bytes
//   k_csr_degree     histogram of src                              16 E read (+ 4 E atomic)
//   scan64           deg -> raw_off                                 4 N read, 8 N write
//   k_csr_partition  (row, col) pairs grouped by row bucket         16 E read, 8 E write
//   k_csr_scatter_part  tmp[raw_off[row] + cursor++] = col, bucket by bucket (L2-sized windows)   8 E read, 4 E write
//   k_csr_sort_*     sort + unique per row, in place                4 E read, <= 4 E write
//   scan64           ucount -> indptr                               4 N read, 8 N write
//   k_csr_compact    indices[indptr[r] ..] = tmp[raw_off[r] ..]     4 nnz read + write
#define GRAPES_PDL_GROUP 1
#include "common.cuh"

#define CB_THREADS 256
#define CB_SCAN_THREADS 1024
#define CB_SCAN_ITEMS 8
#define CB_SCAN_TILE (CB_SCAN_THREADS * CB_SCAN_ITEMS)
#define CB_WARP_MAX 1024             // rows of 129 .. 1024 entries: one warp, a 4 KB strip of shared memory
#define CB_MED_MAX 2048              // rows of 1025 .. 2048 entries: 256-thread CTA, 8 KB of shared memory
#define CB_LONG_SMEM 32768           // rows up to 32768 entries are sorted in shared memory (128 KB), longer ones in HBM
#define CB_MED_THREADS 256
#define CB_LONG_THREADS 1024

static inline size_t cb_align(size_t x) { return (x + 255) & ~(size_t)255; }

// ---------------------------------------------------------------------------------------------------------------------
// 64-bit exclusive scan of int32 counts: tile sums -> one CTA scans the tile sums -> tiles rescan with their offset.
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CB_SCAN_THREADS) k_scan64_tilesum(const int* __restrict__ cnt, int64_t n,
                                                                     long long* __restrict__ tile_sum) {
    __shared__ long long sm[CB_SCAN_THREADS / 32 + 2];
    const int64_t base = (int64_t)blockIdx.x * CB_SCAN_TILE + (int64_t)threadIdx.x * CB_SCAN_ITEMS;
    long long s = 0;
#pragma unroll
    for (int i = 0; i < CB_SCAN_ITEMS; ++i)
        if (base + i < n) s += cnt[base + i];
    long long total;
    block_scan_excl<long long>(s, sm, &total);
    if (threadIdx.x == 0) tile_sum[blockIdx.x] = total;
}

__global__ void __launch_bounds__(CB_SCAN_THREADS) k_scan64_tiles(long long* __restrict__ tile_sum, int tiles,
                                                                   long long* __restrict__ total_out) {
    __shared__ long long sm[CB_SCAN_THREADS / 32 + 2];
    long long run = 0;
    for (int t0 = 0; t0 < tiles; t0 += CB_SCAN_THREADS) {
        const int t = t0 + threadIdx.x;
        const long long v = t < tiles ? tile_sum[t] : 0;
        long long total;
        const long long ex = block_scan_excl<long long>(v, sm, &total);
        if (t < tiles) tile_sum[t] = run + ex;
        run += total;
    }
    if (threadIdx.x == 0 && total_out) *total_out = run;
}

__global__ void __launch_bounds__(CB_SCAN_THREADS) k_scan64_apply(const int* __restrict__ cnt, int64_t n,
                                                                   const long long* __restrict__ tile_off,
                                                                   long long* __restrict__ out /* [n + 1] */) {
    __shared__ long long sm[CB_SCAN_THREADS / 32 + 2];
    const int64_t base = (int64_t)blockIdx.x * CB_SCAN_TILE + (int64_t)threadIdx.x * CB_SCAN_ITEMS;
    int v[CB_SCAN_ITEMS];
    long long s = 0;
#pragma unroll
    for (int i = 0; i < CB_SCAN_ITEMS; ++i) {
        v[i] = (base + i < n) ? cnt[base + i] : 0;
        s += v[i];
    }
    long long total;
    long long run = block_scan_excl<long long>(s, sm, &total) + tile_off[blockIdx.x];
#pragma unroll
    for (int i = 0; i < CB_SCAN_ITEMS; ++i) {
        if (base + i < n) out[base + i] = run;
        run += v[i];
        if (base + i == n - 1) out[n] = run;
    }
}

static void cb_scan64(const int* cnt, int64_t n, long long* tile_sum, long long* out, long long* total_out,
                      cudaStream_t s) {
    const int tiles = (int)((n + CB_SCAN_TILE - 1) / CB_SCAN_TILE);
    pdl(k_scan64_tilesum, tiles, CB_SCAN_THREADS, 0, s)(cnt, n, tile_sum);
    pdl(k_scan64_tiles, 1, CB_SCAN_THREADS, 0, s)(tile_sum, tiles, total_out);
    pdl(k_scan64_apply, tiles, CB_SCAN_THREADS, 0, s)(cnt, n, tile_sum, out);
    grapes_count_launches(3);
}

// ---------------------------------------------------------------------------------------------------------------------
// counting sort by row
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CB_THREADS) k_csr_degree(const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                                            int64_t E, int64_t N, int* __restrict__ deg,
                                                            int* __restrict__ err) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += stride) {
        const int64_t r = src[e], c = dst[e];
        if (r < 0 || r >= N || c < 0 || c >= N) { *err = 1; continue; }     // scipy: "row/column index exceeds matrix dimensions"
        atomicAdd(&deg[r], 1);
    }
}

__global__ void __launch_bounds__(CB_THREADS) k_csr_scatter(const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                                             int64_t E, int64_t N, const long long* __restrict__ raw_off,
                                                             int* __restrict__ cursor, int* __restrict__ tmp) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < E; e += stride) {
        const int64_t r = src[e], c = dst[e];
        if (r < 0 || r >= N || c < 0 || c >= N) continue;
        const int k = atomicAdd(&cursor[r], 1);
        tmp[raw_off[r] + k] = (int)c;
    }
}

// The direct scatter above writes 4 bytes at a random place of a table far larger than L2: every store costs a 32-byte
// sector read + write in DRAM (ncu, products-shape: 6.8 GB read + 3.7 GB written for 2.5 GB of algorithmic traffic).
// Two passes with locality instead: (A) a tile of edges is split by row BUCKET (<= 1024 buckets of 2^shift rows) with a
// shared-memory histogram, each (tile, bucket) run is reserved with one global atomic and written as 8-byte (row, col)
// pairs next to each other -- whole sectors; (B) the CTAs walk the buckets in order, a group of CTAs per bucket, so the
// random 4-byte stores of a bucket fall into a window of a few MB that L2 holds until its sectors are complete.
#define CB_PART_THREADS 512
#define CB_PART_ITEMS 8
#define CB_PART_TILE (CB_PART_THREADS * CB_PART_ITEMS)
#define CB_PART_MAXB 1024

__global__ void __launch_bounds__(CB_PART_THREADS, 2) k_csr_partition(
    const int64_t* __restrict__ src, const int64_t* __restrict__ dst, int64_t E, int64_t N,
    const long long* __restrict__ raw_off, int shift, int B, unsigned long long* __restrict__ bucket_fill,
    unsigned long long* __restrict__ pairs) {
    __shared__ int hist[CB_PART_MAXB];
    __shared__ long long base[CB_PART_MAXB];
    const int64_t tiles = (E + CB_PART_TILE - 1) / CB_PART_TILE;
    for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
        for (int t = threadIdx.x; t < B; t += CB_PART_THREADS) hist[t] = 0;
        __syncthreads();
        int rr[CB_PART_ITEMS], cc[CB_PART_ITEMS], rk[CB_PART_ITEMS];
        int64_t r64[CB_PART_ITEMS], c64[CB_PART_ITEMS];
#pragma unroll
        for (int i = 0; i < CB_PART_ITEMS; ++i) {                   // every load of the tile in flight before the first use
            const int64_t e = tile * CB_PART_TILE + (int64_t)i * CB_PART_THREADS + threadIdx.x;
            r64[i] = e < E ? src[e] : -1;
            c64[i] = e < E ? dst[e] : -1;
        }
#pragma unroll
        for (int i = 0; i < CB_PART_ITEMS; ++i) {
            const int64_t r = r64[i], c = c64[i];
            rr[i] = -1;
            if (r >= 0 && r < N && c >= 0 && c < N) {
                rr[i] = (int)r; cc[i] = (int)c;
                rk[i] = atomicAdd(&hist[(int)(r >> shift)], 1);
            }
        }
        __syncthreads();
        for (int t = threadIdx.x; t < B; t += CB_PART_THREADS) {
            const int n = hist[t];
            if (n > 0) {
                const int64_t first = (int64_t)t << shift;
                base[t] = raw_off[first] + (long long)atomicAdd(&bucket_fill[t], (unsigned long long)n);
            }
        }
        __syncthreads();
#pragma unroll
        for (int i = 0; i < CB_PART_ITEMS; ++i)
            if (rr[i] >= 0)
                pairs[base[rr[i] >> shift] + rk[i]] = ((unsigned long long)(unsigned)rr[i] << 32) | (unsigned)cc[i];
        __syncthreads();
    }
}

__global__ void __launch_bounds__(CB_THREADS) k_csr_scatter_part(const unsigned long long* __restrict__ pairs,
                                                                  const long long* __restrict__ raw_off, int64_t N,
                                                                  int shift, int G, int* __restrict__ cursor,
                                                                  int* __restrict__ tmp) {
    const int b = blockIdx.x / G, g = blockIdx.x - b * G;
    const int64_t r0 = (int64_t)b << shift, r1 = min(N, ((int64_t)b + 1) << shift);
    const long long lo = raw_off[r0], hi = raw_off[r1];
    const long long per = (hi - lo + G - 1) / G;
    const long long s = lo + (long long)g * per, e = min(hi, s + per);
    for (long long p = s + threadIdx.x; p < e; p += CB_THREADS) {
        const unsigned long long pr = pairs[p];
        const int r = (int)(pr >> 32);
        const int k = atomicAdd(&cursor[r], 1);
        tmp[raw_off[r] + k] = (int)(unsigned)pr;
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// per-row sort + unique.  Short rows: one warp per row, the row in one register per lane.
// ---------------------------------------------------------------------------------------------------------------------
// Sort + unique of a row of d <= 32 K entries held K per lane (entry i in register i / 32 of lane i % 32): the ascending-only
// bitonic network with shuffles for strides < 32 and register-to-register exchanges above; +inf pads the tail.
template <int K>
__device__ __forceinline__ void cb_warp_bitonic(int (&v)[K], int lane) {
#pragma unroll
    for (int size = 2; size <= 32 * K; size <<= 1) {
        if (size <= 32) {                                   // flip step inside a register: partner = lane ^ (size - 1)
            const bool lower = (lane & (size - 1)) < (size >> 1);
#pragma unroll
            for (int j = 0; j < K; ++j) {
                const int p = __shfl_xor_sync(GRAPES_FULL_MASK, v[j], size - 1);
                v[j] = lower ? min(v[j], p) : max(v[j], p);
            }
        } else {                                            // flip step across registers: (a, lane) <-> (c, lane ^ 31)
            const int S = size >> 5;
#pragma unroll
            for (int b0 = 0; b0 < K; b0 += S) {
#pragma unroll
                for (int j = 0; j < S / 2; ++j) {
                    const int a = b0 + j, c = b0 + S - 1 - j;
                    const int pa = __shfl_xor_sync(GRAPES_FULL_MASK, v[c], 31);
                    const int pc = __shfl_xor_sync(GRAPES_FULL_MASK, v[a], 31);
                    v[a] = min(v[a], pa);
                    v[c] = max(v[c], pc);
                }
            }
        }
#pragma unroll
        for (int st = size >> 2; st > 0; st >>= 1) {
            if (st >= 32) {
                const int sj = st >> 5;
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    if (!(j & sj)) {
                        const int lo = min(v[j], v[j + sj]), hi = max(v[j], v[j + sj]);
                        v[j] = lo; v[j + sj] = hi;
                    }
                }
            } else {
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    const int p = __shfl_xor_sync(GRAPES_FULL_MASK, v[j], st);
                    v[j] = (lane & st) ? max(v[j], p) : min(v[j], p);
                }
            }
        }
    }
}

template <int K>
__device__ __forceinline__ int cb_warp_sort_unique(int* __restrict__ row, int d, int lane) {
    int v[K];
#pragma unroll
    for (int j = 0; j < K; ++j) v[j] = (j * 32 + lane < d) ? row[j * 32 + lane] : 0x7fffffff;
    cb_warp_bitonic<K>(v, lane);
    int base = 0;
#pragma unroll
    for (int j = 0; j < K; ++j) {
        int prev = __shfl_up_sync(GRAPES_FULL_MASK, v[j], 1);
        if (j > 0) {
            const int last = __shfl_sync(GRAPES_FULL_MASK, v[j - 1], 31);
            if (lane == 0) prev = last;
        }
        const int i = j * 32 + lane;
        const bool keep = i < d && (i == 0 || v[j] != prev);
        const unsigned m = __ballot_sync(GRAPES_FULL_MASK, keep);
        if (keep) row[base + __popc(m & ((1u << lane) - 1u))] = v[j];
        base += __popc(m);
    }
    return base;
}

// ascending-only bitonic network over a[0 .. d) in shared memory, one warp (rows of 129 .. CB_WARP_MAX entries)
__device__ __forceinline__ void cb_warp_bitonic_smem(int* a, int d, int lane) {
    int P = 64;
    while (P < d) P <<= 1;
    for (int size = 2; size <= P; size <<= 1) {
        const int half = size >> 1;
        for (int p = lane; p < (P >> 1); p += 32) {
            const int blk = p / half, off = p - blk * half;
            const int i = blk * size + off, j = blk * size + size - 1 - off;
            if (j < d) { const int x = a[i], y = a[j]; if (x > y) { a[i] = y; a[j] = x; } }
        }
        __syncwarp();
        for (int st = size >> 2; st > 0; st >>= 1) {
            for (int p = lane; p < (P >> 1); p += 32) {
                const int i = 2 * st * (p / st) + (p % st), j = i + st;
                if (j < d) { const int x = a[i], y = a[j]; if (x > y) { a[i] = y; a[j] = x; } }
            }
            __syncwarp();
        }
    }
}

__global__ void __launch_bounds__(CB_THREADS) k_csr_sort_short(int64_t N, const long long* __restrict__ raw_off,
                                                                int* __restrict__ tmp, int* __restrict__ ucount,
                                                                int* __restrict__ worklist, int* __restrict__ wl_count) {
    __shared__ int s_rows[CB_THREADS / 32][CB_WARP_MAX];
    const int lane = lane_id();
    int* a = s_rows[threadIdx.x >> 5];
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < N; r += warps) {
        const long long o = raw_off[r];
        const int d = (int)(raw_off[r + 1] - o);
        if (d > CB_WARP_MAX) {                          // medium rows are listed from the front, long rows from the back
            if (lane == 0) {
                if (d <= CB_MED_MAX) worklist[atomicAdd(&wl_count[0], 1)] = (int)r;
                else worklist[N - 1 - atomicAdd(&wl_count[1], 1)] = (int)r;
            }
            continue;
        }
        if (d == 0) { if (lane == 0) ucount[r] = 0; continue; }
        if (d > 128) {
            // 129 .. CB_WARP_MAX entries: the warp sorts the row in its own shared-memory strip (same ascending-only
            // network as cb_bitonic, __syncwarp between stages), then writes the unique values back in order
            for (int i = lane; i < d; i += 32) a[i] = tmp[o + i];
            __syncwarp();
            cb_warp_bitonic_smem(a, d, lane);
            int base = 0;
            for (int i0 = 0; i0 < d; i0 += 32) {
                const int i = i0 + lane;
                const int v = i < d ? a[i] : 0;
                const bool keep = i < d && (i == 0 || v != a[i - 1]);
                const unsigned m = __ballot_sync(GRAPES_FULL_MASK, keep);
                if (keep) tmp[o + base + __popc(m & ((1u << lane) - 1u))] = v;
                base += __popc(m);
            }
            if (lane == 0) ucount[r] = base;
            __syncwarp();
            continue;
        }
        int u;
        if (d <= 32) u = cb_warp_sort_unique<1>(tmp + o, d, lane);
        else if (d <= 64) u = cb_warp_sort_unique<2>(tmp + o, d, lane);
        else u = cb_warp_sort_unique<4>(tmp + o, d, lane);
        if (lane == 0) ucount[r] = u;
    }
}

// ascending-only bitonic network over a[0 .. n): every compare-exchange leaves the minimum at the lower index, so the
// virtual +inf padding up to the next power of two never moves and pairs whose partner is >= n are skipped.
template <typename Ptr>
__device__ __forceinline__ void cb_bitonic(Ptr a, int n) {
    int P = 1;
    while (P < n) P <<= 1;
    for (int size = 2; size <= P; size <<= 1) {
        const int half = size >> 1;
        for (int p = threadIdx.x; p < (P >> 1); p += blockDim.x) {
            const int blk = p / half, off = p - blk * half;
            const int i = blk * size + off, j = blk * size + size - 1 - off;
            if (j < n) { const int x = a[i], y = a[j]; if (x > y) { a[i] = y; a[j] = x; } }
        }
        __syncthreads();
        for (int st = size >> 2; st > 0; st >>= 1) {
            for (int p = threadIdx.x; p < (P >> 1); p += blockDim.x) {
                const int i = 2 * st * (p / st) + (p % st), j = i + st;
                if (j < n) { const int x = a[i], y = a[j]; if (x > y) { a[i] = y; a[j] = x; } }
            }
            __syncthreads();
        }
    }
}

// ordered unique of the sorted a[0 .. n) into out[0 ..]; `out` may alias `a` (writes trail the reads).  Returns the count.
template <typename Ptr>
__device__ __forceinline__ int cb_unique(Ptr a, int n, int* out, int* sm_scan) {
    __shared__ int s_last;
    int base = 0;
    for (int i0 = 0; i0 < n; i0 += blockDim.x) {
        const int i = i0 + threadIdx.x;
        int v = 0, keep = 0;
        if (i < n) {
            v = a[i];
            const int pv = (i == 0) ? 0 : ((threadIdx.x == 0) ? s_last : a[i - 1]);
            keep = (i == 0 || v != pv) ? 1 : 0;
        }
        __syncthreads();                                  // every read of this chunk (and of s_last) is done
        if (i < n && (threadIdx.x == blockDim.x - 1 || i == n - 1)) s_last = v;
        int total;
        const int ex = block_scan_excl<int>(keep, sm_scan, &total);
        if (keep) out[base + ex] = v;
        base += total;
        __syncthreads();
    }
    return base;
}

template <int THREADS, int SMEM_INTS, bool LONG>
__global__ void __launch_bounds__(THREADS) k_csr_sort_rows(int64_t N, const long long* __restrict__ raw_off,
                                                            int* __restrict__ tmp, int* __restrict__ ucount,
                                                            const int* __restrict__ worklist,
                                                            const int* __restrict__ wl_count) {
    extern __shared__ int cb_sm[];
    __shared__ int sm_scan[THREADS / 32 + 2];
    const int cnt = wl_count[LONG ? 1 : 0];
    for (int w = blockIdx.x; w < cnt; w += gridDim.x) {
        const int r = LONG ? worklist[N - 1 - w] : worklist[w];
        const long long o = raw_off[r];
        const int d = (int)(raw_off[r + 1] - o);
        int* row = tmp + o;
        int u;
        if (d <= SMEM_INTS) {
            for (int i = threadIdx.x; i < d; i += THREADS) cb_sm[i] = row[i];
            __syncthreads();
            cb_bitonic(cb_sm, d);
            u = cb_unique(cb_sm, d, row, sm_scan);
        } else {
            __syncthreads();
            cb_bitonic(row, d);                           // hub row: in place in HBM (L2-resident for anything realistic)
            u = cb_unique(row, d, row, sm_scan);
        }
        if (threadIdx.x == 0) ucount[r] = u;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(CB_THREADS) k_csr_compact(int64_t N, const long long* __restrict__ raw_off,
                                                             const int* __restrict__ tmp,
                                                             const long long* __restrict__ indptr,
                                                             int* __restrict__ indices) {
    const int lane = lane_id();
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < N; r += warps) {
        const long long o = raw_off[r], p = indptr[r];
        const int u = (int)(indptr[r + 1] - p);
        for (int i = lane; i < u; i += 32) indices[p + i] = tmp[o + i];
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Whole-graph gcn_norm structure with int64 offsets (grapes_graph_norm_*): the transposed adjacency, in_off [N+1] int64,
// in_src int32 (sources ascending, stored self-loops dropped, duplicates kept), dinv = (indeg + 1)^-1/2.  A counting sort by
// destination read straight from the input (CSR rows or int64 edge chunks, no expanded copy), then per-row sorts with the
// tiers above, without the unique step.  Scratch: cnt int32 [N] (in-degree -> scatter cursor -> sort worklist), tile sums
// of the 64-bit scan, 4 flags.
// ---------------------------------------------------------------------------------------------------------------------
#define GN_ERR_ID 1                  // an id outside [0, N): the edge is skipped, the caller raises
#define GN_ERR_DEG 2                 // a node with >= 2^31 - 1 in-edges: not representable, the caller raises

template <bool SCATTER>
__device__ __forceinline__ void gn_edge(int64_t r, int64_t c, int64_t N, int* __restrict__ cnt,
                                        const long long* __restrict__ in_off, int* __restrict__ in_src, int* __restrict__ err) {
    if (r < 0 || r >= N || c < 0 || c >= N) { if (!SCATTER) atomicOr(err, GN_ERR_ID); return; }
    if (r == c) return;                                              // stored self-loop: dropped (one is added per node)
    const int k = atomicAdd(&cnt[c], 1);
    if (SCATTER) in_src[in_off[c] + k] = (int)r;
    else if (k == 0x7ffffffe) atomicOr(err, GN_ERR_DEG);
}

// CSR rows [r0, r1): row r is the source, its indices the destinations; one warp per row
template <bool SCATTER>
__global__ void __launch_bounds__(CB_THREADS) k_gn_csr(const long long* __restrict__ indptr, const int* __restrict__ indices,
                                                        int64_t r0, int64_t r1, int64_t N, int* __restrict__ cnt,
                                                        const long long* __restrict__ in_off, int* __restrict__ in_src,
                                                        int* __restrict__ err) {
    const int lane = lane_id();
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = r0 + (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5); r < r1; r += warps) {
        const long long e1 = indptr[r + 1];
        for (long long e = indptr[r] + lane; e < e1; e += 32) gn_edge<SCATTER>(r, indices[e], N, cnt, in_off, in_src, err);
    }
}

// edge chunk: src[e] -> dst[e], e < n (a slice of the int64 rows of edge_index)
template <bool SCATTER>
__global__ void __launch_bounds__(CB_THREADS) k_gn_edges(const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                                          int64_t n, int64_t N, int* __restrict__ cnt,
                                                          const long long* __restrict__ in_off, int* __restrict__ in_src,
                                                          int* __restrict__ err) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride)
        gn_edge<SCATTER>(src[e], dst[e], N, cnt, in_off, in_src, err);
}

// Destination window [lo, hi) of the structure (grapes_graph_norm_window_*): pass 1 scatters only the edges into the window,
// at win_off[c - lo] (offsets local to the window).  Ids were checked by pass 0 over the same input.
__device__ __forceinline__ void gnw_edge(int64_t r, int64_t c, int64_t N, int64_t lo, int64_t hi, int* __restrict__ cnt,
                                         const long long* __restrict__ win_off, int* __restrict__ in_src) {
    if (r < 0 || r >= N || c < lo || c >= hi || r == c) return;
    const int k = atomicAdd(&cnt[c], 1);
    in_src[win_off[c - lo] + k] = (int)r;
}

__global__ void __launch_bounds__(CB_THREADS) k_gnw_csr(const long long* __restrict__ indptr, const int* __restrict__ indices,
                                                         int64_t r0, int64_t r1, int64_t N, int64_t lo, int64_t hi,
                                                         int* __restrict__ cnt, const long long* __restrict__ win_off,
                                                         int* __restrict__ in_src) {
    const int lane = lane_id();
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = r0 + (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5); r < r1; r += warps) {
        const long long e1 = indptr[r + 1];
        for (long long e = indptr[r] + lane; e < e1; e += 32) gnw_edge(r, indices[e], N, lo, hi, cnt, win_off, in_src);
    }
}

__global__ void __launch_bounds__(CB_THREADS) k_gnw_edges(const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                                           int64_t n, int64_t N, int64_t lo, int64_t hi, int* __restrict__ cnt,
                                                           const long long* __restrict__ win_off, int* __restrict__ in_src) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride)
        gnw_edge(src[e], dst[e], N, lo, hi, cnt, win_off, in_src);
}

// Transposed structure (grapes_graph_norm_t_*, the backward of the whole-graph aggregation): row s lists the destinations
// d of the edges s -> d, stored self-loops dropped.  From the graph's CSR, whose row s already holds its destinations
// sorted and unique, that is row s without s itself: a count (pass 0) and an order-keeping warp compaction (pass 1) at
// out_off[s], no cursor and no sort.  From an edge list it is k_gn_edges with the roles of source and destination swapped.
// out_off is read at r - off0: 0 for the whole structure, lo for the offsets of a source window [lo, hi).
template <bool FILL>
__global__ void __launch_bounds__(CB_THREADS) k_gnt_csr(const long long* __restrict__ indptr, const int* __restrict__ indices,
                                                         int64_t r0, int64_t r1, int64_t N, int* __restrict__ cnt,
                                                         const long long* __restrict__ out_off, int64_t off0,
                                                         int* __restrict__ out_dst, int* __restrict__ err) {
    const int lane = lane_id();
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = r0 + (((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5); r < r1; r += warps) {
        const long long e0 = indptr[r], e1 = indptr[r + 1];
        long long base = FILL ? out_off[r - off0] : 0;
        for (long long c0 = e0; c0 < e1; c0 += 32) {
            const long long e = c0 + lane;
            const int64_t v = e < e1 ? (int64_t)indices[e] : (int64_t)r;
            const bool bad = v < 0 || v >= N;
            if (!FILL && bad) atomicOr(err, GN_ERR_ID);
            const unsigned m = __ballot_sync(GRAPES_FULL_MASK, !bad && v != r);
            if (FILL && !bad && v != r) out_dst[base + __popc(m & ((1u << lane) - 1u))] = (int)v;
            base += __popc(m);
        }
        if (!FILL && lane == 0) {
            if (base >= 0x7fffffff) { atomicOr(err, GN_ERR_DEG); base = 0x7ffffffe; }
            cnt[r] = (int)base;
        }
    }
}

// bounds[k] = the least i in [0, N] with (in_off[i] + i) * W >= k * T, T = in_off[N] + N: the prefix of indeg + 1 cut into
// W parts, so every window holds T / W of it to within one row's indeg + 1.  bounds[0] = 0, bounds[W] = N.
__global__ void k_gn_bounds(int64_t N, const long long* __restrict__ in_off, int W, long long* __restrict__ bounds) {
    const long long T = in_off[N] + N;
    for (int k = threadIdx.x; k <= W; k += blockDim.x) {
        const long long target = (long long)k * T;
        long long a = 0, b = N;                                      // invariant: answer in [a, b]
        while (a < b) {
            const long long m = a + ((b - a) >> 1);
            if ((in_off[m] + m) * W >= target) b = m; else a = m + 1;
        }
        bounds[k] = a;
    }
}

// dinv = (indeg + 1)^-1/2 with correctly rounded sqrt and divide (torch's 1.0 / sqrt(float)); cnt becomes the cursor
__global__ void __launch_bounds__(CB_THREADS) k_gn_dinv(int64_t N, int* __restrict__ cnt, float* __restrict__ dinv) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += stride) {
        dinv[i] = __fdiv_rn(1.f, __fsqrt_rn((float)((long long)cnt[i] + 1)));
        cnt[i] = 0;
    }
}

// rows of <= CB_WARP_MAX entries: one warp each, in registers (<= 128) or a shared-memory strip; longer rows are listed
// for k_gn_sort_rows (medium from the front of the worklist, long from the back)
__global__ void __launch_bounds__(CB_THREADS) k_gn_sort_short(int64_t N, const long long* __restrict__ in_off,
                                                               int* __restrict__ in_src, int* __restrict__ worklist,
                                                               int* __restrict__ wl_count) {
    __shared__ int s_rows[CB_THREADS / 32][CB_WARP_MAX];
    const int lane = lane_id();
    int* a = s_rows[threadIdx.x >> 5];
    const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < N; r += warps) {
        const long long o = in_off[r];
        const int d = (int)(in_off[r + 1] - o);
        int* row = in_src + o;
        if (d <= 1) continue;
        if (d > CB_WARP_MAX) {
            if (lane == 0) {
                if (d <= CB_MED_MAX) worklist[atomicAdd(&wl_count[0], 1)] = (int)r;
                else worklist[N - 1 - atomicAdd(&wl_count[1], 1)] = (int)r;
            }
            continue;
        }
        if (d > 128) {
            for (int i = lane; i < d; i += 32) a[i] = row[i];
            __syncwarp();
            cb_warp_bitonic_smem(a, d, lane);
            for (int i = lane; i < d; i += 32) row[i] = a[i];
            __syncwarp();
            continue;
        }
        if (d <= 32) {
            int v[1] = {lane < d ? row[lane] : 0x7fffffff};
            cb_warp_bitonic<1>(v, lane);
            if (lane < d) row[lane] = v[0];
        } else if (d <= 64) {
            int v[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) v[j] = (j * 32 + lane < d) ? row[j * 32 + lane] : 0x7fffffff;
            cb_warp_bitonic<2>(v, lane);
#pragma unroll
            for (int j = 0; j < 2; ++j) if (j * 32 + lane < d) row[j * 32 + lane] = v[j];
        } else {
            int v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) v[j] = (j * 32 + lane < d) ? row[j * 32 + lane] : 0x7fffffff;
            cb_warp_bitonic<4>(v, lane);
#pragma unroll
            for (int j = 0; j < 4; ++j) if (j * 32 + lane < d) row[j * 32 + lane] = v[j];
        }
    }
}

template <int THREADS, int SMEM_INTS, bool LONG>
__global__ void __launch_bounds__(THREADS) k_gn_sort_rows(int64_t N, const long long* __restrict__ in_off,
                                                           int* __restrict__ in_src, const int* __restrict__ worklist,
                                                           const int* __restrict__ wl_count) {
    extern __shared__ int cb_sm[];
    const int cnt = wl_count[LONG ? 1 : 0];
    for (int w = blockIdx.x; w < cnt; w += gridDim.x) {
        const int r = LONG ? worklist[N - 1 - w] : worklist[w];
        const long long o = in_off[r];
        const int d = (int)(in_off[r + 1] - o);
        int* row = in_src + o;
        if (d <= SMEM_INTS) {
            for (int i = threadIdx.x; i < d; i += THREADS) cb_sm[i] = row[i];
            __syncthreads();
            cb_bitonic(cb_sm, d);
            for (int i = threadIdx.x; i < d; i += THREADS) row[i] = cb_sm[i];
        } else {
            __syncthreads();
            cb_bitonic(row, d);                           // hub row: in place in HBM
        }
        __syncthreads();
    }
}

struct GnLayout { size_t cnt, tile_sum, flags, total; };
static GnLayout gn_layout(int64_t N) {
    GnLayout L;
    size_t o = 0;
    L.cnt = o; o += cb_align(sizeof(int) * (size_t)N);
    L.tile_sum = o; o += cb_align(sizeof(long long) * ((size_t)((N + CB_SCAN_TILE - 1) / CB_SCAN_TILE) + 1));
    L.flags = o; o += cb_align(sizeof(int) * 4);
    L.total = o;
    return L;
}

static int gn_sms(int* sms) {
    int dev = 0;
    GRAPES_CUDA_OK(cudaGetDevice(&dev));
    GRAPES_CUDA_OK(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev));
    return GRAPES_OK;
}

int g_csr_direct_scatter = 0;      // 0 = by shape, 1 = single-pass random scatter, 2 = partition + windowed scatter (A/B)

struct CbLayout {
    size_t deg, ucount, raw_off, tile_sum, worklist, flags, bucket_fill, tmp, pairs, total;
};
static CbLayout cb_layout(int64_t N, int64_t E) {
    CbLayout L;
    size_t o = 0;
    const size_t tiles = (size_t)((N + CB_SCAN_TILE - 1) / CB_SCAN_TILE) + 1;
    L.deg = o; o += cb_align(sizeof(int) * (size_t)N);
    L.ucount = o; o += cb_align(sizeof(int) * (size_t)N);
    L.raw_off = o; o += cb_align(sizeof(long long) * (size_t)(N + 1));
    L.tile_sum = o; o += cb_align(sizeof(long long) * tiles);
    L.worklist = o; o += cb_align(sizeof(int) * (size_t)N);
    L.flags = o; o += cb_align(sizeof(int) * 4);
    L.bucket_fill = o; o += cb_align(sizeof(unsigned long long) * CB_PART_MAXB);
    L.tmp = o; o += cb_align(sizeof(int) * (size_t)(E > 0 ? E : 1));
    L.pairs = o; o += cb_align(sizeof(unsigned long long) * (size_t)(E > 0 ? E : 1));
    L.total = o;
    return L;
}

extern "C" {

int grapes_csr_set_direct_scatter(int mode) { g_csr_direct_scatter = (mode == 1 || mode == 2) ? mode : 0; return GRAPES_OK; }

int64_t grapes_csr_workspace_bytes(int64_t num_nodes, int64_t num_edges) {
    if (num_nodes <= 0 || num_edges < 0) return 0;
    return (int64_t)cb_layout(num_nodes, num_edges).total;
}

int grapes_csr_from_edges(const int64_t* src, const int64_t* dst, int64_t num_edges, int64_t num_nodes, int64_t* indptr,
                          int* indices, int64_t* nnz_dev, int* err_dev, void* workspace, int64_t workspace_bytes,
                          void* stream) {
    GRAPES_REQUIRE(num_nodes > 0 && num_nodes < (1ll << 31), "num_nodes must fit int32");
    GRAPES_REQUIRE(num_edges >= 0, "negative edge count");
    GRAPES_REQUIRE(indptr && nnz_dev && err_dev && workspace && (indices || num_edges == 0), "null argument");
    GRAPES_REQUIRE((src && dst) || num_edges == 0, "null edge list");
    const int64_t N = num_nodes, E = num_edges;
    const CbLayout L = cb_layout(N, E);
    GRAPES_REQUIRE(workspace_bytes >= (int64_t)L.total, "workspace smaller than grapes_csr_workspace_bytes()");
    int dev = 0, sms = 0;
    GRAPES_CUDA_OK(cudaGetDevice(&dev));
    GRAPES_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    cudaStream_t s = (cudaStream_t)stream;
    unsigned char* ws = (unsigned char*)workspace;
    int* deg = (int*)(ws + L.deg);
    int* ucount = (int*)(ws + L.ucount);
    long long* raw_off = (long long*)(ws + L.raw_off);
    long long* tile_sum = (long long*)(ws + L.tile_sum);
    int* worklist = (int*)(ws + L.worklist);
    int* flags = (int*)(ws + L.flags);                    // [0] medium rows, [1] long rows
    int* tmp = (int*)(ws + L.tmp);
    GRAPES_CUDA_OK(cudaMemsetAsync(deg, 0, sizeof(int) * (size_t)N, s));
    GRAPES_CUDA_OK(cudaMemsetAsync(flags, 0, sizeof(int) * 4, s));
    GRAPES_CUDA_OK(cudaMemsetAsync(err_dev, 0, sizeof(int), s));
    const int edge_grid = (int)(E > 0 ? ((E + CB_THREADS - 1) / CB_THREADS < (int64_t)sms * 16 ? (E + CB_THREADS - 1) / CB_THREADS
                                                                                                : (int64_t)sms * 16)
                                      : 1);
    const int64_t row_ctas = (N * 32 + CB_THREADS - 1) / CB_THREADS;
    const int row_grid = (int)(row_ctas < (int64_t)sms * 16 ? row_ctas : (int64_t)sms * 16);
    if (E > 0) {
        pdl(k_csr_degree, edge_grid, CB_THREADS, 0, s)(src, dst, E, N, deg, err_dev);
        grapes_count_launches(1);
    }
    cb_scan64(deg, N, tile_sum, raw_off, nullptr, s);
    GRAPES_CUDA_OK(cudaMemsetAsync(deg, 0, sizeof(int) * (size_t)N, s));          // deg becomes the scatter cursor
    // short rows scattered over a table larger than L2 pay a DRAM read-modify-write per store: partition first.  Long rows
    // (Reddit-shape, ~500 entries) and tables that fit L2 do better with the single pass (measured, DESIGN.md section 9).
    const bool direct = g_csr_direct_scatter == 1 || (g_csr_direct_scatter == 0 && (E < (8ll << 20) || E / N >= 128));
    if (E > 0 && direct) {
        pdl(k_csr_scatter, edge_grid, CB_THREADS, 0, s)(src, dst, E, N, raw_off, deg, tmp);
        grapes_count_launches(1);
    } else if (E > 0) {
        unsigned long long* bucket_fill = (unsigned long long*)(ws + L.bucket_fill);
        unsigned long long* pairs = (unsigned long long*)(ws + L.pairs);
        const int max_b = E <= (1ll << 28) ? 256 : CB_PART_MAXB;
        int shift = 0;
        while (((N + (1ll << shift) - 1) >> shift) > max_b) ++shift;
        const int B = (int)((N + (1ll << shift) - 1) >> shift);
        // CTAs per bucket: as many buckets in flight as keep their windows of `tmp` (4 E / B bytes each) inside 32 MB of L2
        const double window = 4.0 * (double)E / B;
        long long conc = (long long)(32.0 * 1024 * 1024 / (window > 1.0 ? window : 1.0));
        if (conc < 1) conc = 1;
        long long G = ((long long)sms * 8 + conc - 1) / conc;
        if (G < 1) G = 1;
        if (G > 4096) G = 4096;
        GRAPES_CUDA_OK(cudaMemsetAsync(bucket_fill, 0, sizeof(unsigned long long) * CB_PART_MAXB, s));
        const int64_t tiles = (E + CB_PART_TILE - 1) / CB_PART_TILE;
        const int part_grid = (int)(tiles < (int64_t)sms * 4 ? tiles : (int64_t)sms * 4);
        pdl(k_csr_partition, part_grid, CB_PART_THREADS, 0, s)(src, dst, E, N, raw_off, shift, B, bucket_fill, pairs);
        pdl(k_csr_scatter_part, (int)(B * G), CB_THREADS, 0, s)(pairs, raw_off, N, shift, (int)G, deg, tmp);
        grapes_count_launches(2);
    }
    pdl(k_csr_sort_short, row_grid, CB_THREADS, 0, s)(N, raw_off, tmp, ucount, worklist, flags);
    {
        static bool configured = false;
        if (!configured) {
            GRAPES_CUDA_OK(cudaFuncSetAttribute(k_csr_sort_rows<CB_LONG_THREADS, CB_LONG_SMEM, true>,
                                                cudaFuncAttributeMaxDynamicSharedMemorySize, CB_LONG_SMEM * 4));
            configured = true;
        }
    }
    pdl((k_csr_sort_rows<CB_MED_THREADS, CB_MED_MAX, false>), sms * 8, CB_MED_THREADS, CB_MED_MAX * 4, s)(
        N, raw_off, tmp, ucount, worklist, flags);
    pdl((k_csr_sort_rows<CB_LONG_THREADS, CB_LONG_SMEM, true>), sms, CB_LONG_THREADS, CB_LONG_SMEM * 4, s)(
        N, raw_off, tmp, ucount, worklist, flags);
    grapes_count_launches(3);
    cb_scan64(ucount, N, tile_sum, (long long*)indptr, (long long*)nnz_dev, s);
    pdl(k_csr_compact, row_grid, CB_THREADS, 0, s)(N, raw_off, tmp, (const long long*)indptr, indices);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}


int64_t grapes_graph_norm_workspace_bytes(int64_t num_nodes) {
    if (num_nodes <= 0) return 0;
    return (int64_t)gn_layout(num_nodes).total;
}

int grapes_graph_norm_begin(int64_t num_nodes, void* workspace, int64_t workspace_bytes, int* err_dev, void* stream) {
    GRAPES_REQUIRE(num_nodes > 0 && num_nodes < (1ll << 31), "num_nodes must fit int32");
    GRAPES_REQUIRE(workspace && err_dev, "null argument");
    const GnLayout L = gn_layout(num_nodes);
    GRAPES_REQUIRE(workspace_bytes >= (int64_t)L.total, "workspace smaller than grapes_graph_norm_workspace_bytes()");
    cudaStream_t s = (cudaStream_t)stream;
    GRAPES_CUDA_OK(cudaMemsetAsync((unsigned char*)workspace + L.cnt, 0, sizeof(int) * (size_t)num_nodes, s));
    GRAPES_CUDA_OK(cudaMemsetAsync((unsigned char*)workspace + L.flags, 0, sizeof(int) * 4, s));
    GRAPES_CUDA_OK(cudaMemsetAsync(err_dev, 0, sizeof(int), s));
    return GRAPES_OK;
}

int grapes_graph_norm_add_csr(int pass, int64_t num_nodes, const int64_t* indptr, const int* indices, int64_t r0, int64_t r1,
                              int64_t* in_off, int* in_src, void* workspace, int* err_dev, void* stream) {
    GRAPES_REQUIRE(pass == 0 || pass == 1, "pass is 0 (count) or 1 (scatter)");
    GRAPES_REQUIRE(indptr && workspace && err_dev && (pass == 0 || (in_off && in_src)), "null argument");
    GRAPES_REQUIRE(0 <= r0 && r0 <= r1 && r1 <= num_nodes, "row range outside [0, N]");
    if (r1 == r0) return GRAPES_OK;
    int sms = 0;
    if (gn_sms(&sms) != GRAPES_OK) return GRAPES_ERR_CUDA;
    int* cnt = (int*)((unsigned char*)workspace + gn_layout(num_nodes).cnt);
    const int64_t ctas = ((r1 - r0) * 32 + CB_THREADS - 1) / CB_THREADS;
    const int grid = (int)(ctas < (int64_t)sms * 16 ? ctas : (int64_t)sms * 16);
    cudaStream_t s = (cudaStream_t)stream;
    if (pass == 0)
        pdl(k_gn_csr<false>, grid, CB_THREADS, 0, s)((const long long*)indptr, indices, r0, r1, num_nodes, cnt, nullptr,
                                                      nullptr, err_dev);
    else
        pdl(k_gn_csr<true>, grid, CB_THREADS, 0, s)((const long long*)indptr, indices, r0, r1, num_nodes, cnt,
                                                     (const long long*)in_off, in_src, err_dev);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_graph_norm_add_edges(int pass, int64_t num_nodes, const int64_t* src, const int64_t* dst, int64_t num_edges,
                                int64_t* in_off, int* in_src, void* workspace, int* err_dev, void* stream) {
    GRAPES_REQUIRE(pass == 0 || pass == 1, "pass is 0 (count) or 1 (scatter)");
    GRAPES_REQUIRE(num_edges >= 0, "negative edge count");
    GRAPES_REQUIRE(workspace && err_dev && (num_edges == 0 || (src && dst)) && (pass == 0 || (in_off && in_src)),
                   "null argument");
    if (num_edges == 0) return GRAPES_OK;
    int sms = 0;
    if (gn_sms(&sms) != GRAPES_OK) return GRAPES_ERR_CUDA;
    int* cnt = (int*)((unsigned char*)workspace + gn_layout(num_nodes).cnt);
    const int64_t ctas = (num_edges + CB_THREADS - 1) / CB_THREADS;
    const int grid = (int)(ctas < (int64_t)sms * 16 ? ctas : (int64_t)sms * 16);
    cudaStream_t s = (cudaStream_t)stream;
    if (pass == 0)
        pdl(k_gn_edges<false>, grid, CB_THREADS, 0, s)(src, dst, num_edges, num_nodes, cnt, nullptr, nullptr, err_dev);
    else
        pdl(k_gn_edges<true>, grid, CB_THREADS, 0, s)(src, dst, num_edges, num_nodes, cnt, (const long long*)in_off, in_src,
                                                       err_dev);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_graph_norm_offsets(int64_t num_nodes, void* workspace, int64_t* in_off, float* dinv, int64_t* nnz_dev,
                              void* stream) {
    GRAPES_REQUIRE(workspace && in_off && dinv && nnz_dev, "null argument");
    int sms = 0;
    if (gn_sms(&sms) != GRAPES_OK) return GRAPES_ERR_CUDA;
    const GnLayout L = gn_layout(num_nodes);
    unsigned char* ws = (unsigned char*)workspace;
    int* cnt = (int*)(ws + L.cnt);
    cudaStream_t s = (cudaStream_t)stream;
    cb_scan64(cnt, num_nodes, (long long*)(ws + L.tile_sum), (long long*)in_off, (long long*)nnz_dev, s);
    const int64_t ctas = (num_nodes + CB_THREADS - 1) / CB_THREADS;
    pdl(k_gn_dinv, (int)(ctas < (int64_t)sms * 16 ? ctas : (int64_t)sms * 16), CB_THREADS, 0, s)(num_nodes, cnt, dinv);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_graph_norm_finish(int64_t num_nodes, const int64_t* in_off, int* in_src, void* workspace, void* stream) {
    GRAPES_REQUIRE(in_off && in_src && workspace, "null argument");
    int sms = 0;
    if (gn_sms(&sms) != GRAPES_OK) return GRAPES_ERR_CUDA;
    const GnLayout L = gn_layout(num_nodes);
    unsigned char* ws = (unsigned char*)workspace;
    int* worklist = (int*)(ws + L.cnt);                   // the cursor is spent after the scatter pass
    int* flags = (int*)(ws + L.flags);
    const long long* off = (const long long*)in_off;
    cudaStream_t s = (cudaStream_t)stream;
    GRAPES_CUDA_OK(cudaMemsetAsync(flags, 0, sizeof(int) * 2, s));
    const int64_t row_ctas = (num_nodes * 32 + CB_THREADS - 1) / CB_THREADS;
    pdl(k_gn_sort_short, (int)(row_ctas < (int64_t)sms * 16 ? row_ctas : (int64_t)sms * 16), CB_THREADS, 0, s)(
        num_nodes, off, in_src, worklist, flags);
    {
        static bool configured = false;
        if (!configured) {
            GRAPES_CUDA_OK(cudaFuncSetAttribute(k_gn_sort_rows<CB_LONG_THREADS, CB_LONG_SMEM, true>,
                                                cudaFuncAttributeMaxDynamicSharedMemorySize, CB_LONG_SMEM * 4));
            configured = true;
        }
    }
    pdl((k_gn_sort_rows<CB_MED_THREADS, CB_MED_MAX, false>), sms * 8, CB_MED_THREADS, CB_MED_MAX * 4, s)(
        num_nodes, off, in_src, worklist, flags);
    pdl((k_gn_sort_rows<CB_LONG_THREADS, CB_LONG_SMEM, true>), sms, CB_LONG_THREADS, CB_LONG_SMEM * 4, s)(
        num_nodes, off, in_src, worklist, flags);
    grapes_count_launches(3);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_graph_norm_t_add_csr(int pass, int64_t num_nodes, const int64_t* indptr, const int* indices, int64_t r0,
                                int64_t r1, int64_t* out_off, int* out_dst, void* workspace, int* err_dev, void* stream) {
    GRAPES_REQUIRE(pass == 0 || pass == 1, "pass is 0 (count) or 1 (compaction)");
    GRAPES_REQUIRE(indptr && workspace && err_dev && (pass == 0 || (out_off && out_dst)), "null argument");
    GRAPES_REQUIRE(0 <= r0 && r0 <= r1 && r1 <= num_nodes, "row range outside [0, N]");
    if (r1 == r0) return GRAPES_OK;
    int sms = 0;
    if (gn_sms(&sms) != GRAPES_OK) return GRAPES_ERR_CUDA;
    int* cnt = (int*)((unsigned char*)workspace + gn_layout(num_nodes).cnt);
    const int64_t ctas = ((r1 - r0) * 32 + CB_THREADS - 1) / CB_THREADS;
    const int grid = (int)(ctas < (int64_t)sms * 16 ? ctas : (int64_t)sms * 16);
    cudaStream_t s = (cudaStream_t)stream;
    if (pass == 0)
        pdl(k_gnt_csr<false>, grid, CB_THREADS, 0, s)((const long long*)indptr, indices, r0, r1, num_nodes, cnt, nullptr,
                                                       (int64_t)0, nullptr, err_dev);
    else
        pdl(k_gnt_csr<true>, grid, CB_THREADS, 0, s)((const long long*)indptr, indices, r0, r1, num_nodes, cnt,
                                                      (const long long*)out_off, (int64_t)0, out_dst, err_dev);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_graph_norm_t_add_edges(int pass, int64_t num_nodes, const int64_t* src, const int64_t* dst, int64_t num_edges,
                                  int64_t* out_off, int* out_dst, void* workspace, int* err_dev, void* stream) {
    // the forward's counting sort keyed by the source: row = src[e], entry = dst[e]
    return grapes_graph_norm_add_edges(pass, num_nodes, dst, src, num_edges, out_off, out_dst, workspace, err_dev, stream);
}

int grapes_graph_norm_t_offsets(int64_t num_nodes, void* workspace, int64_t* out_off, int64_t* nnz_dev, void* stream) {
    GRAPES_REQUIRE(workspace && out_off && nnz_dev, "null argument");
    const GnLayout L = gn_layout(num_nodes);
    unsigned char* ws = (unsigned char*)workspace;
    int* cnt = (int*)(ws + L.cnt);
    cudaStream_t s = (cudaStream_t)stream;
    cb_scan64(cnt, num_nodes, (long long*)(ws + L.tile_sum), (long long*)out_off, (long long*)nnz_dev, s);
    GRAPES_CUDA_OK(cudaMemsetAsync(cnt, 0, sizeof(int) * (size_t)num_nodes, s));    // cnt becomes the scatter cursor
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_graph_norm_window_bounds(int64_t num_nodes, const int64_t* in_off, int world, int64_t* bounds_dev,
                                    void* stream) {
    GRAPES_REQUIRE(in_off && bounds_dev, "null argument");
    GRAPES_REQUIRE(num_nodes > 0 && num_nodes < (1ll << 31), "num_nodes must fit int32");
    GRAPES_REQUIRE(world >= 1 && world <= 1024, "world must be in [1, 1024]");
    pdl(k_gn_bounds, 1, 128, 0, (cudaStream_t)stream)(num_nodes, (const long long*)in_off, world,
                                                                         (long long*)bounds_dev);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_graph_norm_window_add_csr(int64_t num_nodes, const int64_t* indptr, const int* indices, int64_t r0, int64_t r1,
                                     int64_t lo, int64_t hi, const int64_t* win_off, int* in_src, void* workspace,
                                     void* stream) {
    GRAPES_REQUIRE(indptr && workspace && win_off && in_src, "null argument");
    GRAPES_REQUIRE(0 <= r0 && r0 <= r1 && r1 <= num_nodes, "row range outside [0, N]");
    GRAPES_REQUIRE(0 <= lo && lo <= hi && hi <= num_nodes, "window outside [0, N]");
    if (r1 == r0 || hi == lo) return GRAPES_OK;
    int sms = 0;
    if (gn_sms(&sms) != GRAPES_OK) return GRAPES_ERR_CUDA;
    int* cnt = (int*)((unsigned char*)workspace + gn_layout(num_nodes).cnt);
    const int64_t ctas = ((r1 - r0) * 32 + CB_THREADS - 1) / CB_THREADS;
    pdl(k_gnw_csr, (int)(ctas < (int64_t)sms * 16 ? ctas : (int64_t)sms * 16), CB_THREADS, 0, (cudaStream_t)stream)(
        (const long long*)indptr, indices, r0, r1, num_nodes, lo, hi, cnt, (const long long*)win_off, in_src);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_graph_norm_window_add_edges(int64_t num_nodes, const int64_t* src, const int64_t* dst, int64_t num_edges,
                                       int64_t lo, int64_t hi, const int64_t* win_off, int* in_src, void* workspace,
                                       void* stream) {
    GRAPES_REQUIRE(num_edges >= 0, "negative edge count");
    GRAPES_REQUIRE(workspace && win_off && in_src && (num_edges == 0 || (src && dst)), "null argument");
    GRAPES_REQUIRE(0 <= lo && lo <= hi && hi <= num_nodes, "window outside [0, N]");
    if (num_edges == 0 || hi == lo) return GRAPES_OK;
    int sms = 0;
    if (gn_sms(&sms) != GRAPES_OK) return GRAPES_ERR_CUDA;
    int* cnt = (int*)((unsigned char*)workspace + gn_layout(num_nodes).cnt);
    const int64_t ctas = (num_edges + CB_THREADS - 1) / CB_THREADS;
    pdl(k_gnw_edges, (int)(ctas < (int64_t)sms * 16 ? ctas : (int64_t)sms * 16), CB_THREADS, 0, (cudaStream_t)stream)(
        src, dst, num_edges, num_nodes, lo, hi, cnt, (const long long*)win_off, in_src);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_graph_norm_t_window_add_csr(int64_t num_nodes, const int64_t* indptr, const int* indices, int64_t r0,
                                       int64_t r1, int64_t lo, int64_t hi, const int64_t* win_off, int* out_dst,
                                       void* workspace, void* stream) {
    GRAPES_REQUIRE(indptr && workspace && win_off && out_dst, "null argument");
    GRAPES_REQUIRE(0 <= r0 && r0 <= r1 && r1 <= num_nodes, "row range outside [0, N]");
    GRAPES_REQUIRE(0 <= lo && lo <= hi && hi <= num_nodes, "window outside [0, N]");
    // CSR row s is transposed row s: only the input rows inside the window are read
    const int64_t a = r0 > lo ? r0 : lo, b = r1 < hi ? r1 : hi;
    if (b <= a) return GRAPES_OK;
    int sms = 0;
    if (gn_sms(&sms) != GRAPES_OK) return GRAPES_ERR_CUDA;
    const int64_t ctas = ((b - a) * 32 + CB_THREADS - 1) / CB_THREADS;
    pdl(k_gnt_csr<true>, (int)(ctas < (int64_t)sms * 16 ? ctas : (int64_t)sms * 16), CB_THREADS, 0, (cudaStream_t)stream)(
        (const long long*)indptr, indices, a, b, num_nodes, nullptr, (const long long*)win_off, lo, out_dst, nullptr);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_graph_norm_t_window_add_edges(int64_t num_nodes, const int64_t* src, const int64_t* dst, int64_t num_edges,
                                         int64_t lo, int64_t hi, const int64_t* win_off, int* out_dst, void* workspace,
                                         void* stream) {
    // the forward window's scatter keyed by the source: row = src[e] in [lo, hi), entry = dst[e]
    return grapes_graph_norm_window_add_edges(num_nodes, dst, src, num_edges, lo, hi, win_off, out_dst, workspace, stream);
}

}  // extern "C"
