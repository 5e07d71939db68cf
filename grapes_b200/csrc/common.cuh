// Shared device/host helpers for the grapes_b200 sm_100a kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/grapes_b200.h"

#define GRAPES_FULL_MASK 0xffffffffu

struct grapes_ctx {
    int device;
    int sm_count;
    int64_t num_nodes;
    int num_words;                       // ceil(num_nodes / 32)
    // decoupled look-back scratch (self-cleaning, see lookback_* below)
    unsigned long long* scan_status;     // [scan_cap_tiles]
    unsigned int* scan_counters;         // [0] ticket, [1] done
    int scan_cap_tiles;
    // hub-row worklist for the per-row sort
    int* hub_rows;                       // [hub_cap]
    int* hub_count;                      // [1]
    int hub_cap;
    // split-K partial buffer for the TN GEMMs / column reductions
    float* partials;
    size_t partials_bytes;
};

void grapes_set_error(const char* fmt, ...);
void grapes_count_launches(int n);   // bookkeeping for bench.py's gpu_launches

#define GRAPES_CUDA_OK(expr)                                                              \
    do {                                                                                  \
        cudaError_t _e = (expr);                                                          \
        if (_e != cudaSuccess) {                                                          \
            grapes_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr,                \
                             cudaGetErrorString(_e));                                     \
            return GRAPES_ERR_CUDA;                                                       \
        }                                                                                 \
    } while (0)

#define GRAPES_REQUIRE(cond, msg)                                                         \
    do {                                                                                  \
        if (!(cond)) {                                                                    \
            grapes_set_error("%s:%d: %s (%s)", __FILE__, __LINE__, msg, #cond);           \
            return GRAPES_ERR_ARG;                                                        \
        }                                                                                 \
    } while (0)

#define GRAPES_LAUNCH_OK()                                                                \
    do {                                                                                  \
        cudaError_t _e = cudaGetLastError();                                              \
        if (_e != cudaSuccess) {                                                          \
            grapes_set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__,            \
                             cudaGetErrorString(_e));                                     \
            return GRAPES_ERR_CUDA;                                                       \
        }                                                                                 \
    } while (0)

// ---------------------------------------------------------------------------------------
// Programmatic dependent launch: every kernel of the library starts with pdl_begin() and is launched through pdl(),
// so in a stream (or captured graph) the NEXT kernel's launch, block scheduling and prologue overlap this kernel;
// griddepcontrol.wait then blocks until the previous kernel has completed and flushed its writes.
// grapes_set_pdl(0) turns the launch attribute off (plain stream order).
// ---------------------------------------------------------------------------------------
extern int g_grapes_pdl;          // bit mask over source files (GRAPES_PDL_GROUP), off by default
#ifndef GRAPES_PDL_GROUP
#define GRAPES_PDL_GROUP 1
#endif
#ifdef __CUDACC__
#include <utility>
__device__ __forceinline__ void pdl_begin() {
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
}
template <typename K>
struct PdlLaunch {
    K kernel; dim3 grid, block; size_t smem; cudaStream_t stream;
    template <typename... Args>
    void operator()(Args&&... args) const {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at; cfg.numAttrs = (g_grapes_pdl & GRAPES_PDL_GROUP) ? 1 : 0;
        cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
    }
};
template <typename K>
static inline PdlLaunch<K> pdl(K kernel, dim3 grid, dim3 block, size_t smem = 0, cudaStream_t stream = 0) {
    return PdlLaunch<K>{kernel, grid, block, smem, stream};
}
#endif

#ifdef __CUDACC__
// spmm_tma.cu: 0 = launched, 1 = shape not covered (the caller falls back to the register-staged kernels).  in_off is int
// (off64 = 0) or the int64 offsets of a row slab (off64 = 1: n_dev = {R, r0}, out only, no indicator columns)
int grapes_launch_agg_tma(grapes_ctx* ctx, const void* X, int x_bf16, int F, int ldx, const int* nodes, const int* n_dev, int cap_n,
                          const void* in_off, const int* in_src, const float* dinv, const uint32_t* ind_bits, int num_ind,
                          const float* bias, int relu, float* out, int ldo, float* out_hi, float* out_lo, int ones_col,
                          int ec_req, int ctas_per_sm, cudaStream_t s, int off64 = 0);
#endif

static inline int grapes_div_up(long long a, long long b) { return (int)((a + b - 1) / b); }
static inline int grapes_min_i(int a, int b) { return a < b ? a : b; }
static inline int grapes_max_i(int a, int b) { return a > b ? a : b; }

#ifdef __CUDACC__

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

// Philox4x32-10 (Salmon et al. 2011): counter-based, one call = 4 uniforms
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
        const uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
        ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
        key.x += W0; key.y += W1;
    }
    return ctr;
}
// the selection's Gumbel stream: counter (i / 4, 0, offset): word y is always 0
__device__ __forceinline__ float philox_uniform(unsigned long long seed, unsigned long long offset, int i) {
    uint4 ctr = make_uint4((uint32_t)(i >> 2), 0u, (uint32_t)offset, (uint32_t)(offset >> 32));
    const uint4 r = philox4x32_10(ctr, make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const uint32_t x = (i & 3) == 0 ? r.x : (i & 3) == 1 ? r.y : (i & 3) == 2 ? r.z : r.w;
    return (float)(x & 0xffffffu) * (1.0f / 16777216.0f);   // 24-bit mantissa in [0,1), as torch.rand
}

// Inverted dropout of the classifier GCN (modules/gcn.py:33,37).  The keep bit of entry i = row * width + col of site
// `tag` (= 1 + site + 2 * rank; site 0 = hidden layer, 1 = logits) is a pure function of (seed, step, tag, i): Philox
// counter (i / 4, tag, step), key = the seed's two words, keep iff the 24 low bits of word i % 4 are < threshold
// (= llrint((1 - p) * 2^24), computed on the host).  tag >= 1 keeps it apart from the selection stream (y = 0).
// drop_state = {seed, step} in device memory; the step's last reader advances `step` (grapes_classifier_loss_dropout).
struct DropParams {
    unsigned long long* state;          // {seed, step}
    uint32_t tag, threshold;
    float scale;                        // 1 / (1 - p); 0 when p == 1 (nothing is kept)
};
__device__ __forceinline__ uint4 dropout_words(unsigned long long seed, unsigned long long step, uint32_t tag,
                                               unsigned long long i) {
    return philox4x32_10(make_uint4((uint32_t)(i >> 2), tag, (uint32_t)step, (uint32_t)(step >> 32)),
                         make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
}
__device__ __forceinline__ bool dropout_keep(unsigned long long seed, unsigned long long step, uint32_t tag,
                                             uint32_t threshold, unsigned long long i) {
    const uint4 r = dropout_words(seed, step, tag, i);
    const uint32_t x = (i & 3) == 0 ? r.x : (i & 3) == 1 ? r.y : (i & 3) == 2 ? r.z : r.w;
    return (x & 0xffffffu) < threshold;
}
// keep bits of entries i0 .. i0 + 3 (bit j = entry i0 + j); i0 % 4 == 0: one Philox call
__device__ __forceinline__ uint32_t dropout_keep4(unsigned long long seed, unsigned long long step, uint32_t tag,
                                                  uint32_t threshold, unsigned long long i0) {
    const uint4 r = dropout_words(seed, step, tag, i0);
    return ((r.x & 0xffffffu) < threshold ? 1u : 0u) | ((r.y & 0xffffffu) < threshold ? 2u : 0u) |
           ((r.z & 0xffffffu) < threshold ? 4u : 0u) | ((r.w & 0xffffffu) < threshold ? 8u : 0u);
}

// device state words of one data-parallel exchange endpoint (peer_comm.cu; read by grapes_embed_merge_adam)
#define PS_SEQ 0        // steps completed
#define PS_TICKET_A 1   // push ticket
#define PS_TICKET_C 2   // reduce ticket
#define PS_FAILED 3     // sticky failure
#define PS_GO 4         // go word of the current step: seq (arrived) or seq | GO_FAIL
#define GO_FAIL 0x80000000u

// fp32 -> tf32 (10-bit mantissa), round to nearest, ties away from zero: the value cvt.rna.tf32.f32 returns for every
// finite input, in TWO integer instructions (add half an ulp to the magnitude bits, clear the 13 low bits).  ptxas expands
// the cvt into ~6 instructions with NaN / Inf handling; the 3xTF32 operand split calls this twice per element and was
// the largest instruction stream of the tcgen05 kernels (ncu: profiles/r02_topkernels.md).
__device__ __forceinline__ float grapes_tf32_rna(float x) {
    return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
}

// element type of a CSR row-offset array: int for the sampled blocks and graphs below 2^31 entries, int64 (W64) for the
// whole-graph structure of larger graphs (grapes_graph_norm_*)
template <bool W64> struct GrapesOff { typedef int T; };
template <> struct GrapesOff<true> { typedef long long T; };

// local id of global node v: rank of bit v in the bitmap (pref = exclusive popcount prefix per word)
__device__ __forceinline__ int bitmap_rank(const uint32_t* __restrict__ bm, const int* __restrict__ pref, int v) {
    const int w = v >> 5;
    return pref[w] + __popc(bm[w] & ((1u << (v & 31)) - 1u));
}
__device__ __forceinline__ bool bitmap_test(const uint32_t* __restrict__ bm, int v) {
    return (bm[v >> 5] >> (v & 31)) & 1u;
}
__device__ __forceinline__ void bitmap_set(uint32_t* bm, int v) {
    const uint32_t bit = 1u << (v & 31);
    uint32_t* w = bm + (v >> 5);
    if (!(*(volatile uint32_t*)w & bit)) atomicOr(w, bit);
}

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(GRAPES_FULL_MASK, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(GRAPES_FULL_MASK, v, o));
    return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(GRAPES_FULL_MASK, v, o));
    return v;
}

// inclusive warp scan
template <typename T>
__device__ __forceinline__ T warp_scan_incl(T v) {
    const int l = lane_id();
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        T t = __shfl_up_sync(GRAPES_FULL_MASK, v, o);
        if (l >= o) v += t;
    }
    return v;
}

// Block-wide exclusive scan of one value per thread.  `smem` needs (blockDim.x/32 + 1) slots.
// Returns the exclusive prefix; *total receives the block sum (same value in every thread).
template <typename T>
__device__ __forceinline__ T block_scan_excl(T v, T* smem, T* total) {
    const int l = lane_id(), w = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    T incl = warp_scan_incl(v);
    if (l == 31) smem[w] = incl;
    __syncthreads();
    if (w == 0) {
        T s = (l < nw) ? smem[l] : T(0);
        T si = warp_scan_incl(s);
        if (l < nw) smem[l] = si - s;          // exclusive prefix of each warp
        if (l == nw - 1) smem[nw] = si;        // block total
    }
    __syncthreads();
    T res = smem[w] + incl - v;
    *total = smem[nw];
    __syncthreads();                           // smem may be reused by the caller
    return res;
}

// ---------------------------------------------------------------------------------------
// Decoupled look-back (single-pass device-wide scan).  status word: [63:62] flag, [61:0] payload.
// Tiles take a ticket (so a tile's predecessors are always scheduled), publish their aggregate,
// look back for the exclusive prefix, and the last tile to finish zeroes the scratch again so
// the next launch (or CUDA-graph replay) finds it clean.  One scan at a time per ctx/stream.
// ---------------------------------------------------------------------------------------
#define LB_FLAG_AGG (1ull << 62)
#define LB_FLAG_INC (2ull << 62)
#define LB_PAYLOAD ((1ull << 62) - 1ull)

__device__ __forceinline__ unsigned long long lb_load(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.volatile.global.u64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ void lb_store(unsigned long long* p, unsigned long long v) {
    asm volatile("st.volatile.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Call from thread 0 of the block; result broadcast by the caller through shared memory.
__device__ __forceinline__ int lb_take_ticket(unsigned int* counters) { return (int)atomicAdd(&counters[0], 1u); }

// Executed by ALL 32 lanes of warp 0.  Returns the exclusive prefix of `tile` (valid in every lane).
__device__ __forceinline__ unsigned long long lb_exclusive(unsigned long long* status, int tile,
                                                           unsigned long long aggregate) {
    const int l = lane_id();
    if (tile == 0) {
        if (l == 0) lb_store(&status[0], LB_FLAG_INC | aggregate);
        return 0ull;
    }
    if (l == 0) lb_store(&status[tile], LB_FLAG_AGG | aggregate);
    unsigned long long excl = 0ull;
    int look = tile - 1;
    while (true) {
        const int idx = look - l;
        unsigned long long s = (idx >= 0) ? lb_load(&status[idx]) : LB_FLAG_INC;
        while (__any_sync(GRAPES_FULL_MASK, (s >> 62) == 0ull)) {
            s = (idx >= 0) ? lb_load(&status[idx]) : LB_FLAG_INC;
        }
        const unsigned incmask = __ballot_sync(GRAPES_FULL_MASK, (s >> 62) == 2ull);
        const int first = incmask ? (__ffs(incmask) - 1) : 32;
        unsigned long long v = (l <= first) ? (s & LB_PAYLOAD) : 0ull;
        v = warp_sum(v);
        excl += v;
        if (incmask) break;
        look -= 32;
    }
    if (l == 0) lb_store(&status[tile], LB_FLAG_INC | ((excl + aggregate) & LB_PAYLOAD));
    return excl;
}

// Call from thread 0 after the tile is done with lb_exclusive (or skipped it).  Returns true for
// the last tile of the launch, which must then call lb_cleanup with the whole block.
__device__ __forceinline__ bool lb_finish(unsigned int* counters) {
    __threadfence();
    return atomicAdd(&counters[1], 1u) == gridDim.x - 1;
}
__device__ __forceinline__ void lb_cleanup(unsigned long long* status, unsigned int* counters) {
    for (int i = threadIdx.x; i < (int)gridDim.x; i += blockDim.x) status[i] = 0ull;
    if (threadIdx.x == 0) { counters[0] = 0u; counters[1] = 0u; }
}

#endif  // __CUDACC__
