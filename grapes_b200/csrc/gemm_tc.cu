// tcgen05 (5th-gen tensor core) path for the sampler networks' dense transform -- the only true
// contraction on the GRAPES hot path (gcn_gf / gcn_z layer 1: [n x K] . [K x 256], main.py:112-114,210,227).
//
//   z[j] = sum_d relu(Y[j,:] . W1[d,:] + b1[d]) * w2[d]          (hidden activations never leave the SM)
//
// fp32-accurate on TF32 tensor cores by operand splitting (3xTF32): Y = Yh + Yl, W = Wh + Wl with
// Xh = tf32(X), Xl = tf32(X - Xh);  Y.W ~= Yh.Wh + Yh.Wl + Yl.Wh  (error ~2^-21, inside the 1e-5 bar).
//
// Kernel shape (one CTA per SM, persistent over 128-row x 128-col output tiles):
//   warp 0      TMA producer: cp.async.bulk.tensor 2D, SWIZZLE_128B boxes of 32 fp32 x 128 rows, 3-stage ring
//   warp 1      MMA issuer:   one elected lane, tcgen05.mma.cta_group::1.kind::tf32 M128 N128 K8,
//               accumulators in TMEM (2 x 128 columns, double buffered), tcgen05.commit -> mbarriers
//   warps 2..5  epilogue:     tcgen05.ld 32x32b (TMEM lane == output row), bias + relu + dot(w2) per row,
//               relu mask emitted as bits (warp ballot) for the backward
#include <cuda.h>

#define GRAPES_PDL_GROUP 4
#include "common.cuh"

#define TC_BM 128
#define TC_BN 128
#define TC_BK 32                       // fp32 elements per 128-byte swizzle row
#define TC_STAGES 3
#define TC_TILE_BYTES (TC_BM * TC_BK * 4)          // 16 KB: one operand tile of one k-block
#define TC_STAGE_BYTES (4 * TC_TILE_BYTES)         // A_hi, A_lo, B_hi, B_lo
#define TC_THREADS 192
#define TC_SMEM_BYTES (TC_STAGES * TC_STAGE_BYTES + 1024 /*align slack*/ + 256 /*barriers*/)

static int g_tc_debug = 0;      // bit 0: backward operand debug fill; bit 1: force the streaming (non W-resident) forward;
                                // bit 2: forward with BOTH operands in shared memory (k_l1_fwd_tc) instead of the default
                                // A-operand-in-tensor-memory form (k_l1_fwd_ts); bit 3: backward with both operands in shared
                                // memory (k_l1_bwd_tc) instead of the default k_l1_bwd_ts; bit 4: timeline stamps

// ------------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// (try_wait with a 20 us suspend-time hint measured SLOWER: the wake-up of a suspended warp costs more than the issue
// slots its spinning takes; k_l1_fwd_ts 31 -> 37 us per launch.)
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra.uni WAIT_DONE;\n\t"
        "bra.uni WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}\n" ::"r"(addr), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}\n" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// D[tmem] (+)= A[smem desc] . B[smem desc]^T, kind::tf32, issued by ONE thread
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// arrive on an mbarrier once every MMA issued so far by this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_ld_32x32_nowait(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ float tf32_rna_f(float x) { return grapes_tf32_rna(x); }

__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};\n"
        :: "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
           "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),
           "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]),
           "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
        : "memory");
    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}

// Shared-memory matrix descriptor, K-major operand tile stored as [rows][32 fp32] with SWIZZLE_128B
// (what TMA writes): start address >> 4, LBO (unused for swizzled K-major) = 1, SBO = 8 rows * 128 B = 1024 B,
// descriptor version 1 (Blackwell), layout type 2 = SWIZZLE_128B.   (cute/arch/mma_sm100_desc.hpp SmemDescriptor)
__device__ __forceinline__ uint64_t make_kmajor_sw128_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFFu);
    d |= (uint64_t)1u << 16;
    d |= (uint64_t)(1024u >> 4) << 32;
    d |= (uint64_t)1u << 46;
    d |= (uint64_t)2u << 61;
    return d;
}
// Instruction descriptor (InstrDescriptor): c_format F32 (1) @4, a/b_format TF32 (2) @7/@10, K-major A and B,
// N >> 3 @17, M >> 4 @24.
__device__ __forceinline__ constexpr uint32_t make_idesc_tf32(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ------------------------------------------------------------------------------------------------
// forward kernel.  One CTA per SM, persistent over 128-row x 128-column output tiles; 320 threads:
//   warp 0      TMA producer: raw fp32 Y tiles (32 columns x 128 rows, SWIZZLE_128B) into a ring
//   warp 1      MMA issuer (one elected lane), accumulators in TMEM (2 x 128 columns, double buffered)
//   warps 2..5  epilogue: tcgen05.ld, bias + relu + dot(w2) per row, relu mask bits
//   warps 6..9  converters (only when Y arrives as plain fp32, presplit == 0): 3xTF32 operand split of the Y tile IN
//               shared memory (hi in place, lo beside it; elementwise, so the swizzle pattern is irrelevant), then
//               fence.proxy.async -> the tensor core.  Saves the hi/lo copies in HBM at the price of one more
//               pipeline step; with presplit == 1 the aggregation already wrote Y_hi / Y_lo and both are TMA-loaded.
// Two modes:
//   W-resident (K <= 160): the CTA owns ONE 128-column half of the hidden layer and keeps that half of W (hi | lo,
//               all k-blocks) in shared memory for its whole life; only Y streams: 16 KB of L2 traffic per k-block
//               and tile instead of 64 KB (the kernel is L2-feed bound when everything is re-fetched per tile).
//   streaming:  W tiles travel with the Y tile in every stage (any K).
// ------------------------------------------------------------------------------------------------
#define TCF_THREADS 320
#define TC_CHUNK_KB 8                 // k-blocks (256 columns) accumulated in the tensor core before promotion to the master
__global__ void __launch_bounds__(TCF_THREADS, 1) k_l1_fwd_tc(
    const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmA_lo,
    const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo,
    const int* __restrict__ n_dev, int cap_n, int K, int D, int stages, int wres, int presplit,
    const float* __restrict__ b1, const float* __restrict__ w2, float* __restrict__ zpart,
    uint32_t* __restrict__ maskT) {
    pdl_begin();
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);     // SWIZZLE_128B tiles: 1024 B aligned
    const int nkb = (K + TC_BK - 1) / TC_BK;
    const int stage_bytes = wres ? 2 * TC_TILE_BYTES : 4 * TC_TILE_BYTES;            // Y hi | Y lo (| W hi | W lo)
    uint8_t* w_smem = smem;                                                          // W-resident: [nkb][hi | lo]
    uint8_t* ring = smem + (wres ? nkb * 2 * TC_TILE_BYTES : 0);
    uint64_t* bars = (uint64_t*)(ring + stages * stage_bytes);
    uint64_t* raw_bar = bars;                        // [4]  TMA -> converters
    uint64_t* conv_bar = bars + 4;                   // [4]  converters -> MMA
    uint64_t* empty_bar = bars + 8;                  // [4]  MMA -> TMA
    uint64_t* tfull_bar = bars + 12;                 // [2]  MMA -> epilogue
    uint64_t* tempty_bar = bars + 14;                // [2]  epilogue -> MMA
    uint64_t* w_bar = bars + 16;
    uint32_t* tmem_slot = (uint32_t*)(bars + 17);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = min(*n_dev, cap_n);
    const int NH = D / TC_BN;
    const int m_tiles = (n + TC_BM - 1) / TC_BM;
    // tile walk: W-resident -> fixed column half, row tiles strided over the CTAs of that half;
    //            streaming  -> all (row tile, half) pairs strided over the grid
    const int t_first = wres ? (int)blockIdx.x / NH : (int)blockIdx.x;
    const int t_step = wres ? (int)gridDim.x / NH : (int)gridDim.x;
    const int t_count = wres ? m_tiles : m_tiles * NH;
    const int nh_fixed = (int)blockIdx.x % NH;
#define TILE_MT(t) (wres ? (t) : (t) / NH)
#define TILE_NH(t) (wres ? nh_fixed : (t) % NH)

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmB_hi); tma_prefetch_desc(&tmB_lo);
        if (presplit) tma_prefetch_desc(&tmA_lo);
        for (int s = 0; s < stages; ++s) { mbar_init(&raw_bar[s], 1); mbar_init(&conv_bar[s], 4); mbar_init(&empty_bar[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&tfull_bar[s], 1); mbar_init(&tempty_bar[s], 4); }
        mbar_init(w_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(tmem_slot, 512);        // 2 chunk accumulators (2 x 128 columns) + the fp32 master (128)
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ===== TMA producer =====
        if (elect_one()) {
            if (wres && t_first < t_count) {
                mbar_arrive_expect_tx(w_bar, (uint32_t)(nkb * 2 * TC_TILE_BYTES));
                for (int kb = 0; kb < nkb; ++kb) {
                    tma_load_2d(w_smem + kb * 2 * TC_TILE_BYTES, &tmB_hi, w_bar, kb * TC_BK, nh_fixed * TC_BN);
                    tma_load_2d(w_smem + kb * 2 * TC_TILE_BYTES + TC_TILE_BYTES, &tmB_lo, w_bar, kb * TC_BK, nh_fixed * TC_BN);
                }
            }
            int stage = 0; uint32_t phase = 0;
            for (int t = t_first; t < t_count; t += t_step) {
                const int m0 = TILE_MT(t) * TC_BM, n0 = TILE_NH(t) * TC_BN;
                for (int kb = 0; kb < nkb; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    uint8_t* st = ring + stage * stage_bytes;
                    mbar_arrive_expect_tx(&raw_bar[stage], (uint32_t)(((presplit ? 2 : 1) + (wres ? 0 : 2)) * TC_TILE_BYTES));
                    tma_load_2d(st, &tmA, &raw_bar[stage], kb * TC_BK, m0);
                    if (presplit) tma_load_2d(st + TC_TILE_BYTES, &tmA_lo, &raw_bar[stage], kb * TC_BK, m0);
                    if (!wres) {
                        tma_load_2d(st + 2 * TC_TILE_BYTES, &tmB_hi, &raw_bar[stage], kb * TC_BK, n0);
                        tma_load_2d(st + 3 * TC_TILE_BYTES, &tmB_lo, &raw_bar[stage], kb * TC_BK, n0);
                    }
                    if (++stage == stages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (elect_one()) {
            const uint32_t idesc = make_idesc_tf32(TC_BM, TC_BN);
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            if (wres && t_first < t_count) { mbar_wait(w_bar, 0); tc_fence_after(); }
            const uint32_t wa = smem_u32(w_smem);
            for (int t = t_first; t < t_count; t += t_step) {
                for (int kc = 0; kc < nkb; kc += TC_CHUNK_KB) {          // the tensor core adds with truncation: keep chains short
                    mbar_wait(&tempty_bar[acc], acc_phase ^ 1);          // epilogue has drained this accumulator
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + (uint32_t)(acc * TC_BN);
                    const int kend = min(nkb, kc + TC_CHUNK_KB);
                    for (int kb = kc; kb < kend; ++kb) {
                        mbar_wait(presplit ? &raw_bar[stage] : &conv_bar[stage], phase);
                        tc_fence_after();
                        const uint32_t sa = smem_u32(ring + stage * stage_bytes);
                        const uint32_t sb = wres ? wa + kb * 2 * TC_TILE_BYTES : sa + 2 * TC_TILE_BYTES;
                        const uint64_t a_hi = make_kmajor_sw128_desc(sa);
                        const uint64_t a_lo = make_kmajor_sw128_desc(sa + TC_TILE_BYTES);
                        const uint64_t b_hi = make_kmajor_sw128_desc(sb);
                        const uint64_t b_lo = make_kmajor_sw128_desc(sb + TC_TILE_BYTES);
                        const int nks = min(TC_BK / 8, (K - kb * TC_BK + 7) / 8);     // the last k-block may be partly padding
#pragma unroll
                        for (int ks = 0; ks < TC_BK / 8; ++ks) {
                            if (ks >= nks) break;
                            const uint64_t adv = (uint64_t)((ks * 32) >> 4);      // +32 bytes per K=8 slice inside the swizzle row
                            umma_tf32(d_tmem, a_lo + adv, b_hi + adv, idesc, ((kb - kc) | ks) ? 1u : 0u);   // small terms first
                            umma_tf32(d_tmem, a_hi + adv, b_lo + adv, idesc, 1u);
                            umma_tf32(d_tmem, a_hi + adv, b_hi + adv, idesc, 1u);
                        }
                        umma_commit(&empty_bar[stage]);                   // smem slot free once these MMAs retire
                        if (++stage == stages) { stage = 0; phase ^= 1; }
                    }
                    umma_commit(&tfull_bar[acc]);                         // chunk accumulator complete -> epilogue
                    if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                }
            }
        }
    } else if (warp < 6) {
        // ===== epilogue (warps 2..5): TMEM lane quarter = warp % 4 =====
        const int q = warp & 3;
        int acc = 0; uint32_t acc_phase = 0;
        for (int t = t_first; t < t_count; t += t_step) {
            const int mt = TILE_MT(t), nh = TILE_NH(t);
            const int row = mt * TC_BM + q * 32 + lane;
            float zsum = 0.f;
            uint32_t mbits[4] = {0u, 0u, 0u, 0u};
            for (int kc = 0; kc < nkb; kc += TC_CHUNK_KB) {
                const bool first_chunk = (kc == 0), last_chunk = (kc + TC_CHUNK_KB >= nkb);
                mbar_wait(&tfull_bar[acc], acc_phase);
                tc_fence_after();
#pragma unroll
                for (int ch = 0; ch < TC_BN / 32; ++ch) {
                    uint32_t v[32];
                    const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
                    tmem_ld_32x32(lane_base + (uint32_t)(acc * TC_BN + ch * 32), v);
                    if (!first_chunk) {                                   // fp32 master += chunk (round to nearest)
                        uint32_t m[32];
                        tmem_ld_32x32(lane_base + (uint32_t)(2 * TC_BN + ch * 32), m);
#pragma unroll
                        for (int c = 0; c < 32; ++c) v[c] = __float_as_uint(__uint_as_float(v[c]) + __uint_as_float(m[c]));
                    }
                    if (!last_chunk) {
                        tmem_st_32x32(lane_base + (uint32_t)(2 * TC_BN + ch * 32), v);
                        continue;
                    }
#pragma unroll
                    for (int c = 0; c < 32; ++c) {
                        // (read-only-cache loads: the shared-memory pipe is what feeds the tensor core, keep it free)
                        const int col = nh * TC_BN + ch * 32 + c;
                        const float pre = __uint_as_float(v[c]) + __ldg(&b1[col]);
                        zsum = fmaf(fmaxf(pre, 0.f), __ldg(&w2[col]), zsum);
                        if (maskT) {
                            const uint32_t word = __ballot_sync(GRAPES_FULL_MASK, pre > 0.f && row < n);
                            if (lane == c) mbits[ch] = word;
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty_bar[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
            if (row < n) {                                        // two partial rows per half (k_l1_fwd_ts fills both)
                zpart[(size_t)(nh * 2) * cap_n + row] = zsum;
                zpart[(size_t)(nh * 2 + 1) * cap_n + row] = 0.f;
            }
            if (maskT) {
                // maskT[(row group of 32)][D]: bit r of word (g, d) = relu'(pre[32 g + r, d])
                uint32_t* dst = maskT + (size_t)(mt * 4 + q) * D + nh * TC_BN;
#pragma unroll
                for (int ch = 0; ch < 4; ++ch) dst[ch * 32 + lane] = mbits[ch];
            }
        }
    } else if (!presplit) {
        // ===== converters (warps 6..9): Y tile -> (hi, lo) in shared memory =====
        const int ct = threadIdx.x - 6 * 32;                          // 0..127
        int stage = 0; uint32_t phase = 0;
        for (int t = t_first; t < t_count; t += t_step) {
            for (int kb = 0; kb < nkb; ++kb) {
                mbar_wait(&raw_bar[stage], phase);
                uint8_t* st = ring + stage * stage_bytes;
                float4 v[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) v[i] = *reinterpret_cast<const float4*>(st + (size_t)(ct + i * 128) * 16);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    float4 h, l;
                    h.x = tf32_rna_f(v[i].x); h.y = tf32_rna_f(v[i].y); h.z = tf32_rna_f(v[i].z); h.w = tf32_rna_f(v[i].w);
                    l.x = tf32_rna_f(v[i].x - h.x); l.y = tf32_rna_f(v[i].y - h.y);
                    l.z = tf32_rna_f(v[i].z - h.z); l.w = tf32_rna_f(v[i].w - h.w);
                    *reinterpret_cast<float4*>(st + (size_t)(ct + i * 128) * 16) = h;
                    *reinterpret_cast<float4*>(st + TC_TILE_BYTES + (size_t)(ct + i * 128) * 16) = l;
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the tensor core
                __syncwarp();
                if (lane == 0) mbar_arrive(&conv_bar[stage]);
                if (++stage == stages) { stage = 0; phase ^= 1; }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------
// forward kernel, A operand in TENSOR MEMORY (tcgen05.mma ... [d_tmem], [a_tmem], b_desc: "TS" form).
//
// Why: a 128x128x8 tf32 MMA whose two operands both come from shared memory reads 8 KB per 32 tensor-core cycles --
// twice what the shared-memory pipe delivers (128 B/clk) -- and splitting the Y tile in shared memory adds another 48 KB
// of shared-memory traffic per k-block: k_l1_fwd_tc sits at the shared-memory read limit with the tensor pipe 35 % busy.
// Here the raw fp32 Y tile is TMA-loaded into a shared-memory ring and read ONCE by 8 converter warps (thread = tile row:
// with SWIZZLE_128B the 32 rows of a warp hit all 32 banks, 4 wavefronts per 512 bytes, the minimum), which split it into
// the 3xTF32 (hi, lo) pair and store both into a ring of TMEM slots (tcgen05.st; TMEM lane == tile row, which is exactly
// how an M = 128 A operand lives in tensor memory).  The MMA then reads only W from shared memory: 4 KB per 32 cycles,
// exactly the pipe's rate; per k-block 80 KB go through shared memory instead of 160 KB.  Same arithmetic, same
// summation order, same outputs as k_l1_fwd_tc.  (First form of this kernel: the converters read Y from global memory
// directly -- 28 k-blocks per CTA, each waiting ~0.7 us of L2 latency with one k-block of loads in flight: 31.5 vs 35 us.)
//   warp 0       TMA: raw Y tiles through a ring; the CTA's half of W (hi | lo) once (resident, K <= 128 or so), or
//                W tiles through a second ring (any K)
//   warp 1       MMA issuer; accumulators in TMEM (2 x 128 columns, double buffered), fp32 master for long K
//   warps 2..5   epilogue (bias + relu + dot(w2), relu mask bits)
//   warps 6..13  converters: shared memory -> registers -> (hi, lo) -> TMEM slot; lane quarter = warp % 4, column half = (warp-6)/4
// TMEM columns: [0,256) accumulators, [256,384) master when nkb > 8, then the A ring: slots of 64 columns (hi | lo).
// ------------------------------------------------------------------------------------------------
#define TCS_THREADS 448
__device__ __forceinline__ void umma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_st_32x32_x16(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n"
        :: "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
           "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st_32x32_nowait(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};\n"
        :: "r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
           "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),
           "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]),
           "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
        : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// 32 x 32 bit transpose across a warp: in, lane r holds bit c = M[r][c]; out, lane c holds bit r = M[r][c]
__device__ __forceinline__ uint32_t warp_bit_transpose(uint32_t x, int lane) {
#pragma unroll
    for (int j = 16; j >= 1; j >>= 1) {
        const uint32_t m = (j == 16) ? 0x0000ffffu : (j == 8) ? 0x00ff00ffu : (j == 4) ? 0x0f0f0f0fu : (j == 2) ? 0x33333333u : 0x55555555u;
        const uint32_t y = __shfl_xor_sync(GRAPES_FULL_MASK, x, j);
        x = (lane & j) ? ((x & ~m) | ((y >> j) & m)) : ((x & m) | ((y << j) & ~m));
    }
    return x;
}

template <bool LONGK, bool DENSE>
__global__ void __launch_bounds__(TCS_THREADS, 1) k_l1_fwd_ts(
    const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB_hi,
    const __grid_constant__ CUtensorMap tmB_lo, const int* __restrict__ n_dev, int cap_n, int K, int D, int wres,
    int bstages, int ystages, const float* __restrict__ b1, const float* __restrict__ w2, float* __restrict__ zpart,
    uint32_t* __restrict__ maskT, float* __restrict__ hout, int ldh, unsigned long long* dbg) {
    pdl_begin();
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);     // SWIZZLE_128B tiles: 1024 B aligned
    const int nkb = (K + TC_BK - 1) / TC_BK;
    const int nbt = wres ? nkb : bstages;                                            // W tiles (hi | lo) held in shared memory
    uint8_t* w_smem = smem;
    uint8_t* y_ring = smem + (size_t)nbt * 2 * TC_TILE_BYTES;                        // [ystages] raw fp32 Y tiles
    uint64_t* bars = (uint64_t*)(y_ring + (size_t)ystages * TC_TILE_BYTES);
    uint64_t* conv_bar = bars;                       // [4]  converters -> MMA   (A slot filled)
    uint64_t* aempty_bar = bars + 4;                 // [4]  MMA -> converters   (A slot free)
    uint64_t* bfull_bar = bars + 8;                  // [8]  TMA -> MMA          (W tile landed; streaming mode)
    uint64_t* bempty_bar = bars + 16;                // [8]  MMA -> TMA
    uint64_t* tfull_bar = bars + 24;                 // [2]  MMA -> epilogue
    uint64_t* tempty_bar = bars + 26;                // [2]  epilogue -> MMA
    uint64_t* w_bar = bars + 28;
    uint64_t* yfull_bar = bars + 32;                 // [8]  TMA -> converters   (raw Y tile landed)
    uint64_t* yempty_bar = bars + 40;                // [8]  converters -> TMA   (tile read into registers)
    uint32_t* tmem_slot = (uint32_t*)(bars + 29);
    float* s_b1 = (float*)(bars + 48);               // [128] bias of this CTA's hidden half
    float* s_w2 = s_b1 + TC_BN;                      // [128] output weights of the half

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = min(*n_dev, cap_n);
    const int NH = D / TC_BN;
    const int m_tiles = (n + TC_BM - 1) / TC_BM;
    // fixed column half per CTA, row tiles strided over the CTAs of that half
    const int t_first = (int)blockIdx.x / NH, t_step = (int)gridDim.x / NH;
    const int nh = (int)blockIdx.x % NH;
    const bool long_k = nkb > TC_CHUNK_KB;
    const uint32_t a_col0 = long_k ? 384u : 256u;
    const int aslots = long_k ? 2 : 4;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmB_hi); tma_prefetch_desc(&tmB_lo);
        for (int s = 0; s < 4; ++s) { mbar_init(&conv_bar[s], 4); mbar_init(&aempty_bar[s], 1); }
        for (int s = 0; s < 8; ++s) { mbar_init(&yfull_bar[s], 1); mbar_init(&yempty_bar[s], 4); }
        for (int s = 0; s < 8; ++s) { mbar_init(&bfull_bar[s], 1); mbar_init(&bempty_bar[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&tfull_bar[s], 1); mbar_init(&tempty_bar[s], 4); }
        mbar_init(w_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(tmem_slot, 512);
    if (threadIdx.x >= 64 && threadIdx.x < 64 + TC_BN) {
        s_b1[threadIdx.x - 64] = b1[nh * TC_BN + threadIdx.x - 64];
        s_w2[threadIdx.x - 64] = w2[nh * TC_BN + threadIdx.x - 64];
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // grapes_tc_debug bit 4: CTA 0 records globaltimer stamps (MMA issuer: [0] start, [1] W resident, [2 + i] tile i
    // committed; epilogue warp 2: [32 + i] tile i drained; converter warp 6: [64 + i] its i-th k-block stored)
    auto stamp = [&](int slot) {
        if (dbg && blockIdx.x == 0 && slot < 96) {
            unsigned long long tt;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tt));
            dbg[slot] = tt;
        }
    };

    if (warp == 0) {
        // ===== TMA: W (once, or through its ring) and the raw Y tiles =====
        if (elect_one() && t_first < m_tiles) {
            if (wres) {
                mbar_arrive_expect_tx(w_bar, (uint32_t)(nkb * 2 * TC_TILE_BYTES));
                for (int kb = 0; kb < nkb; ++kb) {
                    tma_load_2d(w_smem + kb * 2 * TC_TILE_BYTES, &tmB_hi, w_bar, kb * TC_BK, nh * TC_BN);
                    tma_load_2d(w_smem + kb * 2 * TC_TILE_BYTES + TC_TILE_BYTES, &tmB_lo, w_bar, kb * TC_BK, nh * TC_BN);
                }
            }
            int ys = 0; uint32_t yphase = 0;
            int stage = 0; uint32_t phase = 0;
            for (int t = t_first; t < m_tiles; t += t_step) {
                for (int kb = 0; kb < nkb; ++kb) {
                    mbar_wait(&yempty_bar[ys], yphase ^ 1);
                    mbar_arrive_expect_tx(&yfull_bar[ys], (uint32_t)TC_TILE_BYTES);
                    tma_load_2d(y_ring + ys * TC_TILE_BYTES, &tmA, &yfull_bar[ys], kb * TC_BK, t * TC_BM);
                    if (++ys == ystages) { ys = 0; yphase ^= 1; }
                    if (!wres) {
                        mbar_wait(&bempty_bar[stage], phase ^ 1);
                        uint8_t* st = w_smem + stage * 2 * TC_TILE_BYTES;
                        mbar_arrive_expect_tx(&bfull_bar[stage], (uint32_t)(2 * TC_TILE_BYTES));
                        tma_load_2d(st, &tmB_hi, &bfull_bar[stage], kb * TC_BK, nh * TC_BN);
                        tma_load_2d(st + TC_TILE_BYTES, &tmB_lo, &bfull_bar[stage], kb * TC_BK, nh * TC_BN);
                        if (++stage == bstages) { stage = 0; phase ^= 1; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (elect_one()) {
            const uint32_t idesc = make_idesc_tf32(TC_BM, TC_BN);
            int slot = 0; uint32_t sphase = 0;
            int bst = 0; uint32_t bphase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            stamp(0);
            if (wres && t_first < m_tiles) { mbar_wait(w_bar, 0); tc_fence_after(); }
            stamp(1);
            int tile_no = 0;
            const uint32_t wa = smem_u32(w_smem);
            for (int t = t_first; t < m_tiles; t += t_step) {
                for (int kc = 0; kc < nkb; kc += TC_CHUNK_KB) {          // the tensor core adds with truncation: keep chains short
                    mbar_wait(&tempty_bar[acc], acc_phase ^ 1);          // epilogue has drained this accumulator
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + (uint32_t)(acc * TC_BN);
                    const int kend = min(nkb, kc + TC_CHUNK_KB);
                    for (int kb = kc; kb < kend; ++kb) {
                        mbar_wait(&conv_bar[slot], sphase);               // (hi, lo) of this k-block are in the TMEM slot
                        if (!wres) mbar_wait(&bfull_bar[bst], bphase);
                        tc_fence_after();
                        const uint32_t a_hi = tmem_base + a_col0 + (uint32_t)(slot * 64);
                        const uint32_t a_lo = a_hi + 32u;
                        const uint32_t sb = wa + (uint32_t)((wres ? kb : bst) * 2 * TC_TILE_BYTES);
                        const uint64_t b_hi = make_kmajor_sw128_desc(sb);
                        const uint64_t b_lo = make_kmajor_sw128_desc(sb + TC_TILE_BYTES);
                        const int nks = min(TC_BK / 8, (K - kb * TC_BK + 7) / 8);     // the last k-block may be partly padding
#pragma unroll
                        for (int ks = 0; ks < TC_BK / 8; ++ks) {
                            if (ks >= nks) break;
                            const uint64_t adv = (uint64_t)((ks * 32) >> 4);      // +32 bytes per K=8 slice inside the swizzle row
                            const uint32_t ac = (uint32_t)(ks * 8);               // +8 TMEM columns per K=8 slice
                            umma_tf32_ts(d_tmem, a_lo + ac, b_hi + adv, idesc, ((kb - kc) | ks) ? 1u : 0u);   // small terms first
                            umma_tf32_ts(d_tmem, a_hi + ac, b_lo + adv, idesc, 1u);
                            umma_tf32_ts(d_tmem, a_hi + ac, b_hi + adv, idesc, 1u);
                        }
                        umma_commit(&aempty_bar[slot]);                   // TMEM slot free once these MMAs retire
                        if (++slot == aslots) { slot = 0; sphase ^= 1; }
                        if (!wres) {
                            umma_commit(&bempty_bar[bst]);
                            if (++bst == bstages) { bst = 0; bphase ^= 1; }
                        }
                    }
                    umma_commit(&tfull_bar[acc]);                         // chunk accumulator complete -> epilogue
                    if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                }
                stamp(2 + tile_no++);
            }
        }
    } else if (warp < 6) {
        // ===== epilogue (warps 2..5): TMEM lane quarter = warp % 4.  What the timeline of the first forms showed: the
        // epilogue, not the tensor pipe, set the pace (3 us per tile against 1.3 us of MMA).  Its costs, in order: the
        // ballot / compare / select chain of the relu mask through ONE predicate and ONE register (32 dependent steps per
        // chunk) -> the row's mask word is built locally and the 32 x 32 bits are transposed across the warp with five
        // shuffles; bias / weight loads exposed per column -> float4 loads from shared memory; one accumulator chunk
        // loaded from TMEM at a time -> two in flight =====
        const int q = warp & 3;
        int acc = 0; uint32_t acc_phase = 0;
        int tile_no = 0;
        const uint32_t lane_base = tmem_base + ((uint32_t)(q * 32) << 16);
        for (int t = t_first; t < m_tiles; t += t_step) {
            const int mt = t;
            const int row = mt * TC_BM + q * 32 + lane;
            float zs0 = 0.f, zs1 = 0.f, zs2 = 0.f, zs3 = 0.f;     // four independent chains, combined in a fixed order
            uint32_t mbits[4] = {0u, 0u, 0u, 0u};
            for (int kc = 0; kc < nkb; kc += TC_CHUNK_KB) {
                const bool first_chunk = (kc == 0), last_chunk = (kc + TC_CHUNK_KB >= nkb);
                mbar_wait(&tfull_bar[acc], acc_phase);
                tc_fence_after();
#pragma unroll
                for (int cp = 0; cp < 2; ++cp) {                          // two 32-column chunks per round
                    uint32_t v[2][32];
                    tmem_ld_32x32_nowait(lane_base + (uint32_t)(acc * TC_BN + cp * 64), v[0]);
                    tmem_ld_32x32_nowait(lane_base + (uint32_t)(acc * TC_BN + cp * 64 + 32), v[1]);
                    tmem_wait_ld();
                    if (LONGK) {
#pragma unroll
                        for (int hh = 0; hh < 2; ++hh) {
                            const int ch = cp * 2 + hh;
                            if (!first_chunk) {                           // fp32 master += chunk (round to nearest)
                                uint32_t m[32];
                                tmem_ld_32x32(lane_base + (uint32_t)(2 * TC_BN + ch * 32), m);
#pragma unroll
                                for (int c = 0; c < 32; ++c)
                                    v[hh][c] = __float_as_uint(__uint_as_float(v[hh][c]) + __uint_as_float(m[c]));
                            }
                            if (!last_chunk) tmem_st_32x32(lane_base + (uint32_t)(2 * TC_BN + ch * 32), v[hh]);
                        }
                        if (!last_chunk) continue;
                    }
#pragma unroll
                    for (int hh = 0; hh < 2; ++hh) {
                        const int ch = cp * 2 + hh;
                        uint32_t rowbits = 0u;
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const float4 bb = reinterpret_cast<const float4*>(s_b1)[ch * 8 + i];
                            const float4 ww = reinterpret_cast<const float4*>(s_w2)[ch * 8 + i];
                            const float p0 = __uint_as_float(v[hh][4 * i]) + bb.x;
                            const float p1 = __uint_as_float(v[hh][4 * i + 1]) + bb.y;
                            const float p2 = __uint_as_float(v[hh][4 * i + 2]) + bb.z;
                            const float p3 = __uint_as_float(v[hh][4 * i + 3]) + bb.w;
                            zs0 = fmaf(fmaxf(p0, 0.f), ww.x, zs0);
                            zs1 = fmaf(fmaxf(p1, 0.f), ww.y, zs1);
                            zs2 = fmaf(fmaxf(p2, 0.f), ww.z, zs2);
                            zs3 = fmaf(fmaxf(p3, 0.f), ww.w, zs3);
                            // dense-layer mode (grapes_gemm_bias_relu_tc): the hidden activations themselves, 16 bytes
                            // of the thread's row at a time (a thread covers whole 128-byte lines of its row)
                            if (DENSE && hout && row < n)
                                *reinterpret_cast<float4*>(hout + (size_t)row * ldh + nh * TC_BN + ch * 32 + 4 * i) =
                                    make_float4(fmaxf(p0, 0.f), fmaxf(p1, 0.f), fmaxf(p2, 0.f), fmaxf(p3, 0.f));
                            rowbits |= (p0 > 0.f ? 1u : 0u) << (4 * i) | (p1 > 0.f ? 1u : 0u) << (4 * i + 1) |
                                       (p2 > 0.f ? 1u : 0u) << (4 * i + 2) | (p3 > 0.f ? 1u : 0u) << (4 * i + 3);
                        }
                        // lane r holds its row's 32 relu bits; the backward wants, per column, the word over the 32 rows.
                        // Rows behind n give junk bits: the backward multiplies them by dz = 0.
                        if (maskT) mbits[ch] = warp_bit_transpose(rowbits, lane);
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty_bar[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
            if ((!DENSE || zpart) && row < n) {                   // two partial rows per half: (chains 0, 1) and (chains 2, 3)
                zpart[(size_t)(nh * 2) * cap_n + row] = zs0 + zs1;
                zpart[(size_t)(nh * 2 + 1) * cap_n + row] = zs2 + zs3;
            }
            if (maskT) {
                // maskT[(row group of 32)][D]: bit r of word (g, d) = relu'(pre[32 g + r, d])
                uint32_t* dst = maskT + (size_t)(mt * 4 + q) * D + nh * TC_BN;
#pragma unroll
                for (int ch = 0; ch < 4; ++ch) dst[ch * 32 + lane] = mbits[ch];
            }
            if (warp == 2 && lane == 0) stamp(32 + tile_no);
            ++tile_no;
        }
    } else {
        // ===== converters (warps 6..13): raw Y tile in shared memory -> registers -> (hi, lo) in the TMEM slot.
        // Two groups of four warps (one per TMEM lane quarter) take the k-blocks ALTERNATELY: one k-block costs a warp a
        // chain of latencies (barrier, shared-memory load, tcgen05.st + wait, fence, arrive: ~900 cycles) that is longer
        // than the 786 cycles its MMAs take -- with every warp on every k-block the converters set the pace =====
        const int q = warp & 3;                                       // TMEM lane quarter this warp may touch
        const int grp = (warp - 6) >> 2;                              // k-blocks it == grp (mod 2)
        const int r_in = q * 32 + lane;                               // tile row == TMEM lane
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16) + a_col0;
        int it = 0;                                                   // running k-block count of this CTA
        for (int t = t_first; t < m_tiles; t += t_step) {
            for (int kb = 0; kb < nkb; ++kb, ++it) {
                if ((it & 1) != grp) continue;
                const int ys = it % ystages, slot = it % aslots;
                const uint32_t yphase = (uint32_t)((it / ystages) & 1), sphase = (uint32_t)((it / aslots) & 1);
                mbar_wait(&yfull_bar[ys], yphase);
                const uint8_t* tile = y_ring + ys * TC_TILE_BYTES + r_in * 128;
                float4 cur[8];
#pragma unroll
                for (int i = 0; i < 8; ++i)                            // SWIZZLE_128B: 16-byte chunk index ^ (row % 8)
                    cur[i] = *reinterpret_cast<const float4*>(tile + ((i ^ (r_in & 7)) << 4));
                // The TMA refills the slot through the async proxy as soon as yempty completes, so these generic-proxy
                // reads must be performed first: the proxy fence (MEMBAR + FENCE.VIEW.ASYNC in SASS) holds the arrive
                // until they have returned.  Without it the arrive waited on no load: when the TMA was parked on yempty
                // (W resident, the Y ring full behind a slow epilogue) and the loads queued behind the epilogue's global
                // stores, some 16-byte chunks were read from the NEXT fill of the slot, the k-block `ystages` later.
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(&yempty_bar[ys]);          // the tile is in registers: the slot may be refilled
                uint32_t hi[32], lo[32];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float x[4] = {cur[i].x, cur[i].y, cur[i].z, cur[i].w};
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const float h = tf32_rna_f(x[c]);
                        hi[4 * i + c] = __float_as_uint(h);
                        lo[4 * i + c] = __float_as_uint(x[c] - h);    // exact; the tensor core drops its 13 low bits (2^-21 of x)
                    }
                }
                mbar_wait(&aempty_bar[slot], sphase ^ 1);             // the MMAs that read this slot have retired
                tc_fence_after();
                tmem_st_32x32_nowait(lane_addr + (uint32_t)(slot * 64), hi);      // both stores in flight, ONE wait
                tmem_st_32x32_nowait(lane_addr + (uint32_t)(slot * 64 + 32), lo);
                tmem_wait_st();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&conv_bar[slot]);
                if (warp == 6 && lane == 0) stamp(64 + (it >> 1));
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------
// backward kernel:  S[d, k] = sum_r relu'(pre[r, d]) * dz[r] * Y[r, k]        (k < N; Y[:, K] == 1)
//
// from which   dW1[d,k] = w2[d] S[d,k],   db1[d] = w2[d] S[d,K],   dw2[d] = sum_k W1[d,k] S[d,k] + b1[d] S[d,K]
// (relu(pre) = pre * relu'(pre), so no hidden activation and no dpre matrix is ever stored).
//
// The reduction runs over rows r, split across the persistent CTAs in blocks of 32 rows:
//   A' (M = d, K-major)   built IN the kernel by 4 expander warps from the relu mask BITS the forward emitted
//                         and the 3xTF32 split of dz:  A'_hi[d,r] = bit ? tf32(dz[r]) : 0,  A'_lo likewise
//                         (generic-proxy st.shared in the SWIZZLE_128B pattern + fence.proxy.async)
//   B' (N = k, MN-major)  the aggregated features Y_hi / Y_lo, TMA boxes of 32 rows x 32 columns
//                         (SWIZZLE_128B_ATOM_32B: the only legal MN-major layout for 32-bit operands)
//   D                     [D x N] fp32 in TMEM (NH halves x N columns), accumulated over all the CTA's rows
// ------------------------------------------------------------------------------------------------
#define TCB_ROWS 32                                  // rows per k-block (one 128-byte swizzle row of A')
#define TCB_A_TILE (128 * 128)                       // 128 d x 32 r fp32 = 16 KB
#define TCB_B_TILE (TCB_ROWS * 128)                  // 32 r x 32 k fp32 = 4 KB

// MN-major 32-bit (tf32) operands have exactly one legal shared-memory layout on sm_100: SWIZZLE_128B with a
// 32-byte swizzle atom (layout type 1 = SWIZZLE_128B_BASE32B; TMA mode CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B):
// rows of 128 bytes (32 MN elements), the 32-byte chunk index XORed with (row % 4), K atom = 4 rows (512 B).
__device__ __forceinline__ uint64_t make_mnmajor_sw128_32b_desc(uint32_t smem_addr, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFFu);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;     // stride between 32-column blocks of the MN dimension
    d |= (uint64_t)(512u >> 4) << 32;                      // stride between 4-row atoms of the K dimension
    d |= (uint64_t)1u << 46;
    d |= (uint64_t)1u << 61;
    return d;
}
__device__ __forceinline__ float tf32_rna(float x) { return grapes_tf32_rna(x); }

// v2 of the contraction: the relu mask is 0/1 -- EXACT in tf32 -- so it is the single A operand, and dz is folded into
// the other side: B''[r, k] = fl(dz[r] * Y[r, k]) split into (hi, lo) by the expander warps in shared memory.
//   S = mask^T B''_hi + mask^T B''_lo   ->  with [B''_hi | B''_lo] stored back to back as ONE MN-major operand of
//   N = 2 * NB * 32 columns this is ONE tcgen05.mma per 8-row slice and 128-unit half (instead of three), reading
//   12 KB of operands instead of 24 KB (the kernel is fed at the shared-memory read limit).  The two accumulator halves
//   are added in the epilogue.  Columns [col0, col0 + NB*32) of Y per CTA (NB <= 4): wider Y = several column chunks (blockIdx.y).
// The tensor core adds into its fp32 accumulator with truncation, so a long chain drifts when the terms do not cancel
// (nonnegative features, dz of one sign: 1.9e-4 of the magnitude after 1563 groups in one chain; B200 at 1000 W).
// Both backward kernels therefore cut every CTA's chain each TCBS_FLUSH groups (4 MMAs per group and accumulator; 96
// groups drift 4.5e-6 in the same test): the epilogue stores each interval to its own partial slab
// part[flush][cta][D][N], zero-fills the slabs past the CTA's last interval (the host sizes nflush for cap_n), and
// k_l1_bwd_finalize adds the slabs rounding to nearest.
#define TCBS_FLUSH 96
#define TCB_THREADS 320          // TMA, MMA, 4 mask-expander (+ epilogue) warps, 4 operand-scaling warps
// (register cap: with the interval epilogue inside the expanders' loop ptxas takes 126 registers instead of 85, which
//  leaves less of the register file to the kernels that share the SM in the training step: the Cora-shaped step measured
//  2 % slower on a B200 at 1000 W, with this kernel's own time unchanged.  Launched with TCB_THREADS threads.)
__global__ void __maxnreg__(88) k_l1_bwd_tc(
    const __grid_constant__ CUtensorMap tmY, const __grid_constant__ CUtensorMap tmY_lo, int presplit, int col0,
    const int* __restrict__ n_dev, int cap_n, int NH, int NB, int stages, const uint32_t* __restrict__ maskT, int D,
    const float* __restrict__ dz, float* __restrict__ part, int debug, int ncols, long long chunk_stride, int nflush) {
    pdl_begin();
    // blockIdx.y = column chunk of Y (128 columns each): all chunks of a wide Y (Cora 1437, Reddit 606 columns) run in ONE
    // launch next to each other instead of one launch per chunk; every chunk has its own slab of the partial buffer
    col0 += (int)blockIdx.y * 128;
    NB = min(NB, (ncols - col0 + 31) / 32);
    part += (size_t)blockIdx.y * (size_t)chunk_stride;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int a_bytes = NH * TCB_A_TILE;             // mask tiles of all halves
    const int b_bytes = NB * TCB_B_TILE;             // one of (hi | lo)
    const int stage_bytes = a_bytes + 2 * b_bytes;
    uint64_t* bars = (uint64_t*)(smem + stages * stage_bytes);
    uint64_t* full_bar = bars;                       // [stages] 4 mask-expander + 4 scaling warps -> MMA
    uint64_t* empty_bar = bars + 4;                  // [stages] MMA -> TMA + expanders
    uint64_t* tma_bar = bars + 8;                    // [stages] TMA (Y tile) -> expanders
    uint64_t* done_bar = bars + 12;                  // MMAs of a flush interval retired -> epilogue
    uint32_t* tmem_slot = (uint32_t*)(bars + 13);
    uint64_t* drained_bar = bars + 14;               // epilogue -> MMA: accumulators may be overwritten

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = min(*n_dev, cap_n);
    const int groups = (n + TCB_ROWS - 1) / TCB_ROWS;
    const int N = NB * 32;                           // S columns of this launch; accumulator holds 2N per half
    const int my_groups = (groups > (int)blockIdx.x) ? (groups - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    const int my_flushes = (my_groups + TCBS_FLUSH - 1) / TCBS_FLUSH;     // <= nflush (sized for cap_n on the host)

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmY);
        if (presplit) tma_prefetch_desc(&tmY_lo);
        for (int s = 0; s < stages; ++s) { mbar_init(&full_bar[s], 8); mbar_init(&empty_bar[s], 1); mbar_init(&tma_bar[s], 1); }
        mbar_init(done_bar, 1);
        mbar_init(drained_bar, 4);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        if (elect_one()) {
            int stage = 0; uint32_t phase = 0;
            for (int g = blockIdx.x; g < groups; g += gridDim.x) {
                mbar_wait(&empty_bar[stage], phase ^ 1);
                uint8_t* st = smem + stage * stage_bytes + a_bytes;
                mbar_arrive_expect_tx(&tma_bar[stage], (uint32_t)((presplit ? 2 : 1) * b_bytes));
                for (int nb = 0; nb < NB; ++nb) {
                    tma_load_2d(st + nb * TCB_B_TILE, &tmY, &tma_bar[stage], col0 + nb * 32, g * TCB_ROWS);
                    if (presplit) tma_load_2d(st + b_bytes + nb * TCB_B_TILE, &tmY_lo, &tma_bar[stage], col0 + nb * 32, g * TCB_ROWS);
                }
                if (++stage == stages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        if (elect_one()) {
            // A: K-major, B: MN-major (bit 16), M = 128, N = 2 * NB * 32 (hi block columns, then lo block columns)
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (1u << 16) | ((uint32_t)((2 * N) >> 3) << 17) |
                                   ((uint32_t)(128 >> 4) << 24);
            int stage = 0; uint32_t phase = 0;
            for (int it = 0; it < my_groups; ++it) {
                const int in_flush = it % TCBS_FLUSH;
                if (in_flush == 0 && it > 0) {
                    umma_commit(done_bar);                      // interval done: the epilogue stores it to its slab
                    mbar_wait(drained_bar, (uint32_t)((it / TCBS_FLUSH - 1) & 1));
                    tc_fence_after();
                }
                mbar_wait(&full_bar[stage], phase);
                tc_fence_after();
                const uint32_t sa = smem_u32(smem + stage * stage_bytes);
                const uint64_t bd = make_mnmajor_sw128_32b_desc(sa + a_bytes, TCB_B_TILE);
                for (int h = 0; h < NH; ++h) {
                    const uint64_t ad = make_kmajor_sw128_desc(sa + h * TCB_A_TILE);
                    const uint32_t d_tmem = tmem_base + (uint32_t)(h * 2 * N);
#pragma unroll
                    for (int ks = 0; ks < TCB_ROWS / 8; ++ks) {
                        const uint64_t adv_a = (uint64_t)((ks * 32) >> 4);       // 8 r = 32 bytes along the swizzle row
                        const uint64_t adv_b = (uint64_t)((ks * 1024) >> 4);     // 8 rows of 128 bytes
                        umma_tf32(d_tmem, ad + adv_a, bd + adv_b, idesc, (in_flush == 0 && ks == 0) ? 0u : 1u);
                    }
                }
                umma_commit(&empty_bar[stage]);
                if (++stage == stages) { stage = 0; phase ^= 1; }
            }
            umma_commit(done_bar);
        }
    } else if (warp >= 6) {
        // ===== scaling warps (6..9): B'' = dz * Y split into (hi, lo), in place on the tile(s) the TMA delivered.
        //       MN-major tiles: every 128-byte line holds one row r of a 32-column block, so the row of 16-byte chunk
        //       q is (q / 8) % 32 whatever the swizzle. =====
        const int e = (warp - 6) * 32 + lane;
        int stage = 0; uint32_t phase = 0;
        float dz_nx = 0.f;
        if ((int)blockIdx.x < groups) { const int r0 = blockIdx.x * TCB_ROWS + lane; dz_nx = (r0 < n) ? dz[r0] : 0.f; }
        for (int g = blockIdx.x; g < groups; g += gridDim.x) {
            const float dzr = dz_nx;
            const int gn = g + gridDim.x;
            if (gn < groups) { const int rn = gn * TCB_ROWS + lane; dz_nx = (rn < n) ? dz[rn] : 0.f; }
            uint8_t* bh = smem + stage * stage_bytes + a_bytes;
            mbar_wait(&tma_bar[stage], phase);
            const int n16 = b_bytes >> 4;
            for (int q = e; q < n16; q += 128) {
                const float sc = __shfl_sync(GRAPES_FULL_MASK, dzr, (q >> 3) & 31);
                float4 v = *reinterpret_cast<const float4*>(bh + (size_t)q * 16);
                if (presplit) {
                    const float4 v2 = *reinterpret_cast<const float4*>(bh + b_bytes + (size_t)q * 16);
                    v.x += v2.x; v.y += v2.y; v.z += v2.z; v.w += v2.w;
                }
                v.x *= sc; v.y *= sc; v.z *= sc; v.w *= sc;
                float4 hh, ll;
                hh.x = tf32_rna(v.x); hh.y = tf32_rna(v.y); hh.z = tf32_rna(v.z); hh.w = tf32_rna(v.w);
                ll.x = tf32_rna(v.x - hh.x); ll.y = tf32_rna(v.y - hh.y); ll.z = tf32_rna(v.z - hh.z); ll.w = tf32_rna(v.w - hh.w);
                *reinterpret_cast<float4*>(bh + (size_t)q * 16) = hh;
                *reinterpret_cast<float4*>(bh + b_bytes + (size_t)q * 16) = ll;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(&full_bar[stage]);
            if (++stage == stages) { stage = 0; phase ^= 1; }
        }
    } else {
        // ===== mask expanders (warps 2..5), then epilogue =====
        const int e = (warp - 2) * 32 + lane;            // d index inside a half
        int stage = 0; uint32_t phase = 0;
        // software pipeline: the mask words of the NEXT group are loaded while this group is expanded
        uint32_t words_nx[4] = {0u, 0u, 0u, 0u};
        if ((int)blockIdx.x < groups) {
#pragma unroll
            for (int h = 0; h < 4; ++h) if (h < NH) words_nx[h] = maskT[(size_t)blockIdx.x * D + h * 128 + e];
        }
        // epilogue of flush interval fl: its partial S -> part[fl][cta][NH*128][N]  (hi-part + lo-part accumulators)
        const int q = warp & 3;
        auto slab_row = [&](int fl, int h) {
            return part + (((size_t)fl * gridDim.x + blockIdx.x) * NH * 128 + (size_t)(h * 128 + q * 32 + lane)) * N;
        };
        auto drain = [&](int fl) {
            mbar_wait(done_bar, (uint32_t)(fl & 1));
            tc_fence_after();
            for (int h = 0; h < NH; ++h) {
                float* row = slab_row(fl, h);
                for (int ch = 0; ch < NB; ++ch) {
                    uint32_t v[32], v2[32];
                    tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(h * 2 * N + ch * 32), v);
                    tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(h * 2 * N + N + ch * 32), v2);
#pragma unroll
                    for (int c = 0; c < 32; c += 4)
                        *reinterpret_cast<float4*>(row + ch * 32 + c) =
                            make_float4(__uint_as_float(v[c]) + __uint_as_float(v2[c]),
                                        __uint_as_float(v[c + 1]) + __uint_as_float(v2[c + 1]),
                                        __uint_as_float(v[c + 2]) + __uint_as_float(v2[c + 2]),
                                        __uint_as_float(v[c + 3]) + __uint_as_float(v2[c + 3]));
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(drained_bar);
        };
        int g = blockIdx.x;
        for (int fl = 0; fl < my_flushes; ++fl) {
          const int g_end = min(groups, g + TCBS_FLUSH * (int)gridDim.x);   // the groups of interval fl
          for (; g < g_end; g += gridDim.x) {
            uint32_t words[4];
#pragma unroll
            for (int h = 0; h < 4; ++h) words[h] = words_nx[h];
            const int gn = g + gridDim.x;
            if (gn < groups) {
#pragma unroll
                for (int h = 0; h < 4; ++h) if (h < NH) words_nx[h] = maskT[(size_t)gn * D + h * 128 + e];
            }
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* st = smem + stage * stage_bytes;
            // A: mask bits of hidden unit e (row) over the group's 32 rows (K), 1.0 / 0.0
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const int off = e * 128 + ((c ^ (e & 7)) << 4);          // SWIZZLE_128B: 16-byte chunk index ^ (row % 8)
#pragma unroll
                for (int h = 0; h < 4; ++h) {
                    if (h >= NH) break;
                    const uint32_t w = words[h] >> (c * 4);
                    float4 a;
                    a.x = (w & 1u) ? 1.f : 0.f; a.y = (w & 2u) ? 1.f : 0.f; a.z = (w & 4u) ? 1.f : 0.f; a.w = (w & 8u) ? 1.f : 0.f;
                    if (debug & 1) a = make_float4(1.f, 1.f, 1.f, 1.f);
                    *reinterpret_cast<float4*>(st + h * TCB_A_TILE + off) = a;
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the tensor core
            __syncwarp();
            if (lane == 0) mbar_arrive(&full_bar[stage]);
            if (++stage == stages) { stage = 0; phase ^= 1; }
          }
          drain(fl);
        }
        // flush slabs this CTA did not reach (fewer rows than the capacity the host sized for): zeros
        for (int fl = my_flushes; fl < nflush; ++fl)
            for (int h = 0; h < NH; ++h) {
                float* row = slab_row(fl, h);
                for (int c = 0; c < N; c += 4) *reinterpret_cast<float4*>(row + c) = make_float4(0.f, 0.f, 0.f, 0.f);
            }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------
// backward kernel, scaled-feature operand in TENSOR MEMORY ("TS" form of the contraction, transposed):
//
//     S^T[k, d] = sum_r B''[r, k] * mask[r, d],      B''[r, k] = fl(dz[r] * Y[r, k])  split into (hi, lo)
//
// k_l1_bwd_tc stages both operands in shared memory: per 32-row group the TMA writes the Y tile (16 KB), four warps read
// it, scale, split and write it back twice (48 KB), four warps write the mask tiles (32 KB) and the MMAs read 96 KB --
// 192 KB through a 128 B/clk pipe for 512 tensor-core cycles of work.  Here the Y tile is read from shared memory once:
//   warp 0       TMA: Y tiles (32 rows x 32-column blocks, no swizzle -- no MMA reads them) through a ring
//   warps 6..9   read the tile TRANSPOSED (thread = column k of Y = TMEM lane; for a fixed row the 32 lanes of a warp
//                read one 128-byte line: conflict free), scale by dz, split, and store (hi | lo) into a ring of TMEM
//                slots: the A operand [M = k, K = r] of the MMA lives in tensor memory.
//   warps 2..5   expand the relu-mask bits of the CTA's 128 hidden units into the B operand [N = d, K = r] (1.0 / 0.0,
//                exact in tf32) in shared memory; afterwards they are the epilogue.
//   warp 1       MMA issuer: per 8-row slice one M128 N128 K8 MMA for the hi part and one for the lo part, into two
//                accumulators (added in the epilogue, as in k_l1_bwd_tc).
// Shared-memory traffic per group: 80 KB (Y 16 + 16, mask 16 + 32) instead of 192 KB.  A CTA owns ONE 128-unit half of the hidden layer
// (blockIdx.x % NH) and a strided share of the row groups; blockIdx.y = 128-column chunk of Y.
// Partials: part[chunk][cta / NH][D][N] -- the layout k_l1_bwd_finalize already reads.
// TMEM columns: [0,128) hi accumulator, [128,256) lo accumulator, [256,512) A ring: 4 slots of (hi 32 | lo 32).
// ------------------------------------------------------------------------------------------------
#define TCBS_THREADS 448            // TMA, MMA, 4 mask-expander (+ epilogue) warps, 8 converter warps (two groups)
#define TCBS_STAGES 4
__global__ void __launch_bounds__(TCBS_THREADS, 1) k_l1_bwd_ts(
    const __grid_constant__ CUtensorMap tmY, int ncols, const int* __restrict__ n_dev, int cap_n, int NH,
    const uint32_t* __restrict__ maskT, int D, const float* __restrict__ dz, float* __restrict__ part,
    long long chunk_stride, int ystages, int nflush, unsigned long long* dbg) {
    pdl_begin();
    const int col0 = (int)blockIdx.y * 128;
    const int N = min(4, (ncols - col0 + 31) / 32) * 32;            // S columns of this chunk (a multiple of 32)
    part += (size_t)blockIdx.y * (size_t)chunk_stride;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t* y_ring = smem + TCBS_STAGES * TCB_A_TILE;                // [ystages][4 blocks][32 rows][32 floats]
    uint64_t* bars = (uint64_t*)(y_ring + (size_t)ystages * 4 * TCB_B_TILE);
    uint64_t* full_bar = bars;                       // [4] 4 mask-expander + 4 converter warps -> MMA
    uint64_t* empty_bar = bars + 4;                  // [4] MMA -> producers
    uint64_t* done_bar = bars + 8;                   // MMAs of a flush interval retired -> epilogue
    uint32_t* tmem_slot = (uint32_t*)(bars + 9);
    uint64_t* yfull_bar = bars + 10;                 // [8] TMA -> converters
    uint64_t* yempty_bar = bars + 18;                // [8] converters -> TMA
    uint64_t* drained_bar = bars + 26;               // epilogue -> MMA: accumulators may be overwritten

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n = min(*n_dev, cap_n);
    const int groups = (n + TCB_ROWS - 1) / TCB_ROWS;
    const int h = (int)blockIdx.x % NH;              // hidden half of this CTA
    const int pp = (int)blockIdx.x / NH, per_half = (int)gridDim.x / NH;
    const int g_first = pp, g_step = per_half;
    const int my_groups = (groups > g_first) ? (groups - 1 - g_first) / g_step + 1 : 0;
    const int my_flushes = (my_groups + TCBS_FLUSH - 1) / TCBS_FLUSH;     // <= nflush (sized for cap_n on the host)

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmY);
        for (int s = 0; s < TCBS_STAGES; ++s) { mbar_init(&full_bar[s], 8); mbar_init(&empty_bar[s], 1); }
        for (int s = 0; s < 8; ++s) { mbar_init(&yfull_bar[s], 1); mbar_init(&yempty_bar[s], 4); }
        mbar_init(done_bar, 1);
        mbar_init(drained_bar, 4);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(tmem_slot, 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    auto stamp = [&](int slot) {
        if (dbg && blockIdx.x == 0 && blockIdx.y == 0 && slot < 96) {
            unsigned long long tt;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tt));
            dbg[slot] = tt;
        }
    };

    const int NBk = N / 32;                                           // 32-column blocks of this chunk
    if (warp == 0) {
        if (elect_one()) {
            int ys = 0; uint32_t yphase = 0;
            for (int g = g_first; g < groups; g += g_step) {
                mbar_wait(&yempty_bar[ys], yphase ^ 1);
                mbar_arrive_expect_tx(&yfull_bar[ys], (uint32_t)(NBk * TCB_B_TILE));
                for (int nb = 0; nb < NBk; ++nb)
                    tma_load_2d(y_ring + (size_t)ys * 4 * TCB_B_TILE + nb * TCB_B_TILE, &tmY, &yfull_bar[ys], col0 + nb * 32,
                                g * TCB_ROWS);
                if (++ys == ystages) { ys = 0; yphase ^= 1; }
            }
        }
    } else if (warp == 1) {
        if (elect_one()) {
            const uint32_t idesc = make_idesc_tf32(128, 128);
            int stage = 0; uint32_t phase = 0;
            stamp(0);
            for (int it = 0; it < my_groups; ++it) {
                const int in_flush = it % TCBS_FLUSH;
                if (in_flush == 0 && it > 0) {
                    // the tensor core adds into its fp32 accumulator with truncation: chains are kept short (TCBS_FLUSH).
                    // The epilogue stores the interval's sums to their own partial slab; the finalize adds the slabs
                    umma_commit(done_bar);
                    mbar_wait(drained_bar, (uint32_t)((it / TCBS_FLUSH - 1) & 1));
                    tc_fence_after();
                }
                mbar_wait(&full_bar[stage], phase);
                tc_fence_after();
                const uint64_t bd = make_kmajor_sw128_desc(smem_u32(smem + stage * TCB_A_TILE));
                const uint32_t a_hi = tmem_base + 256u + (uint32_t)(stage * 64);
#pragma unroll
                for (int ks = 0; ks < TCB_ROWS / 8; ++ks) {
                    const uint64_t adv = (uint64_t)((ks * 32) >> 4);          // 8 r = 32 bytes along the swizzle row
                    const uint32_t acc = (in_flush == 0 && ks == 0) ? 0u : 1u;
                    umma_tf32_ts(tmem_base, a_hi + (uint32_t)(ks * 8), bd + adv, idesc, acc);
                    umma_tf32_ts(tmem_base + 128u, a_hi + 32u + (uint32_t)(ks * 8), bd + adv, idesc, acc);
                }
                umma_commit(&empty_bar[stage]);
                if (++stage == TCBS_STAGES) { stage = 0; phase ^= 1; }
                if (it < 30) stamp(2 + it);
            }
            if (my_groups > 0) umma_commit(done_bar);
        }
    } else if (warp >= 6) {
        // ===== converters (warps 6..13): B''^T = (dz * Y)^T split into (hi, lo), shared memory -> registers -> TMEM.
        // Two groups of four warps (one per TMEM lane quarter) take the row groups alternately: one iteration is a chain
        // of latencies (barrier, shared-memory loads, tcgen05.st + wait, fence, arrive) longer than the group's MMAs =====
        const int q = warp & 3;                                       // TMEM lane quarter of this warp == 32-column block
        const int grp = (warp - 6) >> 2;
        const bool blk_valid = q < NBk;                               // blocks behind the chunk's columns hold nothing: zeros
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16) + 256u;
        for (int it = grp; it < my_groups; it += 2) {
            const int g = g_first + it * g_step;
            const int r0 = g * TCB_ROWS;
            const float dzr = (r0 + lane < n) ? __ldg(&dz[r0 + lane]) : 0.f;    // (issued before the wait: latency hidden)
            const int ys = it % ystages, stage = it % TCBS_STAGES;
            const uint32_t yphase = (uint32_t)((it / ystages) & 1), phase = (uint32_t)((it / TCBS_STAGES) & 1);
            mbar_wait(&yfull_bar[ys], yphase);
            const float* tile = reinterpret_cast<const float*>(y_ring + (size_t)ys * 4 * TCB_B_TILE + q * TCB_B_TILE) + lane;
            uint32_t hi[32], lo[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                // rows >= n of the last group are stale in Y: their dz is 0, and 0 * finite = 0 (Y holds finite values only)
                const float y = blk_valid ? tile[i * 32] : 0.f;
                const float v = y * __shfl_sync(GRAPES_FULL_MASK, dzr, i);
                const float hh = tf32_rna(v);
                hi[i] = __float_as_uint(hh);
                lo[i] = __float_as_uint(v - hh);                       // exact; the tensor core drops its 13 low bits
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&yempty_bar[ys]);              // tile consumed: the TMA may refill the slot
            mbar_wait(&empty_bar[stage], phase ^ 1);
            tc_fence_after();
            tmem_st_32x32_nowait(lane_addr + (uint32_t)(stage * 64), hi);      // both stores in flight, ONE wait
            tmem_st_32x32_nowait(lane_addr + (uint32_t)(stage * 64 + 32), lo);
            tmem_wait_st();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&full_bar[stage]);
            if (warp == 6 && lane == 0 && (it >> 1) < 16) stamp(64 + (it >> 1));
        }
    } else if (warp >= 2) {
        // ===== mask expanders (warps 2..5), and the epilogue of every flush interval =====
        const int e = (warp - 2) * 32 + lane;            // hidden unit inside the half: row of the B operand tile
        const int q = warp & 3;
        const int kk = q * 32 + lane;                    // epilogue: TMEM lane = column k of Y
        int stage = 0; uint32_t phase = 0;
        uint32_t word_nx = (my_groups > 0) ? maskT[(size_t)g_first * D + h * 128 + e] : 0u;
        for (int it = 0; it <= my_groups; ++it) {
            if ((it % TCBS_FLUSH == 0 && it > 0) || (it == my_groups && my_groups > 0)) {
                // epilogue of the interval that just ended: TMEM lane = column k of Y, TMEM column = hidden unit; stored
                // transposed -> part[flush][pp][h*128 + d][k]
                const int fl = (it - 1) / TCBS_FLUSH;
                float* dst = part + (((size_t)fl * per_half + pp) * D + (size_t)h * 128) * N;
                mbar_wait(done_bar, (uint32_t)(fl & 1));
                tc_fence_after();
                for (int ch = 0; ch < 4; ++ch) {
                    uint32_t v[32], v2[32];
                    tmem_ld_32x32_nowait(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(ch * 32), v);
                    tmem_ld_32x32_nowait(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(128 + ch * 32), v2);
                    tmem_wait_ld();
                    if (kk < N) {
#pragma unroll
                        for (int c = 0; c < 32; ++c)
                            dst[(size_t)(ch * 32 + c) * N + kk] = __uint_as_float(v[c]) + __uint_as_float(v2[c]);
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(drained_bar);
                if (warp == 2 && lane == 0) stamp(40 + fl);
            }
            if (it == my_groups) break;
            const int g = g_first + it * g_step;
            const uint32_t word = word_nx;
            if (it + 1 < my_groups) word_nx = maskT[(size_t)(g + g_step) * D + h * 128 + e];
            mbar_wait(&empty_bar[stage], phase ^ 1);
            uint8_t* st = smem + stage * TCB_A_TILE;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const int off = e * 128 + ((c ^ (e & 7)) << 4);          // SWIZZLE_128B: 16-byte chunk index ^ (row % 8)
                const uint32_t w = word >> (c * 4);
                float4 a4;
                a4.x = (w & 1u) ? 1.f : 0.f; a4.y = (w & 2u) ? 1.f : 0.f; a4.z = (w & 4u) ? 1.f : 0.f; a4.w = (w & 8u) ? 1.f : 0.f;
                *reinterpret_cast<float4*>(st + off) = a4;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to the tensor core
            __syncwarp();
            if (lane == 0) mbar_arrive(&full_bar[stage]);
            if (++stage == TCBS_STAGES) { stage = 0; phase ^= 1; }
        }
        // flush slabs this CTA did not reach (fewer rows than the capacity the host sized for): zeros
        for (int fl = my_flushes; fl < nflush; ++fl) {
            float* dst = part + (((size_t)fl * per_half + pp) * D + (size_t)h * 128) * N;
            if (kk < N)
                for (int d = 0; d < 128; ++d) dst[(size_t)d * N + kk] = 0.f;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, 512);
}

// Sum the per-CTA partials (fixed order) and turn S into the three gradients, accumulated (+=, times scale).
// One 1024-thread block per hidden unit d.  N/4 threads cover one partial row with float4 loads; the 1024/(N/4)
// thread groups split the partials, each thread keeping 5 independent 16-byte loads in flight, then a fixed-order
// combine through shared memory.
#define FIN_THREADS 1024
__global__ void __launch_bounds__(FIN_THREADS) k_l1_bwd_finalize(
    const float* __restrict__ part_all, int nparts, int D, int ncols, int nchunks, long long chunk_stride, int K,
    const float* __restrict__ W1, int ldw, const float* __restrict__ b1, const float* __restrict__ w2, int ones_col,
    float scale, float* __restrict__ gW1, float* __restrict__ gb1, float* __restrict__ gw2) {
    pdl_begin();
    __shared__ __align__(16) float sums[4 * FIN_THREADS];        // [groups][N], groups * N == 4096
    __shared__ float red[8];
    const int d = blockIdx.x;
    // the column chunks of Y one after the other (fixed order: gw2[d] accumulates chunk by chunk, as separate launches did)
    for (int chunk = 0; chunk < nchunks; ++chunk) {
        const int col0 = chunk * 128;
        const int N = min(4, (ncols - col0 + 31) / 32) * 32;
        const float* part = part_all + (size_t)chunk * (size_t)chunk_stride;
        const int nq = N >> 2;                                   // threads per partial row (N is a multiple of 32, <= 128)
        const int groups = FIN_THREADS / nq;
        const int pg = threadIdx.x / nq, kq = threadIdx.x % nq;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        if (pg < groups) {
            for (int p = pg; p < nparts; p += 5 * groups) {
                float4 v[5];
#pragma unroll
                for (int u = 0; u < 5; ++u) {
                    const int pp = p + u * groups;
                    v[u] = (pp < nparts) ? __ldg(reinterpret_cast<const float4*>(part + ((size_t)pp * D + d) * N) + kq)
                                         : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int u = 0; u < 5; ++u) { acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w; }
            }
            reinterpret_cast<float4*>(sums)[pg * nq + kq] = acc;
        }
        __syncthreads();
        float acc_w2 = 0.f;
        if (threadIdx.x < N) {
            const int k = col0 + threadIdx.x;                    // column of Y / W1 this chunk's column `threadIdx.x` is
            float s = 0.f;
            for (int g = 0; g < groups; ++g) s += sums[g * N + threadIdx.x];   // fixed order
            const float w2d = w2[d];
            if (k < K) {
                gW1[(size_t)d * K + k] += scale * w2d * s;
                acc_w2 = W1[(size_t)d * ldw + k] * s;
            } else if (k == ones_col) {
                gb1[d] += scale * w2d * s;
                acc_w2 = b1[d] * s;
            }
        }
        if (threadIdx.x < 256) {
            acc_w2 = warp_sum(acc_w2);
            if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc_w2;
        }
        __syncthreads();
        if (threadIdx.x == 0)
            gw2[d] += scale * (((red[0] + red[1]) + (red[2] + red[3])) + ((red[4] + red[5]) + (red[6] + red[7])));
        __syncthreads();                                         // sums / red are reused by the next chunk
    }
}

// ------------------------------------------------------------------------------------------------
// operand split: hi = tf32(x), lo = tf32(x - hi); zero padded to ld_dst columns
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float to_tf32(float x) { return grapes_tf32_rna(x); }
__global__ void __launch_bounds__(256) k_split_tf32(const float* __restrict__ src, int ld_src, int R, int K,
                                                    float* __restrict__ hi, float* __restrict__ lo, int ld_dst) {
    pdl_begin();
    const long long total = (long long)R * ld_dst;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(i / ld_dst), c = (int)(i % ld_dst);
        const float x = (c < K) ? src[(size_t)r * ld_src + c] : 0.f;
        const float h = to_tf32(x);
        hi[i] = h;
        lo[i] = to_tf32(x - h);
    }
}

// ------------------------------------------------------------------------------------------------
// host: tensor maps
// ------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (PFN_encodeTiled)p;
    }
    return fn;
}

// row-major fp32 matrix [rows x cols] with row stride ld (elements); box = 32 cols x 128 rows, SWIZZLE_128B
static int make_map(CUtensorMap* m, const float* base, int rows, int cols, int ld, int box_rows = TC_BM,
                    CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
    PFN_encodeTiled enc = get_encode_fn();
    if (!enc) { grapes_set_error("cuTensorMapEncodeTiled not available from the driver"); return GRAPES_ERR_CUDA; }
    if ((((uintptr_t)base) & 15) || (ld % 4)) { grapes_set_error("TMA operand must be 16 B aligned with ld %% 4 == 0"); return GRAPES_ERR_ARG; }
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
    cuuint32_t box[2] = {TC_BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { grapes_set_error("cuTensorMapEncodeTiled failed (%d)", (int)r); return GRAPES_ERR_CUDA; }
    return GRAPES_OK;
}

// A operand in tensor memory (k_l1_fwd_ts): raw Y tiles by TMA, split on the way into TMEM, only W staged for the MMA.
// hout != NULL: the hidden activations relu(Y W^T + b1) are written to hout[n x D] (pitch ldh); zpart / maskT optional.
static int launch_fwd_ts(grapes_ctx* ctx, const float* Y, int ldy, const int* n_dev, int cap_n, int K, const float* W_hi,
                         const float* W_lo, int ldw, int D, const float* b1, const float* w2, float* zpart, uint32_t* maskT,
                         float* hout, int ldh, void* stream) {
    CUtensorMap ma, mb_hi, mb_lo;
    int rc;
        if ((rc = make_map(&mb_hi, W_hi, D, K, ldw)) != GRAPES_OK) return rc;
        if ((rc = make_map(&mb_lo, W_lo, D, K, ldw)) != GRAPES_OK) return rc;
        const int nkb = (K + TC_BK - 1) / TC_BK, NH = D / TC_BN;
        const int m_tiles_cap = (cap_n + TC_BM - 1) / TC_BM;
        if ((rc = make_map(&ma, Y, cap_n, K, ldy)) != GRAPES_OK) return rc;
        const int tail_b = 1024 /*align slack*/ + 1536 /*barriers, bias + output weights of the half*/;
        // W half resident when it leaves room for >= 4 raw Y tiles; otherwise W streams through a 4-stage ring (and with
        // grapes_tc_debug bit 1: both forms sum in the same order, so they give the same bits).  Both instantiations take
        // the same policy.  (The dense layer once had to stream W: with W resident its CTAs read Y chunks from the next
        // fill of a ring slot; see the proxy fence in the converters of k_l1_fwd_ts.)
        const int wres = (nkb * 2 * TC_TILE_BYTES + 4 * TC_TILE_BYTES + tail_b <= 227 * 1024 && ctx->sm_count >= NH &&
                          !(g_tc_debug & 2)) ? 1 : 0;
        const int bstages = 4;
        const int nbt = wres ? nkb : bstages;
        int ystages = (227 * 1024 - tail_b - nbt * 2 * TC_TILE_BYTES) / TC_TILE_BYTES;
        if (ystages > 8) ystages = 8;
        const int smem_bytes = nbt * 2 * TC_TILE_BYTES + ystages * TC_TILE_BYTES + tail_b;
        int per_half = ctx->sm_count / NH;
        if (per_half > m_tiles_cap) per_half = m_tiles_cap;
        if (per_half < 1) per_half = 1;
        static int attr_ts[64] = {0};
        int& have = attr_ts[ctx->device & 63];
        if (smem_bytes > have) {
            GRAPES_CUDA_OK(cudaFuncSetAttribute(k_l1_fwd_ts<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
            GRAPES_CUDA_OK(cudaFuncSetAttribute(k_l1_fwd_ts<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
            GRAPES_CUDA_OK(cudaFuncSetAttribute(k_l1_fwd_ts<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
            GRAPES_CUDA_OK(cudaFuncSetAttribute(k_l1_fwd_ts<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
            have = smem_bytes;
        }
        unsigned long long* dbg = (g_tc_debug & 16) ? reinterpret_cast<unsigned long long*>(ctx->partials) : nullptr;
        const dim3 grid(per_half * NH);
        cudaStream_t cs = (cudaStream_t)stream;
        // the sampler-head form (DENSE = false) and the dense-layer form (hidden activations written out,
        // grapes_gemm_bias_relu_tc; tests/test_gpu_dense_tc.py) are separate instantiations
#define TS_ARGS ma, mb_hi, mb_lo, n_dev, cap_n, K, D, wres, bstages, ystages, b1, w2, zpart, maskT, hout, ldh, dbg
        if (hout) {
            if (nkb > TC_CHUNK_KB) pdl((k_l1_fwd_ts<true, true>), grid, TCS_THREADS, smem_bytes, cs)(TS_ARGS);
            else pdl((k_l1_fwd_ts<false, true>), grid, TCS_THREADS, smem_bytes, cs)(TS_ARGS);
        } else {
            if (nkb > TC_CHUNK_KB) pdl((k_l1_fwd_ts<true, false>), grid, TCS_THREADS, smem_bytes, cs)(TS_ARGS);
            else pdl((k_l1_fwd_ts<false, false>), grid, TCS_THREADS, smem_bytes, cs)(TS_ARGS);
        }
#undef TS_ARGS
        grapes_count_launches(1);
        GRAPES_LAUNCH_OK();
        return GRAPES_OK;
}

extern "C" {

int grapes_tc_debug(int flags) { g_tc_debug = flags; return 0; }
// debugging aid (scripts/trace_fwd_ts.py): device address of the ctx's split-K partial buffer, where grapes_tc_debug bit 4
// parks the phase stamps of k_l1_fwd_ts
int64_t grapes_debug_partials(grapes_ctx* ctx) { return ctx ? (int64_t)(uintptr_t)ctx->partials : 0; }
int64_t grapes_debug_partials_bytes(grapes_ctx* ctx) { return ctx ? (int64_t)ctx->partials_bytes : 0; }

int grapes_split_tf32(grapes_ctx* ctx, const float* src, int ld_src, int R, int K, float* hi, float* lo, int ld_dst,
                      void* stream) {
    GRAPES_REQUIRE(ctx && src && hi && lo, "null argument");
    GRAPES_REQUIRE(ld_dst >= K && ld_src >= K, "bad leading dimension");
    long long total = (long long)R * ld_dst;
    int blocks = (int)((total + 255) / 256);
    if (blocks > ctx->sm_count * 8) blocks = ctx->sm_count * 8;
    if (blocks < 1) blocks = 1;
    pdl((k_split_tf32), blocks, 256, 0, (cudaStream_t)stream)(src, ld_src, R, K, hi, lo, ld_dst);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

// zpart[2 * D/128][cap_n]: partial row dots, two per 128-column half (summed by the caller, e.g. grapes_select_hop).
// Y_lo == NULL: Y is plain fp32 and is split into the 3xTF32 (hi, lo) pair inside the kernel; otherwise (Y, Y_lo) is
// the pair grapes_aggregate wrote (faster: one pipeline step less per k-block).
int grapes_sampler_l1_fwd_tc(grapes_ctx* ctx, const float* Y, const float* Y_lo, int ldy, const int* n_dev, int cap_n,
                             int K, const float* W_hi, const float* W_lo, int ldw, int D, const float* b1,
                             const float* w2, float* zpart, uint32_t* maskT, void* stream) {
    GRAPES_REQUIRE(ctx && Y && n_dev && W_hi && W_lo && b1 && w2 && zpart, "null argument");
    GRAPES_REQUIRE(D % TC_BN == 0 && D >= TC_BN && D <= 512, "hidden dim must be a multiple of 128 (<= 512) for the tcgen05 path");
    GRAPES_REQUIRE(K > 0 && K <= ldy && K <= ldw, "bad K");
    const int presplit = Y_lo ? 1 : 0;
    CUtensorMap ma, ma_lo, mb_hi, mb_lo;
    int rc;
    if (!presplit && !(g_tc_debug & 4))
        return launch_fwd_ts(ctx, Y, ldy, n_dev, cap_n, K, W_hi, W_lo, ldw, D, b1, w2, zpart, maskT, nullptr, 0, stream);
    if ((rc = make_map(&ma, Y, cap_n, K, ldy)) != GRAPES_OK) return rc;
    if ((rc = make_map(&ma_lo, presplit ? Y_lo : Y, cap_n, K, ldy)) != GRAPES_OK) return rc;
    if ((rc = make_map(&mb_hi, W_hi, D, K, ldw)) != GRAPES_OK) return rc;
    if ((rc = make_map(&mb_lo, W_lo, D, K, ldw)) != GRAPES_OK) return rc;
    const int nkb = (K + TC_BK - 1) / TC_BK, NH = D / TC_BN;
    const int m_tiles_cap = (cap_n + TC_BM - 1) / TC_BM;
    const int tail_w = 1024 /*align slack*/ + 256 /*barriers*/;
    const int tail = tail_w;
    // W-resident when one column half of W (hi | lo, all k-blocks) plus >= 3 ring stages of Y fit in shared memory
    int stages = (227 * 1024 - tail_w - nkb * 2 * TC_TILE_BYTES) / (2 * TC_TILE_BYTES);
    if (stages > 4) stages = 4;
    // (measured on B200, K = 104: 26.7 us resident vs 29 us streaming; the 128x128x8 tf32 MMA is fed at the
    //  shared-memory read limit either way.  grapes_tc_debug bit 1 forces streaming.)
    int wres = (stages >= 3 && ctx->sm_count >= NH && !(g_tc_debug & 2)) ? 1 : 0;
    int smem_bytes, blocks;
    if (wres) {
        smem_bytes = (nkb + stages) * 2 * TC_TILE_BYTES + tail_w;
        int per_half = ctx->sm_count / NH;
        if (per_half > m_tiles_cap) per_half = m_tiles_cap;
        if (per_half < 1) per_half = 1;
        blocks = per_half * NH;
    } else {
        stages = 3;
        smem_bytes = stages * 4 * TC_TILE_BYTES + tail;
        const int max_tiles = m_tiles_cap * NH;
        blocks = max_tiles < ctx->sm_count ? max_tiles : ctx->sm_count;
        if (blocks < 1) blocks = 1;
    }
    static int attr_dev[64] = {0};                   // per device: the attribute belongs to the device's copy of the function
    int& attr = attr_dev[ctx->device & 63];
    if (smem_bytes > attr) {
        GRAPES_CUDA_OK(cudaFuncSetAttribute(k_l1_fwd_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
        attr = smem_bytes;
    }
    pdl((k_l1_fwd_tc), blocks, TCF_THREADS, smem_bytes, (cudaStream_t)stream)(ma, ma_lo, mb_hi, mb_lo, n_dev, cap_n, K, D,
                                                                           stages, wres, presplit, b1, w2, zpart, maskT);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}


// Dense GCNConv.lin layer with bias and relu on the tensor cores: H[n x D] = relu(Y[n x K] W^T + b) (3xTF32, fp32-accurate),
// the hidden layer of the full-graph evaluation forward (eval.py:50: gcn_c(x, edge_index) over every node).  W_hi / W_lo from
// grapes_split_tf32; Y 16-byte aligned with ldy % 4 == 0; H 16-byte aligned with ldh % 4 == 0.
int grapes_gemm_bias_relu_tc(grapes_ctx* ctx, const float* Y, int ldy, const int* n_dev, int cap_n, int K, const float* W_hi,
                             const float* W_lo, int ldw, int D, const float* b, float* H, int ldh, void* stream) {
    GRAPES_REQUIRE(ctx && Y && n_dev && W_hi && W_lo && b && H, "null argument");
    GRAPES_REQUIRE(D % TC_BN == 0 && D >= TC_BN && D <= 512, "hidden dim must be a multiple of 128 (<= 512) for the tcgen05 path");
    GRAPES_REQUIRE(K > 0 && K <= ldy && K <= ldw && ldh >= D && ldh % 4 == 0 && (((uintptr_t)H) & 15) == 0, "bad layout");
    return launch_fwd_ts(ctx, Y, ldy, n_dev, cap_n, K, W_hi, W_lo, ldw, D, b, b /* unused weights: zpart == NULL */, nullptr,
                         nullptr, H, ldh, stream);
}

// Gradient DIRECTION of sum_r dz[r] z[r] w.r.t. (W1, b1, w2), accumulated (+=, times `scale`).
// Y must carry a column of ones at index `ones_col` (>= K); maskT from grapes_sampler_l1_fwd_tc.  Y_lo as in the forward.
int grapes_sampler_l1_bwd_tc(grapes_ctx* ctx, const float* Y, const float* Y_lo, int ldy, int ncols,
                             const int* n_dev, int cap_n, int K, int ones_col, const uint32_t* maskT,
                             const float* W1, int ldw, int D, const float* b1, const float* w2, const float* dz,
                             float scale, float* gW1, float* gb1, float* gw2, void* stream) {
    GRAPES_REQUIRE(ctx && Y && n_dev && maskT && W1 && b1 && w2 && dz && gW1 && gb1 && gw2, "null argument");
    GRAPES_REQUIRE(D % 128 == 0 && D >= 128 && D <= 256, "hidden dim must be 128 or 256 for the tcgen05 backward");
    GRAPES_REQUIRE(K <= ones_col && ones_col < ncols && ncols <= ldy, "bad column layout");
    const int NH = D / 128;
    cudaStream_t s = (cudaStream_t)stream;
    // column chunks of <= 128 columns of Y (accumulator: NH halves x (hi | lo) x 128 columns = all 512 TMEM columns): ONE
    // launch, blockIdx.y = chunk, the SMs divided among the chunks; then ONE finalize that walks the chunks in order
    const int nchunks = (ncols + 127) / 128;
    if (!(g_tc_debug & 8) && !Y_lo) {
        // scaled-feature operand in tensor memory (k_l1_bwd_ts): every CTA owns one 128-unit half of the hidden layer
        const int ystages = 6;
        const int smem_ts = TCBS_STAGES * TCB_A_TILE + ystages * 4 * TCB_B_TILE + 1024 + 512;
        CUtensorMap my;
        int rc;
        if ((rc = make_map(&my, Y, cap_n, ncols, ldy, TCB_ROWS, CU_TENSOR_MAP_SWIZZLE_NONE)) != GRAPES_OK) return rc;
        static int attr_ts[64] = {0};
        int& have = attr_ts[ctx->device & 63];
        if (smem_ts > have) {
            GRAPES_CUDA_OK(cudaFuncSetAttribute(k_l1_bwd_ts, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_ts));
            have = smem_ts;
        }
        const int max_groups = (cap_n + TCB_ROWS - 1) / TCB_ROWS;
        int per_half = grapes_max_i(1, ctx->sm_count / nchunks / NH);  // CTAs per chunk and half
        if (per_half > max_groups) per_half = max_groups;
        // accumulator chains are cut every TCBS_FLUSH groups: one partial slab per CTA and flush interval
        int nflush = grapes_div_up(grapes_div_up(max_groups, per_half), TCBS_FLUSH);
        GRAPES_REQUIRE((size_t)nchunks * nflush * per_half * D * 128 * sizeof(float) <= ctx->partials_bytes,
                       "split partial buffer too small");
        const long long chunk_stride = (long long)nflush * per_half * D * 128;
        // (debug stamps: the last KB of the partial buffer, behind every slab)
        unsigned long long* dbg = (g_tc_debug & 16) ? reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(ctx->partials) + ctx->partials_bytes - 1024) : nullptr;
        GRAPES_REQUIRE(!dbg || (size_t)nchunks * nflush * per_half * D * 128 * sizeof(float) + 1024 <= ctx->partials_bytes, "no room for the debug stamps");
        pdl((k_l1_bwd_ts), dim3(per_half * NH, nchunks), TCBS_THREADS, smem_ts, s)(my, ncols, n_dev, cap_n, NH, maskT, D, dz,
                                                                                  ctx->partials, chunk_stride, ystages, nflush, dbg);
        grapes_count_launches(1);
        pdl((k_l1_bwd_finalize), D, FIN_THREADS, 0, s)(ctx->partials, per_half * nflush, D, ncols, nchunks, chunk_stride, K, W1, ldw,
                                                    b1, w2, ones_col, scale, gW1, gb1, gw2);
        grapes_count_launches(1);
        GRAPES_LAUNCH_OK();
        return GRAPES_OK;
    }
    const int NB = (grapes_min_i(ncols, 128) + 31) / 32;              // blocks of 32 columns in a full chunk
    const int stage_bytes = NH * TCB_A_TILE + NB * 2 * TCB_B_TILE;
    int stages = (224 * 1024) / stage_bytes;
    if (stages > 4) stages = 4;
    GRAPES_REQUIRE(stages >= 2, "stage does not fit shared memory");
    const int smem_bytes = stages * stage_bytes + 1024 + 128 + 4 * 32 * (int)sizeof(float);
    CUtensorMap my, my_lo;
    int rc;
    if ((rc = make_map(&my, Y, cap_n, ncols, ldy, TCB_ROWS, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)) != GRAPES_OK) return rc;
    if ((rc = make_map(&my_lo, Y_lo ? Y_lo : Y, cap_n, ncols, ldy, TCB_ROWS, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)) != GRAPES_OK) return rc;
    static int attr_bytes_dev[64] = {0};
    int& attr_bytes = attr_bytes_dev[ctx->device & 63];
    if (smem_bytes > attr_bytes) {
        GRAPES_CUDA_OK(cudaFuncSetAttribute(k_l1_bwd_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
        attr_bytes = smem_bytes;
    }
    const int max_groups = (cap_n + TCB_ROWS - 1) / TCB_ROWS;
    int blocks = grapes_max_i(1, ctx->sm_count / nchunks);           // CTAs per chunk
    if (blocks > max_groups) blocks = max_groups;
    // one partial slab per CTA and flush interval, as in k_l1_bwd_ts
    auto slabs = [&](int b) { return (size_t)b * grapes_div_up(grapes_div_up(max_groups, b), TCBS_FLUSH); };
    while (blocks > 1 && nchunks * slabs(blocks) * D * 128 * sizeof(float) > ctx->partials_bytes) --blocks;
    GRAPES_REQUIRE(nchunks * slabs(blocks) * D * 128 * sizeof(float) <= ctx->partials_bytes, "split partial buffer too small");
    const int nflush = (int)(slabs(blocks) / blocks);
    const long long chunk_stride = (long long)slabs(blocks) * D * 128;
    pdl((k_l1_bwd_tc), dim3(blocks, nchunks), TCB_THREADS, smem_bytes, s)(my, my_lo, Y_lo ? 1 : 0, 0, n_dev, cap_n, NH, NB, stages,
                                                                      maskT, D, dz, ctx->partials, g_tc_debug, ncols, chunk_stride,
                                                                      nflush);
    grapes_count_launches(1);
    pdl((k_l1_bwd_finalize), D, FIN_THREADS, 0, s)(ctx->partials, blocks * nflush, D, ncols, nchunks, chunk_stride, K, W1, ldw, b1,
                                                w2, ones_col, scale, gW1, gb1, gw2);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

}  // extern "C"
