// Gather + SpMM with the feature rows staged through the TMA engine into shared memory (k_agg_tma).
//
// Same contract and the same summation order as k_agg / k_agg_rows in gcn.cu (self term first, then the sources of the
// dst-sorted CSR row in ascending order, one fma each) -> bitwise identical results; what changes is HOW the rows reach
// the SM.  The aggregation is a walk over a flattened entry list
//     row j0: self, src, src, ... | row j0+1: self, src, ... | ...
// in chunks of `ec` (<= 32) entries per warp.  Lane t of a warp owns entry t of a chunk: it finds the entry's row by
// binary search in the warp's row-offset table (shared memory), loads the source id, its node id / weight, and issues ONE
// bulk asynchronous copy (cp.async.bulk, the non-tensor TMA path, SASS UBLKCP) of that feature row into the warp's
// shared-memory slot; an mbarrier with a transaction count tells the warp when all rows of the chunk have landed.
// The four dependent steps (source id -> node id / weights -> row copy -> accumulate) of consecutive chunks are software
// pipelined, two slots per warp, so every warp keeps `ec` rows (ec x 4F bytes) in flight while it accumulates the previous
// chunk from shared memory: the memory-level parallelism no longer depends on registers or on the number of resident
// warps, which is what bounded the register-staged kernels (DESIGN.md section 4).
//
// Replaces (with gcn.cu) the message passing of PyG 2.5.2 GCNConv at the reference's call sites
// /root/reference/modules/gcn.py:18,21,32,36 and the feature gather of /root/reference/main.py:198-204.
#define GRAPES_PDL_GROUP 2
#include "common.cuh"

#define AT_WARPS 8
#define AT_THREADS (AT_WARPS * 32)
#define AT_RB_MAX 256                    // destination rows per warp task (row-offset table in shared memory)
#define AT_POS_STRIDE (AT_RB_MAX + 8)    // ints per warp
#define AT_SELF 0x200
#define AT_LAST 0x400
#define AT_VALID 0x800

__device__ __forceinline__ uint32_t at_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ float at_tf32(float x) { return grapes_tf32_rna(x); }
__device__ __forceinline__ void at_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void at_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void at_mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "AT_WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra.uni AT_WAIT_DONE;\n\t"
        "bra.uni AT_WAIT_LOOP;\n\t"
        "AT_WAIT_DONE:\n\t"
        "}\n" ::"r"(bar), "r"(parity) : "memory");
}
// one feature row, global -> shared, completion counted on the mbarrier
__device__ __forceinline__ void at_bulk_row(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

struct AtA { int sl; int rk; };                                   // source (local id) + packed row / flags
struct AtB { int g; float dsl, dj; uint32_t sb; int rk; };        // node id, deg^-1/2 of source and row, indicator bits

// OUTMODE: 1 = out, 2 = (out_hi, out_lo), 3 = all three.  The kernel is bound by instruction issue, not by memory
// (ncu: issue slots 60 % busy at 25 % DRAM), so the per-entry loop is kept to: one broadcast LDS.128 of the entry's
// metadata, one LDS.128 of the row per 128 columns, 4 FFMA, one branch.
// XB16: the feature table holds bf16 (papers100M-shaped config: 128 bf16 features); rows are staged as stored (2F bytes)
// and widened to fp32 when they are read from shared memory; all arithmetic and the output stay fp32.
// W64: a row slab of the whole-graph structure past 2^31 entries (grapes_aggregate_rows64).  n_dev = {R, r0}: output row j
// (j < R) is graph row r0 + j; in_off is int64 and indexed by graph row; sources, dinv and X rows are graph ids (nodes is
// null).  The summation order is that of the int32 form, so a slab's rows are bit-identical to the same rows of it.
template <int NPASS, bool HAS_IND, int OUTMODE, bool XB16, bool W64 = false>
__global__ void __launch_bounds__(AT_THREADS) k_agg_tma(
    const void* __restrict__ X, int F, int ldx, const int* __restrict__ nodes, const int* __restrict__ n_dev, int cap_n,
    const typename GrapesOff<W64>::T* __restrict__ in_off, const int* __restrict__ in_src, const float* __restrict__ dinv,
    const uint32_t* __restrict__ ind_bits, int num_ind, const float* __restrict__ bias, int relu, float* __restrict__ out,
    int ldo, float* __restrict__ out_hi, float* __restrict__ out_lo, int ones_col, int ec, int rb_min) {
    typedef typename GrapesOff<W64>::T OffT;
    pdl_begin();
    extern __shared__ __align__(128) unsigned char at_smem[];
    const int lane = lane_id();
    const int warp = threadIdx.x >> 5;
    const int n = min(*n_dev, cap_n);
    const int r0 = W64 ? n_dev[1] : 0;
    // bytes staged per row: the row rounded up to a whole float4 (F % 4 != 0: the table's rows are padded, ldx >= round_up(F, 4);
    // the pad values are accumulated into the unused components of the last feature lane and never stored)
    const uint32_t rowbytes = XB16 ? (uint32_t)F * 2u : (uint32_t)((F + 3) & ~3) * 4u;
    const uint32_t slot_bytes = (uint32_t)ec * rowbytes;
    unsigned char* wslots = at_smem + (size_t)warp * 2u * slot_bytes;
    unsigned char* tail = at_smem + (size_t)AT_WARPS * 2u * slot_bytes;
    int4* s_meta = reinterpret_cast<int4*>(tail) + warp * 64;                         // [2 slots][32 entries]
    int* s_pos = reinterpret_cast<int*>(tail + (size_t)AT_WARPS * 64u * 16u) + warp * AT_POS_STRIDE;
    uint64_t* bars = reinterpret_cast<uint64_t*>(tail + (size_t)AT_WARPS * 64u * 16u +
                                                 (size_t)AT_WARPS * AT_POS_STRIDE * 4u) + warp * 2;
    const uint32_t bar0 = at_smem_u32(&bars[0]), bar1 = at_smem_u32(&bars[1]);
    if (lane == 0) { at_mbar_init(bar0, 1); at_mbar_init(bar1, 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncwarp();
    uint32_t ph = 0;                                              // phase parity of the two barriers (bits 0, 1)
    bool act[NPASS];                                              // this lane accumulates and stores columns p*128 + 4*lane .. +3
#pragma unroll
    for (int p = 0; p < NPASS; ++p) act[p] = p * 128 + lane * 4 < F;
    const int cv = F + lane;                                      // this lane's virtual column
    const float vconst = (cv == ones_col) ? 1.f : 0.f;

    const int total_warps = gridDim.x * AT_WARPS;
    int RB = (n + total_warps - 1) / total_warps;
    RB = min(max(RB, rb_min), AT_RB_MAX);
    int top = 1;
    while (top < RB) top <<= 1;                                   // binary-search span (power of two >= RB)
    for (int j0 = (blockIdx.x * AT_WARPS + warp) * RB; j0 < n; j0 += total_warps * RB) {
        const int nr = min(RB, n - j0);
        const OffT base_off = in_off[r0 + j0];
        for (int u = lane; u <= nr; u += 32)                                         // first entry of row u
            s_pos[u] = W64 ? u + (int)(in_off[r0 + j0 + u] - base_off) : u + (int)in_off[j0 + u] - (int)base_off;
        __syncwarp();
        const int T = s_pos[nr];
        const int nchunks = (T + ec - 1) / ec;

        // stage A: entry -> (row, position in the row), source id
        auto stageA = [&](int c) -> AtA {
            AtA a; a.sl = 0; a.rk = 0;
            const int e = c * ec + lane;
            if (c < nchunks && lane < ec && e < T) {
                int r = 0;
                for (int step = top >> 1; step > 0; step >>= 1)
                    if (r + step < nr && s_pos[r + step] <= e) r += step;
                const int first = s_pos[r];
                const int k = e - first;
                a.rk = r | AT_VALID | (k == 0 ? AT_SELF : 0) | (e + 1 == s_pos[r + 1] ? AT_LAST : 0);
                a.sl = (k == 0) ? r : in_src[base_off + first - r + k - 1];
            }
            return a;
        };
        // stage B: node id, deg^-1/2 values, indicator bits of the entry's source
        auto stageB = [&](const AtA& a) -> AtB {
            AtB b; b.g = 0; b.dsl = 0.f; b.dj = 0.f; b.sb = 0u; b.rk = a.rk;
            if (a.rk & AT_VALID) {
                const int j = r0 + j0 + (a.rk & 0x1ff);
                const int sl = (a.rk & AT_SELF) ? j : a.sl;
                b.g = nodes ? nodes[sl] : sl;
                b.dsl = dinv[sl];
                b.dj = dinv[j];
                if (HAS_IND) b.sb = ind_bits[sl];
            }
            return b;
        };
        // stage C: weight + metadata into shared memory, and the row copy into slot (c & 1)
        auto stageC = [&](const AtB& b, int c) {
            if (c < nchunks) {
                const int cnt = min(ec, T - c * ec);
                const uint32_t bar = (c & 1) ? bar1 : bar0;
                if (lane == 0) at_mbar_expect_tx(bar, (uint32_t)cnt * rowbytes);
                s_meta[(c & 1) * 32 + lane] = make_int4(__float_as_int(b.dsl * b.dj), b.rk, (int)b.sb, 0);  // self: dj * dj
                __syncwarp();
                if (b.rk & AT_VALID)
                    at_bulk_row(at_smem_u32(wslots) + (uint32_t)(c & 1) * slot_bytes + (uint32_t)lane * rowbytes,
                                reinterpret_cast<const unsigned char*>(X) + (size_t)b.g * ldx * (XB16 ? 2u : 4u), rowbytes, bar);
            }
        };

        float4 acc[NPASS];
        float aind = 0.f;
#pragma unroll
        for (int p = 0; p < NPASS; ++p) acc[p] = make_float4(0.f, 0.f, 0.f, 0.f);

        // ---- prologue: fill the pipeline (the only place where the dependent chain is exposed).  The metadata stages
        // run 2 + 2 chunks ahead of the row copies, so a frontier-sized task (<= 5 chunks) issues ALL its index loads
        // before the first wait and only the row copies (two slots) remain pipelined. ----
        AtA A0 = stageA(0);
        AtA A1 = stageA(1);
        AtA A2 = stageA(2);
        AtA A3 = stageA(3);
        AtA A4 = stageA(4);
        AtB B0 = stageB(A0);
        AtB B1 = stageB(A1);
        AtB B2 = stageB(A2);
        stageC(B0, 0);
        for (int c = 0; c < nchunks; ++c) {
            const AtA A5 = stageA(c + 5);                    // loads consumed two iterations later
            const AtB B3 = stageB(A3);                       // loads consumed two iterations later
            stageC(B1, c + 1);                               // rows of chunk c+1 in flight while chunk c is accumulated
            // ---- stage D: accumulate chunk c from its slot ----
            const int cnt = min(ec, T - c * ec);
            at_mbar_wait((c & 1) ? bar1 : bar0, (ph >> (c & 1)) & 1u);
            ph ^= 1u << (c & 1);
            // lane l owns columns 4l .. 4l+3 of every 128-column pass: a float4 (fp32 table) or a uint2 (bf16 table)
            const unsigned char* rp = wslots + (size_t)(c & 1) * slot_bytes + (size_t)lane * (XB16 ? 8u : 16u);
            const int4* mp = s_meta + (c & 1) * 32;
            for (int t = 0; t < cnt; ++t, rp += rowbytes) {
                const int4 m = mp[t];                                      // broadcast: weight | row + flags | indicator bits
                const float wt = __int_as_float(m.x);
#pragma unroll
                for (int p = 0; p < NPASS; ++p) {
                    if (act[p]) {
                        float4 v;
                        if (XB16) {
                            const uint2 r = reinterpret_cast<const uint2*>(rp)[p * 32];
                            v.x = __uint_as_float(r.x << 16); v.y = __uint_as_float(r.x & 0xffff0000u);
                            v.z = __uint_as_float(r.y << 16); v.w = __uint_as_float(r.y & 0xffff0000u);
                        } else {
                            v = reinterpret_cast<const float4*>(rp)[p * 32];
                        }
                        acc[p].x = fmaf(wt, v.x, acc[p].x); acc[p].y = fmaf(wt, v.y, acc[p].y);
                        acc[p].z = fmaf(wt, v.z, acc[p].z); acc[p].w = fmaf(wt, v.w, acc[p].w);
                    }
                }
                if (HAS_IND) aind = fmaf(wt, (float)(((uint32_t)m.z >> lane) & 1u), aind);
                if (m.y & AT_LAST) {                               // warp-uniform: the row is complete
                    const size_t orow = (size_t)(j0 + (m.y & 0x1ff)) * ldo;
#pragma unroll
                    for (int p = 0; p < NPASS; ++p) {
                        if (act[p]) {
                            const int c0 = p * 128 + lane * 4;
                            float4 a = acc[p];
                            if (bias) {
                                if (c0 + 4 <= F) { a.x += bias[c0]; a.y += bias[c0 + 1]; a.z += bias[c0 + 2]; a.w += bias[c0 + 3]; }
                                else { a.x += bias[c0]; if (c0 + 1 < F) a.y += bias[c0 + 1]; if (c0 + 2 < F) a.z += bias[c0 + 2]; }
                            }
                            if (relu) { a.x = fmaxf(a.x, 0.f); a.y = fmaxf(a.y, 0.f); a.z = fmaxf(a.z, 0.f); a.w = fmaxf(a.w, 0.f); }
                            if (c0 + 4 > F) {                      // last feature lane of a row with F % 4 != 0: 1..3 valid columns
                                const int nvv = F - c0;
                                auto put = [&](int i, float val) {
                                    if (OUTMODE & 1) out[orow + c0 + i] = val;
                                    if (OUTMODE & 2) {
                                        const float h = at_tf32(val);
                                        out_hi[orow + c0 + i] = h; out_lo[orow + c0 + i] = at_tf32(val - h);
                                    }
                                };
                                put(0, a.x);
                                if (nvv > 1) put(1, a.y);
                                if (nvv > 2) put(2, a.z);
                            } else {
                                if (OUTMODE & 1) *reinterpret_cast<float4*>(out + orow + c0) = a;
                                if (OUTMODE & 2) {                 // 3xTF32 operand split for the tcgen05 GEMM
                                    float4 h, l;
                                    h.x = at_tf32(a.x); h.y = at_tf32(a.y); h.z = at_tf32(a.z); h.w = at_tf32(a.w);
                                    l.x = at_tf32(a.x - h.x); l.y = at_tf32(a.y - h.y);
                                    l.z = at_tf32(a.z - h.z); l.w = at_tf32(a.w - h.w);
                                    *reinterpret_cast<float4*>(out_hi + orow + c0) = h;
                                    *reinterpret_cast<float4*>(out_lo + orow + c0) = l;
                                }
                            }
                        }
                        acc[p] = make_float4(0.f, 0.f, 0.f, 0.f);    // next row starts from fma(w_self, x, 0)
                    }
                    if (cv < ldo) {                                // virtual columns, one scalar lane each
                        const float v = (HAS_IND && lane < num_ind) ? aind : vconst;
                        if (OUTMODE & 1) out[orow + cv] = v;
                        if (OUTMODE & 2) { const float h = at_tf32(v); out_hi[orow + cv] = h; out_lo[orow + cv] = at_tf32(v - h); }
                    }
                    aind = 0.f;
                }
            }
            __syncwarp();                                          // slot (c & 1) is free for chunk c + 2
            A3 = A4; A4 = A5; B1 = B2; B2 = B3;
        }
        __syncwarp();                                              // s_pos is rewritten by the next task
    }
}

size_t grapes_agg_tma_smem(int F, int ec, int es = 4) {
    return (size_t)AT_WARPS * 2u * (size_t)ec * (size_t)F * (size_t)es + (size_t)AT_WARPS * 64u * 16u +
           (size_t)AT_WARPS * AT_POS_STRIDE * 4u + AT_WARPS * 16u;
}

// Returns 0 when the kernel was launched, 1 when the shape is not covered (caller falls back to k_agg_rows / k_agg).
int grapes_launch_agg_tma(grapes_ctx* ctx, const void* X, int x_bf16, int F, int ldx, const int* nodes, const int* n_dev, int cap_n,
                          const void* in_off, const int* in_src, const float* dinv, const uint32_t* ind_bits, int num_ind,
                          const float* bias, int relu, float* out, int ldo, float* out_hi, float* out_lo, int ones_col,
                          int ec_req, int ctas_per_sm, cudaStream_t s, int off64) {
    // fp32 rows must start 16-byte aligned and be readable up to a whole float4: ldx % 4 == 0 and ldx >= round_up(F, 4)
    // (F itself may be any width: Reddit 602, Cora 1433 -- the caller pads the table's row pitch, engine.py)
    if (ldx % 4 != 0 || ldx < ((F + 3) & ~3) || ldo % 4 != 0 || ldo - F > 32 || F > 128 * 12 || F < 4) return 1;
    if (x_bf16 && F % 4 != 0) return 1;
    if (x_bf16 && (F % 8 != 0 || ldx % 8 != 0 || F > 256)) return 1;         // 16-byte rows; bf16 forms built for F <= 256
    const int es = x_bf16 ? 2 : 4;
    const int cps = ctas_per_sm < 1 ? 1 : (ctas_per_sm > 6 ? 6 : ctas_per_sm);       // resident CTAs per SM the shape is sized for
    const size_t budget = cps == 1 ? 226u * 1024u : (cps == 2 ? 113u * 1024u : (size_t)(227u * 1024u / cps - 1024u));
    const int npass = (F + 127) / 128;
    const bool has_ind = ind_bits != nullptr && num_ind > 0;
    const int Fs = x_bf16 ? F : ((F + 3) & ~3);                                       // staged row width
    int ec = ec_req > 0 ? ec_req : 32;
    if (ec > 32) ec = 32;
    while (ec > 1 && grapes_agg_tma_smem(Fs, ec, es) > budget) ec >>= 1;
    const size_t smem = grapes_agg_tma_smem(Fs, ec, es);
    if (smem > 226u * 1024u) return 1;
    const int rb_min = (size_t)Fs * es >= 2048 ? 2 : 8;      // wide rows (Reddit 2.4 KB, Cora 5.7 KB): spread a small frontier over every warp
    long long blocks = ((long long)cap_n + AT_WARPS * rb_min - 1) / (AT_WARPS * rb_min);
    const long long cap = (long long)ctx->sm_count * (smem > 113u * 1024u ? 1 : (cps >= 2 ? cps : 2));
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
#define AT_LAUNCH_W(NP, IND, OM, XB, W)                                                                                 \
    do {                                                                                                                \
        static bool configured = false;                                                                                 \
        if (!configured) {                                                                                              \
            if (cudaFuncSetAttribute(k_agg_tma<NP, IND, OM, XB, W>, cudaFuncAttributeMaxDynamicSharedMemorySize,        \
                                     (int)(226u * 1024u)) != cudaSuccess) return 1;                                     \
            configured = true;                                                                                          \
        }                                                                                                               \
        pdl((k_agg_tma<NP, IND, OM, XB, W>), (int)blocks, AT_THREADS, smem, s)(                                         \
            X, F, ldx, nodes, n_dev, cap_n, (const typename GrapesOff<W>::T*)in_off, in_src, dinv, ind_bits, num_ind,    \
            bias, relu, out, ldo, out_hi, out_lo, ones_col, ec, rb_min);                                                \
    } while (0)
#define AT_LAUNCH_INST(NP, IND, OM, XB) AT_LAUNCH_W(NP, IND, OM, XB, false)
#define AT_LAUNCH2(NP, IND, XB)                                                                                         \
    do {                                                                                                                \
        if (om == 1) AT_LAUNCH_INST(NP, IND, 1, XB); else if (om == 2) AT_LAUNCH_INST(NP, IND, 2, XB);                  \
        else AT_LAUNCH_INST(NP, IND, 3, XB);                                                                            \
    } while (0)
#define AT_LAUNCH(NP)                                                                                                   \
    do {                                                                                                                \
        if (has_ind) AT_LAUNCH2(NP, true, false); else AT_LAUNCH2(NP, false, false);                                    \
    } while (0)
#define AT_LAUNCH_B16(NP)                                                                                               \
    do {                                                                                                                \
        if (has_ind) AT_LAUNCH2(NP, true, true); else AT_LAUNCH2(NP, false, true);                                      \
    } while (0)
    const int om = (out ? 1 : 0) | (out_hi ? 2 : 0);
    if (off64) {                                   // whole-graph row slab: plain output, no indicator columns
        if (om != 1 || has_ind) return 1;
        if (x_bf16) {
            if (npass == 1) AT_LAUNCH_W(1, false, 1, true, true); else AT_LAUNCH_W(2, false, 1, true, true);
        } else if (npass == 1) AT_LAUNCH_W(1, false, 1, false, true);
        else if (npass == 2) AT_LAUNCH_W(2, false, 1, false, true);
        else if (npass <= 5) AT_LAUNCH_W(5, false, 1, false, true);
        else AT_LAUNCH_W(12, false, 1, false, true);
    } else if (x_bf16) {
        if (npass == 1) AT_LAUNCH_B16(1); else AT_LAUNCH_B16(2);
    } else if (npass == 1) AT_LAUNCH(1);
    else if (npass == 2) AT_LAUNCH(2);
    else if (npass <= 5) AT_LAUNCH(5);
    else AT_LAUNCH(12);
#undef AT_LAUNCH_B16
#undef AT_LAUNCH2
#undef AT_LAUNCH_INST
#undef AT_LAUNCH_W
#undef AT_LAUNCH
    return 0;
}
