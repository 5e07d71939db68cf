// gcn_norm + GCNConv aggregation (deterministic CSR SpMM, no fp atomics) and the fp32 SIMT GEMMs.
//
// Restates on the device what PyG 2.5.2 GCNConv does for the reference's call sites
// (/root/reference/modules/gcn.py:18,21,32,36; SURVEY.md section 3.2):
//   out = D^-1/2 (A_noloop + I) D^-1/2 (X W^T) + b,  deg = in-degree incl. the added self-loop.
// Aggregation commutes with the dense transform, so it is done at the NARROWER width
// (features for layer 1, the scalar / class logits for layer 2) -- DESIGN.md section 4.
#define GRAPES_PDL_GROUP 2
#include "common.cuh"

template <int VEC> struct VecT;
template <> struct VecT<1> { typedef float T; };
template <> struct VecT<2> { typedef float2 T; };
template <> struct VecT<4> { typedef float4 T; };

__device__ __forceinline__ float f32_to_tf32(float x) { return grapes_tf32_rna(x); }

template <int VEC>
__device__ __forceinline__ void vec_fma(float (&acc)[VEC], float w, const float* p) {
    typename VecT<VEC>::T v = *reinterpret_cast<const typename VecT<VEC>::T*>(p);
    const float* f = reinterpret_cast<const float*>(&v);
#pragma unroll
    for (int i = 0; i < VEC; ++i) acc[i] = fmaf(w, f[i], acc[i]);
}

// the same for a feature table stored as fp32 (XB16 = false) or bf16 (true; widened to fp32, arithmetic stays fp32)
template <int VEC, bool XB16>
__device__ __forceinline__ void vec_fma_x(float (&acc)[VEC], float w, const void* X, size_t elem) {
    if (!XB16) {
        vec_fma<VEC>(acc, w, reinterpret_cast<const float*>(X) + elem);
    } else {
        const unsigned short* p = reinterpret_cast<const unsigned short*>(X) + elem;
        float f[VEC];
        if (VEC == 4) {
            const uint2 r = *reinterpret_cast<const uint2*>(p);
            f[0] = __uint_as_float(r.x << 16); f[1] = __uint_as_float(r.x & 0xffff0000u);
            f[2 % VEC] = __uint_as_float(r.y << 16); f[3 % VEC] = __uint_as_float(r.y & 0xffff0000u);
        } else if (VEC == 2) {
            const uint32_t r = *reinterpret_cast<const uint32_t*>(p);
            f[0] = __uint_as_float(r << 16); f[1 % VEC] = __uint_as_float(r & 0xffff0000u);
        } else {
            f[0] = __uint_as_float(((uint32_t)p[0]) << 16);
        }
#pragma unroll
        for (int i = 0; i < VEC; ++i) acc[i] = fmaf(w, f[i], acc[i]);
    }
}

// ---------------------------------------------------------------------------------------
// k_agg: one warp per destination row j (local id).
//   out[j, :F] = dinv[j]^2 * X[g(j), :F] + sum_{s in in(j)} dinv[s] dinv[j] * X[g(s), :F]   (+bias)(relu)
//   g(j) = nodes[j] (feature gather fused: reads global feature rows directly, main.py:198-204)
//          or j when nodes == nullptr (plain SpMM on a local matrix).
//   out[j, F + t] (t < num_ind) = the same aggregation of indicator bit t (ind_bits), i.e. the
//   indicator_features columns of main.py:199-202 without materialising the N x (hops+1) matrix.
//   Columns [F + num_ind, ldo) are zero-filled (K padding for the GEMM).
// Sources are preloaded 32 at a time and broadcast by shuffle so the dependent chain
// in_src -> nodes -> X is paid once per 32 sources.
// ---------------------------------------------------------------------------------------
// W64: a row slab of the whole-graph structure past 2^31 entries, as in k_agg_tma (n_dev = {R, r0}, output row j is graph
// row r0 + j, int64 in_off indexed by graph row, nodes null); the same fma chain as the int32 form.
template <int VEC, bool XB16 = false, bool W64 = false>
__global__ void __launch_bounds__(256) k_agg(const void* __restrict__ X, int F, int ldx,
                                             const int* __restrict__ nodes, const int* __restrict__ n_dev, int cap_n,
                                             const typename GrapesOff<W64>::T* __restrict__ in_off,
                                             const int* __restrict__ in_src,
                                             const float* __restrict__ dinv, const uint32_t* __restrict__ ind_bits,
                                             int num_ind, const float* __restrict__ bias, int relu,
                                             float* __restrict__ out, int ldo, float* __restrict__ out_hi,
                                             float* __restrict__ out_lo, int ones_col) {
    typedef typename GrapesOff<W64>::T OffT;
    pdl_begin();
    const int n = min(*n_dev, cap_n);
    const int r0 = W64 ? n_dev[1] : 0;
    const int lane = lane_id();
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < n; j += warps) {
        const int jr = r0 + j;                               // row of in_off / dinv / X
        const float dj = dinv[jr];
        const OffT beg = in_off[jr], end = in_off[jr + 1];
        const size_t gj = nodes ? (size_t)nodes[j] : (size_t)jr;
        float* oj = out ? out + (size_t)j * ldo : nullptr;
        float* ohj = out_hi ? out_hi + (size_t)j * ldo : nullptr;
        float* olj = out_hi ? out_lo + (size_t)j * ldo : nullptr;
        for (int cb = 0; cb < F; cb += 32 * VEC) {           // warp-uniform trip count
            const int c0 = cb + lane * VEC;
            const bool act = c0 < F;
            float acc[VEC];
#pragma unroll
            for (int i = 0; i < VEC; ++i) acc[i] = 0.f;
            if (act) vec_fma_x<VEC, XB16>(acc, dj * dj, X, gj * ldx + c0);
            for (OffT pb = beg; pb < end; pb += 32) {
                const OffT p = pb + lane;
                float w = 0.f; unsigned long long sg = 0ull;
                if (p < end) {
                    const int sl = in_src[p];
                    w = dinv[sl] * dj;
                    sg = nodes ? (unsigned long long)nodes[sl] : (unsigned long long)sl;
                }
                const int cnt = (int)min((OffT)32, end - pb);
                for (int t = 0; t < cnt; ++t) {
                    const float wt = __shfl_sync(GRAPES_FULL_MASK, w, t);
                    const unsigned long long st = __shfl_sync(GRAPES_FULL_MASK, sg, t);
                    if (act) vec_fma_x<VEC, XB16>(acc, wt, X, (size_t)st * ldx + c0);
                }
            }
            if (act) {
#pragma unroll
                for (int i = 0; i < VEC; ++i) {
                    float v = acc[i];
                    if (bias) v += bias[c0 + i];
                    if (relu) v = fmaxf(v, 0.f);
                    acc[i] = v;
                }
                if (oj) *reinterpret_cast<typename VecT<VEC>::T*>(oj + c0) = *reinterpret_cast<typename VecT<VEC>::T*>(acc);
                if (ohj) {                                   // 3xTF32 operand split for the tcgen05 GEMM
                    float h[VEC], l[VEC];
#pragma unroll
                    for (int i = 0; i < VEC; ++i) { h[i] = f32_to_tf32(acc[i]); l[i] = f32_to_tf32(acc[i] - h[i]); }
                    *reinterpret_cast<typename VecT<VEC>::T*>(ohj + c0) = *reinterpret_cast<typename VecT<VEC>::T*>(h);
                    *reinterpret_cast<typename VecT<VEC>::T*>(olj + c0) = *reinterpret_cast<typename VecT<VEC>::T*>(l);
                }
            }
        }
        if (ldo > F) {
            float a = 0.f;
            if (lane < num_ind) {
                a = dj * dj * (float)((ind_bits[j] >> lane) & 1u);
                for (OffT p = beg; p < end; ++p) {
                    const int sl = in_src[p];
                    a = fmaf(dinv[sl] * dj, (float)((ind_bits[sl] >> lane) & 1u), a);
                }
            }
            for (int c = F + lane; c < ldo; c += 32) {
                const float v = (c < F + num_ind) ? a : (c == ones_col ? 1.f : 0.f);
                if (oj) oj[c] = v;
                if (ohj) { const float h = f32_to_tf32(v); ohj[c] = h; olj[c] = f32_to_tf32(v - h); }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
// k_agg_px: k_agg over a table whose rows are partitioned between `world` owners: row s lives at
// base[o] + (s - bound[o]) * ldx for the owner o with bound[o] <= s < bound[o + 1], in this rank's memory or a peer's
// (NVLink).  Serves the hop / classifier gather of a feature table sharded across the data-parallel ranks
// (grapes_aggregate_peer), the same over slabs of the int64 whole-graph structure (grapes_aggregate_rows64_peer_x) and
// the layer 2 of the sharded whole-graph forward (grapes_aggregate_rows64_peer).  The loading lane resolves the owner and
// broadcasts the row address instead of the row id; everything else (nodes indirection, indicator columns by local id,
// bias / relu, out or the 3xTF32 split, ones_col, zero pad, W64 slabs) and the fma chain (self term, then sources
// ascending, bias last) are k_agg's, so the rows are bit-identical to grapes_aggregate / grapes_aggregate_bf16 /
// grapes_aggregate_rows64 over the unpartitioned table.  Register-staged: whether cp.async.bulk reads peer-mapped memory
// is not established.  A kernel of its own rather than a template parameter of k_agg, which would rename every existing
// k_agg instantiation.
// ---------------------------------------------------------------------------------------
#define GRAPES_PEER_MAX 8
struct PeerRows {
    const void* base[GRAPES_PEER_MAX];
    int bound[GRAPES_PEER_MAX];                 // first row of each owner; INT_MAX past the last owner
};

template <bool XB16>
__device__ __forceinline__ const void* peer_row(const PeerRows& P, int s, int ldx) {
    // selects with constant indices (bounds do not decrease: the last window starting at or before s owns it); an index
    // computed at run time would copy the parameter struct to the stack
    const void* b = P.base[0];
    int lo = 0;
#pragma unroll
    for (int k = 1; k < GRAPES_PEER_MAX; ++k)
        if (s >= P.bound[k]) { b = P.base[k]; lo = P.bound[k]; }
    return reinterpret_cast<const char*>(b) + (size_t)(s - lo) * ldx * (XB16 ? 2 : 4);
}

// __maxnreg__ instead of __launch_bounds__(256): with the launch bound alone ptxas settles on 32-40 registers and spills
// the owner select's live values (24-28 bytes); 48 registers hold them (k_agg: 40-48)
template <int VEC, bool XB16, bool W64>
__global__ void __maxnreg__(48) k_agg_px(const PeerRows P, int F, int ldx,
                                                const int* __restrict__ nodes, const int* __restrict__ n_dev, int cap_n,
                                                const typename GrapesOff<W64>::T* __restrict__ in_off,
                                                const int* __restrict__ in_src,
                                                const float* __restrict__ dinv, const uint32_t* __restrict__ ind_bits,
                                                int num_ind, const float* __restrict__ bias, int relu,
                                                float* __restrict__ out, int ldo, float* __restrict__ out_hi,
                                                float* __restrict__ out_lo, int ones_col) {
    typedef typename GrapesOff<W64>::T OffT;
    pdl_begin();
    const int n = min(*n_dev, cap_n);
    const int r0 = W64 ? n_dev[1] : 0;
    const int lane = lane_id();
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < n; j += warps) {
        const int jr = r0 + j;                               // row of in_off / dinv
        const float dj = dinv[jr];
        const OffT beg = in_off[jr], end = in_off[jr + 1];
        const void* xj = peer_row<XB16>(P, nodes ? nodes[j] : jr, ldx);
        float* oj = out ? out + (size_t)j * ldo : nullptr;
        float* ohj = out_hi ? out_hi + (size_t)j * ldo : nullptr;
        float* olj = out_hi ? out_lo + (size_t)j * ldo : nullptr;
        for (int cb = 0; cb < F; cb += 32 * VEC) {           // warp-uniform trip count
            const int c0 = cb + lane * VEC;
            const bool act = c0 < F;
            float acc[VEC];
#pragma unroll
            for (int i = 0; i < VEC; ++i) acc[i] = 0.f;
            if (act) vec_fma_x<VEC, XB16>(acc, dj * dj, xj, c0);
            for (OffT pb = beg; pb < end; pb += 32) {
                const OffT p = pb + lane;
                float w = 0.f; unsigned long long sa = 0ull;
                if (p < end) {
                    const int sl = in_src[p];
                    w = dinv[sl] * dj;
                    sa = (unsigned long long)peer_row<XB16>(P, nodes ? nodes[sl] : sl, ldx);
                }
                const int cnt = (int)min((OffT)32, end - pb);
                for (int t = 0; t < cnt; ++t) {
                    const float wt = __shfl_sync(GRAPES_FULL_MASK, w, t);
                    const unsigned long long st = __shfl_sync(GRAPES_FULL_MASK, sa, t);
                    if (act) vec_fma_x<VEC, XB16>(acc, wt, reinterpret_cast<const void*>(st), c0);
                }
            }
            if (act) {
#pragma unroll
                for (int i = 0; i < VEC; ++i) {
                    float v = acc[i];
                    if (bias) v += bias[c0 + i];
                    if (relu) v = fmaxf(v, 0.f);
                    acc[i] = v;
                }
                if (oj) *reinterpret_cast<typename VecT<VEC>::T*>(oj + c0) = *reinterpret_cast<typename VecT<VEC>::T*>(acc);
                if (ohj) {                                   // 3xTF32 operand split for the tcgen05 GEMM
                    float h[VEC], l[VEC];
#pragma unroll
                    for (int i = 0; i < VEC; ++i) { h[i] = f32_to_tf32(acc[i]); l[i] = f32_to_tf32(acc[i] - h[i]); }
                    *reinterpret_cast<typename VecT<VEC>::T*>(ohj + c0) = *reinterpret_cast<typename VecT<VEC>::T*>(h);
                    *reinterpret_cast<typename VecT<VEC>::T*>(olj + c0) = *reinterpret_cast<typename VecT<VEC>::T*>(l);
                }
            }
        }
        if (ldo > F) {
            float a = 0.f;
            if (lane < num_ind) {
                a = dj * dj * (float)((ind_bits[j] >> lane) & 1u);
                for (OffT p = beg; p < end; ++p) {
                    const int sl = in_src[p];
                    a = fmaf(dinv[sl] * dj, (float)((ind_bits[sl] >> lane) & 1u), a);
                }
            }
            for (int c = F + lane; c < ldo; c += 32) {
                const float v = (c < F + num_ind) ? a : (c == ones_col ? 1.f : 0.f);
                if (oj) oj[c] = v;
                if (ohj) { const float h = f32_to_tf32(v); ohj[c] = h; olj[c] = f32_to_tf32(v - h); }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------
// k_agg_rows: the same aggregation with R destination rows per warp, their dependent load chains interleaved
// (row offsets -> source ids -> source node ids / weights -> feature rows): the chain is 4 memory latencies deep and
// one-row-per-warp pays it once per row and wave; R rows in flight per warp cut the number of waves R-fold.  Same
// summation order as k_agg (self term, then sources ascending) -> bitwise identical results.
// float4 path only (F, ldx, ldo multiples of 4, 16-byte aligned bases); virtual columns (indicators | ones | pad)
// must fit one warp (ldo - F <= 32).
// ---------------------------------------------------------------------------------------
template <int R, int MINB>
__global__ void __launch_bounds__(256, MINB) k_agg_rows(const float* __restrict__ X, int F, int ldx,
                                                     const int* __restrict__ nodes, const int* __restrict__ n_dev,
                                                     int cap_n, const int* __restrict__ in_off,
                                                     const int* __restrict__ in_src, const float* __restrict__ dinv,
                                                     const uint32_t* __restrict__ ind_bits, int num_ind,
                                                     const float* __restrict__ bias, int relu, float* __restrict__ out,
                                                     int ldo, float* __restrict__ out_hi, float* __restrict__ out_lo,
                                                     int ones_col) {
    pdl_begin();
    const int n = min(*n_dev, cap_n);
    const int lane = lane_id();
    const int warps = (gridDim.x * blockDim.x) >> 5;
    const bool has_ind = ind_bits != nullptr && num_ind > 0;
    for (int j0 = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * R; j0 < n; j0 += warps * R) {
        // ---- level 1: per-row metadata (warp-uniform values, R independent loads each) ----
        int beg[R], cnt[R];
        float dj[R];
        size_t gj[R];
        uint32_t ibj[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const int j = min(j0 + r, n - 1);
            beg[r] = in_off[j];
            cnt[r] = (j0 + r < n) ? in_off[j + 1] - beg[r] : 0;
            dj[r] = dinv[j];
            gj[r] = nodes ? (size_t)nodes[j] : (size_t)j;
            ibj[r] = has_ind ? ind_bits[j] : 0u;
        }
        // ---- levels 2-3: lane t of row r preloads source t (first 32 sources; longer rows finish in the hub loop) ----
        float w[R];
        unsigned long long sg[R];
        uint32_t sb[R];
        int sl[R];
#pragma unroll
        for (int r = 0; r < R; ++r) sl[r] = (lane < cnt[r]) ? in_src[beg[r] + lane] : -1;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            w[r] = 0.f; sg[r] = gj[r]; sb[r] = 0u;                 // inactive lanes point at the (cached) self row
            if (sl[r] >= 0) {
                w[r] = dinv[sl[r]] * dj[r];
                sg[r] = nodes ? (unsigned long long)nodes[sl[r]] : (unsigned long long)sl[r];
                sb[r] = has_ind ? ind_bits[sl[r]] : 0u;
            }
        }
        int maxc = 0;
#pragma unroll
        for (int r = 0; r < R; ++r) maxc = max(maxc, min(cnt[r], 32));
        // ---- level 4: feature rows, 128 columns per pass ----
        for (int cb = 0; cb < F; cb += 128) {
            const int c0 = cb + lane * 4;
            const bool act = c0 < F;
            float4 acc[R];
#pragma unroll
            for (int r = 0; r < R; ++r) {
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (act) v = *reinterpret_cast<const float4*>(X + gj[r] * ldx + c0);
                const float ws = dj[r] * dj[r];
                acc[r].x = fmaf(ws, v.x, 0.f); acc[r].y = fmaf(ws, v.y, 0.f);
                acc[r].z = fmaf(ws, v.z, 0.f); acc[r].w = fmaf(ws, v.w, 0.f);
            }
            for (int t = 0; t < maxc; ++t) {
                float wt[R];
                float4 v[R];
#pragma unroll
                for (int r = 0; r < R; ++r) {                      // R independent row loads before any use
                    wt[r] = __shfl_sync(GRAPES_FULL_MASK, w[r], t);
                    const unsigned long long st = __shfl_sync(GRAPES_FULL_MASK, sg[r], t);
                    v[r] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (act && t < cnt[r]) v[r] = *reinterpret_cast<const float4*>(X + (size_t)st * ldx + c0);
                }
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    if (t < cnt[r]) {                               // warp-uniform: keeps the fma chain identical to k_agg
                        acc[r].x = fmaf(wt[r], v[r].x, acc[r].x); acc[r].y = fmaf(wt[r], v[r].y, acc[r].y);
                        acc[r].z = fmaf(wt[r], v[r].z, acc[r].z); acc[r].w = fmaf(wt[r], v[r].w, acc[r].w);
                    }
                }
            }
#pragma unroll
            for (int r = 0; r < R; ++r) {
                for (int pb = beg[r] + 32; pb < beg[r] + cnt[r]; pb += 32) {      // hub rows: sources beyond the first 32
                    const int p = pb + lane;
                    float hw = 0.f; unsigned long long hg = 0ull;
                    if (p < beg[r] + cnt[r]) {
                        const int s2 = in_src[p];
                        hw = dinv[s2] * dj[r];
                        hg = nodes ? (unsigned long long)nodes[s2] : (unsigned long long)s2;
                    }
                    const int c2 = min(32, beg[r] + cnt[r] - pb);
                    for (int t = 0; t < c2; ++t) {
                        const float wt2 = __shfl_sync(GRAPES_FULL_MASK, hw, t);
                        const unsigned long long st2 = __shfl_sync(GRAPES_FULL_MASK, hg, t);
                        if (act) {
                            const float4 v2 = *reinterpret_cast<const float4*>(X + (size_t)st2 * ldx + c0);
                            acc[r].x = fmaf(wt2, v2.x, acc[r].x); acc[r].y = fmaf(wt2, v2.y, acc[r].y);
                            acc[r].z = fmaf(wt2, v2.z, acc[r].z); acc[r].w = fmaf(wt2, v2.w, acc[r].w);
                        }
                    }
                }
                if (act && j0 + r < n) {
                    float4 a = acc[r];
                    if (bias) { a.x += bias[c0]; a.y += bias[c0 + 1]; a.z += bias[c0 + 2]; a.w += bias[c0 + 3]; }
                    if (relu) { a.x = fmaxf(a.x, 0.f); a.y = fmaxf(a.y, 0.f); a.z = fmaxf(a.z, 0.f); a.w = fmaxf(a.w, 0.f); }
                    const size_t o = (size_t)(j0 + r) * ldo + c0;
                    if (out) *reinterpret_cast<float4*>(out + o) = a;
                    if (out_hi) {                                   // 3xTF32 operand split for the tcgen05 GEMM
                        float4 h, l;
                        h.x = f32_to_tf32(a.x); h.y = f32_to_tf32(a.y); h.z = f32_to_tf32(a.z); h.w = f32_to_tf32(a.w);
                        l.x = f32_to_tf32(a.x - h.x); l.y = f32_to_tf32(a.y - h.y);
                        l.z = f32_to_tf32(a.z - h.z); l.w = f32_to_tf32(a.w - h.w);
                        *reinterpret_cast<float4*>(out_hi + o) = h;
                        *reinterpret_cast<float4*>(out_lo + o) = l;
                    }
                }
            }
        }
        // ---- virtual columns [F, ldo): indicator bits aggregated like features, the ones column, zero padding ----
        if (ldo > F) {
#pragma unroll
            for (int r = 0; r < R; ++r) {
                if (j0 + r >= n) continue;                          // warp-uniform
                float a = dj[r] * dj[r] * (float)((ibj[r] >> lane) & 1u);
                for (int t = 0; t < min(cnt[r], 32); ++t) {
                    const float wt = __shfl_sync(GRAPES_FULL_MASK, w[r], t);
                    const uint32_t bt = __shfl_sync(GRAPES_FULL_MASK, sb[r], t);
                    a = fmaf(wt, (float)((bt >> lane) & 1u), a);
                }
                for (int p = beg[r] + 32; p < beg[r] + cnt[r]; ++p) {      // hub rows
                    const int s2 = in_src[p];
                    a = fmaf(dinv[s2] * dj[r], has_ind ? (float)((ind_bits[s2] >> lane) & 1u) : 0.f, a);
                }
                const int c = F + lane;
                if (c < ldo) {
                    const float v = (lane < num_ind) ? a : (c == ones_col ? 1.f : 0.f);
                    const size_t o = (size_t)(j0 + r) * ldo + c;
                    if (out) out[o] = v;
                    if (out_hi) { const float h = f32_to_tf32(v); out_hi[o] = h; out_lo[o] = f32_to_tf32(v - h); }
                }
            }
        }
    }
}

// scalar (width-1) aggregation, one thread per row:  out[j] = dinv[j]^2 z[j] + sum w z[src] + bias
// optional `zero_out[j] = 0` clears a companion vector in the same pass.
__global__ void __launch_bounds__(256) k_agg_scalar(const float* __restrict__ z, int nparts, int part_stride,
                                                    const int* __restrict__ n_dev,
                                                    int cap_n, const int* __restrict__ in_off,
                                                    const int* __restrict__ in_src, const float* __restrict__ dinv,
                                                    const float* __restrict__ bias, float* __restrict__ out,
                                                    float* __restrict__ zero_out) {
    pdl_begin();
    const int n = min(*n_dev, cap_n);
    const float b = bias ? bias[0] : 0.f;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
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
        out[j] = a + b;
        if (zero_out) zero_out[j] = 0.f;
    }
}

// Transposed scalar aggregation for the hop graph, using the row-major edge list the expansion
// already produced (row i of `row_off` = edges whose SOURCE is prev position i):
//   dz[j]  = dinv[j]^2 dl[j]                                   for every row j          (k_dz_self)
//   dz[s] += sum_{e in row i, dst != s} dinv[s] dinv[dst] dl[dst]   s = e_src of row i   (k_dz_rows)
__global__ void __launch_bounds__(256) k_dz_self(const float* __restrict__ dl, const int* __restrict__ n_dev, int cap_n,
                                                 const float* __restrict__ dinv, float* __restrict__ dz) {
    pdl_begin();
    const int n = min(*n_dev, cap_n);
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x)
        dz[j] = dinv[j] * dinv[j] * dl[j];
}
__global__ void __launch_bounds__(256) k_dz_rows(const float* __restrict__ dl, const int* __restrict__ P_dev, int cap_P,
                                                 const int* __restrict__ row_off, const int* __restrict__ e_src,
                                                 const int* __restrict__ e_dst, const float* __restrict__ dinv,
                                                 float* __restrict__ dz) {
    pdl_begin();
    const int P = min(*P_dev, cap_P);
    const int lane = lane_id();
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < P; i += warps) {
        const int beg = row_off[i], end = row_off[i + 1];
        if (beg >= end) continue;
        const int s = e_src[beg];
        float a = 0.f;
        for (int e = beg + lane; e < end; e += 32) {
            const int d = e_dst[e];
            if (d != s) a = fmaf(dinv[d], dl[d], a);
        }
        a = warp_sum(a);
        if (lane == 0) dz[s] += dinv[s] * a;
    }
}

// v[j] = 1 / n for j < n  (d mean(logits) / d logits, main.py:228)
__global__ void __launch_bounds__(256) k_fill_inv_count(float* __restrict__ v, const int* __restrict__ n_dev, int cap_n) {
    pdl_begin();
    const int n = min(*n_dev, cap_n);
    const float inv = n > 0 ? 1.0f / (float)n : 0.f;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) v[j] = inv;
}

// both parts in one launch: blocks [0, nbA) do the self term for rows that are NOT expanded rows with an out-edge
// (the prev bitmap and the graph's CSR degree tell), blocks [nbA, ..) own the expanded rows with out-edges completely
// (self term + their out-edges) -> every row written once, no write race.  An expanded row without out-edges is a
// frontier node only when another row points to it (directed graphs); blocks B skip it, so blocks A take it.
__global__ void __launch_bounds__(256) k_dz_fused(const float* __restrict__ dl, const int* __restrict__ n_dev, int cap_n,
                                                  const int* __restrict__ P_dev, int cap_P,
                                                  const int* __restrict__ row_off, const int* __restrict__ e_src,
                                                  const int* __restrict__ e_dst, const float* __restrict__ dinv,
                                                  const uint32_t* __restrict__ bm_prev,
                                                  const int* __restrict__ batch_nodes,
                                                  const long long* __restrict__ indptr, int nbA,
                                                  float* __restrict__ dz) {
    pdl_begin();
    if ((int)blockIdx.x < nbA) {
        const int n = min(*n_dev, cap_n);
        for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += nbA * blockDim.x) {
            const int g = batch_nodes[j];
            if (!bitmap_test(bm_prev, g) || indptr[g + 1] == indptr[g]) dz[j] = dinv[j] * dinv[j] * dl[j];
        }
        return;
    }
    const int P = min(*P_dev, cap_P);
    const int lane = lane_id();
    const int nbB = gridDim.x - nbA;
    const int warps = (nbB * blockDim.x) >> 5;
    for (int i = (((int)blockIdx.x - nbA) * blockDim.x + threadIdx.x) >> 5; i < P; i += warps) {
        const int beg = row_off[i], end = row_off[i + 1];
        if (beg >= end) continue;
        const int s = e_src[beg];
        float a = 0.f;
        for (int e = beg + lane; e < end; e += 32) {
            const int d = e_dst[e];
            if (d != s) a = fmaf(dinv[d], dl[d], a);
        }
        a = warp_sum(a);
        if (lane == 0) dz[s] = dinv[s] * dinv[s] * dl[s] + dinv[s] * a;
    }
}

// ---------------------------------------------------------------------------------------
// Deterministic reductions
// ---------------------------------------------------------------------------------------
// out[c] (+)= scale * sum_r part[r*ld + c], r < R (R from device or host)
__global__ void __launch_bounds__(256) k_colsum(const float* __restrict__ part, const int* __restrict__ R_dev, int R_cap,
                                                int ld, int C, float scale, int accumulate, float* __restrict__ out) {
    pdl_begin();
    const int R = R_dev ? min(*R_dev, R_cap) : R_cap;
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < C; c += gridDim.x * blockDim.x) {
        float a = 0.f;
#pragma unroll 8
        for (int r = 0; r < R; ++r) a += part[(size_t)r * ld + c];
        a *= scale;
        out[c] = accumulate ? out[c] + a : a;
    }
}

// column sums of a tall matrix M[R x C] in two deterministic stages: slab partials, then k_colsum
__global__ void __launch_bounds__(256) k_colsum_slabs(const float* __restrict__ Mx, const int* __restrict__ R_dev,
                                                      int R_cap, int ld, int C, float* __restrict__ part) {
    pdl_begin();
    const int R = min(*R_dev, R_cap);
    const int slabs = gridDim.y;
    const int rows_per = (R + slabs - 1) / slabs;
    const int r0 = blockIdx.y * rows_per, r1 = min(R, r0 + rows_per);
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < C; c += gridDim.x * blockDim.x) {
        float a = 0.f;
#pragma unroll 8
        for (int r = r0; r < r1; ++r) a += Mx[(size_t)r * ld + c];
        part[(size_t)blockIdx.y * C + c] = a;
    }
}

// deterministic sum of a vector with a device-side length, two stages:
//   k_vec_sum_part: block b sums its fixed 4096-element chunk -> part[b]
//   k_vec_sum_final: one block adds the partials in index order;  *out (+)= scale * sum / (divide_by_n ? n : 1)
#define VS_CHUNK 4096
__global__ void __launch_bounds__(256) k_vec_sum_part(const float* __restrict__ v, const int* __restrict__ n_dev,
                                                      int cap_n, float* __restrict__ part) {
    pdl_begin();
    __shared__ float s[8];
    const int n = min(*n_dev, cap_n);
    const int base = blockIdx.x * VS_CHUNK;
    float a = 0.f;
    for (int i = base + threadIdx.x; i < min(n, base + VS_CHUNK); i += 256) a += v[i];
    a = warp_sum(a);
    if (lane_id() == 0) s[threadIdx.x >> 5] = a;
    __syncthreads();
    if (threadIdx.x == 0) part[blockIdx.x] = ((s[0] + s[1]) + (s[2] + s[3])) + ((s[4] + s[5]) + (s[6] + s[7]));
}
__global__ void __launch_bounds__(1024) k_vec_sum_final(const float* __restrict__ part, int nparts,
                                                        const int* __restrict__ n_dev, int cap_n, float scale,
                                                        int divide_by_n, int accumulate, float* out) {
    pdl_begin();
    __shared__ float s[32];
    const int n = n_dev ? min(*n_dev, cap_n) : cap_n;
    float a = 0.f;
    for (int i = threadIdx.x; i < nparts; i += blockDim.x) a += part[i];
    a = warp_sum(a);
    if (lane_id() == 0) s[threadIdx.x >> 5] = a;
    __syncthreads();
    if (threadIdx.x < 32) {
        float t = (threadIdx.x < (blockDim.x >> 5)) ? s[threadIdx.x] : 0.f;
        t = warp_sum(t);
        if (threadIdx.x == 0) {
            t *= scale;
            if (divide_by_n) t = (n > 0) ? t / (float)n : 0.f;
            *out = accumulate ? *out + t : t;
        }
    }
}

// ---------------------------------------------------------------------------------------
// fp32 SIMT tile GEMM: 128x128x16 CTA tile, 256 threads, 8x8 per thread (two 4-wide groups 64 apart
// so the float4 shared loads are bank-conflict free).  Operands may be K-contiguous ("KC":
// T[m*ld + k]) or MN-contiguous (T[k*ld + m]).  The tcgen05 path (gemm_tc.cu) replaces this for the
// sampler-layer shapes; this one stays as the generic / small-shape fallback ON THE DEVICE.
// ---------------------------------------------------------------------------------------
#define GB_M 128
#define GB_N 128
#define GB_K 16
#define G_THREADS 256
#define G_PAD 4

template <bool KC>
__device__ __forceinline__ void load_tile(const float* __restrict__ T, int ld, int mn0, int MN, int k0, int k1,
                                          float (*S)[GB_M + G_PAD]) {
    // fills S[kk][mm] = T(mn0 + mm, k0 + kk), zero outside [0,MN) x [k0,k1)
    const int tid = threadIdx.x;
    if (KC) {
        const int mm = tid >> 1, kk0 = (tid & 1) * 8;
        const int mrow = mn0 + mm;
        const float* src = T + (size_t)mrow * ld + k0 + kk0;
        const bool vec = ((ld & 3) == 0) && ((((size_t)T) & 15) == 0) && ((k0 & 3) == 0);
        if (mrow < MN && vec && k0 + kk0 + 8 <= k1) {
            const float4 a = *reinterpret_cast<const float4*>(src);
            const float4 b = *reinterpret_cast<const float4*>(src + 4);
            S[kk0 + 0][mm] = a.x; S[kk0 + 1][mm] = a.y; S[kk0 + 2][mm] = a.z; S[kk0 + 3][mm] = a.w;
            S[kk0 + 4][mm] = b.x; S[kk0 + 5][mm] = b.y; S[kk0 + 6][mm] = b.z; S[kk0 + 7][mm] = b.w;
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int k = k0 + kk0 + i;
                S[kk0 + i][mm] = (mrow < MN && k < k1) ? src[i] : 0.f;
            }
        }
    } else {
        const int mm = (tid & 31) * 4;
        const bool vec = ((ld & 3) == 0) && ((((size_t)T) & 15) == 0) && ((mn0 & 3) == 0);
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int kk = (tid >> 5) + r * 8;
            const int k = k0 + kk;
            const float* src = T + (size_t)k * ld + mn0 + mm;
            if (k < k1 && vec && mn0 + mm + 4 <= MN) {
                const float4 a = *reinterpret_cast<const float4*>(src);
                S[kk][mm] = a.x; S[kk][mm + 1] = a.y; S[kk][mm + 2] = a.z; S[kk][mm + 3] = a.w;
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) S[kk][mm + i] = (k < k1 && mn0 + mm + i < MN) ? src[i] : 0.f;
            }
        }
    }
}

__device__ __forceinline__ int g_row(int ty, int r) { return (r < 4) ? ty * 4 + r : 64 + ty * 4 + (r - 4); }
__device__ __forceinline__ int g_col(int tx, int c) { return (c < 4) ? tx * 4 + c : 64 + tx * 4 + (c - 4); }

// acc += A(m0.., k0..k1) * B(n0.., k0..k1)^T
template <bool A_KC, bool B_KC>
__device__ __forceinline__ void gemm_mainloop(const float* __restrict__ A, int lda, int m0, int M,
                                              const float* __restrict__ B, int ldb, int n0, int N, int k0, int k1,
                                              float (*As)[GB_M + G_PAD], float (*Bs)[GB_N + G_PAD],
                                              float (&acc)[8][8]) {
    const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
    for (int k = k0; k < k1; k += GB_K) {
        load_tile<A_KC>(A, lda, m0, M, k, k1, As);
        load_tile<B_KC>(B, ldb, n0, N, k, k1, Bs);
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < GB_K; ++kk) {
            const float4 a0 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 a1 = *reinterpret_cast<const float4*>(&As[kk][64 + ty * 4]);
            const float4 b0 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float4 b1 = *reinterpret_cast<const float4*>(&Bs[kk][64 + tx * 4]);
            const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int r = 0; r < 8; ++r)
#pragma unroll
                for (int c = 0; c < 8; ++c) acc[r][c] = fmaf(a[r], b[c], acc[r][c]);
        }
        __syncthreads();
    }
}

// Generic C[M x N] = A * B^T-like product (+bias[n]) (relu) (* mask: C = (G > 0) ? C : 0).
// M may come from the device (M_dev).  grid = (tiles_n, tiles_m_cap).
template <bool A_KC, bool B_KC>
__global__ void __launch_bounds__(G_THREADS) k_gemm(const float* __restrict__ A, int lda, const float* __restrict__ B,
                                                    int ldb, float* __restrict__ C, int ldc,
                                                    const int* __restrict__ M_dev, int M_cap, int N, int K,
                                                    const float* __restrict__ bias, int relu,
                                                    const float* __restrict__ relu_gate, int ldg) {
    pdl_begin();
    __shared__ __align__(16) float As[GB_K][GB_M + G_PAD];
    __shared__ __align__(16) float Bs[GB_K][GB_N + G_PAD];
    const int M = M_dev ? min(*M_dev, M_cap) : M_cap;
    const int n0 = blockIdx.x * GB_N;
    for (int m0 = blockIdx.y * GB_M; m0 < M; m0 += gridDim.y * GB_M) {
        float acc[8][8];
#pragma unroll
        for (int r = 0; r < 8; ++r)
#pragma unroll
            for (int c = 0; c < 8; ++c) acc[r][c] = 0.f;
        gemm_mainloop<A_KC, B_KC>(A, lda, m0, M, B, ldb, n0, N, 0, K, As, Bs, acc);
        const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int row = m0 + g_row(ty, r);
            if (row >= M) continue;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const int col = n0 + g_col(tx, c);
                if (col >= N) continue;
                float v = acc[r][c];
                if (bias) v += bias[col];
                if (relu) v = fmaxf(v, 0.f);
                if (relu_gate) v = (relu_gate[(size_t)row * ldg + col] > 0.f) ? v : 0.f;
                C[(size_t)row * ldc + col] = v;
            }
        }
    }
}

// keep bits of the 4 consecutive entries i0 .. i0 + 3 of a dropout site (one Philox call when i0 is a multiple of 4)
__device__ __forceinline__ uint32_t drop_bits4(unsigned long long seed, unsigned long long step, const DropParams& dp,
                                               unsigned long long i0) {
    if ((i0 & 3) == 0) return dropout_keep4(seed, step, dp.tag, dp.threshold, i0);
    uint32_t b = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) b |= dropout_keep(seed, step, dp.tag, dp.threshold, i0 + j) ? (1u << j) : 0u;
    return b;
}

// Dropout forms of the classifier's hidden layer (modules/gcn.py:33), kept apart from k_gemm / k_gemm_s so the plain
// products carry no dropout branch.  FWD: C = dropout(relu(A W^T + b)), A [M x K] and W [N x K] K-contiguous (layout 3),
// keep bit of entry (row, col) at i = row * N + col.  !FWD: C = (G > 0) ? s * (A B) : 0, A [M x K] K-contiguous, B [K x N]
// (layout 1): the backward of dropout(relu(.)) when G holds the dropped activations (zero wherever the unit was dropped
// or inactive).
template <bool FWD>
__global__ void __launch_bounds__(G_THREADS) k_gemm_dropout(const float* __restrict__ A, int lda,
                                                            const float* __restrict__ B, int ldb, float* __restrict__ C,
                                                            int ldc, const int* __restrict__ M_dev, int M_cap, int N,
                                                            int K, const float* __restrict__ bias,
                                                            const float* __restrict__ relu_gate, int ldg, DropParams dp) {
    pdl_begin();
    __shared__ __align__(16) float As[GB_K][GB_M + G_PAD];
    __shared__ __align__(16) float Bs[GB_K][GB_N + G_PAD];
    const int M = M_dev ? min(*M_dev, M_cap) : M_cap;
    const int n0 = blockIdx.x * GB_N;
    const unsigned long long seed = FWD ? dp.state[0] : 0ull, step = FWD ? dp.state[1] : 0ull;
    for (int m0 = blockIdx.y * GB_M; m0 < M; m0 += gridDim.y * GB_M) {
        float acc[8][8];
#pragma unroll
        for (int r = 0; r < 8; ++r)
#pragma unroll
            for (int c = 0; c < 8; ++c) acc[r][c] = 0.f;
        gemm_mainloop<true, FWD>(A, lda, m0, M, B, ldb, n0, N, 0, K, As, Bs, acc);
        const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int row = m0 + g_row(ty, r);
            if (row >= M) continue;
            uint32_t keep = 0u;
            if (FWD) {
                const unsigned long long i0 = (unsigned long long)row * N + n0 + tx * 4;
                keep = drop_bits4(seed, step, dp, i0) | (drop_bits4(seed, step, dp, i0 + 64) << 4);
            }
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const int col = n0 + g_col(tx, c);
                if (col >= N) continue;
                float v = acc[r][c];
                if (FWD) {
                    v = fmaxf(v + bias[col], 0.f);
                    v = ((keep >> c) & 1u) ? v * dp.scale : 0.f;
                } else {
                    v = (relu_gate[(size_t)row * ldg + col] > 0.f) ? v * dp.scale : 0.f;
                }
                C[(size_t)row * ldc + col] = v;
            }
        }
    }
}

// Split-K "TN" product for weight gradients:  P[slab][M x N] = sum_{r in slab} A[r, m] * B[r, n]
// (A: R x M row-major, B: R x N row-major, R = rows from the device).  grid = (tiles_n, tiles_m, slabs).
// Slab boundaries are multiples of GB_K so the summation order does not depend on the grid.
__global__ void __launch_bounds__(G_THREADS) k_gemm_tn_splitk(const float* __restrict__ A, int lda,
                                                              const float* __restrict__ B, int ldb,
                                                              const int* __restrict__ R_dev, int R_cap, int M, int N,
                                                              float* __restrict__ part) {
    pdl_begin();
    __shared__ __align__(16) float As[GB_K][GB_M + G_PAD];
    __shared__ __align__(16) float Bs[GB_K][GB_N + G_PAD];
    const int R = R_dev ? min(*R_dev, R_cap) : R_cap;
    const int slabs = gridDim.z;
    int rows_per = (R + slabs - 1) / slabs;
    rows_per = ((rows_per + GB_K - 1) / GB_K) * GB_K;
    const int r0 = min(R, (int)blockIdx.z * rows_per), r1 = min(R, r0 + rows_per);
    const int m0 = blockIdx.y * GB_M, n0 = blockIdx.x * GB_N;
    float acc[8][8];
#pragma unroll
    for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int c = 0; c < 8; ++c) acc[r][c] = 0.f;
    gemm_mainloop<false, false>(A, lda, m0, M, B, ldb, n0, N, r0, r1, As, Bs, acc);
    const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
    float* P = part + (size_t)blockIdx.z * M * N;
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int row = m0 + g_row(ty, r);
        if (row >= M) continue;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            const int col = n0 + g_col(tx, c);
            if (col < N) P[(size_t)row * N + col] = acc[r][c];
        }
    }
}

// ---------------------------------------------------------------------------------------
// Small-tile variant (64x64x16 CTA tile, 256 threads, 4x4 per thread) for the classifier-sized products
// (A = B + hops*k <= a few thousand rows): the 128x128 tiling would leave most of the 148 SMs idle.
// Same summation order over k as the large-tile kernel (k ascending, one fmaf per k).
// ---------------------------------------------------------------------------------------
#define GS_M 64
#define GS_N 64
#define GS_PAD 4

// One 16 x 64 operand tile = one float4 per thread.  fetch_tile_s reads it from global memory into registers (zeros outside
// the matrix), store_tile_s puts it into shared memory: the main loop fetches tile k+1 before it computes on tile k, so the
// global-load latency of these classifier-sized products (a handful of k-steps per CTA) overlaps the FMAs instead of
// being exposed once per k-step.  Same summation order as the unpipelined loop -> bitwise identical results.
template <bool KC>
__device__ __forceinline__ float4 fetch_tile_s(const float* __restrict__ T, int ld, int mn0, int MN, int k0, int k1) {
    const int tid = threadIdx.x;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    if (KC) {
        const int mm = tid >> 2, kk0 = (tid & 3) * 4;
        const int mrow = mn0 + mm;
        const float* src = T + (size_t)mrow * ld + k0 + kk0;
        const bool vec = ((ld & 3) == 0) && ((((size_t)T) & 15) == 0) && ((k0 & 3) == 0);
        if (mrow < MN && vec && k0 + kk0 + 4 <= k1) {
            a = *reinterpret_cast<const float4*>(src);
        } else if (mrow < MN) {
            if (k0 + kk0 + 0 < k1) a.x = src[0];
            if (k0 + kk0 + 1 < k1) a.y = src[1];
            if (k0 + kk0 + 2 < k1) a.z = src[2];
            if (k0 + kk0 + 3 < k1) a.w = src[3];
        }
    } else {
        const int mm = (tid & 15) * 4, kk = tid >> 4;
        const int k = k0 + kk;
        const float* src = T + (size_t)k * ld + mn0 + mm;
        const bool vec = ((ld & 3) == 0) && ((((size_t)T) & 15) == 0) && ((mn0 & 3) == 0);
        if (k < k1 && vec && mn0 + mm + 4 <= MN) {
            a = *reinterpret_cast<const float4*>(src);
        } else if (k < k1) {
            if (mn0 + mm + 0 < MN) a.x = src[0];
            if (mn0 + mm + 1 < MN) a.y = src[1];
            if (mn0 + mm + 2 < MN) a.z = src[2];
            if (mn0 + mm + 3 < MN) a.w = src[3];
        }
    }
    return a;
}
template <bool KC>
__device__ __forceinline__ void store_tile_s(const float4 a, float (*S)[GS_M + GS_PAD]) {
    const int tid = threadIdx.x;
    if (KC) {
        const int mm = tid >> 2, kk0 = (tid & 3) * 4;
        S[kk0 + 0][mm] = a.x; S[kk0 + 1][mm] = a.y; S[kk0 + 2][mm] = a.z; S[kk0 + 3][mm] = a.w;
    } else {
        const int mm = (tid & 15) * 4, kk = tid >> 4;
        S[kk][mm] = a.x; S[kk][mm + 1] = a.y; S[kk][mm + 2] = a.z; S[kk][mm + 3] = a.w;
    }
}

template <bool A_KC, bool B_KC>
__device__ __forceinline__ void gemm_mainloop_s(const float* __restrict__ A, int lda, int m0, int M,
                                                const float* __restrict__ B, int ldb, int n0, int N, int k0, int k1,
                                                float (*As)[GS_M + GS_PAD], float (*Bs)[GS_N + GS_PAD],
                                                float (&acc)[4][4]) {
    const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
    if (k0 >= k1) return;
    float4 ra = fetch_tile_s<A_KC>(A, lda, m0, M, k0, k1);
    float4 rb = fetch_tile_s<B_KC>(B, ldb, n0, N, k0, k1);
    for (int k = k0; k < k1; k += GB_K) {
        store_tile_s<A_KC>(ra, As);
        store_tile_s<B_KC>(rb, Bs);
        __syncthreads();
        if (k + GB_K < k1) {                                       // next tile in flight while this one is multiplied
            ra = fetch_tile_s<A_KC>(A, lda, m0, M, k + GB_K, k1);   // (two tiles ahead measured no better: 0.498 vs 0.494 ms/step)
            rb = fetch_tile_s<B_KC>(B, ldb, n0, N, k + GB_K, k1);
        }
#pragma unroll
        for (int kk = 0; kk < GB_K; ++kk) {
            const float4 a0 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 b0 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float a[4] = {a0.x, a0.y, a0.z, a0.w};
            const float b[4] = {b0.x, b0.y, b0.z, b0.w};
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[r][c] = fmaf(a[r], b[c], acc[r][c]);
        }
        __syncthreads();
    }
}

template <bool A_KC, bool B_KC>
__global__ void __launch_bounds__(G_THREADS) k_gemm_s(const float* __restrict__ A, int lda, const float* __restrict__ B,
                                                      int ldb, float* __restrict__ C, int ldc,
                                                      const int* __restrict__ M_dev, int M_cap, int N, int K,
                                                      const float* __restrict__ bias, int relu,
                                                      const float* __restrict__ relu_gate, int ldg) {
    pdl_begin();
    __shared__ __align__(16) float As[GB_K][GS_M + GS_PAD];
    __shared__ __align__(16) float Bs[GB_K][GS_N + GS_PAD];
    const int M = M_dev ? min(*M_dev, M_cap) : M_cap;
    const int n0 = blockIdx.x * GS_N;
    const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
    for (int m0 = blockIdx.y * GS_M; m0 < M; m0 += gridDim.y * GS_M) {
        float acc[4][4];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[r][c] = 0.f;
        gemm_mainloop_s<A_KC, B_KC>(A, lda, m0, M, B, ldb, n0, N, 0, K, As, Bs, acc);
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int row = m0 + ty * 4 + r;
            if (row >= M) continue;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int col = n0 + tx * 4 + c;
                if (col >= N) continue;
                float v = acc[r][c];
                if (bias) v += bias[col];
                if (relu) v = fmaxf(v, 0.f);
                if (relu_gate) v = (relu_gate[(size_t)row * ldg + col] > 0.f) ? v : 0.f;
                C[(size_t)row * ldc + col] = v;
            }
        }
    }
}

// small-tile form of k_gemm_dropout (classifier-sized products)
template <bool FWD>
__global__ void __launch_bounds__(G_THREADS) k_gemm_s_dropout(const float* __restrict__ A, int lda,
                                                              const float* __restrict__ B, int ldb,
                                                              float* __restrict__ C, int ldc,
                                                              const int* __restrict__ M_dev, int M_cap, int N, int K,
                                                              const float* __restrict__ bias,
                                                              const float* __restrict__ relu_gate, int ldg,
                                                              DropParams dp) {
    pdl_begin();
    __shared__ __align__(16) float As[GB_K][GS_M + GS_PAD];
    __shared__ __align__(16) float Bs[GB_K][GS_N + GS_PAD];
    const int M = M_dev ? min(*M_dev, M_cap) : M_cap;
    const int n0 = blockIdx.x * GS_N;
    const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
    const unsigned long long seed = FWD ? dp.state[0] : 0ull, step = FWD ? dp.state[1] : 0ull;
    for (int m0 = blockIdx.y * GS_M; m0 < M; m0 += gridDim.y * GS_M) {
        float acc[4][4];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[r][c] = 0.f;
        gemm_mainloop_s<true, FWD>(A, lda, m0, M, B, ldb, n0, N, 0, K, As, Bs, acc);
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int row = m0 + ty * 4 + r;
            if (row >= M) continue;
            const uint32_t keep = FWD ? drop_bits4(seed, step, dp, (unsigned long long)row * N + n0 + tx * 4) : 0u;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int col = n0 + tx * 4 + c;
                if (col >= N) continue;
                float v = acc[r][c];
                if (FWD) {
                    v = fmaxf(v + bias[col], 0.f);
                    v = ((keep >> c) & 1u) ? v * dp.scale : 0.f;
                } else {
                    v = (relu_gate[(size_t)row * ldg + col] > 0.f) ? v * dp.scale : 0.f;
                }
                C[(size_t)row * ldc + col] = v;
            }
        }
    }
}

__global__ void __launch_bounds__(G_THREADS) k_gemm_tn_splitk_s(const float* __restrict__ A, int lda,
                                                                const float* __restrict__ B, int ldb,
                                                                const int* __restrict__ R_dev, int R_cap, int M, int N,
                                                                float* __restrict__ part) {
    pdl_begin();
    __shared__ __align__(16) float As[GB_K][GS_M + GS_PAD];
    __shared__ __align__(16) float Bs[GB_K][GS_N + GS_PAD];
    const int R = R_dev ? min(*R_dev, R_cap) : R_cap;
    const int slabs = gridDim.z;
    int rows_per = (R + slabs - 1) / slabs;
    rows_per = ((rows_per + GB_K - 1) / GB_K) * GB_K;
    const int r0 = min(R, (int)blockIdx.z * rows_per), r1 = min(R, r0 + rows_per);
    const int m0 = blockIdx.y * GS_M, n0 = blockIdx.x * GS_N;
    float acc[4][4];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] = 0.f;
    gemm_mainloop_s<false, false>(A, lda, m0, M, B, ldb, n0, N, r0, r1, As, Bs, acc);
    const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
    float* P = part + (size_t)blockIdx.z * M * N;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int row = m0 + ty * 4 + r;
        if (row >= M) continue;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int col = n0 + tx * 4 + c;
            if (col < N) P[(size_t)row * N + col] = acc[r][c];
        }
    }
}

// out[i] (+)= scale * sum_s part[s*size + i]
__global__ void __launch_bounds__(256) k_reduce_slabs(const float* __restrict__ part, int slabs, int size, float scale,
                                                      int accumulate, float* __restrict__ out) {
    pdl_begin();
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < size; i += gridDim.x * blockDim.x) {
        float a = 0.f;
#pragma unroll 8
        for (int s = 0; s < slabs; ++s) a += part[(size_t)s * size + i];
        a *= scale;
        out[i] = accumulate ? out[i] + a : a;
    }
}

// ---------------------------------------------------------------------------------------
// Sampler-network layer 1+2 fused around the GEMM (out_dim == 1: gcn_gf and gcn_z, main.py:112-114).
//   forward : z[j]   = sum_d relu(Y[j,:] . W1[d,:] + b1[d]) * w2[d]           (hidden never stored)
//   backward: recompute pre = Y W1^T + b1;  dpre[j,d] = dz[j] * w2[d] * [pre > 0]      -> dpre (n x D)
//             dw2_part[cta][d] = sum_j dz[j] relu(pre[j,d]);  db1_part[cta][d] = sum_j dpre[j,d]
// One CTA owns 128 rows and walks the hidden dimension in chunks of 128.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(G_THREADS) k_l1_fwd(const float* __restrict__ Y, int ldy, const int* __restrict__ n_dev,
                                                      int cap_n, int K, const float* __restrict__ W1, int ldw, int D,
                                                      const float* __restrict__ b1, const float* __restrict__ w2,
                                                      float* __restrict__ z) {
    pdl_begin();
    __shared__ __align__(16) float As[GB_K][GB_M + G_PAD];
    __shared__ __align__(16) float Bs[GB_K][GB_N + G_PAD];
    const int n = min(*n_dev, cap_n);
    const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
    for (int m0 = blockIdx.x * GB_M; m0 < n; m0 += gridDim.x * GB_M) {
        float zrow[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) zrow[r] = 0.f;
        for (int n0 = 0; n0 < D; n0 += GB_N) {
            float acc[8][8];
#pragma unroll
            for (int r = 0; r < 8; ++r)
#pragma unroll
                for (int c = 0; c < 8; ++c) acc[r][c] = 0.f;
            gemm_mainloop<true, true>(Y, ldy, m0, n, W1, ldw, n0, D, 0, K, As, Bs, acc);
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const int col = n0 + g_col(tx, c);
                const float bb = (col < D) ? b1[col] : 0.f;
                const float ww = (col < D) ? w2[col] : 0.f;
#pragma unroll
                for (int r = 0; r < 8; ++r) zrow[r] = fmaf(fmaxf(acc[r][c] + bb, 0.f), ww, zrow[r]);
            }
        }
        // reduce over the 16 tx lanes that share a row (contiguous half-warp)
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            float v = zrow[r];
            v += __shfl_xor_sync(GRAPES_FULL_MASK, v, 8);
            v += __shfl_xor_sync(GRAPES_FULL_MASK, v, 4);
            v += __shfl_xor_sync(GRAPES_FULL_MASK, v, 2);
            v += __shfl_xor_sync(GRAPES_FULL_MASK, v, 1);
            const int row = m0 + g_row(ty, r);
            if (tx == 0 && row < n) z[row] = v;
        }
    }
}

__global__ void __launch_bounds__(G_THREADS) k_l1_bwd(const float* __restrict__ Y, int ldy, const int* __restrict__ n_dev,
                                                      int cap_n, int K, const float* __restrict__ W1, int ldw, int D,
                                                      const float* __restrict__ b1, const float* __restrict__ w2,
                                                      const float* __restrict__ dz, float* __restrict__ dpre, int ldd,
                                                      float* __restrict__ dw2_part, float* __restrict__ db1_part) {
    pdl_begin();
    __shared__ __align__(16) float As[GB_K][GB_M + G_PAD];
    __shared__ __align__(16) float Bs[GB_K][GB_N + G_PAD];
    __shared__ float red[16][GB_N];
    const int n = min(*n_dev, cap_n);
    const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
    // per-CTA partial sums over all the row tiles this CTA walks (fixed order -> deterministic)
    for (int n0 = 0; n0 < D; n0 += GB_N) {
        float pw2[8], pb1[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) { pw2[c] = 0.f; pb1[c] = 0.f; }
        for (int m0 = blockIdx.x * GB_M; m0 < n; m0 += gridDim.x * GB_M) {
            float acc[8][8];
#pragma unroll
            for (int r = 0; r < 8; ++r)
#pragma unroll
                for (int c = 0; c < 8; ++c) acc[r][c] = 0.f;
            gemm_mainloop<true, true>(Y, ldy, m0, n, W1, ldw, n0, D, 0, K, As, Bs, acc);
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const int row = m0 + g_row(ty, r);
                const float g = (row < n) ? dz[row] : 0.f;
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const int col = n0 + g_col(tx, c);
                    if (col >= D) continue;
                    const float pre = acc[r][c] + b1[col];
                    const float o = fmaxf(pre, 0.f);
                    const float d = (pre > 0.f) ? g * w2[col] : 0.f;
                    pw2[c] = fmaf(g, o, pw2[c]);
                    pb1[c] += d;
                    if (row < n) dpre[(size_t)row * ldd + col] = d;
                }
            }
        }
        // reduce the 16 ty groups column-wise through shared memory, in a fixed order
        for (int which = 0; which < 2; ++which) {
#pragma unroll
            for (int c = 0; c < 8; ++c) red[ty][g_col(tx, c)] = which ? pb1[c] : pw2[c];
            __syncthreads();
            if (threadIdx.x < GB_N) {
                float a = 0.f;
#pragma unroll
                for (int t = 0; t < 16; ++t) a += red[t][threadIdx.x];
                const int col = n0 + threadIdx.x;
                if (col < D) (which ? db1_part : dw2_part)[(size_t)blockIdx.x * D + col] = a;
            }
            __syncthreads();
        }
    }
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

// the two dropout forms of the classifier's hidden layer; same tile choice as grapes_gemm
template <bool FWD>
static int launch_gemm_dropout(grapes_ctx* ctx, const float* A, int lda, const float* B, int ldb, float* C, int ldc,
                               const int* M_dev, int M_cap, int N, int K, const float* bias, const float* relu_gate,
                               int ldg, DropParams dp, cudaStream_t s) {
    if (M_cap == 0) return GRAPES_OK;
    grapes_count_launches(1);
    if ((long long)grapes_div_up(N, GB_N) * grapes_div_up(M_cap, GB_M) < ctx->sm_count) {
        dim3 grid(grapes_div_up(N, GS_N), grapes_min_i(grapes_div_up(M_cap, GS_M), 65535));
        pdl((k_gemm_s_dropout<FWD>), grid, G_THREADS, 0, s)(A, lda, B, ldb, C, ldc, M_dev, M_cap, N, K, bias, relu_gate,
                                                          ldg, dp);
    } else {
        const int tiles_n = grapes_div_up(N, GB_N);
        const int tiles_m = grapes_min_i(grapes_div_up(M_cap, GB_M), grapes_max_i(1, (ctx->sm_count * 4) / tiles_n));
        pdl((k_gemm_dropout<FWD>), dim3(tiles_n, tiles_m), G_THREADS, 0, s)(A, lda, B, ldb, C, ldc, M_dev, M_cap, N, K,
                                                                           bias, relu_gate, ldg, dp);
    }
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

// the owner table of the peer aggregations: HOST arrays of `world` row bases and world + 1 bounds into the parameter struct
static int peer_rows(const void* const* x_rows, const int64_t* bounds, int world, PeerRows& P, size_t& al) {
    GRAPES_REQUIRE(x_rows && bounds, "null argument");
    GRAPES_REQUIRE(world >= 1 && world <= GRAPES_PEER_MAX, "1 to 8 row owners");
    GRAPES_REQUIRE(bounds[0] == 0 && bounds[world] < (1ll << 31), "bounds[0] must be 0 and bounds[world] fit int32");
    P = PeerRows{};
    for (int o = 0; o < GRAPES_PEER_MAX; ++o) P.bound[o] = INT_MAX;
    for (int o = 0; o < world; ++o) {
        GRAPES_REQUIRE(bounds[o] <= bounds[o + 1], "bounds must not decrease");
        GRAPES_REQUIRE(x_rows[o] || bounds[o] == bounds[o + 1], "null row base of a non-empty window");
        P.base[o] = x_rows[o];
        P.bound[o] = (int)bounds[o];
        al |= (size_t)x_rows[o];
    }
    return GRAPES_OK;
}

// one k_agg_px launch in the widest vector form the layout allows (the form k_agg would take)
template <bool W64>
static void launch_agg_px(grapes_ctx* ctx, const PeerRows& P, int x_bf16, int F, int ldx, const int* nodes,
                          const int* n_dev, int cap_n, const typename GrapesOff<W64>::T* in_off, const int* in_src,
                          const float* dinv, const uint32_t* ind_bits, int num_ind, const float* bias, int relu,
                          float* out, int ldo, float* out_hi, float* out_lo, int ones_col, size_t al, cudaStream_t s) {
    const int blocks = grid_for(ctx, (long long)cap_n * 32, 256, 8);
    al |= ((size_t)out) | ((size_t)out_hi) | ((size_t)out_lo);
    const bool v4 = (al & 15) == 0 && (F % 4 == 0) && (ldx % 4 == 0) && (ldo % 4 == 0);
    const bool v2 = (al & 7) == 0 && (F % 2 == 0) && (ldx % 2 == 0) && (ldo % 2 == 0);
#define AGGPX(VEC, XB) pdl((k_agg_px<VEC, XB, W64>), blocks, 256, 0, s)(P, F, ldx, nodes, n_dev, cap_n, in_off, in_src, \
                                                                         dinv, ind_bits, num_ind, bias, relu, out, ldo, \
                                                                         out_hi, out_lo, ones_col)
    if (x_bf16) {
        if (v4) AGGPX(4, true); else if (v2) AGGPX(2, true); else AGGPX(1, true);
    } else {
        if (v4) AGGPX(4, false); else if (v2) AGGPX(2, false); else AGGPX(1, false);
    }
#undef AGGPX
}

static int g_agg_variant = 0;
#define AGG_MIN_ROWS 4096               // smallest row capacity that takes the multi-row / TMA-staged forms (aligned widths)

extern "C" {

// 0 (default): the forms chosen by shape; 1: the register-staged kernels k_agg<4|2|1> only, the bit-exact reference
// that the parity tests compare k_agg_tma with
int grapes_agg_variant(int v) {
    GRAPES_REQUIRE(v == 0 || v == 1, "aggregation variant is 0 (default) or 1 (register-staged)");
    g_agg_variant = v;
    return GRAPES_OK;
}

static int aggregate_impl(grapes_ctx* ctx, const void* Xv, int x_bf16, int F, int ldx, const int* nodes, const int* n_dev,
                          int cap_n, const int* in_off, const int* in_src, const float* dinv, const uint32_t* ind_bits,
                          int num_ind, const float* bias, int relu, float* out, int ldo, float* out_hi, float* out_lo,
                          int ones_col, void* stream) {
    const float* X = reinterpret_cast<const float*>(Xv);
    GRAPES_REQUIRE(ctx && X && n_dev && in_off && in_src && dinv && (out || out_hi), "null argument");
    GRAPES_REQUIRE((out_hi == nullptr) == (out_lo == nullptr), "out_hi and out_lo go together");
    GRAPES_REQUIRE(ones_col < 0 || (ones_col >= F + num_ind && ones_col < ldo), "ones_col must lie in the pad columns");
    GRAPES_REQUIRE(ldo >= F + num_ind, "ldo too small");
    GRAPES_REQUIRE(num_ind == 0 || ind_bits, "indicator columns need ind_bits");
    GRAPES_REQUIRE(num_ind <= 8, "at most 8 indicator columns");
    cudaStream_t s = (cudaStream_t)stream;
    const int blocks = grid_for(ctx, (long long)cap_n * 32, 256, 8);
    const size_t al = ((size_t)X) | ((size_t)out) | ((size_t)out_hi) | ((size_t)out_lo);
    const bool a16 = (al & 15) == 0;
    const bool a8 = (al & 7) == 0;
    if (x_bf16) {
        // bf16 feature table (papers100M-shaped config): TMA-staged form when the shape allows, else one warp per row
        if (a16 && cap_n >= 4096 &&
            grapes_launch_agg_tma(ctx, Xv, 1, F, ldx, nodes, n_dev, cap_n, in_off, in_src, dinv, ind_bits, num_ind, bias, relu,
                                  out, ldo, out_hi, out_lo, ones_col, cap_n > (1 << 19) ? 32 : 16,
                                  cap_n > (1 << 19) ? 1 : 2, s) == 0) {
            grapes_count_launches(1);
            GRAPES_LAUNCH_OK();
            return GRAPES_OK;
        }
        if (a16 && (F % 4 == 0) && (ldx % 4 == 0) && (ldo % 4 == 0))
            pdl((k_agg<4, true>), blocks, 256, 0, s)(Xv, F, ldx, nodes, n_dev, cap_n, in_off, in_src, dinv, ind_bits, num_ind,
                                                     bias, relu, out, ldo, out_hi, out_lo, ones_col);
        else if ((F % 2 == 0) && (ldx % 2 == 0) && (ldo % 2 == 0) && a8)
            pdl((k_agg<2, true>), blocks, 256, 0, s)(Xv, F, ldx, nodes, n_dev, cap_n, in_off, in_src, dinv, ind_bits, num_ind,
                                                     bias, relu, out, ldo, out_hi, out_lo, ones_col);
        else
            pdl((k_agg<1, true>), blocks, 256, 0, s)(Xv, F, ldx, nodes, n_dev, cap_n, in_off, in_src, dinv, ind_bits, num_ind,
                                                     bias, relu, out, ldo, out_hi, out_lo, ones_col);
        grapes_count_launches(1);
        GRAPES_LAUNCH_OK();
        return GRAPES_OK;
    }
    const bool shaped = g_agg_variant == 0;
    const bool whole = cap_n > (1 << 19);
    if (shaped && a16 && (F % 4 != 0) && (ldx % 4 == 0) && ldx >= ((F + 3) & ~3) && (ldo % 4 == 0) && (ldo - F <= 32) &&
        cap_n >= 256) {
        // rows whose width is not a multiple of 4 (Reddit 602, Cora 1433) on a table with a padded row pitch: TMA-staged
        // form with a partial last feature lane.  Reddit-shape hop: 2 CTAs/SM 0.236, 1 CTA/SM 0.272 ms/step
        if (grapes_launch_agg_tma(ctx, X, 0, F, ldx, nodes, n_dev, cap_n, in_off, in_src, dinv, ind_bits, num_ind, bias, relu,
                                  out, ldo, out_hi, out_lo, ones_col, whole ? 32 : 16, whole ? 1 : 2, s) == 0) {
            grapes_count_launches(1);
            GRAPES_LAUNCH_OK();
            return GRAPES_OK;
        }
    }
    if (shaped && a16 && (F % 4 == 0) && (ldx % 4 == 0) && (ldo % 4 == 0) && (ldo - F <= 32) && cap_n >= AGG_MIN_ROWS) {
        // rows staged by TMA bulk copies (spmm_tma.cu).  Measured on B200 (scripts/bench_spmm.py): frontier-sized
        // launches are best with 8-entry chunks and 3 CTAs/SM (ncu: 21.8 us against 23.3 at 2 CTAs/SM, 24.6 at 4), wide
        // rows with 2 CTAs/SM, whole-graph launches with 32-entry chunks and 1 CTA/SM.
        const int ec = whole ? 32 : (F > 256 ? 16 : 8), cps = whole ? 1 : (F > 256 ? 2 : 3);
        if (grapes_launch_agg_tma(ctx, X, 0, F, ldx, nodes, n_dev, cap_n, in_off, in_src, dinv, ind_bits, num_ind, bias, relu,
                                  out, ldo, out_hi, out_lo, ones_col, ec, cps, s) == 0) {
            grapes_count_launches(1);
            GRAPES_LAUNCH_OK();
            return GRAPES_OK;
        }
        // shapes k_agg_tma does not cover: 2 rows per warp with interleaved load chains, the best register-staged form
        // (products-shaped hop, 65k rows)
        pdl((k_agg_rows<2, 4>), grid_for(ctx, (long long)grapes_div_up(cap_n, 2) * 32, 256, 4), 256, 0, s)(
            X, F, ldx, nodes, n_dev, cap_n, in_off, in_src, dinv, ind_bits, num_ind, bias, relu, out, ldo, out_hi, out_lo,
            ones_col);
    } else if (a16 && (F % 4 == 0) && (ldx % 4 == 0) && (ldo % 4 == 0))
        pdl((k_agg<4>), blocks, 256, 0, s)(X, F, ldx, nodes, n_dev, cap_n, in_off, in_src, dinv, ind_bits, num_ind, bias,
                                        relu, out, ldo, out_hi, out_lo, ones_col);
    else if (a8 && (F % 2 == 0) && (ldx % 2 == 0) && (ldo % 2 == 0))
        pdl((k_agg<2>), blocks, 256, 0, s)(X, F, ldx, nodes, n_dev, cap_n, in_off, in_src, dinv, ind_bits, num_ind, bias,
                                        relu, out, ldo, out_hi, out_lo, ones_col);
    else
        pdl((k_agg<1>), blocks, 256, 0, s)(X, F, ldx, nodes, n_dev, cap_n, in_off, in_src, dinv, ind_bits, num_ind, bias,
                                        relu, out, ldo, out_hi, out_lo, ones_col);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_aggregate(grapes_ctx* ctx, const float* X, int F, int ldx, const int* nodes, const int* n_dev, int cap_n,
                     const int* in_off, const int* in_src, const float* dinv, const uint32_t* ind_bits, int num_ind,
                     const float* bias, int relu, float* out, int ldo, float* out_hi, float* out_lo, int ones_col,
                     void* stream) {
    return aggregate_impl(ctx, X, 0, F, ldx, nodes, n_dev, cap_n, in_off, in_src, dinv, ind_bits, num_ind, bias, relu, out,
                          ldo, out_hi, out_lo, ones_col, stream);
}

int grapes_aggregate_bf16(grapes_ctx* ctx, const void* X_bf16, int F, int ldx, const int* nodes, const int* n_dev,
                          int cap_n, const int* in_off, const int* in_src, const float* dinv, const uint32_t* ind_bits,
                          int num_ind, const float* bias, int relu, float* out, int ldo, float* out_hi, float* out_lo,
                          int ones_col, void* stream) {
    return aggregate_impl(ctx, X_bf16, 1, F, ldx, nodes, n_dev, cap_n, in_off, in_src, dinv, ind_bits, num_ind, bias, relu,
                          out, ldo, out_hi, out_lo, ones_col, stream);
}

int grapes_aggregate_rows64(grapes_ctx* ctx, const void* X, int x_bf16, int F, int ldx, const int* slab_dev, int cap_r,
                            const int64_t* in_off, const int* in_src, const float* dinv, const float* bias, float* out,
                            int ldo, void* stream) {
    GRAPES_REQUIRE(ctx && X && slab_dev && in_off && in_src && dinv && out, "null argument");
    GRAPES_REQUIRE(F > 0 && ldx >= F && ldo >= F, "bad shape");
    if (cap_r <= 0) return GRAPES_OK;
    cudaStream_t s = (cudaStream_t)stream;
    const long long* off = reinterpret_cast<const long long*>(in_off);
    const bool shaped = g_agg_variant == 0;
    const bool whole = cap_r > (1 << 19);
    const size_t al = ((size_t)X) | ((size_t)out);
    const bool a16 = (al & 15) == 0, a8 = (al & 7) == 0;
    // the forms and launch shapes grapes_aggregate / grapes_aggregate_bf16 pick for a whole graph of cap_r rows
    bool launched = false;
    if (shaped && a16) {
        if (x_bf16) {
            if (cap_r >= 4096)
                launched = grapes_launch_agg_tma(ctx, X, 1, F, ldx, nullptr, slab_dev, cap_r, off, in_src, dinv, nullptr, 0,
                                                 bias, 0, out, ldo, nullptr, nullptr, -1, whole ? 32 : 16, whole ? 1 : 2, s,
                                                 1) == 0;
        } else if ((F % 4 != 0) && (ldx % 4 == 0) && ldx >= ((F + 3) & ~3) && (ldo % 4 == 0) && (ldo - F <= 32) &&
                   cap_r >= 256) {
            launched = grapes_launch_agg_tma(ctx, X, 0, F, ldx, nullptr, slab_dev, cap_r, off, in_src, dinv, nullptr, 0,
                                             bias, 0, out, ldo, nullptr, nullptr, -1, whole ? 32 : 16, whole ? 1 : 2, s, 1) == 0;
        } else if ((F % 4 == 0) && (ldx % 4 == 0) && (ldo % 4 == 0) && (ldo - F <= 32) && cap_r >= AGG_MIN_ROWS) {
            const int ec = whole ? 32 : (F > 256 ? 16 : 8), cps = whole ? 1 : (F > 256 ? 2 : 3);
            launched = grapes_launch_agg_tma(ctx, X, 0, F, ldx, nullptr, slab_dev, cap_r, off, in_src, dinv, nullptr, 0,
                                             bias, 0, out, ldo, nullptr, nullptr, -1, ec, cps, s, 1) == 0;
        }
    }
    if (!launched) {                       // register-staged: layouts the TMA form does not take, and agg variant 1
        const int blocks = grid_for(ctx, (long long)cap_r * 32, 256, 8);
#define AGG64(VEC, XB) pdl((k_agg<VEC, XB, true>), blocks, 256, 0, s)(X, F, ldx, nullptr, slab_dev, cap_r, off, in_src, dinv, \
                                                                       nullptr, 0, bias, 0, out, ldo, nullptr, nullptr, -1)
        const bool v4 = a16 && (F % 4 == 0) && (ldx % 4 == 0) && (ldo % 4 == 0);
        const bool v2 = a8 && (F % 2 == 0) && (ldx % 2 == 0) && (ldo % 2 == 0);
        if (x_bf16) {
            if (v4) AGG64(4, true); else if (v2) AGG64(2, true); else AGG64(1, true);
        } else {
            if (v4) AGG64(4, false); else if (v2) AGG64(2, false); else AGG64(1, false);
        }
#undef AGG64
    }
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_aggregate_peer(grapes_ctx* ctx, const void* const* x_rows, const int64_t* bounds, int world, int x_bf16, int F,
                          int ldx, const int* nodes, const int* n_dev, int cap_n, const int* in_off, const int* in_src,
                          const float* dinv, const uint32_t* ind_bits, int num_ind, const float* bias, int relu,
                          float* out, int ldo, float* out_hi, float* out_lo, int ones_col, void* stream) {
    GRAPES_REQUIRE(ctx && n_dev && in_off && in_src && dinv && (out || out_hi), "null argument");
    GRAPES_REQUIRE((out_hi == nullptr) == (out_lo == nullptr), "out_hi and out_lo go together");
    GRAPES_REQUIRE(F > 0 && ldx >= F, "bad shape");
    GRAPES_REQUIRE(ones_col < 0 || (ones_col >= F + num_ind && ones_col < ldo), "ones_col must lie in the pad columns");
    GRAPES_REQUIRE(ldo >= F + num_ind, "ldo too small");
    GRAPES_REQUIRE(num_ind == 0 || ind_bits, "indicator columns need ind_bits");
    GRAPES_REQUIRE(num_ind <= 8, "at most 8 indicator columns");
    PeerRows P;
    size_t al = 0;
    const int rc = peer_rows(x_rows, bounds, world, P, al);
    if (rc != GRAPES_OK) return rc;
    if (cap_n > 0)
        launch_agg_px<false>(ctx, P, x_bf16, F, ldx, nodes, n_dev, cap_n, in_off, in_src, dinv, ind_bits, num_ind, bias,
                             relu, out, ldo, out_hi, out_lo, ones_col, al, (cudaStream_t)stream);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_aggregate_rows64_peer_x(grapes_ctx* ctx, const void* const* x_rows, const int64_t* bounds, int world,
                                   int x_bf16, int F, int ldx, const int* slab_dev, int cap_r, const int64_t* in_off,
                                   const int* in_src, const float* dinv, const float* bias, float* out, int ldo,
                                   void* stream) {
    if (cap_r <= 0) return GRAPES_OK;                    // an empty window: nothing to read or write
    GRAPES_REQUIRE(ctx && slab_dev && in_off && in_src && dinv && out, "null argument");
    GRAPES_REQUIRE(F > 0 && ldx >= F && ldo >= F, "bad shape");
    PeerRows P;
    size_t al = 0;
    const int rc = peer_rows(x_rows, bounds, world, P, al);
    if (rc != GRAPES_OK) return rc;
    launch_agg_px<true>(ctx, P, x_bf16, F, ldx, nullptr, slab_dev, cap_r, reinterpret_cast<const long long*>(in_off),
                        in_src, dinv, nullptr, 0, bias, 0, out, ldo, nullptr, nullptr, -1, al, (cudaStream_t)stream);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_aggregate_rows64_peer(grapes_ctx* ctx, const void* const* z_rows, const int64_t* bounds, int world, int F,
                                 int ldz, const int* slab_dev, int cap_r, const int64_t* in_off, const int* in_src,
                                 const float* dinv, const float* bias, float* out, int ldo, void* stream) {
    return grapes_aggregate_rows64_peer_x(ctx, z_rows, bounds, world, 0, F, ldz, slab_dev, cap_r, in_off, in_src, dinv,
                                          bias, out, ldo, stream);
}

int grapes_aggregate_scalar(grapes_ctx* ctx, const float* z, int nparts, int part_stride, const int* n_dev, int cap_n, const int* in_off,
                            const int* in_src, const float* dinv, const float* bias, float* out, float* zero_out,
                            void* stream) {
    GRAPES_REQUIRE(ctx && z && n_dev && in_off && in_src && dinv && out, "null argument");
    GRAPES_REQUIRE(nparts >= 1, "nparts >= 1");
    pdl((k_agg_scalar), grid_for(ctx, cap_n, 256), 256, 0, (cudaStream_t)stream)(z, nparts, part_stride, n_dev, cap_n, in_off, in_src, dinv,
                                                                              bias, out, zero_out);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_aggregate_scalar_T(grapes_ctx* ctx, const float* dl, const int* n_dev, int cap_n, const int* P_dev,
                              int cap_P, const int* row_off, const int* e_src, const int* e_dst, const float* dinv,
                              const uint32_t* bm_prev, const int* batch_nodes, const int64_t* indptr, float* dz,
                              void* stream) {
    GRAPES_REQUIRE(ctx && dl && n_dev && P_dev && row_off && e_src && e_dst && dinv && dz, "null argument");
    GRAPES_REQUIRE(!bm_prev == !batch_nodes && !bm_prev == !indptr, "bm_prev, batch_nodes and indptr go together");
    cudaStream_t s = (cudaStream_t)stream;
    if (bm_prev) {
        const int nbA = grid_for(ctx, cap_n, 256), nbB = grid_for(ctx, (long long)cap_P * 32, 256);
        pdl((k_dz_fused), nbA + nbB, 256, 0, s)(dl, n_dev, cap_n, P_dev, cap_P, row_off, e_src, e_dst, dinv, bm_prev,
                                             batch_nodes, reinterpret_cast<const long long*>(indptr), nbA, dz);
        grapes_count_launches(1);
        GRAPES_LAUNCH_OK();
        return GRAPES_OK;
    }
    pdl((k_dz_self), grid_for(ctx, cap_n, 256), 256, 0, s)(dl, n_dev, cap_n, dinv, dz);
    grapes_count_launches(1);
    pdl((k_dz_rows), grid_for(ctx, (long long)cap_P * 32, 256), 256, 0, s)(dl, P_dev, cap_P, row_off, e_src, e_dst, dinv,
                                                                         dz);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_fill_inv_count(grapes_ctx* ctx, float* v, const int* n_dev, int cap_n, void* stream) {
    GRAPES_REQUIRE(ctx && v && n_dev, "null argument");
    pdl((k_fill_inv_count), grid_for(ctx, cap_n, 256), 256, 0, (cudaStream_t)stream)(v, n_dev, cap_n);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_vec_sum(grapes_ctx* ctx, const float* v, const int* n_dev, int cap_n, float scale, int divide_by_n,
                   int accumulate, float* out, void* stream) {
    GRAPES_REQUIRE(ctx && v && n_dev && out, "null argument");
    const int nparts = grapes_max_i(1, grapes_div_up(cap_n, VS_CHUNK));
    GRAPES_REQUIRE((size_t)nparts * sizeof(float) <= ctx->partials_bytes, "partial buffer too small");
    pdl((k_vec_sum_part), nparts, 256, 0, (cudaStream_t)stream)(v, n_dev, cap_n, ctx->partials);
    grapes_count_launches(1);
    pdl((k_vec_sum_final), 1, 1024, 0, (cudaStream_t)stream)(ctx->partials, nparts, n_dev, cap_n, scale, divide_by_n,
                                                          accumulate, out);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

// layout: bit0 = A is K-contiguous, bit1 = B is K-contiguous
int grapes_gemm(grapes_ctx* ctx, int layout, const float* A, int lda, const float* B, int ldb, float* C, int ldc,
                const int* M_dev, int M_cap, int N, int K, const float* bias, int relu, const float* relu_gate,
                int ldg, void* stream) {
    GRAPES_REQUIRE(ctx && A && B && C, "null argument");
    GRAPES_REQUIRE(M_cap >= 0 && N > 0 && K > 0, "bad shape");
    if (M_cap == 0) return GRAPES_OK;
    cudaStream_t s = (cudaStream_t)stream;
    grapes_count_launches(1);
    if ((long long)grapes_div_up(N, GB_N) * grapes_div_up(M_cap, GB_M) < ctx->sm_count) {
        // classifier-sized product: 64x64 tiles so the grid covers the GPU
        dim3 grid(grapes_div_up(N, GS_N), grapes_min_i(grapes_div_up(M_cap, GS_M), 65535));
        switch (layout & 3) {
            case 3: pdl((k_gemm_s<true, true>), grid, G_THREADS, 0, s)(A, lda, B, ldb, C, ldc, M_dev, M_cap, N, K, bias, relu, relu_gate, ldg); break;
            case 1: pdl((k_gemm_s<true, false>), grid, G_THREADS, 0, s)(A, lda, B, ldb, C, ldc, M_dev, M_cap, N, K, bias, relu, relu_gate, ldg); break;
            case 2: pdl((k_gemm_s<false, true>), grid, G_THREADS, 0, s)(A, lda, B, ldb, C, ldc, M_dev, M_cap, N, K, bias, relu, relu_gate, ldg); break;
            default: pdl((k_gemm_s<false, false>), grid, G_THREADS, 0, s)(A, lda, B, ldb, C, ldc, M_dev, M_cap, N, K, bias, relu, relu_gate, ldg); break;
        }
        GRAPES_LAUNCH_OK();
        return GRAPES_OK;
    }
    const int tiles_n = grapes_div_up(N, GB_N);
    int tiles_m = grapes_div_up(M_cap, GB_M);
    const int max_y = grapes_max_i(1, (ctx->sm_count * 4) / tiles_n);
    tiles_m = grapes_min_i(tiles_m, max_y);
    dim3 grid(tiles_n, tiles_m);
    switch (layout & 3) {
        case 3: pdl((k_gemm<true, true>), grid, G_THREADS, 0, s)(A, lda, B, ldb, C, ldc, M_dev, M_cap, N, K, bias, relu, relu_gate, ldg); break;
        case 1: pdl((k_gemm<true, false>), grid, G_THREADS, 0, s)(A, lda, B, ldb, C, ldc, M_dev, M_cap, N, K, bias, relu, relu_gate, ldg); break;
        case 2: pdl((k_gemm<false, true>), grid, G_THREADS, 0, s)(A, lda, B, ldb, C, ldc, M_dev, M_cap, N, K, bias, relu, relu_gate, ldg); break;
        default: pdl((k_gemm<false, false>), grid, G_THREADS, 0, s)(A, lda, B, ldb, C, ldc, M_dev, M_cap, N, K, bias, relu, relu_gate, ldg); break;
    }
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_gemm_bias_relu_dropout(grapes_ctx* ctx, const float* A, int lda, const float* W, int ldw, float* H, int ldh,
                                  const int* M_dev, int M_cap, int N, int K, const float* bias,
                                  unsigned long long* drop_state, uint32_t tag, uint32_t threshold, float scale,
                                  void* stream) {
    GRAPES_REQUIRE(ctx && A && W && H && bias && drop_state, "null argument");
    GRAPES_REQUIRE(M_cap >= 0 && N > 0 && K > 0 && tag >= 1u && threshold <= (1u << 24), "bad shape or dropout parameters");
    DropParams dp = {drop_state, tag, threshold, scale};
    return launch_gemm_dropout<true>(ctx, A, lda, W, ldw, H, ldh, M_dev, M_cap, N, K, bias, nullptr, 0, dp,
                                     (cudaStream_t)stream);
}

int grapes_gemm_gated_scaled(grapes_ctx* ctx, const float* A, int lda, const float* B, int ldb, float* C, int ldc,
                             const int* M_dev, int M_cap, int N, int K, const float* gate, int ldg, float scale,
                             void* stream) {
    GRAPES_REQUIRE(ctx && A && B && C && gate, "null argument");
    GRAPES_REQUIRE(M_cap >= 0 && N > 0 && K > 0, "bad shape");
    DropParams dp = {nullptr, 0u, 0u, scale};
    return launch_gemm_dropout<false>(ctx, A, lda, B, ldb, C, ldc, M_dev, M_cap, N, K, nullptr, gate, ldg, dp,
                                      (cudaStream_t)stream);
}

// out[M x N] (+)= scale * A[R x M]^T B[R x N]   (weight gradients; deterministic split over rows)
int grapes_gemm_tn(grapes_ctx* ctx, const float* A, int lda, const float* B, int ldb, const int* R_dev, int R_cap,
                   int M, int N, float scale, int accumulate, float* out, void* stream) {
    GRAPES_REQUIRE(ctx && A && B && out, "null argument");
    cudaStream_t s = (cudaStream_t)stream;
    const bool small = R_cap <= 16384;                 // classifier-sized: 64x64 tiles, fewer / shorter slabs
    const int tiles_n = grapes_div_up(N, small ? GS_N : GB_N), tiles_m = grapes_div_up(M, small ? GS_M : GB_M);
    int slabs = grapes_max_i(1, (small ? 2 * ctx->sm_count : ctx->sm_count) / (tiles_n * tiles_m));
    slabs = grapes_min_i(slabs, grapes_max_i(1, grapes_div_up(R_cap, 4 * GB_K)));
    const size_t need = (size_t)slabs * M * N * sizeof(float);
    GRAPES_REQUIRE(need <= ctx->partials_bytes, "split-K partial buffer too small");
    dim3 grid(tiles_n, tiles_m, slabs);
    if (small) pdl((k_gemm_tn_splitk_s), grid, G_THREADS, 0, s)(A, lda, B, ldb, R_dev, R_cap, M, N, ctx->partials);
    else pdl((k_gemm_tn_splitk), grid, G_THREADS, 0, s)(A, lda, B, ldb, R_dev, R_cap, M, N, ctx->partials);
    grapes_count_launches(1);
    pdl((k_reduce_slabs), grid_for(ctx, (long long)M * N, 256), 256, 0, s)(ctx->partials, slabs, M * N, scale, accumulate,
                                                                       out);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

// out[c] (+)= scale * sum_r Mx[r, c]
int grapes_colsum(grapes_ctx* ctx, const float* Mx, const int* R_dev, int R_cap, int ld, int C, float scale,
                  int accumulate, float* out, void* stream) {
    GRAPES_REQUIRE(ctx && Mx && out, "null argument");
    GRAPES_REQUIRE(R_dev != nullptr, "R_dev required");
    cudaStream_t s = (cudaStream_t)stream;
    const int slabs = grapes_max_i(1, grapes_min_i(ctx->sm_count, grapes_div_up(R_cap, 64)));
    GRAPES_REQUIRE((size_t)slabs * C * sizeof(float) <= ctx->partials_bytes, "partial buffer too small");
    dim3 grid(grapes_div_up(C, 256), slabs);
    pdl((k_colsum_slabs), grid, 256, 0, s)(Mx, R_dev, R_cap, ld, C, ctx->partials);
    grapes_count_launches(1);
    pdl((k_colsum), grapes_div_up(C, 256), 256, 0, s)(ctx->partials, nullptr, slabs, C, C, scale, accumulate, out);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_sampler_l1_fwd(grapes_ctx* ctx, const float* Y, int ldy, const int* n_dev, int cap_n, int K,
                          const float* W1, int ldw, int D, const float* b1, const float* w2, float* z, void* stream) {
    GRAPES_REQUIRE(ctx && Y && n_dev && W1 && b1 && w2 && z, "null argument");
    const int blocks = grapes_max_i(1, grapes_min_i(grapes_div_up(cap_n, GB_M), ctx->sm_count * 2));
    pdl((k_l1_fwd), blocks, G_THREADS, 0, (cudaStream_t)stream)(Y, ldy, n_dev, cap_n, K, W1, ldw, D, b1, w2, z);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

// Gradient DIRECTION of sum(dz . z) w.r.t. (W1, b1, w2): accumulated (+=, times `scale`) into gW1/gb1/gw2.
int grapes_sampler_l1_bwd(grapes_ctx* ctx, const float* Y, int ldy, const int* n_dev, int cap_n, int K,
                          const float* W1, int ldw, int D, const float* b1, const float* w2, const float* dz,
                          float* dpre_scratch, float scale, int accumulate, float* gW1, int ldgw, float* gb1,
                          float* gw2, void* stream) {
    GRAPES_REQUIRE(ctx && Y && n_dev && W1 && b1 && w2 && dz && dpre_scratch && gW1 && gb1 && gw2, "null argument");
    GRAPES_REQUIRE(ldgw == K, "gW1 must be dense [D x K]");
    cudaStream_t s = (cudaStream_t)stream;
    const int blocks = grapes_max_i(1, grapes_min_i(grapes_div_up(cap_n, GB_M), ctx->sm_count));
    GRAPES_REQUIRE((size_t)2 * blocks * D * sizeof(float) <= ctx->partials_bytes, "partial buffer too small");
    float* dw2_part = ctx->partials;
    float* db1_part = ctx->partials + (size_t)blocks * D;
    pdl((k_l1_bwd), blocks, G_THREADS, 0, s)(Y, ldy, n_dev, cap_n, K, W1, ldw, D, b1, w2, dz, dpre_scratch, D, dw2_part,
                                          db1_part);
    grapes_count_launches(1);
    // a CTA whose first tile is past n writes zeros (its loops do not run), so all `blocks` rows are valid
    pdl((k_colsum), grapes_div_up(D, 256), 256, 0, s)(dw2_part, nullptr, blocks, D, D, scale, accumulate, gw2);
    grapes_count_launches(1);
    pdl((k_colsum), grapes_div_up(D, 256), 256, 0, s)(db1_part, nullptr, blocks, D, D, scale, accumulate, gb1);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    // gW1[D x K] += scale * dpre^T Y   (uses ctx->partials again, stream-ordered after the colsums)
    return grapes_gemm_tn(ctx, dpre_scratch, D, Y, ldy, n_dev, cap_n, D, K, scale, accumulate, gW1, stream);
}

}  // extern "C"
