// The tail of a training step as ONE launch: GFlowNet / REINFORCE gradient scale (main.py:271-287), the gradient
// exchange of the data-parallel path (mean over ranks, NVLink peer memory) and both Adam updates (main.py:268,289).
// The reference is single-process, so the exchange replaces nothing in /root/reference: it is
// `optimizer_c.step(); optimizer_gf.step()` applied to the mean of the per-rank gradients.
//
// Exchange (world > 1): every rank owns one symmetric buffer (torch.distributed._symmetric_memory hands each rank the
// peers' device pointers):  [parity 0: world slots | parity 1: world slots | flags].  Step s = *seq + 1, parity s & 1:
//   push     every rank WRITES its flat gradient into slot[rank] of EVERY rank's buffer (posted NVLink stores, no
//            round trip); the last block to finish stores s into flags[rank] of every peer (st.release.sys).
//   wait     block 0 polls its OWN flags (local memory) until flags[r] >= s for all r -- bounded, never a hang -- and
//            releases the rest of the grid through a device-scope go word, so the verdict is uniform over the grid.
//   reduce   every rank sums the world slots of its own buffer in rank order (identical bits on every rank, run-to-run
//            deterministic), divides by world, writes the mean gradient back and applies both Adam groups.
// Two parities suffice: a rank can push step s + 2 only after its reduce of step s + 1, which needed every peer's push
// of s + 1, which follows that peer's reduce of step s in stream order -- nobody still reads parity s & 1.
// A peer that never arrives (timeout) raises GRAPES_OVF_PEER_TIMEOUT, and the step is a NO-OP on this rank: parameters,
// moments, step counts and the sequence number stay untouched, and the failure is sticky (every later launch is a
// no-op too) until the host sees the flag.  No per-step host argument: the launch is captured into the step's CUDA graph.
//
// Learned node features (grapes_step_tail_embed): the table gradient is non-zero only on the step's all_nodes rows, so
// each rank also pushes (A, all_nodes[:A], dXc[:A, :F]) into slot[rank] of a SECOND symmetric buffer
// [parity 0: world slots | parity 1: world slots] of every rank (grapes_embed_slot_floats per slot).  Those stores sit
// before the block's __threadfence_system() and ticket, so the one per-step flag of the first buffer covers both
// payloads: no second flag, wait or timeout.  grapes_embed_merge_adam then reads this rank's own second buffer in a
// LATER launch of the same stream (union of the id lists, rank-order mean rows, dense table Adam).  Two parities still
// suffice, but only because that merge launch sits between this rank's tails of steps s and s + 1 on one stream: a rank
// can push step s + 2 into slot parity s & 1 of peer p only after its tail of s + 1 saw p's flag of s + 1, which p's
// tail of s + 1 releases after (stream order) p's merge of step s has finished reading parity s & 1.
//
// Learned table sharded by rows (grapes_embed_merge_adam_rows over rank r's rows [lo_r, hi_r) only): rank r's step
// s + 1 gathers rows of every shard o (hop aggregations, classifier layer 1, predict), so those reads must follow o's
// table walk of step s.  The exchange's flag of step s does not order them: o releases it in its tail, BEFORE its merge.
// Every rank therefore owns a small symmetric epoch buffer [world words | own count] (grapes_embed_epoch_words):
//   post     after this rank's shard walk, same stream: count += 1, then st.release.sys of the count into word[rank] of
//            every rank's epoch buffer.  Skipped when the step's exchange failed (go word GO_FAIL): nothing was applied.
//   wait     before the first read of the table of a step or of predict, same stream: ld.acquire.sys spin until word[p]
//            of this rank's own buffer has reached the own count for every p -- every peer has applied as many table
//            steps as this rank -- bounded like the tail's wait.  A timeout raises GRAPES_OVF_PEER_TIMEOUT and sets the
//            exchange's sticky failure, so that step's tail and merge are no-ops on this rank (as for a missing flag).
// The count lives in device memory, so a replayed graph advances it; a step enqueued without the optimiser (the graph
// warm-up) waits but never posts.  No deadlock: r's wait before step s + 1 needs o's post of s, which follows o's merge and
// tail of s, which needed only the flags of step s -- released by every rank's tail of s, which precedes that rank's
// wait of s + 1 in its stream.  Writes after reads are ordered already: o's walk of step s + 1 follows o's tail of s + 1,
// which waited for r's flag of s + 1, released after all of r's reads of step s + 1 (with the NCCL exchange the
// all-gather of s + 1 orders them the same way).  The two-parity argument above is unchanged: the merge still sits
// between this rank's tails on one stream, and the post after it changes no slot.
#define GRAPES_PDL_GROUP 8
#include "common.cuh"

#define PEER_MAX 8
struct PeerTable {
    float* buf[PEER_MAX];              // base of every rank's symmetric buffer (peer-mapped device pointers)
};

__device__ __forceinline__ void st_release_sys_u32(unsigned int* p, unsigned int v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys_u32(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu_u32(unsigned int* p, unsigned int v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_gpu_u32(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

struct TailArgs {
    // exchange
    PeerTable pt; int rank, world, n, n_pad;
    unsigned int* state; int* err_flag; unsigned int spin_limit;
    // GFlowNet / REINFORCE scale (do_scale == 0: the gradients are final already); scal may be null without it
    float* scal; int do_scale; float loss_coef, log_z_init; int reinforce, have_log_z;
    const float* dir; int gf_off, n_gf, z_off, n_z;
    // Adam (two groups over the flat buffers)
    float* p; float* g; float* m; float* v; int off0, n0; float lr0; int off1, n1; float lr1;
    float beta1, beta2, eps; float* steps;
};

// table payload of the learned node features (k_step_tail_embed)
struct EmbedPush {
    float* buf[PEER_MAX];              // base of every rank's second symmetric buffer
    const int* count;                  // A: rows of this step (device)
    const int* ids;                    // all_nodes[:A], ascending
    const float* rows; int ldg;        // dXc[:A, :F], pitch ldg floats
    int F, cap;                        // row width (multiple of 4), rows per slot (cap_A)
    long long slot;                    // floats per slot (grapes_embed_slot_floats)
};

template <bool PEER, bool EMBED>
__device__ __forceinline__ void step_tail(const TailArgs& a, const EmbedPush* e) {
    pdl_begin();
    __shared__ float s_step_size[2], s_bc2_sqrt[2];
    __shared__ int s_last, s_go;
    const int tid = threadIdx.x;
    __builtin_assume(tid < 256);                           // __launch_bounds__(256) of both kernels below
    const int gtid = blockIdx.x * blockDim.x + tid, gsz = gridDim.x * blockDim.x;
    // ---- loss_gfn and the scale of the accumulated gradient directions (every thread, from read-only inputs) ----
    float g_gf = 0.f, g_z = 0.f;
    if (a.do_scale) {
        const float loss_c = a.scal[GRAPES_SCAL_LOSS_C];
        const float tot = a.scal[GRAPES_SCAL_TOT_LOG_PROB];
        const float log_z = a.have_log_z ? a.scal[GRAPES_SCAL_LOG_Z_MEAN] - a.log_z_init : 0.f;
        float loss_gfn;
        if (a.reinforce) { loss_gfn = -tot * loss_c; g_gf = -loss_c; g_z = 0.f; }                       // main.py:279
        else { const float r = log_z + tot + a.loss_coef * loss_c; loss_gfn = r * r; g_gf = g_z = 2.0f * r; }   // :282
        if (gtid == 0) {
            a.scal[GRAPES_SCAL_LOG_Z] = log_z;
            a.scal[GRAPES_SCAL_LOSS_GFN] = loss_gfn;
            a.scal[GRAPES_SCAL_G_GF] = g_gf;
            a.scal[GRAPES_SCAL_G_Z] = g_z;
        }
    }
    if (tid >= 32 && tid < 34) {
        const int q = tid - 32;
        const double t = (double)a.steps[q] + 1.0;
        const double bc1 = 1.0 - pow((double)a.beta1, t), bc2 = 1.0 - pow((double)a.beta2, t);
        s_step_size[q] = (float)((double)(q ? a.lr1 : a.lr0) / bc1);
        s_bc2_sqrt[q] = (float)sqrt(bc2);
    }
    // this rank's gradient of element i: scaled direction inside the sampler-net ranges, the stored value elsewhere
    auto own_grad = [&](int i) -> float {
        if (a.do_scale) {
            if (i >= a.gf_off && i < a.gf_off + a.n_gf) return g_gf * a.dir[i];
            if (i >= a.z_off && i < a.z_off + a.n_z) return g_z * a.dir[i];
        }
        return a.g[i];
    };
    unsigned int seq = 0u;
    size_t par_base = 0;
    if (PEER) {
        seq = a.state[PS_SEQ] + 1u;
        par_base = (size_t)(seq & 1u) * a.world * a.n_pad;
        const bool failed = a.state[PS_FAILED] != 0u;
        // ---- push ----
        if (!failed) {
            const size_t my_slot = par_base + (size_t)a.rank * a.n_pad;
            for (int i = gtid; i < a.n; i += gsz) {
                const float gi = own_grad(i);
#pragma unroll
                for (int r = 0; r < PEER_MAX; ++r)
                    if (r < a.world) a.pt.buf[r][my_slot + i] = gi;
            }
            if (EMBED) {
                // slot: [A, 3 pad | ids, cap rounded up to 4 | rows, cap x F]
                const int A = min(*e->count, e->cap), F4 = e->F >> 2, cap4 = (e->cap + 3) & ~3;
                const size_t es = (size_t)(seq & 1u) * a.world * e->slot + (size_t)a.rank * e->slot;
                for (int i = gtid; i < A; i += gsz) {
                    const int v = e->ids[i];
#pragma unroll
                    for (int r = 0; r < PEER_MAX; ++r)
                        if (r < a.world) reinterpret_cast<int*>(e->buf[r] + es)[4 + i] = v;
                }
                if (gtid == 0) {
#pragma unroll
                    for (int r = 0; r < PEER_MAX; ++r)
                        if (r < a.world) reinterpret_cast<int*>(e->buf[r] + es)[0] = A;
                }
                const float4* g4 = reinterpret_cast<const float4*>(e->rows);
                const int ldg4 = e->ldg >> 2;
                for (int i = gtid; i < A * F4; i += gsz) {
                    const int row = i / F4, c = i - row * F4;
                    const float4 gv = g4[(size_t)row * ldg4 + c];
#pragma unroll
                    for (int r = 0; r < PEER_MAX; ++r)
                        if (r < a.world) reinterpret_cast<float4*>(e->buf[r] + es + 4 + cap4)[i] = gv;
                }
            }
        }
        __threadfence_system();
        __syncthreads();
        if (tid == 0) s_last = (atomicAdd(&a.state[PS_TICKET_A], 1u) == gridDim.x - 1) ? 1 : 0;
        __syncthreads();
        if (s_last) {                                        // last block: every block's stores are fenced
            __threadfence_system();
            if (tid < a.world && !failed) {
                unsigned int* flags = reinterpret_cast<unsigned int*>(a.pt.buf[tid] + 2 * (size_t)a.world * a.n_pad);
                st_release_sys_u32(flags + a.rank, seq);
            }
            if (tid == 0) a.state[PS_TICKET_A] = 0u;
        }
        // ---- wait: block 0 polls this rank's own flag words, then releases the grid ----
        if (blockIdx.x == 0) {
            int arrived = 1;
            if (tid < a.world && !failed) {
                const unsigned int* flags =
                    reinterpret_cast<const unsigned int*>(a.pt.buf[a.rank] + 2 * (size_t)a.world * a.n_pad);
                unsigned int it = 0;
                while (ld_acquire_sys_u32(flags + tid) < seq) {
                    if (++it > a.spin_limit) { arrived = 0; break; }             // never hang the GPU
                    __nanosleep(32);
                }
            }
            const int ok = __syncthreads_and(arrived) && !failed;
            if (tid == 0) {
                if (!ok) {
                    const int bits = atomicOr(a.err_flag, GRAPES_OVF_PEER_TIMEOUT) | GRAPES_OVF_PEER_TIMEOUT;
                    a.state[PS_FAILED] = 1u;
                    if (a.scal) a.scal[GRAPES_SCAL_FLAGS] = (float)bits;
                }
                __threadfence();
                st_release_gpu_u32(&a.state[PS_GO], ok ? seq : (seq | GO_FAIL));
            }
        }
        if (tid == 0) {
            unsigned int go, it = 0;
            while (((go = ld_acquire_gpu_u32(&a.state[PS_GO])) & ~GO_FAIL) != seq) {
                if (++it > 4u * a.spin_limit) { go = seq | GO_FAIL; break; }
                __nanosleep(32);
            }
            s_go = (go & GO_FAIL) ? 0 : 1;
        }
        __syncthreads();
        if (!s_go) return;                                 // a peer is missing: this step does not happen on this rank
    } else {
        __syncthreads();
    }
    // ---- reduce (rank order) + Adam ----
    const float inv_w = 1.0f / (float)a.world;
    for (int i = gtid; i < a.n; i += gsz) {
        float gi;
        if (PEER) {
            const float* mine = a.pt.buf[a.rank] + par_base + i;
            float s = 0.f;
#pragma unroll
            for (int r = 0; r < PEER_MAX; ++r)
                if (r < a.world) s += __ldcg(mine + (size_t)r * a.n_pad);        // written by the peers: read at L2
            gi = s * inv_w;
            a.g[i] = gi;
        } else {
            gi = own_grad(i);
            if (a.do_scale) a.g[i] = gi;
        }
        int grp = -1;
        if (i >= a.off0 && i < a.off0 + a.n0) grp = 0;
        else if (i >= a.off1 && i < a.off1 + a.n1) grp = 1;
        if (grp >= 0) {                                                  // torch.optim.Adam single-tensor arithmetic (k_adam2)
            const float mi = adam_exp_avg(a.m[i], gi, a.beta1);
            const float vi = adam_exp_avg_sq(a.v[i], gi, a.beta2);
            a.m[i] = mi; a.v[i] = vi;
            const float denom = sqrtf(vi) / s_bc2_sqrt[grp] + a.eps;
            a.p[i] = a.p[i] - s_step_size[grp] * (mi / denom);
        }
    }
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        s_last = (atomicAdd(&a.state[PS_TICKET_C], 1u) == gridDim.x - 1) ? 1 : 0;
    }
    __syncthreads();
    if (s_last && tid == 0) {
        if (a.n0 > 0) a.steps[0] += 1.0f;
        if (a.n1 > 0) a.steps[1] += 1.0f;
        if (PEER) a.state[PS_SEQ] = seq;
        a.state[PS_TICKET_C] = 0u;
        if (a.scal && a.err_flag) a.scal[GRAPES_SCAL_FLAGS] = (float)(*(volatile int*)a.err_flag);
    }
}

template <bool PEER>
__global__ void __launch_bounds__(256) k_step_tail(const TailArgs a) {
    step_tail<PEER, false>(a, nullptr);
}

__global__ void __launch_bounds__(256) k_step_tail_embed(const TailArgs a, const EmbedPush e) {
    step_tail<true, true>(a, &e);
}

// ---- epoch of a learned table sharded by rows (grapes_embed_epoch_post / _wait); epoch: [world words | own count] ----
struct EpochBufs {
    unsigned int* buf[PEER_MAX];       // every rank's epoch buffer (peer-mapped)
};

__global__ void __launch_bounds__(32) k_embed_epoch_post(const EpochBufs e, unsigned int* own, int rank, int world,
                                                          const unsigned int* state) {
    pdl_begin();
    if (state && (*(volatile const unsigned int*)(state + PS_GO) & GO_FAIL)) return;    // the step was not applied
    const unsigned int c = *(volatile unsigned int*)(own + world) + 1u;
    __syncwarp();
    if (threadIdx.x == 0) own[world] = c;
    __threadfence_system();                           // this rank's walk (earlier launches of the stream) before the words
#pragma unroll
    for (int r = 0; r < PEER_MAX; ++r)                // lane r -> rank r; constant indices keep the table in parameters
        if (r == (int)threadIdx.x && r < world) st_release_sys_u32(e.buf[r] + rank, c);
}

__global__ void __launch_bounds__(32) k_embed_epoch_wait(const unsigned int* epoch, int world, unsigned int* state,
                                                          int* err_flag, unsigned int spin_limit) {
    pdl_begin();
    const int tid = threadIdx.x;
    const bool failed = state && *(volatile const unsigned int*)(state + PS_FAILED) != 0u;
    const unsigned int c = *(volatile const unsigned int*)(epoch + world);
    int arrived = 1;
    if (tid < world && !failed) {
        unsigned int it = 0;
        while ((int)(ld_acquire_sys_u32(epoch + tid) - c) < 0) {
            if (++it > spin_limit) { arrived = 0; break; }                       // never hang the GPU
            __nanosleep(32);
        }
    }
    const bool ok = __all_sync(0xffffffffu, arrived) && !failed;
    if (tid == 0 && !ok) {
        atomicOr(err_flag, GRAPES_OVF_PEER_TIMEOUT);
        if (state) state[PS_FAILED] = 1u;
        __threadfence();
    }
}

static int launch_tail(grapes_ctx* ctx, TailArgs& a, void* const* peer_bufs, void* stream,
                       const EmbedPush* embed = nullptr) {
    for (int r = 0; r < PEER_MAX; ++r)
        a.pt.buf[r] = (peer_bufs && r < a.world) ? reinterpret_cast<float*>(peer_bufs[r]) : nullptr;
    a.n_pad = (a.n + 63) / 64 * 64;
    // a few seconds of polling (about 1 us per try: one system-scope load + a short sleep) before a rank gives up on a
    // peer and raises the error flag
    a.spin_limit = 3000000u;
    int blocks = (a.n + 255) / 256;
    // every block spins on the go word while the push of the others is in flight: the grid must be co-resident
    if (blocks > ctx->sm_count * 2) blocks = ctx->sm_count * 2;
    cudaStream_t s = (cudaStream_t)stream;
    if (embed) pdl((k_step_tail_embed), blocks, 256, 0, s)(a, *embed);
    else if (peer_bufs && a.world > 1) pdl((k_step_tail<true>), blocks, 256, 0, s)(a);
    else pdl((k_step_tail<false>), blocks, 256, 0, s)(a);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

extern "C" {

int64_t grapes_peer_buffer_floats(int n, int world) {
    const int64_t n_pad = ((int64_t)n + 63) / 64 * 64;
    return 2 * (int64_t)(world < 1 ? 1 : world) * n_pad + 64;
}

int grapes_peer_state_words(void) { return 8; }

// peer_bufs: HOST array of `world` device pointers (the peers' symmetric buffers, own buffer at index `rank`), each of
// grapes_peer_buffer_floats(n, world) floats, zero-initialised once.  state: grapes_peer_state_words() uint32 on the
// device, zero-initialised.  err_flag: the engine's overflow word.
int grapes_allreduce_adam_peer(grapes_ctx* ctx, void* const* peer_bufs, int rank, int world, const float* grads, int n,
                               float* params, float* grads_mean_out, float* exp_avg, float* exp_avg_sq, int off0,
                               int n0, float lr0, int off1, int n1, float lr1, float beta1, float beta2, float eps,
                               float* steps_dev, unsigned int* state, int* err_flag, void* stream) {
    GRAPES_REQUIRE(ctx && peer_bufs && grads && params && grads_mean_out && exp_avg && exp_avg_sq && steps_dev && state &&
                       err_flag, "null argument");
    GRAPES_REQUIRE(grads == grads_mean_out, "the mean gradient replaces the local one in place");
    GRAPES_REQUIRE(world >= 1 && world <= PEER_MAX && rank >= 0 && rank < world, "1 <= world <= 8");
    GRAPES_REQUIRE(n > 0, "empty gradient");
    TailArgs a;
    memset(&a, 0, sizeof(a));
    a.rank = rank; a.world = world; a.n = n; a.state = state; a.err_flag = err_flag;
    a.p = params; a.g = grads_mean_out; a.m = exp_avg; a.v = exp_avg_sq;
    a.off0 = off0; a.n0 = n0; a.lr0 = lr0; a.off1 = off1; a.n1 = n1; a.lr1 = lr1;
    a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.steps = steps_dev;
    return launch_tail(ctx, a, peer_bufs, stream);
}

// The whole tail of a step in one launch (main.py:271-291): loss_gfn + gradient scale of the accumulated directions
// (dir is indexed like the flat parameter buffer; ranges [gf_off, gf_off + n_gf) and [z_off, z_off + n_z)), the mean
// over ranks when peer_bufs != NULL and world > 1, then both Adam groups.  grads holds the classifier gradient on entry
// and the step's (mean) gradient of every parameter on exit.
int grapes_step_tail(grapes_ctx* ctx, float* scal, int do_scale, float loss_coef, float log_z_init, int reinforce,
                     int have_log_z, const float* dir, int gf_off, int n_gf, int z_off, int n_z, void* const* peer_bufs,
                     int rank, int world, int n, float* params, float* grads, float* exp_avg, float* exp_avg_sq, int off0,
                     int n0, float lr0, int off1, int n1, float lr1, float beta1, float beta2, float eps, float* steps_dev,
                     unsigned int* state, int* err_flag, void* stream) {
    GRAPES_REQUIRE(ctx && params && grads && exp_avg && exp_avg_sq && steps_dev && state, "null argument");
    GRAPES_REQUIRE(!do_scale || (scal && dir), "a gradient scale needs the scalar block and the direction buffer");
    GRAPES_REQUIRE(!peer_bufs || (world >= 1 && world <= PEER_MAX && rank >= 0 && rank < world && err_flag),
                   "1 <= world <= 8");
    GRAPES_REQUIRE(n > 0 && n0 >= 0 && n1 >= 0, "empty gradient");
    TailArgs a;
    memset(&a, 0, sizeof(a));
    a.rank = peer_bufs ? rank : 0; a.world = peer_bufs ? world : 1; a.n = n; a.state = state; a.err_flag = err_flag;
    a.scal = scal; a.do_scale = do_scale; a.loss_coef = loss_coef; a.log_z_init = log_z_init; a.reinforce = reinforce; a.have_log_z = have_log_z;
    a.dir = dir; a.gf_off = gf_off; a.n_gf = n_gf; a.z_off = z_off; a.n_z = n_z;
    a.p = params; a.g = grads; a.m = exp_avg; a.v = exp_avg_sq;
    a.off0 = off0; a.n0 = n0; a.lr0 = lr0; a.off1 = off1; a.n1 = n1; a.lr1 = lr1;
    a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.steps = steps_dev;
    return launch_tail(ctx, a, peer_bufs, stream);
}

int64_t grapes_embed_slot_floats(int cap_rows, int F) {
    return 4 + ((int64_t)cap_rows + 3) / 4 * 4 + (int64_t)cap_rows * F;
}

int64_t grapes_embed_peer_buffer_floats(int cap_rows, int F, int world) {
    return 2 * (int64_t)(world < 1 ? 1 : world) * grapes_embed_slot_floats(cap_rows, F);
}

// grapes_step_tail with peers, plus the learned table's payload of this step (A = *count_dev rows: ids[:A] ascending,
// rows[:A, :F] at pitch ldg) pushed into slot[rank] of every rank's second symmetric buffer (embed_bufs, each of
// grapes_embed_peer_buffer_floats(cap_rows, F, world) floats) under the same per-step flag.
int grapes_step_tail_embed(grapes_ctx* ctx, float* scal, int do_scale, float loss_coef, float log_z_init, int reinforce,
                           int have_log_z, const float* dir, int gf_off, int n_gf, int z_off, int n_z,
                           void* const* peer_bufs, void* const* embed_bufs, int rank, int world, int n, float* params,
                           float* grads, float* exp_avg, float* exp_avg_sq, int off0, int n0, float lr0, int off1, int n1,
                           float lr1, float beta1, float beta2, float eps, float* steps_dev, unsigned int* state,
                           int* err_flag, const int* count_dev, const int* ids, const float* rows, int ldg, int F,
                           int cap_rows, void* stream) {
    GRAPES_REQUIRE(ctx && params && grads && exp_avg && exp_avg_sq && steps_dev && state && err_flag && peer_bufs &&
                       embed_bufs && count_dev && ids && rows, "null argument");
    GRAPES_REQUIRE(!do_scale || (scal && dir), "a gradient scale needs the scalar block and the direction buffer");
    GRAPES_REQUIRE(world >= 1 && world <= PEER_MAX && rank >= 0 && rank < world, "1 <= world <= 8");
    GRAPES_REQUIRE(n > 0 && n0 >= 0 && n1 >= 0, "empty gradient");
    GRAPES_REQUIRE(F > 0 && F % 4 == 0 && ldg % 4 == 0 && ldg >= F && cap_rows > 0,
                   "table width and row pitch must be multiples of 4");
    GRAPES_REQUIRE((reinterpret_cast<uintptr_t>(rows) & 15) == 0, "rows must be 16-byte aligned");
    TailArgs a;
    memset(&a, 0, sizeof(a));
    a.rank = rank; a.world = world; a.n = n; a.state = state; a.err_flag = err_flag;
    a.scal = scal; a.do_scale = do_scale; a.loss_coef = loss_coef; a.log_z_init = log_z_init; a.reinforce = reinforce; a.have_log_z = have_log_z;
    a.dir = dir; a.gf_off = gf_off; a.n_gf = n_gf; a.z_off = z_off; a.n_z = n_z;
    a.p = params; a.g = grads; a.m = exp_avg; a.v = exp_avg_sq;
    a.off0 = off0; a.n0 = n0; a.lr0 = lr0; a.off1 = off1; a.n1 = n1; a.lr1 = lr1;
    a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.steps = steps_dev;
    EmbedPush e;
    memset(&e, 0, sizeof(e));
    for (int r = 0; r < PEER_MAX; ++r) e.buf[r] = r < world ? reinterpret_cast<float*>(embed_bufs[r]) : nullptr;
    e.count = count_dev; e.ids = ids; e.rows = rows; e.ldg = ldg; e.F = F; e.cap = cap_rows;
    e.slot = grapes_embed_slot_floats(cap_rows, F);
    return launch_tail(ctx, a, peer_bufs, stream, &e);
}

int grapes_embed_epoch_words(int world) {
    return (world < 1 ? 1 : world) + 1;
}

int grapes_embed_epoch_post(grapes_ctx* ctx, void* const* epoch_bufs, int rank, int world, const unsigned int* state,
                            void* stream) {
    GRAPES_REQUIRE(ctx && epoch_bufs, "null argument");
    GRAPES_REQUIRE(world >= 1 && world <= PEER_MAX && rank >= 0 && rank < world, "1 <= world <= 8");
    EpochBufs e;
    memset(&e, 0, sizeof(e));
    for (int r = 0; r < world; ++r) {
        GRAPES_REQUIRE(epoch_bufs[r], "null epoch buffer");
        e.buf[r] = reinterpret_cast<unsigned int*>(epoch_bufs[r]);
    }
    pdl((k_embed_epoch_post), 1, 32, 0, (cudaStream_t)stream)(e, e.buf[rank], rank, world, state);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

int grapes_embed_epoch_wait(grapes_ctx* ctx, const unsigned int* epoch, int world, unsigned int* state, int* err_flag,
                            uint32_t spin_limit, void* stream) {
    GRAPES_REQUIRE(ctx && epoch && err_flag, "null argument");
    GRAPES_REQUIRE(world >= 1 && world <= PEER_MAX, "1 <= world <= 8");
    // 0: the tail's bound (a few seconds of polling, about 1 us per try)
    pdl((k_embed_epoch_wait), 1, 32, 0, (cudaStream_t)stream)(epoch, world, state, err_flag,
                                                             spin_limit ? spin_limit : 3000000u);
    grapes_count_launches(1);
    GRAPES_LAUNCH_OK();
    return GRAPES_OK;
}

}  // extern "C"
