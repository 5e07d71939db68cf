// Context (library-owned workspace), error reporting.
#include <stdarg.h>

#include "common.cuh"

static thread_local char g_err[512] = "";
static long long g_launches = 0;
int g_grapes_pdl = 0;   // measured on B200: slower or neutral per group and unsafe in combination (DESIGN.md section 9)
void grapes_count_launches(int n) { g_launches += n; }

void grapes_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" {

const char* grapes_last_error(void) { return g_err; }
int grapes_abi_version(void) { return 1; }
#ifndef GRAPES_BUILD_ID
#define GRAPES_BUILD_ID "unknown"
#endif
// the marker prefix lets the host read the id out of the file without loading it
static const char g_build_id[] = "GRAPES_BUILD_ID=" GRAPES_BUILD_ID;
const char* grapes_build_id(void) { return g_build_id + 16; }
int grapes_set_pdl(int mask) { g_grapes_pdl = mask; return 0; }
int64_t grapes_kernel_launches(void) { return (int64_t)g_launches; }

int grapes_ctx_set_sm_limit(grapes_ctx* ctx, int sms) {
    GRAPES_REQUIRE(ctx != nullptr, "null ctx");
    cudaDeviceProp prop;
    GRAPES_CUDA_OK(cudaGetDeviceProperties(&prop, ctx->device));
    ctx->sm_count = (sms > 0 && sms < prop.multiProcessorCount) ? sms : prop.multiProcessorCount;
    return GRAPES_OK;
}

int grapes_ctx_create(int device, int64_t num_nodes, int64_t max_frontier, int64_t partials_bytes, grapes_ctx** out) {
    GRAPES_REQUIRE(out != nullptr, "null out");
    GRAPES_REQUIRE(num_nodes > 0 && num_nodes < (1ll << 31), "num_nodes must fit int32");
    GRAPES_REQUIRE(max_frontier > 0 && max_frontier < (1ll << 31), "max_frontier must fit int32");
    int ndev = 0;
    GRAPES_CUDA_OK(cudaGetDeviceCount(&ndev));
    GRAPES_REQUIRE(device >= 0 && device < ndev, "no such CUDA device (there is no CPU fallback)");
    int prev_device = device;
    GRAPES_CUDA_OK(cudaGetDevice(&prev_device));
    struct Restore { int d; ~Restore() { cudaSetDevice(d); } } restore{prev_device};   // the caller's current device is left as found
    GRAPES_CUDA_OK(cudaSetDevice(device));
    cudaDeviceProp prop;
    GRAPES_CUDA_OK(cudaGetDeviceProperties(&prop, device));
    GRAPES_REQUIRE(prop.major >= 10, "grapes_b200 kernels are built for sm_100a (Blackwell) only");
    grapes_ctx* c = new grapes_ctx();
    memset(c, 0, sizeof(*c));
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->num_nodes = num_nodes;
    c->num_words = (int)((num_nodes + 31) / 32);
    long long tiles_nodes = (c->num_words + 1023) / 1024 + 1;
    long long tiles_front = (max_frontier + 1023) / 1024 + 1;
    c->scan_cap_tiles = (int)(tiles_nodes > tiles_front ? tiles_nodes : tiles_front) + 8;
    c->hub_cap = 1 << 16;
    c->partials_bytes = (size_t)(partials_bytes > (1 << 20) ? partials_bytes : (1 << 20));
    cudaError_t e;
    if ((e = cudaMalloc(&c->scan_status, sizeof(unsigned long long) * c->scan_cap_tiles)) != cudaSuccess ||
        (e = cudaMalloc(&c->scan_counters, sizeof(unsigned int) * 4)) != cudaSuccess ||
        (e = cudaMalloc(&c->hub_rows, sizeof(int) * c->hub_cap)) != cudaSuccess ||
        (e = cudaMalloc(&c->hub_count, sizeof(int))) != cudaSuccess ||
        (e = cudaMalloc(&c->partials, c->partials_bytes)) != cudaSuccess) {
        grapes_set_error("grapes_ctx_create: cudaMalloc -> %s", cudaGetErrorString(e));
        grapes_ctx_destroy(c);
        return GRAPES_ERR_NOMEM;
    }
    GRAPES_CUDA_OK(cudaMemset(c->scan_status, 0, sizeof(unsigned long long) * c->scan_cap_tiles));
    GRAPES_CUDA_OK(cudaMemset(c->scan_counters, 0, sizeof(unsigned int) * 4));
    GRAPES_CUDA_OK(cudaMemset(c->hub_count, 0, sizeof(int)));
    *out = c;
    return GRAPES_OK;
}

int grapes_ctx_destroy(grapes_ctx* c) {
    if (!c) return GRAPES_OK;
    cudaFree(c->scan_status);
    cudaFree(c->scan_counters);
    cudaFree(c->hub_rows);
    cudaFree(c->hub_count);
    cudaFree(c->partials);
    delete c;
    return GRAPES_OK;
}

int grapes_zero(grapes_ctx* ctx, void* ptr, int64_t bytes, void* stream) {
    GRAPES_REQUIRE(ctx && (ptr || bytes == 0), "null argument");
    if (bytes > 0) GRAPES_CUDA_OK(cudaMemsetAsync(ptr, 0, (size_t)bytes, (cudaStream_t)stream));
    return GRAPES_OK;
}

}  // extern "C"
