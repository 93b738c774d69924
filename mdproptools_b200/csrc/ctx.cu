// Context, scratch arena and error reporting of libmdprop_b200.
#include <stdarg.h>

#include "common.cuh"
#include "scratch_plan.h"

static thread_local char g_err[1024] = "";

void mdp_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int mdp_ctx::arena_reserve(size_t bytes)
{
    bytes = mdp_scratch_reserved(bytes);   // batch sizes are planned on this same total (scratch_plan.h)
    if (bytes <= slab_bytes) return 0;
    if (bytes > slab_limit) {
        mdp_set_error("scratch request %zu B exceeds the context limit %zu B", bytes, slab_limit);
        return MDP_ERR_OOM;
    }
    // grow geometrically; cudaFree synchronises the device, which also retires every user of the old slab
    size_t want = slab_bytes ? slab_bytes : ((size_t)64 << 20);
    while (want < bytes) want *= 2;
    if (want > slab_limit) want = slab_limit;
    if (slab) MDP_CUDA(cudaFree(slab));
    slab = nullptr;
    slab_bytes = 0;
    cudaError_t e = cudaMalloc((void **)&slab, want);
    if (e != cudaSuccess && want > bytes) {
        (void)cudaGetLastError();
        want = bytes;
        e = cudaMalloc((void **)&slab, want);
    }
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        mdp_set_error("cudaMalloc of %zu B scratch failed: %s", want, cudaGetErrorString(e));
        return MDP_ERR_OOM;
    }
    slab_bytes = want;
    return 0;
}

extern "C" {

int mdp_version(void) { return MDP_VERSION; }

const char *mdp_last_error(void) { return g_err; }

int mdp_ctx_create(int device, mdp_ctx **out)
{
    MDP_REQUIRE(out != nullptr, "mdp_ctx_create: out is NULL");
    int ndev = 0;
    MDP_CUDA(cudaGetDeviceCount(&ndev));
    MDP_REQUIRE(device >= 0 && device < ndev, "mdp_ctx_create: device %d out of range (%d devices)", device, ndev);
    MDP_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    MDP_CUDA(cudaGetDeviceProperties(&prop, device));
    MDP_REQUIRE(prop.major == 10, "libmdprop_b200 is built for sm_100a only; device %d is sm_%d%d", device,
                prop.major, prop.minor);
    mdp_ctx *c = new mdp_ctx();
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->smem_optin = prop.sharedMemPerBlockOptin;
    cudaError_t e = cudaMalloc((void **)&c->d_stats, 8 * sizeof(unsigned long long));
    if (e != cudaSuccess) {
        mdp_set_error("cudaMalloc stats: %s", cudaGetErrorString(e));
        delete c;
        return MDP_ERR_OOM;
    }
    cudaMemset(c->d_stats, 0, 8 * sizeof(unsigned long long));
    *out = c;
    return 0;
}

void mdp_ctx_destroy(mdp_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    if (ctx->slab) cudaFree(ctx->slab);
    if (ctx->d_stats) cudaFree(ctx->d_stats);
    delete ctx;
}

int64_t mdp_ctx_scratch_bytes(mdp_ctx *ctx) { return ctx ? (int64_t)ctx->slab_bytes : 0; }

int mdp_ctx_set_scratch_limit(mdp_ctx *ctx, int64_t bytes)
{
    MDP_REQUIRE(ctx && bytes > 0, "mdp_ctx_set_scratch_limit: bad argument");
    ctx->slab_limit = (size_t)bytes;
    return 0;
}

int64_t mdp_ctx_launch_count(mdp_ctx *ctx) { return ctx ? ctx->launches : 0; }

int mdp_ctx_timing(mdp_ctx *ctx, int enable)
{
    MDP_REQUIRE(ctx, "mdp_ctx_timing: NULL context");
    ctx->timing = enable != 0;
    return 0;
}

int mdp_ctx_timing_read(mdp_ctx *ctx, int tag, double *ms_total, int64_t *count)
{
    MDP_REQUIRE(ctx && ms_total && count, "mdp_ctx_timing_read: NULL argument");
    double total = 0.0;
    int64_t n = 0;
    std::vector<mdp_ctx::Timed> keep;
    for (auto &t : ctx->timed) {
        if (t.tag != tag) {
            keep.push_back(t);
            continue;
        }
        MDP_CUDA(cudaEventSynchronize(t.e1));
        float ms = 0.f;
        MDP_CUDA(cudaEventElapsedTime(&ms, t.e0, t.e1));
        total += ms;
        ++n;
        cudaEventDestroy(t.e0);
        cudaEventDestroy(t.e1);
    }
    ctx->timed.swap(keep);
    *ms_total = total;
    *count = n;
    return 0;
}

int mdp_ctx_pair_stats(mdp_ctx *ctx, int64_t out[4])
{
    MDP_REQUIRE(ctx && out, "mdp_ctx_pair_stats: bad argument");
    unsigned long long h[4];
    MDP_CUDA(cudaMemcpy(h, ctx->d_stats, sizeof(h), cudaMemcpyDeviceToHost));
    for (int k = 0; k < 4; ++k) out[k] = (int64_t)h[k];
    return 0;
}

} // extern "C"
