// context.cu -- zkb_ctx lifetime, error reporting, device-memory wrappers, scratch arenas.
#include "common.cuh"
#include <stdarg.h>
#include <string.h>

namespace zkb {
static thread_local char g_err[512] = "";
void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
int32_t scratch_get(zkb_ctx *ctx, int slot, size_t bytes, void **out) {
    DeviceBuffer &b = ctx->scratch[slot];
    if (b.bytes < bytes) {
        if (b.ptr) {
            ZKB_CUDA(cudaStreamSynchronize(ctx->stream));
            ZKB_CUDA(cudaFree(b.ptr));
            b.ptr = nullptr;
            b.bytes = 0;
        }
        size_t want = bytes + (bytes >> 3);  // 12.5 % headroom against repeated regrowth
        cudaError_t e = cudaMalloc(&b.ptr, want);
        if (e != cudaSuccess) {
            want = bytes;
            e = cudaMalloc(&b.ptr, want);
        }
        if (e != cudaSuccess) {
            set_error("scratch slot %d: cudaMalloc(%zu) failed: %s", slot, want, cudaGetErrorString(e));
            b.ptr = nullptr;
            return ZKB_ERR_ALLOC;
        }
        b.bytes = want;
    }
    *out = b.ptr;
    return ZKB_OK;
}
int32_t block_alloc(zkb_ctx *ctx, size_t bytes, void **out, size_t *got) {
    if (bytes < 256) bytes = 256;
    bytes = (bytes + 255) & ~(size_t)255;
    auto it = ctx->block_cache.lower_bound(bytes);
    if (it != ctx->block_cache.end() && it->first <= bytes + (bytes >> 2) + 4096) {  // reuse a block at most 25 % larger
        *out = it->second;
        *got = it->first;
        ctx->block_cache_bytes -= it->first;
        ctx->block_cache.erase(it);
        return ZKB_OK;
    }
    cudaError_t e = cudaMalloc(out, bytes);
    if (e != cudaSuccess) {
        // release the cache and retry once
        cudaStreamSynchronize(ctx->stream);
        for (auto &kv : ctx->block_cache) cudaFree(kv.second);
        ctx->block_cache.clear();
        ctx->block_cache_bytes = 0;
        e = cudaMalloc(out, bytes);
    }
    if (e != cudaSuccess) {
        set_error("cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
        return ZKB_ERR_ALLOC;
    }
    *got = bytes;
    return ZKB_OK;
}
void block_free(zkb_ctx *ctx, void *p, size_t bytes) {
    if (!p) return;
    ctx->block_cache.emplace(bytes, p);
    ctx->block_cache_bytes += bytes;
}

}  // namespace zkb

using namespace zkb;

extern "C" const char *zkb_last_error(void) { return g_err; }
extern "C" uint32_t zkb_version(void) { return (1u << 16) | 2u; }

extern "C" int32_t zkb_init(int32_t device, zkb_ctx **out) {
    ZKB_ARG(out != nullptr);
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        set_error("no CUDA device available (%s); libzkb200 has no CPU fallback", e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
        return ZKB_ERR_CUDA;
    }
    ZKB_ARG(device >= 0 && device < count);
    ZKB_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    ZKB_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        set_error("device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
        return ZKB_ERR_CUDA;
    }
    zkb_ctx *ctx = new zkb_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ZKB_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    ZKB_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
    *out = ctx;
    return ZKB_OK;
}

extern "C" int32_t zkb_destroy(zkb_ctx *ctx) {
    if (!ctx) return ZKB_OK;
    cudaSetDevice(ctx->device);
    zkb_comm_destroy(ctx);
    cudaStreamSynchronize(ctx->stream);
    for (auto &kv : ctx->ntt_plans) {
        NttPlan &p = kv.second;
        if (p.tw_lo) cudaFree(p.tw_lo);
        if (p.tw_hi) cudaFree(p.tw_hi);
        for (int i = 0; i < 2; ++i)
            if (p.tw_b[i]) cudaFree(p.tw_b[i]);
        if (p.tw_b_scaled) cudaFree(p.tw_b_scaled);
        for (int i = 0; i < 3; ++i)
            if (p.loc[i]) cudaFree(p.loc[i]);
    }
    for (auto &pp : ctx->prof_pending) { cudaEventDestroy(pp.a); cudaEventDestroy(pp.b); }
    for (auto e : ctx->prof_free) cudaEventDestroy(e);
    for (auto &b : ctx->scratch)
        if (b.ptr) cudaFree(b.ptr);
    for (auto &kv : ctx->block_cache) cudaFree(kv.second);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    cudaStreamDestroy(ctx->copy_stream);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
    return ZKB_OK;
}

// per-kernel-class device time (bench.py's roofline: average launch duration of the dominant kernel measured live, on the stream)
extern "C" int32_t zkb_prof_enable(zkb_ctx *ctx, int32_t on) {
    ZKB_ARG(ctx);
    ctx->prof_on = on != 0;
    return ZKB_OK;
}
extern "C" int32_t zkb_prof_read(zkb_ctx *ctx, int32_t cls, uint64_t *launches, double *ms, int32_t reset) {
    ZKB_ARG(ctx && cls >= 0 && cls < 4);
    ZKB_CUDA(cudaSetDevice(ctx->device));
    for (auto &pp : ctx->prof_pending) {
        ZKB_CUDA(cudaEventSynchronize(pp.b));
        float t = 0;
        ZKB_CUDA(cudaEventElapsedTime(&t, pp.a, pp.b));
        ctx->prof_ms[pp.cls] += t;
        ctx->prof_count[pp.cls]++;
        ctx->prof_free.push_back(pp.a);
        ctx->prof_free.push_back(pp.b);
    }
    ctx->prof_pending.clear();
    if (launches) *launches = ctx->prof_count[cls];
    if (ms) *ms = ctx->prof_ms[cls];
    if (reset) { for (int i = 0; i < 4; ++i) { ctx->prof_ms[i] = 0; ctx->prof_count[i] = 0; } }
    return ZKB_OK;
}

extern "C" uint64_t zkb_launch_count(const zkb_ctx *ctx) { return ctx ? ctx->launches : 0; }
extern "C" uint64_t zkb_msm_last_adds(const zkb_ctx *ctx) { return ctx ? ctx->msm_last_adds : 0; }
extern "C" uint32_t zkb_msm_last_levels(const zkb_ctx *ctx) { return ctx ? ctx->msm_last_levels : 0; }
extern "C" void *zkb_stream(zkb_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }
extern "C" int32_t zkb_sync(zkb_ctx *ctx) {
    ZKB_ARG(ctx);
    ZKB_CUDA(cudaStreamSynchronize(ctx->stream));
    return ZKB_OK;
}
extern "C" int32_t zkb_malloc(zkb_ctx *ctx, uint64_t bytes, void **dptr) {
    ZKB_ARG(ctx && dptr);
    ZKB_CUDA(cudaSetDevice(ctx->device));
    ZKB_CUDA(cudaMalloc(dptr, bytes ? bytes : 1));
    return ZKB_OK;
}
extern "C" int32_t zkb_free(zkb_ctx *ctx, void *dptr) {
    ZKB_ARG(ctx);
    if (dptr) ZKB_CUDA(cudaFree(dptr));
    return ZKB_OK;
}
extern "C" int32_t zkb_h2d(zkb_ctx *ctx, void *dst_dev, const void *src_host, uint64_t bytes) {
    ZKB_ARG(ctx && dst_dev && src_host);
    ZKB_CUDA(cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    ZKB_CUDA(cudaStreamSynchronize(ctx->stream));
    return ZKB_OK;
}
extern "C" int32_t zkb_d2h(zkb_ctx *ctx, void *dst_host, const void *src_dev, uint64_t bytes) {
    ZKB_ARG(ctx && dst_host && src_dev);
    ZKB_CUDA(cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    ZKB_CUDA(cudaStreamSynchronize(ctx->stream));
    return ZKB_OK;
}
