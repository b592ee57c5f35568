// comm.cu -- NCCL communicator of a context (one process per GPU) for the multi-GPU create_proof.
//
// The proving session stays replicated (every rank runs the same host code on the same inputs and therefore produces
// the same transcript and the same proof bytes); only the two heavy, embarrassingly parallel stages are dealt across
// ranks (SURVEY.md 8e): commitment batches (column i is committed by rank i mod P) and the quotient's coset parts (part j
// by rank j mod P).  Results are exchanged with ONE all-reduce each over NVLink: every rank writes its share into a
// zero-initialised buffer, so a u64 sum of the disjoint supports is an exact gather (no 256-bit NCCL type exists).
// NCCL is resolved at run time (dlopen of libnccl.so.2: inside a torch process that is torch's bundled copy).
#include "common.cuh"
#include <dlfcn.h>
#include <nccl.h>
#include <string.h>

namespace zkb {

struct NcclApi {
    void *handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
};

static NcclApi *nccl_api() {
    static NcclApi api;
    if (api.handle) return &api;
    void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) { set_error("cannot load libnccl.so.2: %s", dlerror()); return nullptr; }
    api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(h, "ncclGetUniqueId");
    api.CommInitRank = (decltype(api.CommInitRank))dlsym(h, "ncclCommInitRank");
    api.CommDestroy = (decltype(api.CommDestroy))dlsym(h, "ncclCommDestroy");
    api.AllReduce = (decltype(api.AllReduce))dlsym(h, "ncclAllReduce");
    api.GetErrorString = (decltype(api.GetErrorString))dlsym(h, "ncclGetErrorString");
    api.AllGather = (decltype(api.AllGather))dlsym(h, "ncclAllGather");
    api.Send = (decltype(api.Send))dlsym(h, "ncclSend");
    api.Recv = (decltype(api.Recv))dlsym(h, "ncclRecv");
    api.GroupStart = (decltype(api.GroupStart))dlsym(h, "ncclGroupStart");
    api.GroupEnd = (decltype(api.GroupEnd))dlsym(h, "ncclGroupEnd");
    if (!api.GetUniqueId || !api.CommInitRank || !api.CommDestroy || !api.AllReduce || !api.AllGather || !api.Send || !api.Recv || !api.GroupStart || !api.GroupEnd) { set_error("libnccl.so.2 lacks required symbols"); return nullptr; }
    api.handle = h;
    return &api;
}

#define ZKB_NCCL(api, expr)                                                                                           \
    do {                                                                                                              \
        ncclResult_t _r = (expr);                                                                                     \
        if (_r != ncclSuccess) {                                                                                      \
            zkb::set_error("%s:%d NCCL: %s", __FILE__, __LINE__, (api)->GetErrorString ? (api)->GetErrorString(_r) : "error"); \
            return ZKB_ERR_CUDA;                                                                                      \
        }                                                                                                             \
    } while (0)

// in-place sum of `count` u64 words on the device (disjoint supports -> exact gather)
int32_t comm_allreduce_u64(zkb_ctx *ctx, void *dev_buf, size_t count, cudaStream_t st) {
    if (ctx->nranks <= 1) return ZKB_OK;
    NcclApi *api = nccl_api();
    if (!api || !ctx->nccl_comm) { set_error("communicator not initialised"); return ZKB_ERR_STATE; }
    ZKB_NCCL(api, api->AllReduce(dev_buf, dev_buf, count, ncclUint64, ncclSum, (ncclComm_t)ctx->nccl_comm, st));
    return ZKB_OK;
}

int32_t comm_allgather(zkb_ctx *ctx, const void *send, void *recv, size_t bytes_per_rank, cudaStream_t st) {
    if (ctx->nranks <= 1) {
        if (send != recv) ZKB_CUDA(cudaMemcpyAsync(recv, send, bytes_per_rank, cudaMemcpyDeviceToDevice, st));
        return ZKB_OK;
    }
    NcclApi *api = nccl_api();
    if (!api || !ctx->nccl_comm) { set_error("communicator not initialised"); return ZKB_ERR_STATE; }
    ZKB_NCCL(api, api->AllGather(send, recv, bytes_per_rank, ncclUint8, (ncclComm_t)ctx->nccl_comm, st));
    return ZKB_OK;
}

int32_t comm_allgather_host(zkb_ctx *ctx, void *host, size_t bytes_per_rank, cudaStream_t st) {
    if (ctx->nranks <= 1) return ZKB_OK;
    uint8_t *d = nullptr;
    const size_t own = (size_t)ctx->rank * bytes_per_rank;
    ZKB_TRY(scratch_get(ctx, SCR_COMM, (size_t)ctx->nranks * bytes_per_rank, (void **)&d));
    ZKB_CUDA(cudaMemcpyAsync(d + own, (const uint8_t *)host + own, bytes_per_rank, cudaMemcpyHostToDevice, st));
    ZKB_TRY(comm_allgather(ctx, d + own, d, bytes_per_rank, st));
    ZKB_CUDA(cudaMemcpyAsync(host, d, (size_t)ctx->nranks * bytes_per_rank, cudaMemcpyDeviceToHost, st));
    ZKB_CUDA(cudaStreamSynchronize(st));
    return ZKB_OK;
}

int32_t comm_alltoall(zkb_ctx *ctx, const void *send, void *recv, size_t bytes_per_block, cudaStream_t st) {
    if (ctx->nranks <= 1) {
        if (send != recv) ZKB_CUDA(cudaMemcpyAsync(recv, send, bytes_per_block, cudaMemcpyDeviceToDevice, st));
        return ZKB_OK;
    }
    NcclApi *api = nccl_api();
    if (!api || !ctx->nccl_comm) { set_error("communicator not initialised"); return ZKB_ERR_STATE; }
    ncclComm_t comm = (ncclComm_t)ctx->nccl_comm;
    ZKB_NCCL(api, api->GroupStart());
    for (int j = 0; j < ctx->nranks; ++j) {
        ZKB_NCCL(api, api->Send((const uint8_t *)send + (size_t)j * bytes_per_block, bytes_per_block, ncclUint8, j, comm, st));
        ZKB_NCCL(api, api->Recv((uint8_t *)recv + (size_t)j * bytes_per_block, bytes_per_block, ncclUint8, j, comm, st));
    }
    ZKB_NCCL(api, api->GroupEnd());
    return ZKB_OK;
}

int32_t comm_barrier(zkb_ctx *ctx, cudaStream_t st) {
    if (ctx->nranks <= 1) return ZKB_OK;
    void *w = nullptr;
    ZKB_TRY(scratch_get(ctx, SCR_COMM_FLAG, 64, &w));
    return comm_allreduce_u64(ctx, w, 1, st);
}

// Exchange window: one cudaMalloc block per rank, exported with cudaIpcGetMemHandle, the 64-byte handles all-gathered over the
// communicator and opened by every other rank (cudaIpcMemLazyEnablePeerAccess): afterwards ctx->win_peers[j] is a pointer that
// kernels on THIS device can load from / store to; the traffic goes over NVLink / NVSwitch as plain peer accesses.
int32_t comm_window(zkb_ctx *ctx, size_t bytes, cudaStream_t st) {
    if (ctx->win_bytes >= bytes && ctx->win_local) return ZKB_OK;
    // every rank must be past its last use of the old windows before anyone unmaps them
    ZKB_TRY(comm_barrier(ctx, st));
    ZKB_CUDA(cudaStreamSynchronize(st));
    for (int j = 0; j < ctx->nranks; ++j)
        if (j != ctx->rank && ctx->win_peers[j]) { cudaIpcCloseMemHandle(ctx->win_peers[j]); ctx->win_peers[j] = nullptr; }
    if (ctx->nranks > 1) { ZKB_TRY(comm_barrier(ctx, st)); ZKB_CUDA(cudaStreamSynchronize(st)); }   // all peers unmapped before the owner frees
    if (ctx->win_local) { ZKB_CUDA(cudaFree(ctx->win_local)); ctx->win_local = nullptr; ctx->win_bytes = 0; }
    const size_t want = (bytes + (2u << 20) - 1) & ~(size_t)((2u << 20) - 1);
    ZKB_CUDA(cudaMalloc(&ctx->win_local, want));
    ctx->win_bytes = want;
    ctx->win_peers[ctx->rank] = ctx->win_local;
    if (ctx->nranks <= 1) return ZKB_OK;
    cudaIpcMemHandle_t all[16];
    ZKB_CUDA(cudaIpcGetMemHandle(&all[ctx->rank], ctx->win_local));
    ZKB_TRY(comm_allgather_host(ctx, all, sizeof(cudaIpcMemHandle_t), st));
    for (int j = 0; j < ctx->nranks; ++j) {
        if (j == ctx->rank) continue;
        ZKB_CUDA(cudaIpcOpenMemHandle(&ctx->win_peers[j], all[j], cudaIpcMemLazyEnablePeerAccess));
    }
    return ZKB_OK;
}

}  // namespace zkb
using namespace zkb;

extern "C" int32_t zkb_comm_unique_id(uint8_t out[128]) {
    ZKB_ARG(out != nullptr);
    NcclApi *api = nccl_api();
    if (!api) return ZKB_ERR_CUDA;
    ncclUniqueId id;
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    ZKB_NCCL(api, api->GetUniqueId(&id));
    memcpy(out, &id, 128);
    return ZKB_OK;
}

extern "C" int32_t zkb_comm_init(zkb_ctx *ctx, const uint8_t unique_id[128], int32_t rank, int32_t nranks) {
    ZKB_ARG(ctx && unique_id && nranks >= 1 && rank >= 0 && rank < nranks);
    if (ctx->nccl_comm) { set_error("communicator already initialised"); return ZKB_ERR_STATE; }
    ZKB_CUDA(cudaSetDevice(ctx->device));
    NcclApi *api = nccl_api();
    if (!api) return ZKB_ERR_CUDA;
    ncclUniqueId id;
    memcpy(&id, unique_id, 128);
    ncclComm_t comm = nullptr;
    ZKB_NCCL(api, api->CommInitRank(&comm, nranks, id, rank));
    ctx->nccl_comm = comm;
    ctx->rank = rank;
    ctx->nranks = nranks;
    return ZKB_OK;
}

extern "C" int32_t zkb_comm_destroy(zkb_ctx *ctx) {
    ZKB_ARG(ctx);
    // exchange window: unmap the peers' blocks, free the own one (the peers close their mappings in their own destroy)
    for (int j = 0; j < 16; ++j)
        if (j != ctx->rank && ctx->win_peers[j]) { cudaIpcCloseMemHandle(ctx->win_peers[j]); ctx->win_peers[j] = nullptr; }
    if (ctx->nccl_comm) {
        NcclApi *api = nccl_api();
        cudaStreamSynchronize(ctx->stream);
        if (api) api->CommDestroy((ncclComm_t)ctx->nccl_comm);
        ctx->nccl_comm = nullptr;
    }
    if (ctx->win_local) { cudaFree(ctx->win_local); ctx->win_local = nullptr; ctx->win_bytes = 0; }
    ctx->win_peers[ctx->rank] = nullptr;
    for (auto &kv : ctx->shard_tw) cudaFree(kv.second);
    ctx->shard_tw.clear();
    ctx->rank = 0;
    ctx->nranks = 1;
    return ZKB_OK;
}
