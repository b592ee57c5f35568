// common.cuh -- context, error plumbing and launch accounting shared by all translation units of libzkb200.so
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <map>
#include <string>
#include <vector>
#include <array>
#include "../../include/zkb200.h"
#include "ff.cuh"
#include "g1.cuh"

namespace zkb {

void set_error(const char *fmt, ...);

#define ZKB_CUDA(expr)                                                                                   \
    do {                                                                                                 \
        cudaError_t _e = (expr);                                                                         \
        if (_e != cudaSuccess) {                                                                         \
            zkb::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e));         \
            return _e == cudaErrorMemoryAllocation ? ZKB_ERR_ALLOC : ZKB_ERR_CUDA;                       \
        }                                                                                                \
    } while (0)

#define ZKB_TRY(expr)                    \
    do {                                 \
        int32_t _r = (expr);             \
        if (_r != ZKB_OK) return _r;     \
    } while (0)

#define ZKB_ARG(cond)                                                            \
    do {                                                                         \
        if (!(cond)) {                                                           \
            zkb::set_error("%s:%d invalid argument: %s", __FILE__, __LINE__, #cond); \
            return ZKB_ERR_ARG;                                                  \
        }                                                                        \
    } while (0)

// One cached NTT plan per (log_n, omega): twiddle tables on the device (see ntt.cu for the tile / pass structure).
struct NttPlan {
    uint32_t log_n = 0;
    int npass = 0;
    int bits[3] = {0, 0, 0};
    Fr *tw_lo = nullptr;   // omega^i,           i < 2^min(log_n, 12)   (source of the boundary tables)
    Fr *tw_hi = nullptr;   // omega^(i * 2^12),  i < 2^(log_n - 12)     (log_n > 12)
    Fr *loc[3] = {nullptr, nullptr, nullptr};  // per pass: (omega_{2^a})^i, i < 2^(a-1); TMA-staged into shared memory once per CTA
    // inter-pass twiddle tables, one per pass boundary, stored TILE-MAJOR in the order the consuming tile reads them
    // (tile = cblk, then bit-reversed row q, then column c) so that one cp.async.bulk stages a tile's 64 KB of twiddles:
    //   boundary p: 2^(bits[p]) * 2^(log_inner_p) entries = n for the first boundary, A2*A3 for the second of a 3-pass plan.
    Fr *tw_b[2] = {nullptr, nullptr};
    // the LAST boundary's table with a caller scale folded in (1/n of the inverse transforms), rebuilt when the scale changes
    Fr *tw_b_scaled = nullptr;
    Fr scaled_key;
    bool has_scaled = false;
};

struct DeviceBuffer {
    void *ptr = nullptr;
    size_t bytes = 0;
};

}  // namespace zkb

struct zkb_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;  // H2D of witness columns overlaps the MSMs of the previous batch
    int sm_count = 148;
    // multi-GPU: NCCL communicator of this rank (comm.cu); nranks == 1 -> everything local
    void *nccl_comm = nullptr;
    int rank = 0, nranks = 1;
    // peer-memory exchange window of this rank (sharded.cu): cudaMalloc'ed, exported with cudaIpc, mapped by every other rank
    void *win_local = nullptr;
    size_t win_bytes = 0;
    void *win_peers[16] = {nullptr};   // win_peers[rank] == win_local
    std::map<std::array<uint64_t, 6>, void *> shard_tw;   // cached twiddle tables of the sharded transforms
    uint64_t launches = 0;
    // optional per-kernel-class timing (zkb_prof_*): CUDA event pairs around the launches of the three hot kernels, on the
    // launching stream; off by default (two event records per launch when on)
    bool prof_on = false;
    struct ProfPair { cudaEvent_t a, b; int cls; };
    std::vector<ProfPair> prof_pending;
    std::vector<cudaEvent_t> prof_free;
    double prof_ms[4] = {0, 0, 0, 0};
    uint64_t prof_count[4] = {0, 0, 0, 0};
    bool ntt_ready = false;   // per-device kernel attributes / constants of ntt.cu are set (a context owns one device)
    uint64_t msm_last_adds = 0;
    uint32_t msm_last_levels = 0;   // reduction levels >= 1 the last MSM actually executed (device-side decision)
    std::map<std::array<uint64_t, 5>, zkb::NttPlan> ntt_plans;
    // grow-only scratch arenas (device), keyed by purpose; avoids cudaMalloc in steady state
    zkb::DeviceBuffer scratch[14];
    // cached device blocks (size -> pointers) recycled between proving sessions: cudaMalloc/cudaFree of tens of GB per proof
    // costs seconds and is wildly variable; blocks go back to the driver only at zkb_destroy
    std::multimap<size_t, void *> block_cache;
    size_t block_cache_bytes = 0;
    void *pinned = nullptr;  // small pinned staging buffer
    size_t pinned_bytes = 0;
};

// ParamsKZG<Bn256> resident on the device (srs.cu): g (monomial basis), g_lagrange, and -- memory permitting -- the
// window-shifted copies the one-bucket-set Pippenger variant gathers from.  One handle per context, shared by proving keys.
struct zkb_srs {
    zkb_ctx *ctx = nullptr;
    uint32_t k = 0;
    uint64_t n = 0;
    zkb::G1Affine *g = nullptr, *g_lagrange = nullptr;
    zkb::G1Affine *g_shift = nullptr, *g_lagrange_shift = nullptr;   // msm_shift_copies(n) x n points each, or null
    std::vector<std::pair<void *, size_t>> blocks;
};

namespace zkb {
// returns a device scratch buffer of at least `bytes` (slot-indexed, grow-only)
int32_t scratch_get(zkb_ctx *ctx, int slot, size_t bytes, void **out);
// cached block allocator (see zkb_ctx::block_cache)
int32_t block_alloc(zkb_ctx *ctx, size_t bytes, void **out, size_t *got);
void block_free(zkb_ctx *ctx, void *p, size_t bytes);
inline cudaStream_t pick_stream(zkb_ctx *ctx, void *stream) { return stream ? (cudaStream_t)stream : ctx->stream; }
// kernel classes of zkb_prof_read: 0 ntt_tile_kernel, 1 msm_acc_chunk_kernel, 2 expr_kernel (quotient / lookup interpreter)
enum ProfClass { PROF_NTT = 0, PROF_MSM_ACC = 1, PROF_EXPR = 2, PROF_OTHER = 3 };
struct ProfScope {   // records an event pair around the launches issued while it is alive (no-op unless profiling is on)
    zkb_ctx *ctx;
    cudaStream_t st;
    cudaEvent_t a = nullptr, b = nullptr;
    int cls;
    ProfScope(zkb_ctx *c, int cl, cudaStream_t s) : ctx(c), st(s), cls(cl) {
        if (!ctx->prof_on) return;
        auto get = [&]() { cudaEvent_t e = nullptr; if (!ctx->prof_free.empty()) { e = ctx->prof_free.back(); ctx->prof_free.pop_back(); } else cudaEventCreate(&e); return e; };
        a = get(); b = get();
        cudaEventRecord(a, st);
    }
    ~ProfScope() {
        if (!a) return;
        cudaEventRecord(b, st);
        ctx->prof_pending.push_back({a, b, cls});
    }
};

// ---- cross-translation-unit device-side services (all launch on `st`, none synchronises unless stated) ----------------
Fr host_root_of_unity(uint32_t k);
Fr host_zeta();
// dst <- NTT_omega(src * in_scale) * scale ; src == dst allowed; coset_zeta as in zkb_ntt_fr_dev
int32_t ntt_fr_device(zkb_ctx *ctx, const Fr *src, Fr *dst, uint32_t log_n, const Fr &omega, const Fr *scale_host, int coset_zeta,
                      const Fr *d_in_scale, cudaStream_t st);
// `count` transforms in one launch per pass: column y reads h_src[y], writes h_dst[y] (HOST arrays of device pointers; may alias)
int32_t ntt_fr_batch_device(zkb_ctx *ctx, const Fr *const *h_src, Fr *const *h_dst, uint32_t count, uint32_t log_n,
                            const Fr &omega, const Fr *scale_host, int coset_zeta, const Fr *d_in_scale, cudaStream_t st);
// final-pass routing of a domain-sharded transform: element i of the result is multiplied by out_tw[i] and stored into
// peers[i >> log_blk] at offset (rank << log_blk) + (i mod 2^log_blk)   (peers: device pointers valid on this device, own window included)
struct NttPeerRoute {
    const Fr *out_tw;
    bool routed;          // false: twiddle only, plain store (the NCCL all-to-all variant)
    uint32_t log_blk, rank;
    int nranks;
    Fr *peers[16];
};
int32_t ntt_fr_batch_device_ex(zkb_ctx *ctx, const Fr *const *h_src, Fr *const *h_dst, uint32_t count, uint32_t log_n, const Fr &omega,
                               const Fr *scale_host, int coset_zeta, const Fr *d_in_scale, const NttPeerRoute *route, cudaStream_t st);
// synchronises: the result point is returned to the host
int32_t msm_g1_device(zkb_ctx *ctx, const Fr *scalars, const G1Affine *bases, uint64_t n, G1Affine *out_affine_host, cudaStream_t st);
// `batch` MSMs over the same bases in one pass (d_scalar_cols: DEVICE array of device pointers; batch <= msm_max_batch(n))
uint32_t msm_max_batch(uint64_t n);
// window-shifted precomputed bases (copy w = 2^(c w) P_i): one bucket set per column, no Horner
uint32_t msm_shift_copies(uint64_t n);
int32_t msm_build_shifted_bases(zkb_ctx *ctx, const G1Affine *bases, uint64_t n, G1Affine *out, cudaStream_t st);
int32_t msm_g1_batch_device_ex(zkb_ctx *ctx, const Fr *const *d_scalar_cols, uint32_t batch, const G1Affine *bases, uint64_t n,
                               G1Affine *out_affine_host, bool shifted, cudaStream_t st);
int32_t msm_g1_batch_device(zkb_ctx *ctx, const Fr *const *d_scalar_cols, uint32_t batch, const G1Affine *bases, uint64_t n,
                            G1Affine *out_affine_host, cudaStream_t st);
// SRS handle (srs.cu): sources on the host or on the device; g_lagrange == nullptr -> derived on the device (g_to_lagrange)
int32_t srs_create(zkb_ctx *ctx, uint32_t k, const G1Affine *g, bool g_on_device, const G1Affine *g_lagrange, bool gl_on_device, zkb_srs **out);
// `count` commitments against basis 0 (g) / 1 (g_lagrange); cols = HOST array of device pointers; synchronises (results on the host)
int32_t srs_commit_many(zkb_srs *s, int basis, const Fr *const *cols, uint32_t count, uint64_t len, G1Affine *out_host, cudaStream_t st);
int32_t fr_powers_device(zkb_ctx *ctx, const Fr &base, uint64_t n, Fr *out, cudaStream_t st);
int32_t poly_eval_device(zkb_ctx *ctx, const Fr *const *d_polys, uint32_t num, uint64_t n, const Fr &x, Fr *out_host, cudaStream_t st);
int32_t prefix_product_device(zkb_ctx *ctx, const Fr *in, uint64_t n, const Fr &init, Fr *out, cudaStream_t st);
int32_t prefix_sum_device(zkb_ctx *ctx, const Fr *in, uint64_t n, const Fr &init, Fr *out, cudaStream_t st);
int32_t kate_division_device(zkb_ctx *ctx, const Fr *a, uint64_t n, const Fr &u, Fr *q, cudaStream_t st);
int32_t lincomb_device(zkb_ctx *ctx, const Fr *const *d_polys, const Fr *d_coefs, uint32_t num, uint64_t n, Fr *out, bool accumulate, cudaStream_t st);
int32_t batch_invert_device(zkb_ctx *ctx, const Fr *a, Fr *out, uint64_t n, cudaStream_t st);
// in-place u64 sum across the context's ranks (exact gather when the supports are disjoint); no-op for a single rank
int32_t comm_allreduce_u64(zkb_ctx *ctx, void *dev_buf, size_t count, cudaStream_t st);
// all-gather: every rank contributes bytes_per_rank; recv holds nranks blocks in rank order (send may be recv + rank * bytes_per_rank)
int32_t comm_allgather(zkb_ctx *ctx, const void *send, void *recv, size_t bytes_per_rank, cudaStream_t st);
// the same for small HOST buffers: host holds nranks blocks, this rank's block goes out, all come back; synchronises
int32_t comm_allgather_host(zkb_ctx *ctx, void *host, size_t bytes_per_rank, cudaStream_t st);
// point-range sharded MSM (cross.cu): every rank passes its own slice of scalars and bases; the full sum lands on every rank's host
int32_t msm_g1_sharded(zkb_ctx *ctx, const Fr *scalars, const G1Affine *bases, uint64_t n_local, G1Affine *out_host, cudaStream_t st);
// all-to-all: block s of `send` (bytes_per_block each) goes to rank s; block j of `recv` came from rank j
int32_t comm_alltoall(zkb_ctx *ctx, const void *send, void *recv, size_t bytes_per_block, cudaStream_t st);
// stream-ordered barrier across the ranks (a 8-byte all-reduce): work queued before it on every rank is complete when it completes
int32_t comm_barrier(zkb_ctx *ctx, cudaStream_t st);
// peer-memory window of at least `bytes` on every rank, mapped into every rank (cudaIpc); COLLECTIVE, same `bytes` everywhere
int32_t comm_window(zkb_ctx *ctx, size_t bytes, cudaStream_t st);

struct DevPool {  // owns device allocations of a pk / session; blocks are recycled through the context's block cache
    zkb_ctx *ctx = nullptr;
    std::vector<std::pair<void *, size_t>> ptrs;
    ~DevPool() {
        if (!ctx) return;
        cudaStreamSynchronize(ctx->stream);
        for (auto &p : ptrs) block_free(ctx, p.first, p.second);
    }
    int32_t alloc(size_t bytes, void **out) {
        size_t got = 0;
        ZKB_TRY(block_alloc(ctx, bytes ? bytes : 32, out, &got));
        ptrs.push_back({*out, got});
        return ZKB_OK;
    }
    int32_t fr(uint64_t n, Fr **out) { return alloc(n * sizeof(Fr), (void **)out); }
};

enum ScratchSlot { SCR_NTT = 0, SCR_MSM_A = 1, SCR_MSM_B = 2, SCR_MSM_C = 3, SCR_HOSTIO_A = 4, SCR_HOSTIO_B = 5, SCR_MISC = 6, SCR_MISC2 = 7, SCR_MSM_TBL = 8, SCR_COMM = 9, SCR_NTT_DESC = 10, SCR_MSM_D = 11, SCR_COMM_FLAG = 12, SCR_SHARD = 13 };
}  // namespace zkb
