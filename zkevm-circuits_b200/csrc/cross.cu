// cross.cu -- multi-GPU building blocks (SURVEY.md section 8e): the size-P transform ACROSS ranks that follows the
// all-to-all of a domain-sharded NTT, and the host-side sum of per-rank MSM partial results.
//
// Sharding of one huge NTT (n = P * M, P ranks; halo2's best_fft has no distributed form, this is new):
//   input  : rank r holds the cyclic subsequence x[r + P t], t < M
//   step A : local size-M NTT with omega^P                       (existing kernels)
//   step B : multiply element t by omega^(r t)                   (fr_powers + element-wise multiply)
//   step C : ONE all-to-all: rank s receives, from every rank j, the block t in [s M/P, (s+1) M/P)
//   step D : zkb_ntt_cross_dev: out[k][t] = sum_j in[j][t] * omega_P^(j k)  (this file; log2 P radix-2 stages in registers, P <= 16)
//   output : rank s holds X[k M + s M/P + t] for k < P, t < M/P  ("strips"; zkb200.parallel.strips_to_natural documents it)
// MSM shards by point range (no exchange of points); partial sums are all-gathered as 64-byte affine points and added
// with zkb_g1_sum_affine_host (pure host code, also usable on a box without a GPU).
#include "common.cuh"
#include <string.h>
#include <stdlib.h>

namespace zkb {

struct CrossTw { Fr w[16]; };  // omega_P^i, i < P

// log2(P) radix-2 decimation-in-frequency stages in registers: (P/2) log2 P multiplies per t (12 at P = 8, 32 at P = 16; the
// earlier direct O(P^2) form needed 56 / 240 and spilled); outputs leave in bit-reversed register order.
template <int P>
__global__ void __launch_bounds__(128) ntt_cross_kernel(const Fr *__restrict__ in, Fr *__restrict__ out, uint64_t len, CrossTw tw) {
    const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (t >= len) return;
    Fr v[P];
#pragma unroll
    for (int j = 0; j < P; ++j) v[j] = fp_load(in + (size_t)j * len + t);
#pragma unroll
    for (int half = P / 2; half >= 1; half >>= 1) {
#pragma unroll
        for (int b = 0; b < P; b += 2 * half) {
#pragma unroll
            for (int j = 0; j < half; ++j) {
                const Fr u = v[b + j], w = v[b + j + half];
                v[b + j] = fp_add(u, w);
                const Fr d = fp_sub(u, w);
                const int e = j * (P / (2 * half));   // omega_P^e
                v[b + j + half] = e == 0 ? d : fp_mul(d, tw.w[e]);
            }
        }
    }
#pragma unroll
    for (int i = 0; i < P; ++i) {
        int k = 0;
#pragma unroll
        for (int bit = 1, rb = P >> 1; bit < P; bit <<= 1, rb >>= 1) if (i & bit) k |= rb;
        fp_store(out + (size_t)k * len + t, v[i]);
    }
}

}  // namespace zkb
using namespace zkb;

extern "C" int32_t zkb_ntt_cross_dev(zkb_ctx *ctx, const uint64_t *in_dev, uint64_t *out_dev, uint32_t p, uint64_t len, const uint64_t omega_p[4],
                                     void *stream) {
    ZKB_ARG(ctx && in_dev && out_dev && omega_p && in_dev != out_dev);
    ZKB_ARG(p == 1 || p == 2 || p == 4 || p == 8 || p == 16);
    if (len == 0) return ZKB_OK;
    cudaStream_t st = pick_stream(ctx, stream);
    Fr w;
    memcpy(w.l, omega_p, 32);
    // order check: w^p == 1 and (p > 1) w^(p/2) == -1
    if (!(fp_pow_u64(w, p) == Fr::one()) || (p > 1 && !fp_add(fp_pow_u64(w, p / 2), Fr::one()).is_zero())) {
        set_error("omega_p does not have order %u", p);
        return ZKB_ERR_ARG;
    }
    CrossTw tw;
    tw.w[0] = Fr::one();
    for (uint32_t i = 1; i < 16; ++i) tw.w[i] = i < p ? fp_mul(tw.w[i - 1], w) : Fr::zero();
    const unsigned blocks = (unsigned)((len + 127) / 128);
    const Fr *in = (const Fr *)in_dev;
    Fr *out = (Fr *)out_dev;
    switch (p) {
    case 1: ZKB_CUDA(cudaMemcpyAsync(out, in, len * sizeof(Fr), cudaMemcpyDeviceToDevice, st)); break;
    case 2: ntt_cross_kernel<2><<<blocks, 128, 0, st>>>(in, out, len, tw); break;
    case 4: ntt_cross_kernel<4><<<blocks, 128, 0, st>>>(in, out, len, tw); break;
    case 8: ntt_cross_kernel<8><<<blocks, 128, 0, st>>>(in, out, len, tw); break;
    default: ntt_cross_kernel<16><<<blocks, 128, 0, st>>>(in, out, len, tw); break;
    }
    ctx->launches++;
    ZKB_CUDA(cudaGetLastError());
    return ZKB_OK;
}

// sum of `count` affine points (host buffers); pure host arithmetic, no CUDA device needed
extern "C" int32_t zkb_g1_sum_affine_host(const uint64_t *points, uint64_t count, uint64_t out_affine[8], uint8_t *out_compressed) {
    ZKB_ARG(out_affine && (points || count == 0));
    G1Xyzz acc = G1Xyzz::identity();
    for (uint64_t i = 0; i < count; ++i) {
        G1Affine p;
        memcpy(&p, points + 8 * i, 64);
        g1_add_mixed(acc, p);
    }
    const G1Affine r = g1_to_affine(acc);
    memcpy(out_affine, &r, 64);
    if (out_compressed) g1_compress(r, out_compressed);
    return ZKB_OK;
}

// ======================================================================================================================
// Domain-sharded NTT and point-range sharded MSM behind the C ABI (SURVEY.md 8e; one process per GPU, communicator from
// zkb_comm_init).  halo2's best_fft / best_multiexp have no distributed form; what is reproduced is their RESULT.
//
//   n = P * M, rank r.  "cyclic" layout: rank r holds x[r + P t], t < M.  "strips" layout: rank s holds X[k1 M + s B + t] at row
//   k1 B + t (B = M / P, k1 < P, t < B).  With j = r + P t and k = k2 + M k1:  omega^(j k) = omega_M^(t k2) omega^(r k2) omega_P^(r k1).
//
//   direction 0 (cyclic in -> strips out):  local size-M transform, twiddle omega^(r k2), EXCHANGE (block s of rank r -> row r of
//        rank s), size-P transform across the rows.  The twiddle and the exchange are FUSED into the store phase of the local
//        transform's last pass: every result is multiplied by its twiddle and stored straight into the owner's window over
//        NVLink (peer store), tile by tile, while the butterflies of the following tiles run -- one kernel, no staging copy.
//   direction 1 (strips in -> cyclic out):  size-P transform across the rows fused with the twiddle and the peer stores
//        (ntt_cross_kernel<P, true>), then the local size-M transform reads the window.
//   The only NCCL traffic on this path is the 8-byte all-reduce used as a stream-ordered barrier on both sides of the exchange.
//   ZKB_SHARDED_EXCHANGE=nccl selects the baseline instead (twiddle kernel, ncclSend/ncclRecv all-to-all, cross kernel) so that
//   bench.py can print both.
namespace zkb {

struct Pow2Tab { Fr p[28]; };   // base^(2^j)
// out[i] = first * base^i
__global__ void geometric_kernel(Fr first, Pow2Tab tab, uint64_t n, Fr *__restrict__ out) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fr acc = first;
    for (int j = 0; j < 28; ++j)
        if ((i >> j) & 1) acc = fp_mul(acc, tab.p[j]);
    fp_store(out + i, acc);
}
static int32_t geometric_device(zkb_ctx *ctx, const Fr &first, const Fr &base, uint64_t n, Fr *out, cudaStream_t st) {
    ZKB_ARG(n <= (1ull << 28));
    Pow2Tab t;
    t.p[0] = base;
    for (int j = 1; j < 28; ++j) t.p[j] = fp_sqr(t.p[j - 1]);
    geometric_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(first, t, n, out);
    ctx->launches++;
    ZKB_CUDA(cudaGetLastError());
    return ZKB_OK;
}

struct CrossRoute {
    const Fr *tw;        // [k][t]: multiplier of output row k, column t
    uint32_t log_blk;    // log2 B
    uint32_t rank;       // this rank s: row k goes to peers[k] at offset s * B + t
    Fr *peers[16];
};
// the cross transform of direction 1: rows in, every output row k multiplied by tw[k][t] and stored into rank k's window
template <int P>
__global__ void __launch_bounds__(128) ntt_cross_scatter_kernel(const Fr *__restrict__ in, uint64_t len, CrossTw tw, CrossRoute rt) {
    const uint64_t t = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (t >= len) return;
    Fr v[P];
#pragma unroll
    for (int j = 0; j < P; ++j) v[j] = fp_load(in + (size_t)j * len + t);
#pragma unroll
    for (int half = P / 2; half >= 1; half >>= 1) {
#pragma unroll
        for (int b = 0; b < P; b += 2 * half) {
#pragma unroll
            for (int j = 0; j < half; ++j) {
                const Fr u = v[b + j], w = v[b + j + half];
                v[b + j] = fp_add(u, w);
                const Fr d = fp_sub(u, w);
                const int e = j * (P / (2 * half));
                v[b + j + half] = e == 0 ? d : fp_mul(d, tw.w[e]);
            }
        }
    }
#pragma unroll
    for (int i = 0; i < P; ++i) {
        int k = 0;
#pragma unroll
        for (int bit = 1, rb = P >> 1; bit < P; bit <<= 1, rb >>= 1) if (i & bit) k |= rb;
        const Fr r = k == 0 ? v[i] : fp_mul(v[i], fp_load(rt.tw + (size_t)k * len + t));   // omega^(0 * k2) = 1
        fp_store_stream(rt.peers[k] + ((uint64_t)rt.rank << rt.log_blk) + t, r);
    }
}

static Fr fr_pow(const Fr &b, uint64_t e) { return fp_pow_u64(b, e); }

// cached table of a sharded transform: kind 0 -> omega^(rank * k2), k2 < M;  kind 1 -> [k][t] = omega^(k * (rank * B + t))
static int32_t shard_table(zkb_ctx *ctx, int kind, uint32_t log_n, const Fr &omega, Fr **out, cudaStream_t st) {
    std::array<uint64_t, 6> key;
    key[0] = ((uint64_t)kind << 32) | log_n;
    for (int i = 0; i < 4; ++i) key[1 + i] = (uint64_t)omega.l[2 * i] | ((uint64_t)omega.l[2 * i + 1] << 32);
    key[5] = ((uint64_t)ctx->rank << 32) | (uint64_t)ctx->nranks;
    auto it = ctx->shard_tw.find(key);
    if (it != ctx->shard_tw.end()) { *out = (Fr *)it->second; return ZKB_OK; }
    const uint32_t P = (uint32_t)ctx->nranks;
    const uint64_t M = (1ull << log_n) / P, B = M / P;
    Fr *tbl = nullptr;
    ZKB_CUDA(cudaMalloc((void **)&tbl, M * sizeof(Fr)));
    if (kind == 0) {
        ZKB_TRY(geometric_device(ctx, Fr::one(), fr_pow(omega, (uint64_t)ctx->rank), M, tbl, st));
    } else {
        for (uint32_t k = 0; k < P; ++k) {
            const Fr ratio = fr_pow(omega, k);
            ZKB_TRY(geometric_device(ctx, fr_pow(ratio, (uint64_t)ctx->rank * B), ratio, B, tbl + (size_t)k * B, st));
        }
    }
    ctx->shard_tw.emplace(key, tbl);
    *out = tbl;
    return ZKB_OK;
}

static bool exchange_over_nccl() {
    const char *e = getenv("ZKB_SHARDED_EXCHANGE");
    return e && (e[0] == 'n' || e[0] == 'N');
}

template <int P>
static void launch_cross_scatter(const Fr *in, uint64_t len, const CrossTw &tw, const CrossRoute &rt, cudaStream_t st) {
    ntt_cross_scatter_kernel<P><<<(unsigned)((len + 127) / 128), 128, 0, st>>>(in, len, tw, rt);
}

}  // namespace zkb

extern "C" int32_t zkb_ntt_fr_sharded_dev(zkb_ctx *ctx, const uint64_t *in_dev, uint64_t *out_dev, uint32_t log_n, const uint64_t omega[4],
                                          const uint64_t *scale, int32_t direction, void *stream) {
    ZKB_ARG(ctx && in_dev && out_dev && omega && (direction == 0 || direction == 1) && in_dev != out_dev);
    ZKB_CUDA(cudaSetDevice(ctx->device));
    const uint32_t P = (uint32_t)ctx->nranks;
    uint32_t log_p = 0;
    while ((1u << log_p) < P) ++log_p;
    ZKB_ARG((1u << log_p) == P && P <= 16 && log_n <= 28 && log_n >= 2 * log_p);
    cudaStream_t st = pick_stream(ctx, stream);
    Fr w, sc;
    memcpy(w.l, omega, 32);
    if (scale) memcpy(sc.l, scale, 32);
    const uint32_t log_m = log_n - log_p;
    const uint64_t M = 1ull << log_m, B = M >> log_p;
    const Fr w_m = fp_pow_u64(w, P);          // order M
    const Fr w_p = fp_pow_u64(w, M);          // order P
    if (P == 1) return ntt_fr_device(ctx, (const Fr *)in_dev, (Fr *)out_dev, log_n, w, scale ? &sc : nullptr, 0, nullptr, st);
    {   // order check of omega_P (the local plan checks omega_M): catches a root of the wrong order before anything is exchanged
        if (!(fp_pow_u64(w_p, P) == Fr::one()) || !fp_add(fp_pow_u64(w_p, P / 2), Fr::one()).is_zero()) { set_error("omega does not have order 2^%u", log_n); return ZKB_ERR_ARG; }
    }
    CrossTw ctw;
    ctw.w[0] = Fr::one();
    for (uint32_t i = 1; i < 16; ++i) ctw.w[i] = i < P ? fp_mul(ctw.w[i - 1], w_p) : Fr::zero();
    const bool nccl = exchange_over_nccl();
    ZKB_TRY(comm_window(ctx, M * sizeof(Fr), st));
    Fr *win = (Fr *)ctx->win_local;
    Fr *tbl = nullptr;
    ZKB_TRY(shard_table(ctx, direction, log_n, w, &tbl, st));
    const Fr *in = (const Fr *)in_dev;
    Fr *out = (Fr *)out_dev;
    ZKB_TRY(comm_barrier(ctx, st));   // every rank is done reading its window (previous call) before anyone stores into it
    if (direction == 0) {
        NttPeerRoute rt;
        rt.out_tw = tbl;
        rt.routed = !nccl;
        rt.log_blk = log_m - log_p;
        rt.rank = (uint32_t)ctx->rank;
        rt.nranks = (int)P;
        for (uint32_t j = 0; j < 16; ++j) rt.peers[j] = j < P ? (Fr *)ctx->win_peers[j] : nullptr;
        const Fr *src = in;
        Fr *dst = out;   // nccl variant: twiddled result lands in `out`, blocks in destination order
        ZKB_TRY(ntt_fr_batch_device_ex(ctx, &src, &dst, 1, log_m, w_m, scale ? &sc : nullptr, 0, nullptr, &rt, st));   // the caller's scale rides on the local transform (linear)
        if (nccl) ZKB_TRY(comm_alltoall(ctx, out, win, B * sizeof(Fr), st));
        else ZKB_TRY(comm_barrier(ctx, st));   // all peer stores into this rank's window have landed
        // rows of the window -> strips
        switch (P) {
        case 2: ntt_cross_kernel<2><<<(unsigned)((B + 127) / 128), 128, 0, st>>>(win, out, B, ctw); break;
        case 4: ntt_cross_kernel<4><<<(unsigned)((B + 127) / 128), 128, 0, st>>>(win, out, B, ctw); break;
        case 8: ntt_cross_kernel<8><<<(unsigned)((B + 127) / 128), 128, 0, st>>>(win, out, B, ctw); break;
        default: ntt_cross_kernel<16><<<(unsigned)((B + 127) / 128), 128, 0, st>>>(win, out, B, ctw); break;
        }
        ctx->launches++;
        ZKB_CUDA(cudaGetLastError());
    } else {
        if (nccl) {
            // baseline: cross transform into scratch, twiddle multiply, all-to-all, local transform
            Fr *tmp = nullptr;
            ZKB_TRY(scratch_get(ctx, SCR_SHARD, M * sizeof(Fr), (void **)&tmp));
            ZKB_TRY(zkb_ntt_cross_dev(ctx, in_dev, (uint64_t *)tmp, P, B, (const uint64_t *)w_p.l, st));
            ZKB_TRY(zkb_field_binop_dev(ctx, 0, 2, (const uint64_t *)tmp, (const uint64_t *)tbl, (uint64_t *)tmp, M, st));
            ZKB_TRY(comm_alltoall(ctx, tmp, win, B * sizeof(Fr), st));
        } else {
            CrossRoute rt;
            rt.tw = tbl;
            rt.log_blk = log_m - log_p;
            rt.rank = (uint32_t)ctx->rank;
            for (uint32_t j = 0; j < 16; ++j) rt.peers[j] = j < P ? (Fr *)ctx->win_peers[j] : nullptr;
            switch (P) {
            case 2: launch_cross_scatter<2>(in, B, ctw, rt, st); break;
            case 4: launch_cross_scatter<4>(in, B, ctw, rt, st); break;
            case 8: launch_cross_scatter<8>(in, B, ctw, rt, st); break;
            default: launch_cross_scatter<16>(in, B, ctw, rt, st); break;
            }
            ctx->launches++;
            ZKB_CUDA(cudaGetLastError());
            ZKB_TRY(comm_barrier(ctx, st));
        }
        ZKB_TRY(ntt_fr_device(ctx, win, out, log_m, w_m, scale ? &sc : nullptr, 0, nullptr, st));
    }
    return ZKB_OK;
}

namespace zkb {
// point-range sharded MSM: this rank's slice -> local Pippenger -> all-gather of the 64-byte partial sums -> host add.
// Identical result on every rank.  No point crosses NVLink (SURVEY 8e).
int32_t msm_g1_sharded(zkb_ctx *ctx, const Fr *scalars, const G1Affine *bases, uint64_t n_local, G1Affine *out_host, cudaStream_t st) {
    G1Affine all[16];
    ZKB_TRY(msm_g1_device(ctx, scalars, bases, n_local, &all[ctx->rank], st));
    ZKB_TRY(comm_allgather_host(ctx, all, sizeof(G1Affine), st));
    return zkb_g1_sum_affine_host((const uint64_t *)all, (uint64_t)ctx->nranks, (uint64_t *)out_host, nullptr);
}
}  // namespace zkb

extern "C" int32_t zkb_msm_g1_sharded_dev(zkb_ctx *ctx, const uint64_t *scalars_shard_dev, const uint64_t *bases_shard_dev, uint64_t n_local,
                                          uint64_t out_affine[8], uint8_t *out_compressed, void *stream) {
    ZKB_ARG(ctx && out_affine && (n_local == 0 || (scalars_shard_dev && bases_shard_dev)));
    ZKB_CUDA(cudaSetDevice(ctx->device));
    G1Affine r;
    ZKB_TRY(msm_g1_sharded(ctx, (const Fr *)scalars_shard_dev, (const G1Affine *)bases_shard_dev, n_local, &r, pick_stream(ctx, stream)));
    memcpy(out_affine, &r, 64);
    if (out_compressed) g1_compress(r, out_compressed);
    return ZKB_OK;
}
