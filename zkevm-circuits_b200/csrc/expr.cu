// expr.cu -- device interpreter for constraint-expression programs (see expr.cuh).
#include "common.cuh"
#include "expr.cuh"
#include <stdlib.h>

namespace zkb {

struct ExprLaunch {
    const Instr *code;
    uint32_t ncode;
    const Fr *const *cols;   // column slot -> device array of (1 << log_n) elements
    const Fr *consts;
    Fr *const *outs;         // output slot -> device array
    uint32_t log_n;
    uint32_t out_stride;     // output index = row * out_stride + out_offset
    uint32_t out_offset;
};

// Register file of the interpreter.  SMEM = true: in SHARED memory, two 16-byte planes indexed [reg][thread] (adjacent lanes touch
// adjacent 16-byte slots: conflict free).  The first version kept it in local memory: 512 B per thread x ~150 k resident threads is
// L2-sized, so the "registers" and the column data evicted each other and one coset part of the k = 20 quotient moved 107 GB
// through HBM for 7.8 GB of algorithmic traffic (profiles/r02_expr_kernel_k20_ncu.txt).  SMEM = false: local memory (NREGS = 64).
template <int NREGS, int THREADS, bool SMEM>
struct RegFile {
    uint4 *lo, *hi;
    Fr loc[SMEM ? 1 : NREGS];
    __device__ __forceinline__ RegFile(uint4 *base) : lo(base + threadIdx.x), hi(base + NREGS * THREADS + threadIdx.x) {}
    __device__ __forceinline__ Fr get(uint32_t r) const {
        if (!SMEM) return loc[r];
        const uint4 a = lo[r * THREADS], b = hi[r * THREADS];
        Fr v;
        v.l[0] = a.x; v.l[1] = a.y; v.l[2] = a.z; v.l[3] = a.w;
        v.l[4] = b.x; v.l[5] = b.y; v.l[6] = b.z; v.l[7] = b.w;
        return v;
    }
    __device__ __forceinline__ void set(uint32_t r, const Fr &v) {
        if (!SMEM) { loc[r] = v; return; }
        lo[r * THREADS] = make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]);
        hi[r * THREADS] = make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]);
    }
};

// one instruction for the thread owning `row`; `cols` is the slot table the program reads (one circuit's table in a batched launch)
template <int NREGS, int THREADS, bool SMEM>
__device__ __forceinline__ void expr_step(const ExprLaunch &L, const Instr in, const Fr *const *cols, uint32_t row, uint32_t mask,
                                          RegFile<NREGS, THREADS, SMEM> &regs, Fr &acc, Fr &acc2) {
    switch (in.op) {
    case OP_LOADCOL: {
        const int32_t rot = (int32_t)(int16_t)(in.imm >> 16);
        const uint32_t r = (row + (uint32_t)rot) & mask;
        regs.set(in.dst, fp_load(cols[in.imm & 0xffffu] + r));
    } break;
    case OP_LOADCONST: regs.set(in.dst, fp_load(L.consts + in.imm)); break;
    case OP_ADD: { Fr a = regs.get(in.a), b = regs.get(in.b); regs.set(in.dst, fp_add(a, b)); } break;
    case OP_SUB: { Fr a = regs.get(in.a), b = regs.get(in.b); regs.set(in.dst, fp_sub(a, b)); } break;
    case OP_MUL: { Fr a = regs.get(in.a), b = regs.get(in.b); regs.set(in.dst, fp_mul(a, b)); } break;
    case OP_NEG: { Fr a = regs.get(in.a); regs.set(in.dst, fp_neg(a)); } break;
    case OP_HORNER: acc = fp_add(fp_mul(acc, fp_load(L.consts + in.imm)), regs.get(in.a)); break;
    case OP_STORE: fp_store(L.outs[in.imm] + (size_t)row * L.out_stride + L.out_offset, regs.get(in.a)); break;
    case OP_STOREACC:
        fp_store(L.outs[in.imm & 0xffu] + (size_t)row * L.out_stride + L.out_offset, fp_mul(acc, fp_load(L.consts + (in.imm >> 8))));
        break;
    case OP_CLEARACC: acc = Fr::zero(); break;
    case OP_HORNER2: acc2 = fp_add(fp_mul(acc2, fp_load(L.consts + in.imm)), regs.get(in.a)); break;
    case OP_FOLD:
        acc = fp_add(fp_mul(acc, fp_load(L.consts + in.imm)), fp_mul(regs.get(in.a), acc2));
        acc2 = Fr::zero();
        break;
    default: break;
    }
}

template <int NREGS, int THREADS, bool SMEM>
__global__ void __launch_bounds__(THREADS) expr_kernel(ExprLaunch L) {
    extern __shared__ uint4 expr_smem[];
    const uint32_t n = 1u << L.log_n, mask = n - 1;
    const uint32_t row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n) return;
    RegFile<NREGS, THREADS, SMEM> regs(expr_smem);
    Fr acc = Fr::zero(), acc2 = Fr::zero();
    for (uint32_t pc = 0; pc < L.ncode; ++pc) expr_step(L, L.code[pc], L.cols, row, mask, regs, acc, acc2);
}

// Several circuits of one constraint system (create_proof with C circuits): the body code[0, body_len) runs once per circuit,
// run c reading the slot table at cols + c * stride, and acc / acc2 carry over from one run to the next, so circuit c's
// constraints continue the Horner chain in y where circuit c - 1 stopped.  The tail code[body_len, ncode) runs once, after the
// last circuit.  A separate kernel, so the single-circuit launches keep their code.
struct ExprCircuits {
    uint32_t count, body_len, stride;
};
template <int NREGS, int THREADS, bool SMEM>
__global__ void __launch_bounds__(THREADS) expr_circuits_kernel(ExprLaunch L, ExprCircuits C) {
    extern __shared__ uint4 expr_smem[];
    const uint32_t n = 1u << L.log_n, mask = n - 1;
    const uint32_t row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n) return;
    RegFile<NREGS, THREADS, SMEM> regs(expr_smem);
    Fr acc = Fr::zero(), acc2 = Fr::zero();
    for (uint32_t c = 0; c < C.count; ++c) {
        const Fr *const *cols = L.cols + (size_t)c * C.stride;
        for (uint32_t pc = 0; pc < C.body_len; ++pc) expr_step(L, L.code[pc], cols, row, mask, regs, acc, acc2);
    }
    for (uint32_t pc = C.body_len; pc < L.ncode; ++pc) expr_step(L, L.code[pc], L.cols, row, mask, regs, acc, acc2);
}

// CIRCUITS: the batched kernel (expr_circuits_kernel, C != nullptr), else expr_kernel
template <int NREGS, int THREADS, bool SMEM, bool CIRCUITS>
static int32_t launch(const ExprLaunch &L, const ExprCircuits *C, uint32_t n, cudaStream_t st) {
    constexpr size_t bytes = SMEM ? (size_t)NREGS * THREADS * 32 : 0;
    static bool attr_set[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (bytes > 48 * 1024 && dev < 64 && !attr_set[dev]) {
        if (CIRCUITS) ZKB_CUDA(cudaFuncSetAttribute(expr_circuits_kernel<NREGS, THREADS, SMEM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        else ZKB_CUDA(cudaFuncSetAttribute(expr_kernel<NREGS, THREADS, SMEM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        attr_set[dev] = true;
    }
    const unsigned blocks = (n + THREADS - 1) / THREADS;
    if (CIRCUITS) expr_circuits_kernel<NREGS, THREADS, SMEM><<<blocks, THREADS, bytes, st>>>(L, *C);
    else expr_kernel<NREGS, THREADS, SMEM><<<blocks, THREADS, bytes, st>>>(L);
    return ZKB_OK;
}

template <bool CIRCUITS>
static int32_t expr_launch(zkb_ctx *ctx, const ExprLaunch &L, const ExprCircuits *C, int nregs, cudaStream_t st) {
    const uint32_t n = 1u << L.log_n;
    ProfScope ps_(ctx, PROF_EXPR, st);
    // Register file placement, measured on the k = 20 quotient (profiles/r02_expr_kernel_k20_ncu.txt, _smem_ncu.txt):
    //   local memory, 16 registers : 65 ms per coset part, 107 GB of DRAM traffic (registers and columns evict each other from L2), pipe 75 %
    //   shared memory, 16 registers: 92 ms per part,  12.6 GB of DRAM traffic (1.6x algorithmic) -- but 64 KB per 128 threads leaves 12
    //                                warps per SM and the multiplier pipe drops to 52 %
    // so programs of <= 8 registers (32 KB per block, 7 blocks per SM) run from shared memory, larger ones from local memory unless
    // ZKB_EXPR_SMEM_REGS=1 asks for the low-traffic variant; the hybrid (8 registers in shared memory, the rest local) is the next step.
    static const bool smem_regs = getenv("ZKB_EXPR_SMEM_REGS") && getenv("ZKB_EXPR_SMEM_REGS")[0] == '1';
    if (nregs <= 8) ZKB_TRY((launch<8, 128, true, CIRCUITS>(L, C, n, st)));
    else if (nregs <= 16 && smem_regs) ZKB_TRY((launch<16, 128, true, CIRCUITS>(L, C, n, st)));
    else if (nregs <= 16) ZKB_TRY((launch<16, 128, false, CIRCUITS>(L, C, n, st)));
    else ZKB_TRY((launch<64, 128, false, CIRCUITS>(L, C, n, st)));
    ctx->launches++;
    ZKB_CUDA(cudaGetLastError());
    return ZKB_OK;
}

// d_code / d_cols / d_consts / d_outs are device pointers
int32_t expr_run_device(zkb_ctx *ctx, const Instr *d_code, uint32_t ncode, int nregs, const Fr *const *d_cols, const Fr *d_consts,
                        Fr *const *d_outs, uint32_t log_n, uint32_t out_stride, uint32_t out_offset, cudaStream_t st) {
    const ExprLaunch L{d_code, ncode, d_cols, d_consts, d_outs, log_n, out_stride, out_offset};
    return expr_launch<false>(ctx, L, nullptr, nregs, st);
}
// the same program over `count` circuits: d_cols holds count slot tables of `stride` slots; code[0, body_len) runs per circuit,
// code[body_len, ncode) once at the end (expr_circuits_kernel)
int32_t expr_run_circuits_device(zkb_ctx *ctx, const Instr *d_code, uint32_t ncode, uint32_t body_len, int nregs, const Fr *const *d_cols,
                                 uint32_t count, uint32_t stride, const Fr *d_consts, Fr *const *d_outs, uint32_t log_n, uint32_t out_stride,
                                 uint32_t out_offset, cudaStream_t st) {
    const ExprLaunch L{d_code, ncode, d_cols, d_consts, d_outs, log_n, out_stride, out_offset};
    const ExprCircuits C{count, body_len, stride};
    return expr_launch<true>(ctx, L, &C, nregs, st);
}

}  // namespace zkb
