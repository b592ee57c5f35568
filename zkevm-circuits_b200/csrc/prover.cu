// prover.cu -- device-resident create_proof: host orchestration (C++) over the CUDA kernels.
//
// Mirrors halo2_proofs 1.1.0 (scroll-tech/halo2 v1.1 @ e5ddf67) plonk/prover.rs `create_proof` for
// KZGCommitmentScheme<Bn256> + ProverSHPLONK + Blake2bWrite/Challenge255, the instantiation the reference uses at
// circuit-benchmarks/src/super_circuit.rs:117-132 and circuit-benchmarks/src/packed_multi_keccak.rs:72-87:
//   transcript order, mv-lookup (logUp) argument (plonk/mv_lookup/prover.rs), permutation argument
//   (plonk/permutation/prover.rs), vanishing argument (plonk/vanishing/prover.rs), quotient numerator term order
//   (plonk/evaluation.rs evaluate_h), evaluation order and SHPLONK multi-open (poly/kzg/multiopen/shplonk/prover.rs).
// The proof layout / evaluation order / constraint formulas are the ones visible in the reference fixture
// aggregator/data/batch-task.json (see tests/golden and SURVEY.md appendix B).
//
// What crosses the boundary (include/zkb200.h, `zkb_pk_*`, `zkb_prove_*`): the constraint system as a flat "CSF" blob,
// fixed / sigma column values, the SRS, per-phase advice columns (already blinded by the caller), blinding scalars and
// vk.transcript_repr (Rust-specific derivations, SURVEY.md hard part 1).  Everything else stays in HBM: columns,
// polynomials, coset evaluations, the quotient; only 64-byte commitments and 32-byte evaluations return to the host.
//
// B200 design points (not upstream's): the quotient is evaluated coset-part by coset-part (extended domain = E cosets of
// size n, SURVEY 8e) by ONE fused interpreter kernel per part; all scans / inversions / evaluations are parallel kernels.
#include "common.cuh"
#include "expr.cuh"
#include "blake2b.h"
#include "poseidon.h"
#include "keccak.h"
#include <algorithm>
#include <memory>
#include <string.h>
#include <stdlib.h>
#include <time.h>

namespace zkb {

int32_t expr_run_device(zkb_ctx *ctx, const Instr *d_code, uint32_t ncode, int nregs, const Fr *const *d_cols, const Fr *d_consts,
                        Fr *const *d_outs, uint32_t log_n, uint32_t out_stride, uint32_t out_offset, cudaStream_t st);
int32_t expr_run_circuits_device(zkb_ctx *ctx, const Instr *d_code, uint32_t ncode, uint32_t body_len, int nregs, const Fr *const *d_cols,
                                 uint32_t count, uint32_t stride, const Fr *d_consts, Fr *const *d_outs, uint32_t log_n, uint32_t out_stride,
                                 uint32_t out_offset, cudaStream_t st);

// ---------------------------------------------------------------------------------------------------------- CSF
enum { N_CONST = 0, N_FIXED = 1, N_ADVICE = 2, N_INSTANCE = 3, N_CHALLENGE = 4, N_NEG = 5, N_ADD = 6, N_MUL = 7, N_SCALED = 8 };
constexpr uint32_t CSF_MAGIC = 0x3146535au;

struct CsfLookup {
    std::vector<std::vector<uint32_t>> inputs;
    std::vector<uint32_t> table;
};
struct Csf {
    uint32_t k = 0, nf = 0, na = 0, ni = 0, nch = 0, bf = 0, d = 0, nphases = 0;
    std::vector<uint32_t> adv_phase, ch_phase;
    std::vector<std::array<uint32_t, 3>> nodes;
    std::vector<Fr> consts;
    std::vector<uint32_t> gates;
    std::vector<CsfLookup> lookups;
    std::vector<std::array<uint32_t, 2>> perm;
    std::vector<std::array<int32_t, 2>> advq, fixq, instq;
};

static bool parse_csf(const uint32_t *w, uint64_t nw, Csf &c) {
    if (nw < 18 || w[0] != CSF_MAGIC) { set_error("CSF: bad magic / too short"); return false; }
    c.k = w[1]; c.nf = w[2]; c.na = w[3]; c.ni = w[4]; c.nch = w[5]; c.bf = w[6]; c.d = w[7]; c.nphases = w[8];
    const uint32_t n_nodes = w[9], n_consts = w[10], n_gates = w[11], n_lookups = w[12], n_perm = w[13], n_aq = w[14], n_fq = w[15], n_iq = w[16];
    uint64_t p = 18;
    auto need = [&](uint64_t cnt) { return p + cnt <= nw; };
    if (!need(c.na + c.nch)) { set_error("CSF: truncated"); return false; }
    c.adv_phase.assign(w + p, w + p + c.na); p += c.na;
    c.ch_phase.assign(w + p, w + p + c.nch); p += c.nch;
    if (!need(3ull * n_nodes)) { set_error("CSF: truncated nodes"); return false; }
    c.nodes.resize(n_nodes);
    for (uint32_t i = 0; i < n_nodes; ++i) { c.nodes[i] = {w[p], w[p + 1], w[p + 2]}; p += 3; }
    if (!need(8ull * n_consts)) { set_error("CSF: truncated consts"); return false; }
    c.consts.resize(n_consts);
    for (uint32_t i = 0; i < n_consts; ++i) { memcpy(c.consts[i].l, w + p, 32); p += 8; }
    if (!need(n_gates)) { set_error("CSF: truncated gates"); return false; }
    c.gates.assign(w + p, w + p + n_gates); p += n_gates;
    c.lookups.resize(n_lookups);
    for (uint32_t l = 0; l < n_lookups; ++l) {
        if (!need(2)) { set_error("CSF: truncated lookups"); return false; }
        const uint32_t nsets = w[p], width = w[p + 1];
        p += 2;
        if (nsets == 0 || width == 0 || nsets > 4096 || width > 4096) { set_error("CSF: lookup %u has an implausible shape (%u input sets x %u)", l, nsets, width); return false; }
        if (!need(((uint64_t)nsets + 1) * (uint64_t)width)) { set_error("CSF: truncated lookup body"); return false; }
        c.lookups[l].inputs.resize(nsets);
        for (uint32_t s = 0; s < nsets; ++s) { c.lookups[l].inputs[s].assign(w + p, w + p + width); p += width; }
        c.lookups[l].table.assign(w + p, w + p + width); p += width;
    }
    if (!need(2ull * (n_perm + n_aq + n_fq + n_iq))) { set_error("CSF: truncated tail"); return false; }
    c.perm.resize(n_perm);
    for (uint32_t i = 0; i < n_perm; ++i) { c.perm[i] = {w[p], w[p + 1]}; p += 2; }
    auto rdq = [&](std::vector<std::array<int32_t, 2>> &q, uint32_t cnt) {
        q.resize(cnt);
        for (uint32_t i = 0; i < cnt; ++i) { q[i] = {(int32_t)w[p], (int32_t)w[p + 1]}; p += 2; }
    };
    rdq(c.advq, n_aq); rdq(c.fixq, n_fq); rdq(c.instq, n_iq);
    for (auto &nd : c.nodes) {
        if (nd[0] > N_SCALED) { set_error("CSF: bad node op"); return false; }
    }
    if (c.k < 1 || c.k > 26 || c.d < 3 || c.bf < 5) { set_error("CSF: bad k / degree / blinding factors"); return false; }
    return true;
}

// ---------------------------------------------------------------------------------------------------------- small kernels
__global__ void set_one_kernel(Fr *a, uint64_t idx) { fp_store(a + idx, Fr::one()); }
__global__ void fill_range_one_kernel(Fr *a, uint64_t from, uint64_t to) {
    uint64_t i = from + blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i < to) fp_store(a + i, Fr::one());
}
__global__ void mul_arrays_kernel(const Fr *__restrict__ a, const Fr *__restrict__ b, Fr *__restrict__ out, uint64_t n) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i < n) fp_store(out + i, fp_mul(fp_load(a + i), fp_load(b + i)));
}
// a[i] *= c
__global__ void scale_const_kernel(Fr *__restrict__ a, Fr c, uint64_t n) {
    uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i < n) fp_store(a + i, fp_mul(fp_load(a + i), c));
}
// out[i] -= low[i] for i < k (subtract a low-degree polynomial given on the device)
__global__ void sub_low_kernel(Fr *__restrict__ out, const Fr *__restrict__ low, uint32_t k) {
    uint32_t i = threadIdx.x;   // one block of 256 threads: a rotation set has at most 256 points
    if (i < k) fp_store(out + i, fp_sub(fp_load(out + i), fp_load(low + i)));
}

// out[j + E * i] = parts[j * n + i]  (coset parts gathered as rows -> extended-domain order)
__global__ void interleave_parts_kernel(const Fr *__restrict__ parts, Fr *__restrict__ out, uint32_t log_n, uint32_t E) {
    const uint64_t idx = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (idx >= ((uint64_t)E << log_n)) return;
    const uint64_t j = idx % E, i = idx / E;
    fp_store(out + idx, fp_load(parts + (j << log_n) + i));
}

// ---- multiplicities of the mv-lookup: open-addressing hash table keyed by the 32-byte compressed table value --------
__device__ __forceinline__ uint32_t key_hash(const Fr &k) {
    uint32_t h = 0x9e3779b9u;
#pragma unroll
    for (int i = 0; i < 8; ++i) { h ^= k.l[i]; h *= 0x85ebca6bu; h ^= h >> 13; }
    return h;
}
__global__ void m_insert_kernel(const Fr *__restrict__ t, uint32_t usable, uint32_t *slots, uint32_t mask) {
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= usable) return;
    const uint32_t i = usable - 1 - tid;  // descending row order: the winning (last) duplicate tends to arrive first
    const Fr key = fp_load(t + i);
    uint32_t h = key_hash(key) & mask;
    while (true) {
        const uint32_t s = atomicCAS(&slots[h], 0u, i + 1);
        if (s == 0) return;
        if (fp_load(t + (s - 1)) == key) {   // BTreeMap collect(): the last duplicate table row wins
            if (s < i + 1) atomicMax(&slots[h], i + 1);
            return;
        }
        h = (h + 1) & mask;
    }
}
__global__ void m_count_kernel(const Fr *__restrict__ f, const Fr *__restrict__ t, uint32_t usable, const uint32_t *__restrict__ slots,
                               uint32_t mask, uint32_t *counts, int *err) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t target = 0xffffffffu;
    if (i < usable) {
        const Fr key = fp_load(f + i);
        uint32_t h = key_hash(key) & mask;
        while (true) {
            const uint32_t s = slots[h];
            if (s == 0) { atomicExch(err, 1); break; }  // input not in table: unsatisfied lookup
            if (fp_load(t + (s - 1)) == key) { target = s - 1; break; }
            h = (h + 1) & mask;
        }
    }
    // most rows of a zkEVM lookup hit the same few table rows (selector off -> the all-zero row): aggregate per warp
    const uint32_t peers = __match_any_sync(0xffffffffu, target);
    if (target != 0xffffffffu && (threadIdx.x & 31) == (uint32_t)(__ffs(peers) - 1)) atomicAdd(&counts[target], (uint32_t)__popc(peers));
}
__global__ void counts_to_fr_kernel(const uint32_t *__restrict__ counts, uint32_t n, Fr *__restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) fp_store(out + i, fp_from_u64<FrParams>(counts[i]));
}

// ---------------------------------------------------------------------------------------------------------- helpers
static Fr fr_from_u64(uint64_t v) { return fp_from_u64<FrParams>(v); }
static bool fr_less(const Fr &a, const Fr &b) {  // halo2curves Ord: canonical integer comparison
    Fr x = fp_to_canonical(a), y = fp_to_canonical(b);
    for (int i = 7; i >= 0; --i) {
        if (x.l[i] != y.l[i]) return x.l[i] < y.l[i];
    }
    return false;
}
static Fr fr_pow_i64(const Fr &base, const Fr &base_inv, int64_t e) { return e >= 0 ? fp_pow_u64(base, (uint64_t)e) : fp_pow_u64(base_inv, (uint64_t)(-e)); }
// DELTA = 7^(2^28), the generator of the permutation argument's column cosets (permutation/keygen.rs)
static Fr perm_delta() {
    Fr delta = fr_from_u64(7);
    for (int i = 0; i < 28; ++i) delta = fp_sqr(delta);
    return delta;
}

// ---------------------------------------------------------------------------------------------------------- transcript
// base-field coordinate (canonical limbs, < q) -> scalar-field element (x mod r), Montgomery form: snark-verifier's fe_to_fe
static Fr fq_canonical_to_fr(const Fq &c) {
    uint32_t v[8];
    for (int i = 0; i < 8; ++i) v[i] = c.l[i];
    bool ge = true;
    for (int i = 7; i >= 0; --i) {
        if (v[i] != FrParams::P(i)) { ge = v[i] > FrParams::P(i); break; }
    }
    if (ge) {  // q < 2r: one subtraction suffices
        int64_t br = 0;
        for (int i = 0; i < 8; ++i) { int64_t d = (int64_t)v[i] - FrParams::P(i) + br; v[i] = (uint32_t)d; br = d >> 32; }
    }
    Fr out;
    for (int i = 0; i < 8; ++i) out.l[i] = v[i];
    return fp_from_canonical(out);
}
// 32-byte big-endian image of a canonical field element (EvmTranscript absorbs and writes `to_repr()` reversed)
template <class F>
static void push_be32(std::vector<uint8_t> &dst, const F &canonical) {
    const uint8_t *b = (const uint8_t *)canonical.l;
    for (int i = 31; i >= 0; --i) dst.push_back(b[i]);
}
// Challenge255 of a Blake2b("Halo2-Transcript") state: absorb the 0x00 prefix, then Fr::from_uniform_bytes of the 64-byte
// digest, (lo + hi * 2^256) mod r, computed with Montgomery multiplications by R^2
static Fr blake2b_challenge(Blake2b &h) {
    const uint8_t pre = 0;
    h.update(&pre, 1);
    uint8_t d[64];
    h.finalize_copy(d);
    Fr lo, hi;
    memcpy(lo.l, d, 32);
    memcpy(hi.l, d + 32, 32);
    const Fr r2 = Fr::r2();
    return fp_add(fp_mul(lo, r2), fp_mul(fp_mul(hi, r2), r2));
}

// The transcript of one proof.  The kind values are those of the C ABI (zkb_prove_begin_ex, zkb_transcript_script_host).
enum TranscriptKind : int32_t {
    TR_BLAKE2B = 0,    // Blake2bWrite<_, G1Affine, Challenge255<_>> (benches)
    TR_POSEIDON = 1,   // snark-verifier-sdk PoseidonTranscript (gen_snark_shplonk)
    TR_EVM = 2,        // snark-verifier EvmTranscript over Keccak-256 (gen_evm_proof_shplonk)
    TR_CALLER = 3,     // the caller's transcript through zkb_transcript_vtable (create_proof's generic `T: TranscriptWrite`: the
                       // shim forwards the four operations to the Rust object it was handed)
};
struct Transcript {
    TranscriptKind kind = TR_BLAKE2B;
    zkb_transcript_vtable vt{};
    int32_t cb_error = 0;   // first non-zero return of a caller callback (checked after every stage)
    Blake2b blake{"Halo2-Transcript"};
    PoseidonSponge pos;
    std::vector<uint8_t> evm_buf;
    std::vector<uint8_t> proof;

    void callback(int32_t r) {
        if (r && !cb_error) cb_error = r;
    }
    // ZKB_ERR_STATE once a caller callback has failed
    int32_t status() const {
        if (!cb_error) return ZKB_OK;
        set_error("the caller's transcript callback failed (%d)", cb_error);
        return ZKB_ERR_STATE;
    }
    void common_scalar(const Fr &v) {
        if (kind == TR_CALLER) { callback(vt.common_scalar(vt.user, (const uint64_t *)v.l)); return; }
        if (kind == TR_POSEIDON) { pos.update(v); return; }
        if (kind == TR_EVM) { push_be32(evm_buf, fp_to_canonical(v)); return; }
        const uint8_t pre = 2;
        Fr c = fp_to_canonical(v);
        blake.update(&pre, 1);
        blake.update(c.l, 32);
    }
    void write_scalar(const Fr &v) {
        if (kind == TR_CALLER) { callback(vt.write_scalar(vt.user, (const uint64_t *)v.l)); return; }
        common_scalar(v);
        Fr c = fp_to_canonical(v);
        if (kind == TR_EVM) { push_be32(proof, c); return; }
        const uint8_t *b = (const uint8_t *)c.l;
        proof.insert(proof.end(), b, b + 32);
    }
    int32_t write_point(const G1Affine &p) {
        if (p.is_identity()) { set_error("cannot write points at infinity to the transcript"); return ZKB_ERR_STATE; }
        if (kind == TR_CALLER) {
            const int32_t r = vt.write_point(vt.user, (const uint64_t *)&p);
            if (r) { set_error("the caller's transcript refused a point (callback returned %d)", r); callback(r); return ZKB_ERR_STATE; }
            return ZKB_OK;
        }
        Fq x = fp_to_canonical(p.x), y = fp_to_canonical(p.y);
        if (kind == TR_EVM) {  // absorbed and written uncompressed: x || y, big-endian
            push_be32(evm_buf, x); push_be32(evm_buf, y);
            push_be32(proof, x); push_be32(proof, y);
            return ZKB_OK;
        }
        if (kind == TR_POSEIDON) {
            pos.update(fq_canonical_to_fr(x));
            pos.update(fq_canonical_to_fr(y));
        } else {
            const uint8_t pre = 1;
            blake.update(&pre, 1);
            blake.update(x.l, 32);
            blake.update(y.l, 32);
        }
        uint8_t comp[32];
        g1_compress(p, comp);
        proof.insert(proof.end(), comp, comp + 32);
        return ZKB_OK;
    }
    Fr squeeze() {
        if (kind == TR_CALLER) {
            Fr c = Fr::zero();
            callback(vt.squeeze_challenge(vt.user, (uint64_t *)c.l));
            return c;
        }
        if (kind == TR_POSEIDON) return pos.squeeze();
        if (kind == TR_EVM) {
            // hash the buffer (plus a 0x01 byte when it holds just the previous digest), keep the digest as the new buffer,
            // challenge = digest as a big-endian integer mod r
            if (evm_buf.size() == 32) evm_buf.push_back(1);
            uint8_t h[32];
            keccak256(evm_buf.data(), evm_buf.size(), h);
            evm_buf.assign(h, h + 32);
            Fr v;
            uint8_t *b = (uint8_t *)v.l;
            for (int i = 0; i < 32; ++i) b[i] = h[31 - i];
            return fp_mul(v, Fr::r2());  // Montgomery multiply reduces any 256-bit value: v * R^2 / R = v R mod r
        }
        return blake2b_challenge(blake);
    }
};

}  // namespace zkb
using namespace zkb;

struct zkb_pk {
    zkb_ctx *ctx = nullptr;
    Csf cs;
    uint32_t k = 0, ext_k = 0, E = 0, qdeg = 0, chunk = 0, nsets = 0;
    uint64_t n = 0, N = 0;
    Fr omega, omega_inv, ext_omega, ext_omega_inv, n_inv, N_inv, zeta;
    std::vector<Fr> t_inv;
    DevPool pool;
    std::vector<Fr *> fixed_values, fixed_polys, sigma_values, sigma_polys;
    Fr *l0_poly = nullptr, *llast_poly = nullptr, *lblind_poly = nullptr, *xid_poly = nullptr, *omega_pows = nullptr;
    zkb_srs *srs = nullptr;       // shared ParamsKZG handle (owned when the pk was made by the legacy zkb_pk_create)
    bool owns_srs = false;
    // coset evaluations of the proof-independent polynomials (fixed, sigma, l_0, l_last, l_blind, X) for every coset part,
    // like upstream's pk.fixed_cosets / permutation cosets / l0 / l_last / l_active_row: [part][poly] -> n elements
    std::vector<std::vector<Fr *>> coset_cache;
    ~zkb_pk() {
        if (owns_srs && srs) zkb_srs_destroy(srs);
    }
};

// One proof of `nc` circuits of the same constraint system (create_proof's `circuits: &[C]`).  Per-circuit columns are
// circuit-major: circuit c's instance column i is inst_values[c * ni + i], its advice column j is adv_values[c * na + j].
struct zkb_session {
    zkb_pk *pk = nullptr;
    uint32_t nc = 1;
    Transcript tr;
    DevPool pool;
    std::vector<Fr *> inst_values, inst_polys, adv_values;
    // columns handed over ahead of their phase (zkb_prove_upload_advice), keyed by c * na + column: staged device copies, consumed
    // by zkb_prove_advice_phase
    std::map<uint32_t, Fr *> early_cols;
    std::vector<Fr> challenges;
    uint32_t next_phase = 0;
    bool finished = false;
};

namespace zkb {

// ---------------------------------------------------------------------------------------------------------- basis changes
static int32_t lagrange_to_coeff(zkb_pk *pk, const Fr *values, Fr *poly, cudaStream_t st) {
    return ntt_fr_device(pk->ctx, values, poly, pk->k, pk->omega_inv, &pk->n_inv, 0, nullptr, st);
}
// generator of coset part j of the extended domain: zeta * omega_ext^j
static Fr coset_gen(const zkb_pk *pk, uint32_t j) { return fp_mul(pk->zeta, fp_pow_u64(pk->ext_omega, j)); }

// multi-GPU dealing of independent units (columns, lookup arguments, coset parts): the `count` units are cut into P contiguous
// blocks of blk = ceil(count / P), rank r computes block r.  Results live in a slab of P * blk unit slots (the tail of the last
// blocks is padding), so ONE in-place ncclAllGather (every rank contributes its own block, 1/P of the slab) completes it -- no
// zero filling, no arithmetic on the wire (round 1 used an all-reduce over a zero-initialised slab: P times the bytes).
struct Deal {
    size_t count = 0, blk = 0;
    int P = 1, rank = 0;
    bool on = false;
    Deal(const zkb_ctx *c, size_t n) : count(n), P(c->nranks), rank(c->rank) {
        on = P > 1 && n >= 2;
        blk = on ? (n + P - 1) / P : n;
    }
    bool mine(size_t i) const { return !on || (int)(i / blk) == rank; }
    size_t padded() const { return on ? (size_t)P * blk : count; }
    size_t first() const { return on ? (size_t)rank * blk : 0; }   // index of this rank's first unit
};
static int32_t deal_gather(zkb_ctx *ctx, const Deal &d, void *slab, size_t unit_bytes, cudaStream_t st) {
    if (!d.on) return ZKB_OK;
    return comm_allgather(ctx, (const uint8_t *)slab + d.first() * unit_bytes, slab, d.blk * unit_bytes, st);
}
// the same for a slab of small values on the host (padded() units of unit_bytes; synchronises)
static int32_t deal_gather_host(zkb_ctx *ctx, const Deal &d, void *slab, size_t unit_bytes, cudaStream_t st) {
    if (!d.on) return ZKB_OK;
    return comm_allgather_host(ctx, slab, d.blk * unit_bytes, st);
}

enum { BASIS_G = 0, BASIS_LAGRANGE = 1 };   // the bases of srs_commit_many
// commit several columns of n scalars against one basis of the SRS with batched MSMs.  With a communicator the columns
// are dealt in contiguous blocks (Deal) and the 64-byte results are all-gathered; a single commitment (random polynomial, SHPLONK's
// h and the final quotient) cannot be dealt: it is sharded by point range instead (SURVEY 8e).
static int32_t commit_many(zkb_pk *pk, int basis, const std::vector<Fr *> &cols, std::vector<G1Affine> &out, cudaStream_t st) {
    zkb_ctx *ctx = pk->ctx;
    const uint64_t n = pk->n;
    if (ctx->nranks > 1 && cols.size() == 1 && n >= (1u << 14)) {
        const uint64_t P = (uint64_t)ctx->nranks, lo = n * (uint64_t)ctx->rank / P, hi = n * ((uint64_t)ctx->rank + 1) / P;
        const G1Affine *bases = basis == BASIS_G ? pk->srs->g : pk->srs->g_lagrange;
        out.resize(1);
        return msm_g1_sharded(ctx, cols[0] + lo, bases + lo, hi - lo, out.data(), st);
    }
    const Deal d(ctx, cols.size());
    std::vector<const Fr *> mine;
    for (size_t i = 0; i < cols.size(); ++i)
        if (d.mine(i)) mine.push_back(cols[i]);
    out.resize(d.padded());
    if (!mine.empty()) ZKB_TRY(srs_commit_many(pk->srs, basis, mine.data(), (uint32_t)mine.size(), n, out.data() + d.first(), st));
    ZKB_TRY(deal_gather_host(ctx, d, out.data(), sizeof(G1Affine), st));
    out.resize(cols.size());
    return ZKB_OK;
}
// commit_many, then write every commitment to the session's transcript
static int32_t commit_write(zkb_session *s, int basis, const std::vector<Fr *> &cols, cudaStream_t st) {
    std::vector<G1Affine> cms;
    ZKB_TRY(commit_many(s->pk, basis, cols, cms, st));
    for (auto &cm : cms) ZKB_TRY(s->tr.write_point(cm));
    return ZKB_OK;
}

// program bundle uploaded to the device
struct DeviceProgram {
    Instr *code = nullptr;
    uint32_t ncode = 0;
    int nregs = 0;
    Fr *consts = nullptr;
};
static int32_t upload_program(DevPool &pool, const ProgramBuilder &pb, const ExprBuilder &eb, DeviceProgram &dp, cudaStream_t st) {
    dp.ncode = (uint32_t)pb.code.size();
    dp.nregs = pb.max_regs_used;
    ZKB_TRY(pool.alloc(pb.code.size() * sizeof(Instr) + 8, (void **)&dp.code));
    ZKB_TRY(pool.alloc(eb.consts.size() * sizeof(Fr) + 32, (void **)&dp.consts));
    ZKB_CUDA(cudaMemcpyAsync(dp.code, pb.code.data(), pb.code.size() * sizeof(Instr), cudaMemcpyHostToDevice, st));
    ZKB_CUDA(cudaMemcpyAsync(dp.consts, eb.consts.data(), eb.consts.size() * sizeof(Fr), cudaMemcpyHostToDevice, st));
    ZKB_CUDA(cudaStreamSynchronize(st));  // host vectors may die after return
    return ZKB_OK;
}
template <class T>
static int32_t upload_table(DevPool &pool, const std::vector<T *> &host, T ***dev, cudaStream_t st) {
    ZKB_TRY(pool.alloc(host.size() * sizeof(T *) + 8, (void **)dev));
    ZKB_CUDA(cudaMemcpyAsync(*dev, host.data(), host.size() * sizeof(T *), cudaMemcpyHostToDevice, st));
    ZKB_CUDA(cudaStreamSynchronize(st));
    return ZKB_OK;
}

// translate CSF nodes into ExprBuilder nodes; column slot numbering is supplied by the caller
struct SlotMap { uint32_t fixed0, advice0, instance0; };
static uint32_t translate(const Csf &cs, uint32_t node, ExprBuilder &eb, const SlotMap &sm, const std::vector<Fr> &challenges, std::vector<int64_t> &memo) {
    if (memo[node] >= 0) return (uint32_t)memo[node];
    const auto &nd = cs.nodes[node];
    uint32_t r = 0;
    switch (nd[0]) {
    case N_CONST: r = eb.constant(cs.consts[nd[1]]); break;
    case N_FIXED: r = eb.col(sm.fixed0 + nd[1], (int32_t)nd[2]); break;
    case N_ADVICE: r = eb.col(sm.advice0 + nd[1], (int32_t)nd[2]); break;
    case N_INSTANCE: r = eb.col(sm.instance0 + nd[1], (int32_t)nd[2]); break;
    case N_CHALLENGE: r = eb.constant(challenges[nd[1]]); break;
    case N_NEG: r = eb.neg(translate(cs, nd[1], eb, sm, challenges, memo)); break;
    case N_ADD: { uint32_t a = translate(cs, nd[1], eb, sm, challenges, memo), b = translate(cs, nd[2], eb, sm, challenges, memo); r = eb.add(a, b); } break;
    case N_MUL: { uint32_t a = translate(cs, nd[1], eb, sm, challenges, memo), b = translate(cs, nd[2], eb, sm, challenges, memo); r = eb.mul(a, b); } break;
    case N_SCALED: { uint32_t a = translate(cs, nd[1], eb, sm, challenges, memo); r = eb.mul(a, eb.constant(cs.consts[nd[2]])); } break;
    }
    memo[node] = r;
    return r;
}
// compressed = fold(exprs, acc * theta + e), first term taken as is (0 * theta + e0 == e0)
static uint32_t compress_exprs(const Csf &cs, const std::vector<uint32_t> &exprs, ExprBuilder &eb, const SlotMap &sm, const std::vector<Fr> &ch,
                               std::vector<int64_t> &memo, const Fr &theta) {
    uint32_t acc = translate(cs, exprs[0], eb, sm, ch, memo);
    for (size_t i = 1; i < exprs.size(); ++i) acc = eb.add(eb.mul(acc, eb.constant(theta)), translate(cs, exprs[i], eb, sm, ch, memo));
    return acc;
}
// slot of a permutation column (kind, index) in a table numbered by `sm`
static uint32_t perm_slot(const SlotMap &sm, const std::array<uint32_t, 2> &c) {
    return c[0] == N_FIXED ? sm.fixed0 + c[1] : c[0] == N_ADVICE ? sm.advice0 + c[1] : sm.instance0 + c[1];
}

// upload an interpreter program and its output table, run it over the n rows of the columns in d_cols
static int32_t run_program(zkb_session *s, const ProgramBuilder &pb, const ExprBuilder &eb, Fr *const *d_cols, const std::vector<Fr *> &outs, cudaStream_t st) {
    DeviceProgram dp;
    ZKB_TRY(upload_program(s->pool, pb, eb, dp, st));
    Fr **d_outs = nullptr;
    ZKB_TRY(upload_table(s->pool, outs, &d_outs, st));
    return expr_run_device(s->pk->ctx, dp.code, dp.ncode, dp.nregs, d_cols, dp.consts, d_outs, s->pk->k, 1, 0, st);
}
// out (+)= sum_i coefs[i] polys[i] over n coefficients.  Does not synchronise: `coefs` must stay alive until the stream is.
static int32_t lincomb(zkb_session *s, const std::vector<Fr *> &polys, const std::vector<Fr> &coefs, Fr *out, bool accumulate, cudaStream_t st) {
    Fr **d_p = nullptr;
    Fr *d_c = nullptr;
    ZKB_TRY(upload_table(s->pool, polys, &d_p, st));
    ZKB_TRY(s->pool.fr(coefs.size(), &d_c));
    ZKB_CUDA(cudaMemcpyAsync(d_c, coefs.data(), coefs.size() * sizeof(Fr), cudaMemcpyHostToDevice, st));
    return lincomb_device(s->pk->ctx, d_p, d_c, (uint32_t)polys.size(), s->pk->n, out, accumulate, st);
}

}  // namespace zkb

// ================================================================================================ C ABI: proving key
// Builds the device-resident proving key.  sigma columns come either from the host (sigma_values) or are already on the
// device (sigma_dev, keygen path).  The SRS handle is shared, not copied.
static int32_t pk_build(zkb_ctx *ctx, const uint32_t *csf, uint64_t csf_words, const uint64_t *const *fixed_values, const uint64_t *const *sigma_values,
                        const std::vector<Fr *> *sigma_dev, zkb_srs *srs, bool owns_srs, zkb_pk **out) {
    ZKB_ARG(ctx && csf && srs && out);
    ZKB_CUDA(cudaSetDevice(ctx->device));
    std::unique_ptr<zkb_pk> pk(new zkb_pk());
    pk->ctx = ctx;
    pk->pool.ctx = ctx;
    pk->srs = srs;
    pk->owns_srs = owns_srs;
    ZKB_TRY(zkb_csf_validate(csf, csf_words));
    if (!parse_csf(csf, csf_words, pk->cs)) return ZKB_ERR_ARG;
    const Csf &cs = pk->cs;
    ZKB_ARG((cs.nf == 0 || fixed_values) && (cs.perm.empty() || sigma_values || sigma_dev));
    if (srs->ctx != ctx || srs->k != cs.k) { set_error("the SRS handle is for k = %u on another context or size (circuit k = %u): downsize it first", srs->k, cs.k); return ZKB_ERR_ARG; }
    cudaStream_t st = ctx->stream;
    pk->k = cs.k;
    pk->n = 1ull << cs.k;
    const uint64_t n = pk->n;
    // EvaluationDomain::new(j = cs.degree(), k)
    pk->qdeg = cs.d - 1;
    pk->ext_k = cs.k;
    while ((1ull << pk->ext_k) < n * pk->qdeg) pk->ext_k++;
    ZKB_ARG(pk->ext_k <= 28);
    pk->N = 1ull << pk->ext_k;
    pk->E = (uint32_t)(pk->N / n);
    pk->chunk = cs.d - 2;
    pk->nsets = (uint32_t)((cs.perm.size() + pk->chunk - 1) / pk->chunk);
    pk->ext_omega = host_root_of_unity(pk->ext_k);
    pk->omega = pk->ext_omega;
    for (uint32_t i = cs.k; i < pk->ext_k; ++i) pk->omega = fp_sqr(pk->omega);
    pk->omega_inv = fp_inv(pk->omega);
    pk->ext_omega_inv = fp_inv(pk->ext_omega);
    pk->n_inv = fp_inv(fr_from_u64(n));
    pk->N_inv = fp_inv(fr_from_u64(pk->N));
    pk->zeta = host_zeta();
    pk->t_inv.resize(pk->E);
    for (uint32_t j = 0; j < pk->E; ++j) pk->t_inv[j] = fp_inv(fp_sub(fp_pow_u64(coset_gen(pk.get(), j), n), Fr::one()));
    // fixed / sigma columns (host or device sources): values and coefficient form
    auto ingest = [&](const void *const *src, size_t cnt, std::vector<Fr *> &vals, std::vector<Fr *> &polys) -> int32_t {
        vals.resize(cnt);
        polys.resize(cnt);
        for (size_t i = 0; i < cnt; ++i) {
            ZKB_TRY(pk->pool.fr(n, &vals[i]));
            ZKB_TRY(pk->pool.fr(n, &polys[i]));
            ZKB_CUDA(cudaMemcpyAsync(vals[i], src[i], n * sizeof(Fr), cudaMemcpyDefault, st));
            ZKB_TRY(lagrange_to_coeff(pk.get(), vals[i], polys[i], st));
        }
        return ZKB_OK;
    };
    ZKB_TRY(ingest((const void *const *)fixed_values, cs.nf, pk->fixed_values, pk->fixed_polys));
    ZKB_ARG(!sigma_dev || sigma_dev->size() == cs.perm.size());
    std::vector<const void *> sigma_src(cs.perm.size());
    for (size_t i = 0; i < cs.perm.size(); ++i) sigma_src[i] = sigma_dev ? (const void *)(*sigma_dev)[i] : (const void *)sigma_values[i];
    ZKB_TRY(ingest(sigma_src.data(), cs.perm.size(), pk->sigma_values, pk->sigma_polys));
    // l_0, l_last, l_blind (Lagrange indicator vectors -> coefficient form), X (identity polynomial), omega^i
    ZKB_TRY(pk->pool.fr(n, &pk->l0_poly));
    ZKB_TRY(pk->pool.fr(n, &pk->llast_poly));
    ZKB_TRY(pk->pool.fr(n, &pk->lblind_poly));
    ZKB_TRY(pk->pool.fr(n, &pk->xid_poly));
    ZKB_TRY(pk->pool.fr(n, &pk->omega_pows));
    ZKB_CUDA(cudaMemsetAsync(pk->l0_poly, 0, n * sizeof(Fr), st));
    ZKB_CUDA(cudaMemsetAsync(pk->llast_poly, 0, n * sizeof(Fr), st));
    ZKB_CUDA(cudaMemsetAsync(pk->lblind_poly, 0, n * sizeof(Fr), st));
    ZKB_CUDA(cudaMemsetAsync(pk->xid_poly, 0, n * sizeof(Fr), st));
    ZKB_ARG(n > cs.bf + 1);
    set_one_kernel<<<1, 1, 0, st>>>(pk->l0_poly, 0);
    set_one_kernel<<<1, 1, 0, st>>>(pk->llast_poly, n - cs.bf - 1);
    fill_range_one_kernel<<<(cs.bf + 127) / 128, 128, 0, st>>>(pk->lblind_poly, n - cs.bf, n);
    if (n > 1) set_one_kernel<<<1, 1, 0, st>>>(pk->xid_poly, 1);
    ctx->launches += 4;
    ZKB_TRY(lagrange_to_coeff(pk.get(), pk->l0_poly, pk->l0_poly, st));
    ZKB_TRY(lagrange_to_coeff(pk.get(), pk->llast_poly, pk->llast_poly, st));
    ZKB_TRY(lagrange_to_coeff(pk.get(), pk->lblind_poly, pk->lblind_poly, st));
    ZKB_TRY(fr_powers_device(ctx, pk->omega, n, pk->omega_pows, st));
    {
        // cache the coset evaluations of the static polynomials unless that would take more than ZKB_COSET_CACHE_GB (default 48)
        std::vector<Fr *> stat;
        for (auto q : pk->fixed_polys) stat.push_back(q);
        for (auto q : pk->sigma_polys) stat.push_back(q);
        stat.push_back(pk->l0_poly); stat.push_back(pk->llast_poly); stat.push_back(pk->lblind_poly); stat.push_back(pk->xid_poly);
        const char *env = getenv("ZKB_COSET_CACHE_GB");
        const double budget = (env ? atof(env) : 48.0) * 1e9;
        if ((double)stat.size() * pk->N * sizeof(Fr) <= budget) {
            Fr *pows = nullptr;
            ZKB_TRY(pk->pool.fr(n, &pows));
            pk->coset_cache.resize(pk->E);
            for (uint32_t j = 0; j < pk->E; ++j) {
                ZKB_TRY(fr_powers_device(ctx, coset_gen(pk.get(), j), n, pows, st));
                pk->coset_cache[j].resize(stat.size());
                for (size_t i = 0; i < stat.size(); ++i) {
                    ZKB_TRY(pk->pool.fr(n, &pk->coset_cache[j][i]));
                    ZKB_TRY(ntt_fr_device(ctx, stat[i], pk->coset_cache[j][i], cs.k, pk->omega, nullptr, 0, pows, st));
                }
            }
        }
    }
    ZKB_CUDA(cudaStreamSynchronize(st));
    *out = pk.release();
    return ZKB_OK;
}

extern "C" int32_t zkb_pk_create(zkb_ctx *ctx, const uint32_t *csf, uint64_t csf_words, const uint64_t *const *fixed_values,
                                 const uint64_t *const *sigma_values, const uint64_t *g, const uint64_t *g_lagrange, zkb_pk **out) {
    ZKB_ARG(ctx && csf && csf_words >= 18 && g && g_lagrange && out);
    ZKB_CUDA(cudaSetDevice(ctx->device));
    ZKB_TRY(zkb_csf_validate(csf, csf_words));
    zkb_srs *srs = nullptr;
    ZKB_TRY(srs_create(ctx, csf[1], (const G1Affine *)g, false, (const G1Affine *)g_lagrange, false, &srs));
    const int32_t r = pk_build(ctx, csf, csf_words, fixed_values, sigma_values, nullptr, srs, true, out);
    if (r != ZKB_OK) zkb_srs_destroy(srs);
    return r;
}
extern "C" int32_t zkb_pk_create_with_srs(zkb_ctx *ctx, const uint32_t *csf, uint64_t csf_words, const uint64_t *const *fixed_values,
                                          const uint64_t *const *sigma_values, zkb_srs *srs, zkb_pk **out) {
    return pk_build(ctx, csf, csf_words, fixed_values, sigma_values, nullptr, srs, false, out);
}

// ---- keygen: permutation assembly + sigma columns (plonk/permutation/keygen.rs Assembly::copy, build_pk) -------------------
// sigma_i[j] = DELTA^(mapping column) * omega^(mapping row): the cycle structure is merged on the host exactly like upstream
// (mapping / aux / sizes with union by size -- inherently sequential), the n x P field values are produced on the device.
__global__ void sigma_from_mapping_kernel(const uint32_t *__restrict__ map_col, const uint32_t *__restrict__ map_row, const Fr *__restrict__ omega_pows,
                                          const Fr *__restrict__ delta_pows, uint64_t n, Fr *__restrict__ out) {
    const uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    if (i < n) fp_store(out + i, fp_mul(fp_load(delta_pows + map_col[i]), fp_load(omega_pows + map_row[i])));
}

// copies: n_copies x 4 u32 = (left column, left row, right column, right row); columns are indices into the CSF's permutation column list
extern "C" int32_t zkb_keygen_pk(zkb_ctx *ctx, const uint32_t *csf, uint64_t csf_words, const uint64_t *const *fixed_values, const uint32_t *copies,
                                 uint64_t n_copies, zkb_srs *srs, zkb_pk **out) {
    ZKB_ARG(ctx && csf && srs && out && (copies || n_copies == 0));
    ZKB_CUDA(cudaSetDevice(ctx->device));
    ZKB_TRY(zkb_csf_validate(csf, csf_words));
    Csf cs;
    if (!parse_csf(csf, csf_words, cs)) return ZKB_ERR_ARG;
    const uint64_t n = 1ull << cs.k;
    const size_t P = cs.perm.size();
    ZKB_ARG(P * n < (1ull << 32));
    // Assembly: mapping[c][r] = next cell of the cycle, aux = cycle representative, sizes = cycle length at the representative
    std::vector<uint32_t> map_col(P * n), map_row(P * n), aux_col(P * n), aux_row(P * n), sizes(P * n, 1);
    for (size_t c = 0; c < P; ++c)
        for (uint64_t r = 0; r < n; ++r) { map_col[c * n + r] = aux_col[c * n + r] = (uint32_t)c; map_row[c * n + r] = aux_row[c * n + r] = (uint32_t)r; }
    for (uint64_t i = 0; i < n_copies; ++i) {
        const uint32_t lc = copies[4 * i], lr = copies[4 * i + 1], rc = copies[4 * i + 2], rr = copies[4 * i + 3];
        if (lc >= P || rc >= P || lr >= n || rr >= n) { set_error("copy constraint %llu is out of range", (unsigned long long)i); return ZKB_ERR_ARG; }
        const size_t a = lc * n + lr, b = rc * n + rr;
        size_t lcy = aux_col[a] * n + aux_row[a], rcy = aux_col[b] * n + aux_row[b];
        if (lcy == rcy) continue;
        if (sizes[lcy] < sizes[rcy]) std::swap(lcy, rcy);
        sizes[lcy] += sizes[rcy];
        size_t cur = rcy;
        do {   // relabel the smaller cycle
            aux_col[cur] = (uint32_t)(lcy / n);
            aux_row[cur] = (uint32_t)(lcy % n);
            cur = map_col[cur] * n + map_row[cur];
        } while (cur != rcy);
        std::swap(map_col[a], map_col[b]);
        std::swap(map_row[a], map_row[b]);
    }
    cudaStream_t st = ctx->stream;
    DevPool tmp;
    tmp.ctx = ctx;
    uint32_t *d_mc = nullptr, *d_mr = nullptr;
    Fr *d_om = nullptr, *d_dl = nullptr;
    ZKB_TRY(tmp.alloc(P * n * 4 + 4, (void **)&d_mc));
    ZKB_TRY(tmp.alloc(P * n * 4 + 4, (void **)&d_mr));
    ZKB_TRY(tmp.fr(n, &d_om));
    ZKB_TRY(tmp.fr(P + 1, &d_dl));
    ZKB_CUDA(cudaMemcpyAsync(d_mc, map_col.data(), P * n * 4, cudaMemcpyHostToDevice, st));
    ZKB_CUDA(cudaMemcpyAsync(d_mr, map_row.data(), P * n * 4, cudaMemcpyHostToDevice, st));
    Fr omega = host_root_of_unity(cs.k);
    ZKB_TRY(fr_powers_device(ctx, omega, n, d_om, st));
    ZKB_TRY(fr_powers_device(ctx, perm_delta(), P + 1, d_dl, st));
    std::vector<Fr *> sig(P);
    for (size_t c = 0; c < P; ++c) {
        ZKB_TRY(tmp.fr(n, &sig[c]));
        sigma_from_mapping_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_mc + c * n, d_mr + c * n, d_om, d_dl, n, sig[c]);
        ctx->launches++;
    }
    ZKB_CUDA(cudaGetLastError());
    ZKB_CUDA(cudaStreamSynchronize(st));   // host vectors die at return
    return pk_build(ctx, csf, csf_words, fixed_values, nullptr, &sig, srs, false, out);
}
// sigma column values of a proving key (n x 32 B each, Lagrange basis) back to the host: lets a caller persist / inspect keygen output
extern "C" int32_t zkb_pk_sigma_read(zkb_pk *pk, uint32_t column, uint64_t *out_host) {
    ZKB_ARG(pk && out_host && column < pk->sigma_values.size());
    ZKB_CUDA(cudaSetDevice(pk->ctx->device));
    ZKB_CUDA(cudaMemcpyAsync(out_host, pk->sigma_values[column], pk->n * sizeof(Fr), cudaMemcpyDeviceToHost, pk->ctx->stream));
    ZKB_CUDA(cudaStreamSynchronize(pk->ctx->stream));
    return ZKB_OK;
}

// ---- host-only transcript primitives (no device needed): let the CPU test-suite pin the two hashers of the proving session ----
// absorb n Fr elements (Montgomery) into a fresh Poseidon sponge (PoseidonTranscript::common_scalar) and squeeze one challenge
extern "C" int32_t zkb_poseidon_hash_host(const uint64_t *inputs, uint64_t n, uint64_t out[4]) {
    ZKB_ARG(out && (inputs || n == 0));
    PoseidonSponge sp;
    for (uint64_t i = 0; i < n; ++i) {
        Fr v;
        memcpy(v.l, inputs + 4 * i, 32);
        sp.update(v);
    }
    const Fr c = sp.squeeze();
    memcpy(out, c.l, 32);
    return ZKB_OK;
}
// Host-only: replay a scripted sequence of transcript operations through the session's own transcript code (no device work).
// ops[i]: 0 = common_scalar, 1 = write_scalar, 2 = write_point, 3 = squeeze_challenge; operands are consumed in order (scalar:
// 4 limbs, point: 8 limbs, Montgomery form); challenges are appended to `challenges` (4 limbs each).  Lets the CPU suite pin the
// framing of every transcript kind against the oracle's transcripts.
extern "C" int32_t zkb_transcript_script_host(int32_t kind, const uint8_t *ops, uint64_t n_ops, const uint64_t *operands, uint8_t *proof, uint64_t cap,
                                              uint64_t *proof_len, uint64_t *challenges) {
    ZKB_ARG(kind >= TR_BLAKE2B && kind <= TR_EVM && (ops || n_ops == 0) && proof_len);
    Transcript t;
    t.kind = (TranscriptKind)kind;
    const uint64_t *op = operands;
    for (uint64_t i = 0; i < n_ops; ++i) {
        switch (ops[i]) {
            case 0:
            case 1: {
                ZKB_ARG(op);
                Fr v;
                memcpy(v.l, op, 32);
                op += 4;
                if (ops[i] == 0) t.common_scalar(v); else t.write_scalar(v);
                break;
            }
            case 2: {
                ZKB_ARG(op);
                G1Affine p;
                memcpy(&p, op, 64);
                op += 8;
                ZKB_TRY(t.write_point(p));
                break;
            }
            case 3: {
                ZKB_ARG(challenges);
                const Fr c = t.squeeze();
                memcpy(challenges, c.l, 32);
                challenges += 4;
                break;
            }
            default: ZKB_ARG(false);
        }
    }
    *proof_len = t.proof.size();
    if (proof) {
        ZKB_ARG(cap >= t.proof.size());
        if (!t.proof.empty()) memcpy(proof, t.proof.data(), t.proof.size());
    }
    return ZKB_OK;
}
extern "C" int32_t zkb_keccak256_host(const uint8_t *bytes, uint64_t len, uint8_t out[32]) {
    ZKB_ARG(out && (bytes || len == 0));
    keccak256(bytes, len, out);
    return ZKB_OK;
}
// feed raw bytes to a fresh Blake2b("Halo2-Transcript") state and squeeze one Challenge255 (prefix 0x00, 64-byte digest mod r)
extern "C" int32_t zkb_blake2b_challenge_host(const uint8_t *bytes, uint64_t len, uint64_t out[4]) {
    ZKB_ARG(out && (bytes || len == 0));
    Blake2b st("Halo2-Transcript");
    if (len) st.update(bytes, len);
    const Fr c = blake2b_challenge(st);
    memcpy(out, c.l, 32);
    return ZKB_OK;
}

// VerifyingKey::write(SerdeFormat::Processed) (halo2_proofs plonk.rs): u32 BE k || u32 BE num_fixed || fixed commitments ||
// permutation commitments, points compressed -- the layout of the reference fixture's `vk` (aggregator/data/batch-task.json:
// 0x19, 4, 4 + 3 points = 232 B).  Commitments = commit_lagrange of the fixed / sigma columns (keygen.rs), batched MSMs.
extern "C" int32_t zkb_pk_vk_bytes(zkb_pk *pk, uint8_t *out, uint64_t cap, uint64_t *len) {
    ZKB_ARG(pk && len);
    const Csf &cs = pk->cs;
    const uint64_t need = 8 + 32ull * (cs.nf + cs.perm.size());
    *len = need;
    if (!out) return ZKB_OK;
    ZKB_ARG(cap >= need);
    ZKB_CUDA(cudaSetDevice(pk->ctx->device));
    cudaStream_t st = pk->ctx->stream;
    std::vector<Fr *> cols;
    for (auto c : pk->fixed_values) cols.push_back(c);
    for (auto c : pk->sigma_values) cols.push_back(c);
    std::vector<G1Affine> cms;
    if (!cols.empty()) ZKB_TRY(commit_many(pk, BASIS_LAGRANGE, cols, cms, st));
    auto be32 = [](uint8_t *p, uint32_t v) { p[0] = (uint8_t)(v >> 24); p[1] = (uint8_t)(v >> 16); p[2] = (uint8_t)(v >> 8); p[3] = (uint8_t)v; };
    be32(out, cs.k);
    be32(out + 4, cs.nf);
    for (size_t i = 0; i < cms.size(); ++i) g1_compress(cms[i], out + 8 + 32 * i);
    return ZKB_OK;
}

// host-only structural check of a CSF blob (no device needed)
extern "C" int32_t zkb_csf_validate(const uint32_t *csf, uint64_t csf_words) {
    ZKB_ARG(csf != nullptr);
    Csf c;
    if (!parse_csf(csf, csf_words, c)) return ZKB_ERR_ARG;
    // node references must point backwards; column / challenge / constant indices must be in range
    for (size_t i = 0; i < c.nodes.size(); ++i) {
        const auto &nd = c.nodes[i];
        bool ok = true;
        switch (nd[0]) {
        case N_CONST: ok = nd[1] < c.consts.size(); break;
        case N_FIXED: ok = nd[1] < c.nf; break;
        case N_ADVICE: ok = nd[1] < c.na; break;
        case N_INSTANCE: ok = nd[1] < c.ni; break;
        case N_CHALLENGE: ok = nd[1] < c.nch; break;
        case N_NEG: ok = nd[1] < i; break;
        case N_ADD: case N_MUL: ok = nd[1] < i && nd[2] < i; break;
        case N_SCALED: ok = nd[1] < i && nd[2] < c.consts.size(); break;
        }
        if (!ok) { set_error("CSF: node %zu has an out-of-range operand", i); return ZKB_ERR_ARG; }
    }
    auto in_nodes = [&](uint32_t v) { return v < c.nodes.size(); };
    for (auto g : c.gates) if (!in_nodes(g)) { set_error("CSF: gate references a missing node"); return ZKB_ERR_ARG; }
    for (auto &lk : c.lookups) {
        if (lk.inputs.empty() || lk.table.empty()) { set_error("CSF: empty lookup"); return ZKB_ERR_ARG; }
        for (auto &inp : lk.inputs) for (auto v : inp) if (!in_nodes(v)) { set_error("CSF: lookup references a missing node"); return ZKB_ERR_ARG; }
        for (auto v : lk.table) if (!in_nodes(v)) { set_error("CSF: lookup references a missing node"); return ZKB_ERR_ARG; }
    }
    for (auto &pc : c.perm) {
        const uint32_t lim = pc[0] == N_FIXED ? c.nf : pc[0] == N_ADVICE ? c.na : pc[0] == N_INSTANCE ? c.ni : 0;
        if (pc[1] >= lim) { set_error("CSF: permutation column out of range"); return ZKB_ERR_ARG; }
    }
    // queries: column in range, rotation representable in the interpreter's 16-bit field (also for expression nodes)
    auto chkq = [&](const std::vector<std::array<int32_t, 2>> &q, uint32_t lim, const char *what) {
        for (auto &e : q) {
            if (e[0] < 0 || (uint32_t)e[0] >= lim) { set_error("CSF: %s query references column %d of %u", what, e[0], lim); return false; }
            if (e[1] < -32767 || e[1] > 32767) { set_error("CSF: %s query rotation %d does not fit 16 bits", what, e[1]); return false; }
        }
        return true;
    };
    if (!chkq(c.advq, c.na, "advice") || !chkq(c.fixq, c.nf, "fixed") || !chkq(c.instq, c.ni, "instance")) return ZKB_ERR_ARG;
    for (auto &nd : c.nodes) {
        if (nd[0] == N_FIXED || nd[0] == N_ADVICE || nd[0] == N_INSTANCE) {
            const int32_t rot = (int32_t)nd[2];
            if (rot < -32767 || rot > 32767) { set_error("CSF: node rotation %d does not fit 16 bits", rot); return ZKB_ERR_ARG; }
        }
    }
    if ((uint64_t)c.nf + c.na + c.ni + c.perm.size() + 1 >= 65536) { set_error("CSF: more than 65535 column slots"); return ZKB_ERR_ARG; }
    for (uint32_t ph : c.adv_phase) if (ph >= c.nphases) { set_error("CSF: advice phase out of range"); return ZKB_ERR_ARG; }
    for (uint32_t ph : c.ch_phase) if (ph >= c.nphases) { set_error("CSF: challenge phase out of range"); return ZKB_ERR_ARG; }
    return ZKB_OK;
}

extern "C" int32_t zkb_pk_destroy(zkb_pk *pk) {
    if (pk) {
        cudaSetDevice(pk->ctx->device);
        cudaStreamSynchronize(pk->ctx->stream);
        delete pk;
    }
    return ZKB_OK;
}

// ================================================================================================ C ABI: proof session
extern "C" int32_t zkb_prove_begin_ex(zkb_pk *pk, int32_t transcript_kind, const uint64_t transcript_repr[4], const uint64_t *const *instance_values,
                                      const uint32_t *instance_lens, zkb_session **out);
extern "C" int32_t zkb_prove_begin(zkb_pk *pk, const uint64_t transcript_repr[4], const uint64_t *const *instance_values, const uint32_t *instance_lens,
                                   zkb_session **out) {
    return zkb_prove_begin_ex(pk, 0, transcript_repr, instance_values, instance_lens, out);
}
static int32_t prove_begin_common(zkb_pk *pk, int32_t transcript_kind, const zkb_transcript_vtable *vt, const uint64_t transcript_repr[4],
                                  uint32_t num_circuits, const uint64_t *const *instance_values, const uint32_t *instance_lens, zkb_session **out);
extern "C" int32_t zkb_prove_begin_ex(zkb_pk *pk, int32_t transcript_kind, const uint64_t transcript_repr[4], const uint64_t *const *instance_values,
                                      const uint32_t *instance_lens, zkb_session **out) {
    ZKB_ARG(transcript_kind >= TR_BLAKE2B && transcript_kind <= TR_EVM);
    return prove_begin_common(pk, transcript_kind, nullptr, transcript_repr, 1, instance_values, instance_lens, out);
}
extern "C" int32_t zkb_prove_begin_cb(zkb_pk *pk, const zkb_transcript_vtable *vt, const uint64_t transcript_repr[4],
                                      const uint64_t *const *instance_values, const uint32_t *instance_lens, zkb_session **out) {
    ZKB_ARG(vt && vt->common_scalar && vt->write_scalar && vt->write_point && vt->squeeze_challenge);
    return prove_begin_common(pk, TR_CALLER, vt, transcript_repr, 1, instance_values, instance_lens, out);
}
extern "C" int32_t zkb_prove_begin_multi(zkb_pk *pk, int32_t transcript_kind, const zkb_transcript_vtable *vt, const uint64_t transcript_repr[4],
                                         uint32_t num_circuits, const uint64_t *const *instance_values, const uint32_t *instance_lens,
                                         zkb_session **out) {
    ZKB_ARG(transcript_kind >= TR_BLAKE2B && transcript_kind <= TR_CALLER && num_circuits >= 1);
    if (transcript_kind == TR_CALLER) ZKB_ARG(vt && vt->common_scalar && vt->write_scalar && vt->write_point && vt->squeeze_challenge);
    else ZKB_ARG(vt == nullptr);
    return prove_begin_common(pk, transcript_kind, vt, transcript_repr, num_circuits, instance_values, instance_lens, out);
}
static int32_t prove_begin_common(zkb_pk *pk, int32_t transcript_kind, const zkb_transcript_vtable *vt, const uint64_t transcript_repr[4],
                                  uint32_t num_circuits, const uint64_t *const *instance_values, const uint32_t *instance_lens, zkb_session **out) {
    ZKB_ARG(pk && transcript_repr && out && (pk->cs.ni == 0 || (instance_values && instance_lens)));
    ZKB_ARG((uint64_t)num_circuits * (pk->cs.na + pk->cs.ni + pk->cs.lookups.size() + pk->nsets) < (1ull << 31));
    ZKB_CUDA(cudaSetDevice(pk->ctx->device));
    std::unique_ptr<zkb_session> s(new zkb_session());
    s->pk = pk;
    s->nc = num_circuits;
    s->tr.kind = (TranscriptKind)transcript_kind;
    if (vt) s->tr.vt = *vt;
    s->pool.ctx = pk->ctx;
    const Csf &cs = pk->cs;
    const uint64_t n = pk->n;
    cudaStream_t st = pk->ctx->stream;
    Fr repr;
    memcpy(repr.l, transcript_repr, 32);
    s->tr.common_scalar(repr);  // vk.hash_into(transcript)
    // instance values circuit-major: for each circuit, for each instance column, every value
    const uint32_t ninst = num_circuits * cs.ni;
    s->inst_values.resize(ninst);
    s->inst_polys.resize(ninst);
    for (uint32_t c = 0; c < ninst; ++c) {
        ZKB_ARG(instance_lens[c] <= n - (cs.bf + 1));
        ZKB_TRY(s->pool.fr(n, &s->inst_values[c]));
        ZKB_TRY(s->pool.fr(n, &s->inst_polys[c]));
        ZKB_CUDA(cudaMemsetAsync(s->inst_values[c], 0, n * sizeof(Fr), st));
        for (uint32_t i = 0; i < instance_lens[c]; ++i) {  // KZG: QUERY_INSTANCE = false -> values are absorbed as scalars
            Fr v;
            memcpy(v.l, instance_values[c] + 4 * i, 32);
            s->tr.common_scalar(v);
        }
        if (instance_lens[c]) ZKB_CUDA(cudaMemcpyAsync(s->inst_values[c], instance_values[c], (size_t)instance_lens[c] * sizeof(Fr), cudaMemcpyHostToDevice, st));
        ZKB_TRY(lagrange_to_coeff(pk, s->inst_values[c], s->inst_polys[c], st));
    }
    s->adv_values.assign((size_t)num_circuits * cs.na, nullptr);
    s->challenges.assign(cs.nch, Fr::zero());
    ZKB_CUDA(cudaStreamSynchronize(st));
    ZKB_TRY(s->tr.status());
    *out = s.release();
    return ZKB_OK;
}

// Witness-side overlap (SURVEY 8f row 4): `synthesize` assigns sub-circuit after sub-circuit (super_circuit.rs:714-806), so the columns
// of a phase become final one at a time.  The shim may hand each finished column over immediately: the copy runs on the copy stream
// while Rust keeps synthesising, and zkb_prove_advice_phase later finds the column already in HBM (its pointer may then be NULL).
// In a session of C circuits `column` is c * num_advice + the column of circuit c.
extern "C" int32_t zkb_prove_upload_advice(zkb_session *s, uint32_t column, const uint64_t *values) {
    ZKB_ARG(s && values && (uint64_t)column < (uint64_t)s->nc * s->pk->cs.na);
    zkb_pk *pk = s->pk;
    if (s->finished || pk->cs.adv_phase[column % pk->cs.na] < s->next_phase) { set_error("column %u belongs to a phase that is already committed", column); return ZKB_ERR_STATE; }
    ZKB_CUDA(cudaSetDevice(pk->ctx->device));
    Fr *&d = s->early_cols[column];
    if (!d) ZKB_TRY(s->pool.fr(pk->n, &d));
    ZKB_CUDA(cudaMemcpyAsync(d, values, pk->n * sizeof(Fr), cudaMemcpyDefault, pk->ctx->copy_stream));
    return ZKB_OK;
}

extern "C" int32_t zkb_prove_advice_phase(zkb_session *s, uint32_t phase, const uint64_t *const *advice_columns, uint64_t *challenges_out) {
    ZKB_ARG(s && advice_columns);
    zkb_pk *pk = s->pk;
    const Csf &cs = pk->cs;
    if (phase != s->next_phase || phase >= cs.nphases || s->finished) { set_error("advice phases must be submitted in order"); return ZKB_ERR_STATE; }
    ZKB_CUDA(cudaSetDevice(pk->ctx->device));
    cudaStream_t st = pk->ctx->stream;
    const uint64_t n = pk->n;
    // H2D on the copy stream, batch by batch; the MSM of batch b waits only for batch b's event, so the copies of the
    // following batches overlap it (pinned caller buffers; pageable ones are staged synchronously by the driver anyway).
    // Multi-GPU: a rank uploads and commits only the columns it owns, then the column data is gathered over NVLink.
    // circuit-major: circuit 0's columns of this phase, then circuit 1's, ... (the order of the commitments in the transcript)
    std::vector<const uint64_t *> phase_src;
    std::vector<uint32_t> phase_idx;
    for (uint32_t c = 0; c < s->nc * cs.na; ++c) {
        if (cs.adv_phase[c % cs.na] != phase) continue;
        auto early = s->early_cols.find(c);
        const uint64_t *src = advice_columns[c] ? advice_columns[c] : (early != s->early_cols.end() ? (const uint64_t *)early->second : nullptr);
        if (!src) {
            if (s->nc == 1) set_error("advice column %u of phase %u was neither passed nor uploaded ahead", c, phase);
            else set_error("advice column %u of circuit %u (phase %u) was neither passed nor uploaded ahead", c % cs.na, c / cs.na, phase);
            return ZKB_ERR_ARG;
        }
        phase_src.push_back(src);   // a staged copy is a device pointer: the gather into the phase slab below is then device-to-device
        phase_idx.push_back(c);
    }
    const size_t ncols = phase_src.size();
    const Deal deal(pk->ctx, ncols);
    Fr *slab = nullptr;
    ZKB_TRY(s->pool.fr(std::max<size_t>(1, deal.padded()) * n, &slab));
    std::vector<Fr *> phase_cols(ncols);
    for (size_t i = 0; i < ncols; ++i) { phase_cols[i] = slab + i * n; s->adv_values[phase_idx[i]] = phase_cols[i]; }
    const bool dealt = deal.on;
    ZKB_CUDA(cudaStreamSynchronize(st));  // the destination block may still be in use by work queued on `st`
    const uint32_t maxb = msm_max_batch(n);
    const size_t nbatch = dealt ? 1 : (ncols + maxb - 1) / maxb;
    struct EventList {   // destroyed on every exit path
        std::vector<cudaEvent_t> v;
        ~EventList() { for (auto e : v) if (e) cudaEventDestroy(e); }
    } evl;
    evl.v.assign(nbatch, nullptr);
    std::vector<cudaEvent_t> &evs = evl.v;
    for (size_t b = 0; b < nbatch; ++b) {
        ZKB_CUDA(cudaEventCreateWithFlags(&evs[b], cudaEventDisableTiming));
        const size_t lo = dealt ? 0 : b * maxb, hi = dealt ? ncols : std::min(ncols, (b + 1) * (size_t)maxb);
        for (size_t i = lo; i < hi; ++i)
            if (deal.mine(i))
                ZKB_CUDA(cudaMemcpyAsync(phase_cols[i], phase_src[i], n * sizeof(Fr), cudaMemcpyDefault, pk->ctx->copy_stream));   // host (pinned or pageable) or device-resident columns
        ZKB_CUDA(cudaEventRecord(evs[b], pk->ctx->copy_stream));
    }
    for (size_t b = 0; b < nbatch; ++b) {
        ZKB_CUDA(cudaStreamWaitEvent(st, evs[b], 0));
        const size_t lo = dealt ? 0 : b * maxb, hi = dealt ? ncols : std::min(ncols, (b + 1) * (size_t)maxb);
        const std::vector<Fr *> part(phase_cols.begin() + lo, phase_cols.begin() + hi);
        ZKB_TRY(commit_write(s, BASIS_LAGRANGE, part, st));   // dealt: the same contiguous blocks as the uploads (same unit count)
    }
    ZKB_TRY(deal_gather(pk->ctx, deal, slab, n * sizeof(Fr), st));   // column data of the other ranks' blocks over NVLink
    for (uint32_t i = 0; i < cs.nch; ++i) {
        if (cs.ch_phase[i] == phase) {
            s->challenges[i] = s->tr.squeeze();
            if (challenges_out) memcpy(challenges_out + 4 * i, s->challenges[i].l, 32);
        }
    }
    s->next_phase++;
    return s->tr.status();
}

extern "C" int32_t zkb_session_destroy(zkb_session *s) {
    if (s) {
        cudaSetDevice(s->pk->ctx->device);
        cudaStreamSynchronize(s->pk->ctx->stream);
        delete s;
    }
    return ZKB_OK;
}

namespace zkb {

// stage timing (ZKB_TRACE=1): wall clock per create_proof stage after a stream synchronise, printed to stderr
struct StageTrace {
    bool on;
    cudaStream_t st;
    double t0;
    explicit StageTrace(cudaStream_t s) : st(s) {
        const char *e = getenv("ZKB_TRACE");
        on = e && e[0] == '1';
        t0 = now();
    }
    static double now() {
        timespec ts;
        clock_gettime(CLOCK_MONOTONIC, &ts);
        return ts.tv_sec + 1e-9 * ts.tv_nsec;
    }
    void mark(const char *name) {
        if (!on) return;
        cudaStreamSynchronize(st);
        const double t = now();
        fprintf(stderr, "[zkb trace] %-28s %9.3f ms\n", name, (t - t0) * 1e3);
        t0 = t;
    }
};

struct OpenQuery {
    int poly_id;        // identity of the committed polynomial
    const Fr *poly;     // device coefficients (n)
    int64_t rot;        // point = x * omega^rot
    Fr point;
    Fr eval;
};
// SHPLONK: a committed polynomial with the rotations it is opened at, and a set of polynomials opened at the same rotations
struct ShplonkCommit { int id; const Fr *poly; std::vector<int64_t> rots; };
struct RotationSet {
    std::vector<int64_t> rots;
    std::vector<const ShplonkCommit *> comms;
    std::vector<Fr> pts;                       // x * omega^rot of every rotation
    std::vector<std::vector<Fr>> r_coeffs;     // per commitment: low-degree interpolant through (pts, evaluations)
};

// What the stages of one create_proof hand to each other; lives for one call of prove_finish_impl.  With C circuits every
// per-circuit vector (lookups, permutation sets, their polynomials) is circuit-major: unit u belongs to circuit u / count.
struct ProofState {
    zkb_session *s;
    zkb_pk *pk;
    zkb_ctx *ctx;
    const Csf &cs;
    uint64_t n;
    uint32_t k, bf, nc;
    cudaStream_t st;
    DevPool &pool;
    Deal lk_deal;   // multi-GPU: the lookup arguments of all circuits are dealt, prepared and summed by the rank that owns them
    Fr theta, beta, gamma, y, x, sy, sv, su;   // sy, sv, su: SHPLONK's y, v, u
    // value-domain column tables, one per circuit (circuit c's at d_vcols + c * vstride): [fixed | advice | instance | sigma | omega_pows]
    Fr **d_vcols = nullptr;
    uint32_t vstride = 0;
    std::vector<std::vector<Fr *>> lk_f;      // compressed inputs per lookup / input set
    std::vector<Fr *> lk_t, lk_m, zs, phis;   // compressed tables, multiplicities, permutation grand products, lookup grand sums
    Fr *random_poly = nullptr;
    std::vector<Fr *> adv_polys, z_polys, phi_polys, m_polys;   // coefficient forms
    // quotient: coset-domain slot table of one circuit [fixed | advice | instance | sigma | z | phi | m | l0 | l_last | l_blind | X]
    // (q_stride slots; C circuits: C tables, the shared slots repeat); qpolys holds every distinct polynomial once, q_slot maps each
    // table entry to it; the program (common body + one trailing STOREACC slot rewritten per coset part); h on the extended
    // domain, then its d - 1 pieces
    std::vector<Fr *> qpolys;
    std::vector<uint32_t> q_slot;
    uint32_t q_sigma0 = 0, q_z0 = 0, q_phi0 = 0, q_m0 = 0, q_l0 = 0, q_stride = 0;
    DeviceProgram qdp;
    size_t q_base_len = 0;
    std::vector<uint32_t> tinv_idx;
    Fr *h_ext = nullptr;
    // openings: queries in multiopen order, the point of every rotation, the evaluation of every (polynomial, rotation)
    std::vector<OpenQuery> queries;
    std::map<int64_t, Fr> point_of;
    std::map<std::pair<int, int64_t>, Fr> eval_of;
    // SHPLONK: commitments (the sets point into this vector), rotation sets, the union of their rotations, h_x, work buffers
    std::vector<ShplonkCommit> sh_commits;
    std::vector<RotationSet> rsets;
    std::vector<int64_t> super_rots;
    Fr *hx = nullptr, *work = nullptr, *work2 = nullptr, *d_small = nullptr;

    explicit ProofState(zkb_session *sess)
        : s(sess), pk(sess->pk), ctx(pk->ctx), cs(pk->cs), n(pk->n), k(pk->cs.k), bf(pk->cs.bf), nc(sess->nc), st(pk->ctx->stream), pool(sess->pool),
          lk_deal(pk->ctx, (size_t)sess->nc * pk->cs.lookups.size()) {}
};

// mv_lookup/prover.rs::prepare: compress inputs and table with theta, multiplicities m over the usable rows, commit m
static int32_t lookups_prepare(ProofState &p) {
    zkb_session *s = p.s;
    const Csf &cs = p.cs;
    const uint64_t n = p.n;
    const uint32_t usable = (uint32_t)(n - p.bf - 1);
    const size_t nl = cs.lookups.size(), nu = p.nc * nl;   // nu: lookup arguments of all circuits
    cudaStream_t st = p.st;
    DevPool &pool = p.pool;
    const SlotMap vsm{0, cs.nf, cs.nf + cs.na};
    std::vector<Fr *> vcols;
    for (uint32_t c = 0; c < p.nc; ++c) {
        for (auto q : p.pk->fixed_values) vcols.push_back(q);
        for (uint32_t i = 0; i < cs.na; ++i) vcols.push_back(s->adv_values[(size_t)c * cs.na + i]);
        for (uint32_t i = 0; i < cs.ni; ++i) vcols.push_back(s->inst_values[(size_t)c * cs.ni + i]);
        for (auto q : p.pk->sigma_values) vcols.push_back(q);
        vcols.push_back(p.pk->omega_pows);
    }
    p.vstride = (uint32_t)(vcols.size() / p.nc);
    ZKB_TRY(upload_table(pool, vcols, &p.d_vcols, st));

    p.lk_f.resize(nu);
    p.lk_t.resize(nu);
    p.lk_m.resize(nu);
    // m columns live in one slab, completed by one all-gather when dealt
    const Deal &deal = p.lk_deal;
    Fr *m_slab = nullptr;
    if (nu) {
        ZKB_TRY(pool.fr(deal.padded() * n, &m_slab));
        for (size_t u = 0; u < nu; ++u) p.lk_m[u] = m_slab + u * n;
    }
    uint64_t lookup_errors = 0;
    for (size_t u = 0; u < nu; ++u) {
        if (!deal.mine(u)) continue;
        const size_t c = u / nl, l = u % nl;
        const CsfLookup &lk = cs.lookups[l];
        ExprBuilder eb;
        ProgramBuilder pb(eb);
        std::vector<int64_t> memo(cs.nodes.size(), -1);
        std::vector<ProgramBuilder::Root> roots;
        std::vector<Fr *> outs;
        for (size_t j = 0; j < lk.inputs.size(); ++j) {
            Fr *a;
            ZKB_TRY(pool.fr(n, &a));
            p.lk_f[u].push_back(a);
            outs.push_back(a);
            roots.push_back({compress_exprs(cs, lk.inputs[j], eb, vsm, s->challenges, memo, p.theta), ProgramBuilder::STORE, (uint32_t)j});
        }
        ZKB_TRY(pool.fr(n, &p.lk_t[u]));
        outs.push_back(p.lk_t[u]);
        roots.push_back({compress_exprs(cs, lk.table, eb, vsm, s->challenges, memo, p.theta), ProgramBuilder::STORE, (uint32_t)lk.inputs.size()});
        if (!pb.scope(roots)) { set_error("lookup %zu: %s", l, pb.error.c_str()); return ZKB_ERR_ARG; }
        ZKB_TRY(run_program(s, pb, eb, p.d_vcols + c * p.vstride, outs, st));
        // multiplicities over the usable rows
        uint32_t tsize = 1;
        while (tsize < 2 * usable) tsize <<= 1;
        uint32_t *slots = nullptr, *counts = nullptr;
        int *d_err = nullptr;
        ZKB_TRY(pool.alloc((size_t)tsize * 4, (void **)&slots));
        ZKB_TRY(pool.alloc((size_t)n * 4 + 16, (void **)&counts));
        d_err = (int *)(counts + n);
        ZKB_CUDA(cudaMemsetAsync(slots, 0, (size_t)tsize * 4, st));
        ZKB_CUDA(cudaMemsetAsync(counts, 0, (size_t)n * 4 + 16, st));
        const unsigned ub = (usable + 255) / 256;
        m_insert_kernel<<<ub, 256, 0, st>>>(p.lk_t[u], usable, slots, tsize - 1);
        for (size_t j = 0; j < lk.inputs.size(); ++j) m_count_kernel<<<ub, 256, 0, st>>>(p.lk_f[u][j], p.lk_t[u], usable, slots, tsize - 1, counts, d_err);
        counts_to_fr_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(counts, (uint32_t)n, p.lk_m[u]);
        p.ctx->launches += 2 + lk.inputs.size();
        int herr = 0;
        ZKB_CUDA(cudaMemcpyAsync(&herr, d_err, 4, cudaMemcpyDeviceToHost, st));
        ZKB_CUDA(cudaStreamSynchronize(st));
        if (herr) {
            if (p.nc == 1) set_error("lookup %zu: an input row is not in the table (unsatisfied witness)", l);
            else set_error("circuit %zu, lookup %zu: an input row is not in the table (unsatisfied witness)", c, l);
            if (!deal.on) return ZKB_ERR_ARG;
            lookup_errors++;   // multi-GPU: every rank must learn about it before anyone leaves the collective sequence
        }
    }
    if (deal.on) {
        ZKB_TRY(deal_gather(p.ctx, deal, m_slab, n * sizeof(Fr), st));
        uint64_t *d_errw = nullptr;   // every rank learns about an unsatisfied lookup before anyone leaves the collective sequence
        ZKB_TRY(scratch_get(p.ctx, SCR_COMM_FLAG, 64, (void **)&d_errw));
        ZKB_CUDA(cudaMemcpyAsync(d_errw + 1, &lookup_errors, 8, cudaMemcpyHostToDevice, st));
        ZKB_TRY(comm_allreduce_u64(p.ctx, d_errw + 1, 1, st));
        uint64_t total_err = 0;
        ZKB_CUDA(cudaMemcpyAsync(&total_err, d_errw + 1, 8, cudaMemcpyDeviceToHost, st));
        ZKB_CUDA(cudaStreamSynchronize(st));
        if (total_err) {
            if (!lookup_errors) set_error("a lookup input row is not in the table (reported by another rank)");
            return ZKB_ERR_ARG;
        }
    }
    return commit_write(s, BASIS_LAGRANGE, p.lk_m, st);
}

// permutation/prover.rs: grand products z of the permutation sets (z_blinds: bf values per set), commit z
static int32_t permutation_commit(ProofState &p, const uint64_t *z_blinds) {
    zkb_pk *pk = p.pk;
    zkb_ctx *ctx = p.ctx;
    const Csf &cs = p.cs;
    const uint64_t n = p.n;
    const uint32_t bf = p.bf;
    cudaStream_t st = p.st;
    const Fr one = Fr::one();
    const SlotMap vsm{0, cs.nf, cs.nf + cs.na};
    const uint32_t v_sigma0 = cs.nf + cs.na + cs.ni, v_omega = v_sigma0 + (uint32_t)cs.perm.size();
    const Fr delta = perm_delta();
    // Multi-GPU: the sets of all circuits are dealt.  Upstream chains a circuit's sets (z_i[0] = last value of z_{i-1}; every
    // circuit's first set starts at 1), which is sequential; here every set is scanned from 1 and rescaled afterwards by c_i = product
    // of the same circuit's previous sets' last values -- the same field elements (z_i = c_i * z'_i row by row), with only the last
    // values crossing the ranks before the columns are gathered.
    const uint32_t nsets = pk->nsets, nu = p.nc * nsets;   // unit u = set u % nsets of circuit u / nsets
    const Deal dp_sets(ctx, nu);
    p.zs.resize(nu);
    Fr *z_slab = nullptr;
    ZKB_TRY(p.pool.fr(std::max<size_t>(1, dp_sets.padded()) * n, &z_slab));
    for (uint32_t u = 0; u < nu; ++u) p.zs[u] = z_slab + (size_t)u * n;
    Fr *num, *den, *tmp;
    ZKB_TRY(p.pool.fr(n, &num));
    ZKB_TRY(p.pool.fr(n, &den));
    ZKB_TRY(p.pool.fr(n, &tmp));
    std::vector<Fr> lasts(std::max<size_t>(1, dp_sets.padded()), one);
    Fr last_z = one;
    for (uint32_t u = 0; u < nu; ++u) {
        const uint32_t c = u / nsets, si = u % nsets;
        if (si == 0) last_z = one;
        if (!dp_sets.mine(u)) continue;
        ExprBuilder eb;
        ProgramBuilder pb(eb);
        uint32_t nnum = 0, nden = 0;
        bool first = true;
        Fr delta_pow = fp_pow_u64(delta, (uint64_t)si * pk->chunk);
        for (uint32_t j = si * pk->chunk; j < std::min<size_t>((si + 1) * pk->chunk, cs.perm.size()); ++j) {
            const uint32_t v = eb.col(perm_slot(vsm, cs.perm[j]), 0);
            const uint32_t dterm = eb.add(eb.add(v, eb.mul(eb.col(v_sigma0 + j, 0), eb.constant(p.beta))), eb.constant(p.gamma));
            const uint32_t nterm = eb.add(eb.add(v, eb.mul(eb.col(v_omega, 0), eb.constant(fp_mul(p.beta, delta_pow)))), eb.constant(p.gamma));
            nden = first ? dterm : eb.mul(nden, dterm);
            nnum = first ? nterm : eb.mul(nnum, nterm);
            first = false;
            delta_pow = fp_mul(delta_pow, delta);
        }
        if (!pb.scope({{nnum, ProgramBuilder::STORE, 0}, {nden, ProgramBuilder::STORE, 1}})) { set_error("permutation: %s", pb.error.c_str()); return ZKB_ERR_ARG; }
        ZKB_TRY(run_program(p.s, pb, eb, p.d_vcols + (size_t)c * p.vstride, {num, den}, st));
        ZKB_TRY(batch_invert_device(ctx, den, tmp, n, st));
        mul_arrays_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(num, tmp, den, n);  // den <- modified values
        ctx->launches++;
        // one GPU: chained exactly like upstream (init = previous last value); dealt: from 1, rescaled below
        ZKB_TRY(prefix_product_device(ctx, den, n, dp_sets.on ? one : last_z, p.zs[u], st));
        ZKB_CUDA(cudaMemcpyAsync(&last_z, p.zs[u] + (n - bf - 1), sizeof(Fr), cudaMemcpyDeviceToHost, st));
        ZKB_CUDA(cudaStreamSynchronize(st));
        lasts[u] = last_z;
        if (!dp_sets.on) ZKB_CUDA(cudaMemcpyAsync(p.zs[u] + (n - bf), z_blinds + 4ull * bf * u, (size_t)bf * sizeof(Fr), cudaMemcpyHostToDevice, st));
    }
    if (dp_sets.on) {
        ZKB_TRY(deal_gather_host(ctx, dp_sets, lasts.data(), sizeof(Fr), st));
        Fr c = one;   // c_i = prod_{j < i} last'_j over the sets of the same circuit
        for (uint32_t u = 0; u < nu; ++u) {
            if (u % nsets == 0) c = one;
            if (dp_sets.mine(u)) {
                if (!(c == one)) { scale_const_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(p.zs[u], c, n); ctx->launches++; }
                ZKB_CUDA(cudaMemcpyAsync(p.zs[u] + (n - bf), z_blinds + 4ull * bf * u, (size_t)bf * sizeof(Fr), cudaMemcpyHostToDevice, st));
            }
            c = fp_mul(c, lasts[u]);
        }
        ZKB_TRY(deal_gather(ctx, dp_sets, z_slab, n * sizeof(Fr), st));
    }
    return commit_write(p.s, BASIS_LAGRANGE, p.zs, st);
}

// mv_lookup/prover.rs::commit_grand_sum: phi = prefix sum of sum_j 1/(f_j + beta) - m/(t + beta) (phi_blinds: bf values per lookup)
static int32_t lookups_commit_sums(ProofState &p, const uint64_t *phi_blinds) {
    const uint64_t n = p.n;
    const size_t nl = p.lk_m.size();   // lookup arguments of all circuits, circuit-major
    cudaStream_t st = p.st;
    DevPool &pool = p.pool;
    p.phis.resize(nl);
    Fr *phi_slab = nullptr;
    if (nl) {
        ZKB_TRY(pool.fr(p.lk_deal.padded() * n, &phi_slab));
        for (size_t l = 0; l < nl; ++l) p.phis[l] = phi_slab + l * n;
    }
    for (size_t l = 0; l < nl; ++l) {
        if (!p.lk_deal.mine(l)) continue;
        const size_t J = p.lk_f[l].size();
        // denominators (f_j + beta), (t + beta) into one contiguous array, inverted at once
        Fr *dens, *invs, *dterm;
        ZKB_TRY(pool.fr((J + 1) * n, &dens));
        ZKB_TRY(pool.fr((J + 1) * n, &invs));
        ZKB_TRY(pool.fr(n, &dterm));
        std::vector<Fr *> cols;
        for (auto q : p.lk_f[l]) cols.push_back(q);
        cols.push_back(p.lk_t[l]);          // slot J
        cols.push_back(p.lk_m[l]);          // slot J + 1
        for (size_t j = 0; j <= J; ++j) cols.push_back(invs + j * n);  // slots J + 2 ..
        Fr **d_cols = nullptr;
        ZKB_TRY(upload_table(pool, cols, &d_cols, st));
        {
            ExprBuilder eb;
            ProgramBuilder pb(eb);
            std::vector<ProgramBuilder::Root> roots;
            std::vector<Fr *> outs;
            for (size_t j = 0; j <= J; ++j) {
                roots.push_back({eb.add(eb.col((uint32_t)j, 0), eb.constant(p.beta)), ProgramBuilder::STORE, (uint32_t)j});
                outs.push_back(dens + j * n);
            }
            if (!pb.scope(roots)) { set_error("lookup sum: %s", pb.error.c_str()); return ZKB_ERR_ARG; }
            ZKB_TRY(run_program(p.s, pb, eb, d_cols, outs, st));
        }
        ZKB_TRY(batch_invert_device(p.ctx, dens, invs, (J + 1) * n, st));
        {
            ExprBuilder eb;
            ProgramBuilder pb(eb);
            uint32_t acc = eb.neg(eb.mul(eb.col((uint32_t)J + 1, 0), eb.col((uint32_t)(J + 2 + J), 0)));  // - m / (t + beta)
            for (size_t j = 0; j < J; ++j) acc = eb.add(acc, eb.col((uint32_t)(J + 2 + j), 0));
            if (!pb.scope({{acc, ProgramBuilder::STORE, 0}})) { set_error("lookup sum: %s", pb.error.c_str()); return ZKB_ERR_ARG; }
            ZKB_TRY(run_program(p.s, pb, eb, d_cols, {dterm}, st));
        }
        ZKB_TRY(prefix_sum_device(p.ctx, dterm, n, Fr::zero(), p.phis[l], st));
        ZKB_CUDA(cudaMemcpyAsync(p.phis[l] + (n - p.bf), phi_blinds + 4ull * p.bf * l, (size_t)p.bf * sizeof(Fr), cudaMemcpyHostToDevice, st));
    }
    if (nl) ZKB_TRY(deal_gather(p.ctx, p.lk_deal, phi_slab, n * sizeof(Fr), st));
    return commit_write(p.s, BASIS_LAGRANGE, p.phis, st);
}

// vanishing/prover.rs commit: the caller's random polynomial (n coefficients), committed with g
static int32_t vanishing_commit_random(ProofState &p, const uint64_t *random_poly_host) {
    ZKB_TRY(p.pool.fr(p.n, &p.random_poly));
    ZKB_CUDA(cudaMemcpyAsync(p.random_poly, random_poly_host, p.n * sizeof(Fr), cudaMemcpyHostToDevice, p.st));
    return commit_write(p.s, BASIS_G, {p.random_poly}, p.st);
}

// size-n transforms of src[i] into dst[i], batched with at most 2 GiB of NTT scratch per launch
static int32_t ntt_many(ProofState &p, const std::vector<Fr *> &src, const std::vector<Fr *> &dst, const Fr &w, const Fr *scale, const Fr *in_scale) {
    const uint32_t chunk = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(256, (1ull << 31) / (p.n * sizeof(Fr))));
    for (size_t done = 0; done < src.size(); done += chunk) {
        const uint32_t cur = (uint32_t)std::min<size_t>(chunk, src.size() - done);
        std::vector<Fr *> a(src.begin() + done, src.begin() + done + cur), b(dst.begin() + done, dst.begin() + done + cur);
        ZKB_TRY(ntt_fr_batch_device(p.ctx, a.data(), b.data(), cur, p.k, w, scale, 0, in_scale, p.st));
    }
    return ZKB_OK;
}
// coefficient forms of `vals` in a new slab; multi-GPU: contiguous blocks of columns per rank, completed by one all-gather
static int32_t to_coeff_new(ProofState &p, const std::vector<Fr *> &vals, std::vector<Fr *> &polys) {
    polys.resize(vals.size());
    if (vals.empty()) return ZKB_OK;
    Fr *pslab = nullptr;
    const Deal dc(p.ctx, vals.size());
    ZKB_TRY(p.pool.fr(dc.padded() * p.n, &pslab));
    for (size_t i = 0; i < vals.size(); ++i) polys[i] = pslab + i * p.n;
    std::vector<Fr *> src, dst;
    for (size_t i = 0; i < vals.size(); ++i)
        if (dc.mine(i)) { src.push_back(vals[i]); dst.push_back(polys[i]); }
    if (!src.empty()) ZKB_TRY(ntt_many(p, src, dst, p.pk->omega_inv, &p.pk->n_inv, nullptr));
    return deal_gather(p.ctx, dc, pslab, p.n * sizeof(Fr), p.st);
}
static int32_t to_coefficients(ProofState &p) {
    ZKB_TRY(to_coeff_new(p, p.s->adv_values, p.adv_polys));
    ZKB_TRY(to_coeff_new(p, p.zs, p.z_polys));
    ZKB_TRY(to_coeff_new(p, p.phis, p.phi_polys));
    return to_coeff_new(p, p.lk_m, p.m_polys);
}

// evaluation.rs::evaluate_h: the quotient numerator as ONE interpreter program over the coset-domain slot table, every constraint
// folded in with Horner in y, in upstream's order (gates, permutation, lookups).  With C circuits upstream loops over the circuits
// and keeps folding into the same accumulator; here the kernel runs the same program once per circuit's slot table and carries the
// accumulator over, so h = sum_c A_c y^(K (C - 1 - c)) for the single-circuit numerators A_c of K folded constraints each.
static int32_t quotient_program(ProofState &p) {
    zkb_pk *pk = p.pk;
    const Csf &cs = p.cs;
    const std::vector<Fr> &challenges = p.s->challenges;
    const Fr one = Fr::one();
    const uint32_t ns = pk->nsets, nl = (uint32_t)cs.lookups.size();
    p.q_sigma0 = cs.nf + cs.na + cs.ni;
    p.q_z0 = p.q_sigma0 + (uint32_t)cs.perm.size();
    p.q_phi0 = p.q_z0 + ns;
    p.q_m0 = p.q_phi0 + nl;
    p.q_l0 = p.q_m0 + nl;
    p.q_stride = p.q_l0 + 4;
    const uint32_t q_l0 = p.q_l0, q_llast = q_l0 + 1, q_lblind = q_l0 + 2, q_x = q_l0 + 3;
    ZKB_ARG(p.q_stride < 65536);
    auto table_of = [&](uint32_t c) {   // the slot table of circuit c (coefficient forms)
        std::vector<Fr *> t(pk->fixed_polys);
        auto add = [&](const std::vector<Fr *> &v, size_t first, size_t count) { t.insert(t.end(), v.begin() + first, v.begin() + first + count); };
        add(p.adv_polys, (size_t)c * cs.na, cs.na);
        add(p.s->inst_polys, (size_t)c * cs.ni, cs.ni);
        add(pk->sigma_polys, 0, cs.perm.size());
        add(p.z_polys, (size_t)c * ns, ns);
        add(p.phi_polys, (size_t)c * nl, nl);
        add(p.m_polys, (size_t)c * nl, nl);
        t.insert(t.end(), {pk->l0_poly, pk->llast_poly, pk->lblind_poly, pk->xid_poly});
        return t;
    };
    auto scoped = [&](uint32_t slot) { return (slot >= cs.nf && slot < p.q_sigma0) || (slot >= p.q_z0 && slot < p.q_l0); };
    p.qpolys = table_of(0);
    for (uint32_t i = 0; i < p.q_stride; ++i) p.q_slot.push_back(i);
    for (uint32_t c = 1; c < p.nc; ++c) {
        const std::vector<Fr *> t = table_of(c);
        for (uint32_t i = 0; i < p.q_stride; ++i) {
            if (!scoped(i)) { p.q_slot.push_back(i); continue; }
            p.q_slot.push_back((uint32_t)p.qpolys.size());
            p.qpolys.push_back(t[i]);
        }
    }
    const SlotMap qsm{0, cs.nf, cs.nf + cs.na};

    ExprBuilder qeb;
    ProgramBuilder qpb(qeb);
    const uint32_t y_idx = qeb.const_slot(p.y);
    std::vector<int64_t> memo(cs.nodes.size(), -1);
    // Gate polynomials, Horner in y in constraint-system order.  Circuits multiply whole groups of constraints by one selector
    // (`q_enable * constraint`), so runs of CONSECUTIVE gates of the form fixed(col, rot) * t_j are folded exactly:
    //   (..(acc y + f t_1) y + ..) y + f t_r  =  acc y^r + f (t_1 y^(r-1) + .. + t_r)
    // -- the same field element (distributivity is exact mod r), one multiply per gate less than the term-by-term form.
    auto selector_split = [&](uint32_t gnode, uint32_t &sel, uint32_t &rest) -> bool {
        const auto &nd = cs.nodes[gnode];
        if (nd[0] != N_MUL) return false;
        for (int side = 0; side < 2; ++side) {
            const uint32_t a = nd[1 + side], b = nd[2 - side];
            if (cs.nodes[a][0] == N_FIXED) { sel = a; rest = b; return true; }
        }
        return false;
    };
    auto same_query = [&](uint32_t a, uint32_t b) { return cs.nodes[a][1] == cs.nodes[b][1] && cs.nodes[a][2] == cs.nodes[b][2]; };
    for (size_t gi = 0; gi < cs.gates.size();) {
        uint32_t sel = 0, rest = 0;
        size_t run = 1;
        if (selector_split(cs.gates[gi], sel, rest)) {
            uint32_t s2 = 0, r2 = 0;
            while (gi + run < cs.gates.size() && run < 4096 && selector_split(cs.gates[gi + run], s2, r2) && same_query(sel, s2)) ++run;
        }
        if (run < 2) {
            if (!qpb.scope({{translate(cs, cs.gates[gi], qeb, qsm, challenges, memo), ProgramBuilder::HORNER, y_idx}})) { set_error("gate: %s", qpb.error.c_str()); return ZKB_ERR_ARG; }
            ++gi;
            continue;
        }
        for (size_t t = 0; t < run; ++t) {
            uint32_t s2 = 0, r2 = 0;
            selector_split(cs.gates[gi + t], s2, r2);
            if (!qpb.scope({{translate(cs, r2, qeb, qsm, challenges, memo), ProgramBuilder::HORNER2, y_idx}})) { set_error("gate: %s", qpb.error.c_str()); return ZKB_ERR_ARG; }
        }
        const uint32_t yr_idx = qeb.const_slot(fp_pow_u64(p.y, run));
        if (!qpb.scope({{translate(cs, sel, qeb, qsm, challenges, memo), ProgramBuilder::FOLD, yr_idx}})) { set_error("gate: %s", qpb.error.c_str()); return ZKB_ERR_ARG; }
        gi += run;
    }
    auto lactive = [&]() { return qeb.sub(qeb.sub(qeb.constant(one), qeb.col(q_llast, 0)), qeb.col(q_lblind, 0)); };
    if (pk->nsets) {
        const uint32_t z0 = qeb.col(p.q_z0, 0), zl = qeb.col(p.q_z0 + pk->nsets - 1, 0);
        if (!qpb.scope({{qeb.mul(qeb.sub(qeb.constant(one), z0), qeb.col(q_l0, 0)), ProgramBuilder::HORNER, y_idx}})) return ZKB_ERR_ARG;
        if (!qpb.scope({{qeb.mul(qeb.sub(qeb.mul(zl, zl), zl), qeb.col(q_llast, 0)), ProgramBuilder::HORNER, y_idx}})) return ZKB_ERR_ARG;
        for (uint32_t i = 1; i < pk->nsets; ++i) {
            const uint32_t t = qeb.mul(qeb.sub(qeb.col(p.q_z0 + i, 0), qeb.col(p.q_z0 + i - 1, -(int32_t)(p.bf + 1))), qeb.col(q_l0, 0));
            if (!qpb.scope({{t, ProgramBuilder::HORNER, y_idx}})) return ZKB_ERR_ARG;
        }
        const Fr delta = perm_delta();
        Fr delta_pow = one;
        for (uint32_t si = 0; si < pk->nsets; ++si) {
            uint32_t left = qeb.col(p.q_z0 + si, 1), right = qeb.col(p.q_z0 + si, 0);
            for (uint32_t j = si * pk->chunk; j < std::min<size_t>((si + 1) * pk->chunk, cs.perm.size()); ++j) {
                const uint32_t v = qeb.col(perm_slot(qsm, cs.perm[j]), 0);
                left = qeb.mul(left, qeb.add(qeb.add(v, qeb.mul(qeb.col(p.q_sigma0 + j, 0), qeb.constant(p.beta))), qeb.constant(p.gamma)));
                right = qeb.mul(right, qeb.add(qeb.add(v, qeb.mul(qeb.col(q_x, 0), qeb.constant(fp_mul(p.beta, delta_pow)))), qeb.constant(p.gamma)));
                delta_pow = fp_mul(delta_pow, delta);
            }
            if (!qpb.scope({{qeb.mul(qeb.sub(left, right), lactive()), ProgramBuilder::HORNER, y_idx}})) { set_error("permutation: %s", qpb.error.c_str()); return ZKB_ERR_ARG; }
        }
    }
    for (size_t l = 0; l < cs.lookups.size(); ++l) {
        const CsfLookup &lk = cs.lookups[l];
        std::vector<uint32_t> fsb;
        for (auto &inp : lk.inputs) fsb.push_back(qeb.add(compress_exprs(cs, inp, qeb, qsm, challenges, memo, p.theta), qeb.constant(p.beta)));
        const uint32_t tb = qeb.add(compress_exprs(cs, lk.table, qeb, qsm, challenges, memo, p.theta), qeb.constant(p.beta));
        uint32_t prod = fsb[0];
        for (size_t j = 1; j < fsb.size(); ++j) prod = qeb.mul(prod, fsb[j]);
        uint32_t ssum = 0;
        bool have_sum = false;
        for (size_t i = 0; i < fsb.size(); ++i) {
            uint32_t pr = 0;
            bool have = false;
            for (size_t j = 0; j < fsb.size(); ++j) {
                if (j == i) continue;
                pr = have ? qeb.mul(pr, fsb[j]) : fsb[j];
                have = true;
            }
            if (!have) pr = qeb.constant(one);
            ssum = have_sum ? qeb.add(ssum, pr) : pr;
            have_sum = true;
        }
        const uint32_t phi = qeb.col(p.q_phi0 + (uint32_t)l, 0), phi_next = qeb.col(p.q_phi0 + (uint32_t)l, 1), m = qeb.col(p.q_m0 + (uint32_t)l, 0);
        const uint32_t lhs = qeb.mul(qeb.mul(tb, prod), qeb.sub(phi_next, phi));
        const uint32_t rhs = qeb.sub(qeb.mul(tb, ssum), qeb.mul(m, prod));
        std::vector<ProgramBuilder::Root> roots = {{qeb.mul(phi, qeb.col(q_l0, 0)), ProgramBuilder::HORNER, y_idx},
                                                   {qeb.mul(phi, qeb.col(q_llast, 0)), ProgramBuilder::HORNER, y_idx},
                                                   {qeb.mul(qeb.sub(lhs, rhs), lactive()), ProgramBuilder::HORNER, y_idx}};
        if (!qpb.scope(roots)) { set_error("lookup %zu: %s", l, qpb.error.c_str()); return ZKB_ERR_ARG; }
    }
    // one STOREACC per coset part (the scale constant differs): the device code buffer holds the common body + one trailing
    // STOREACC slot that is rewritten per part
    p.tinv_idx.resize(pk->E);
    for (uint32_t j = 0; j < pk->E; ++j) p.tinv_idx[j] = qeb.const_slot(pk->t_inv[j]);
    p.q_base_len = qpb.code.size();
    qpb.store_acc(0, p.tinv_idx[0]);
    return upload_program(p.pool, qpb, qeb, p.qdp, p.st);
}

// evaluate h on the extended domain, coset part by coset part: size-n NTTs of every polynomial not in the pk's coset cache, one
// interpreter launch, x 1/((zeta omega_ext^j)^n - 1)
static int32_t quotient_evaluate(ProofState &p) {
    zkb_pk *pk = p.pk;
    zkb_ctx *ctx = p.ctx;
    const uint64_t n = p.n;
    cudaStream_t st = p.st;
    DevPool &pool = p.pool;
    const std::vector<Fr *> &qpolys = p.qpolys;
    Fr *slab, *pows;   // slab: coset values of every distinct polynomial of the slot tables
    ZKB_TRY(pool.fr(qpolys.size() * n, &slab));
    ZKB_TRY(pool.fr(n, &pows));
    ZKB_TRY(pool.fr(pk->N, &p.h_ext));
    std::vector<Fr *> qcols(qpolys.size());
    for (size_t i = 0; i < qpolys.size(); ++i) qcols[i] = slab + i * n;
    // slots served from the pk's coset cache: fixed [0, nf), sigma, l0 / l_last / l_blind / X
    const bool cached = !pk->coset_cache.empty();
    std::vector<int> cache_idx(qpolys.size(), -1);
    if (cached) {
        int ci = 0;
        for (uint32_t i = 0; i < p.cs.nf; ++i) cache_idx[i] = ci++;
        for (size_t i = 0; i < p.cs.perm.size(); ++i) cache_idx[p.q_sigma0 + i] = ci++;
        for (uint32_t i = 0; i < 4; ++i) cache_idx[p.q_l0 + i] = ci++;
    }
    std::vector<Fr *> ntt_src, ntt_dst;
    for (size_t i = 0; i < qpolys.size(); ++i) {
        if (cache_idx[i] < 0) { ntt_src.push_back(qpolys[i]); ntt_dst.push_back(qcols[i]); }
    }
    Fr **d_qcols = nullptr, **d_hout = nullptr;   // d_qcols: the slot tables of all circuits
    ZKB_TRY(pool.alloc(p.q_slot.size() * sizeof(Fr *) + 8, (void **)&d_qcols));
    // multi-GPU: coset parts are dealt in contiguous blocks; a rank writes its parts as contiguous n-element rows of h_parts, the rows
    // are all-gathered and interleaved into the extended-domain order h_ext[j + E i] the inverse transform expects
    const Deal dq(ctx, pk->E);
    Fr *h_parts = nullptr;
    if (dq.on) ZKB_TRY(pool.fr(dq.padded() * n, &h_parts));
    ZKB_TRY(upload_table(pool, std::vector<Fr *>{dq.on ? h_parts : p.h_ext}, &d_hout, st));
    const DeviceProgram &qdp = p.qdp;
    for (uint32_t j = 0; j < pk->E; ++j) {
        if (!dq.mine(j)) continue;
        ZKB_TRY(fr_powers_device(ctx, coset_gen(pk, j), n, pows, st));
        ZKB_TRY(ntt_many(p, ntt_src, ntt_dst, pk->omega, nullptr, pows));
        std::vector<Fr *> cols_j = qcols;
        if (cached)
            for (size_t i = 0; i < qpolys.size(); ++i)
                if (cache_idx[i] >= 0) cols_j[i] = pk->coset_cache[j][cache_idx[i]];
        std::vector<Fr *> tables(p.q_slot.size());
        for (size_t t = 0; t < tables.size(); ++t) tables[t] = cols_j[p.q_slot[t]];
        Instr tail{OP_STOREACC, 0, 0, 0, 0u | (p.tinv_idx[j] << 8)};
        ZKB_CUDA(cudaMemcpyAsync(d_qcols, tables.data(), tables.size() * sizeof(Fr *), cudaMemcpyHostToDevice, st));
        ZKB_CUDA(cudaMemcpyAsync(qdp.code + p.q_base_len, &tail, sizeof(Instr), cudaMemcpyHostToDevice, st));
        const uint32_t out_stride = dq.on ? 1 : pk->E, out_offset = dq.on ? (uint32_t)((uint64_t)j * n) : j;
        if (p.nc == 1) ZKB_TRY(expr_run_device(ctx, qdp.code, qdp.ncode, qdp.nregs, d_qcols, qdp.consts, d_hout, p.k, out_stride, out_offset, st));
        else ZKB_TRY(expr_run_circuits_device(ctx, qdp.code, qdp.ncode, (uint32_t)p.q_base_len, qdp.nregs, d_qcols, p.nc, p.q_stride, qdp.consts, d_hout,
                                              p.k, out_stride, out_offset, st));
        ZKB_CUDA(cudaStreamSynchronize(st));  // `tail` and `tables` live on the stack
    }
    if (dq.on) {
        ZKB_TRY(deal_gather(ctx, dq, h_parts, n * sizeof(Fr), st));
        interleave_parts_kernel<<<(unsigned)((pk->N + 255) / 256), 256, 0, st>>>(h_parts, p.h_ext, p.k, pk->E);
        ctx->launches++;
    }
    return ZKB_OK;
}

// vanishing::construct: extended_to_coeff (inverse NTT over the extended domain, 1/N, undo the zeta coset), the d - 1 pieces of
// n coefficients, committed with g
static int32_t quotient_commit(ProofState &p) {
    zkb_pk *pk = p.pk;
    ZKB_TRY(ntt_fr_device(p.ctx, p.h_ext, p.h_ext, pk->ext_k, pk->ext_omega_inv, &pk->N_inv, 2, nullptr, p.st));
    std::vector<Fr *> pieces;
    for (uint32_t i = 0; i < pk->qdeg; ++i) pieces.push_back(p.h_ext + (size_t)i * p.n);
    return commit_write(p.s, BASIS_G, pieces, p.st);
}

// the evaluations written to the transcript (prover.rs order), then the multiopen queries (prover.rs order)
static int32_t evaluate(ProofState &p) {
    zkb_pk *pk = p.pk;
    const Csf &cs = p.cs;
    const size_t nl = cs.lookups.size();
    const uint64_t n = p.n;
    cudaStream_t st = p.st;
    // h(X) = sum_i x^(n i) piece_i
    const Fr xn = fp_pow_u64(p.x, n);
    Fr *h_poly;
    ZKB_TRY(p.pool.fr(n, &h_poly));
    {
        std::vector<Fr *> pieces;
        std::vector<Fr> cf;
        Fr cur = Fr::one();
        for (uint32_t i = 0; i < pk->qdeg; ++i) { pieces.push_back(p.h_ext + (size_t)i * n); cf.push_back(cur); cur = fp_mul(cur, xn); }
        ZKB_TRY(lincomb(p.s, pieces, cf, h_poly, false, st));
        ZKB_CUDA(cudaStreamSynchronize(st));
    }
    const uint32_t nc = p.nc, na = cs.na, ns = pk->nsets;
    int next_id = 0;   // identities of the committed polynomials, in this order; per-circuit ones circuit-major
    auto ids = [&](size_t count) { std::vector<int> v(count); for (auto &e : v) e = next_id++; return v; };
    const std::vector<int> adv_id = ids(nc * na), fix_id = ids(cs.nf), sig_id = ids(cs.perm.size()), z_id = ids(nc * ns), phi_id = ids(nc * nl),
                           m_id = ids(nc * nl);
    const int h_id = next_id++, rand_id = next_id++;
    const int64_t rot_last = -(int64_t)(p.bf + 1);
    // (1) the evaluations written to the transcript, in order: every circuit's advice queries, the fixed queries, the random
    // polynomial, sigma, every circuit's z evaluations, every circuit's lookup evaluations; the queries are built afterwards in
    // the multiopen order
    struct EvalReq { int poly_id; const Fr *poly; int64_t rot; };
    std::vector<EvalReq> reqs;
    for (uint32_t c = 0; c < nc; ++c)
        for (auto &q : cs.advq) reqs.push_back({adv_id[c * na + q[0]], p.adv_polys[c * na + q[0]], q[1]});
    for (auto &q : cs.fixq) reqs.push_back({fix_id[q[0]], pk->fixed_polys[q[0]], q[1]});
    reqs.push_back({rand_id, p.random_poly, 0});
    for (size_t i = 0; i < cs.perm.size(); ++i) reqs.push_back({sig_id[i], pk->sigma_polys[i], 0});
    for (uint32_t u = 0; u < nc * ns; ++u) {
        reqs.push_back({z_id[u], p.z_polys[u], 0});
        reqs.push_back({z_id[u], p.z_polys[u], 1});
        if (u % ns + 1 != ns) reqs.push_back({z_id[u], p.z_polys[u], rot_last});
    }
    for (size_t u = 0; u < nc * nl; ++u) {
        reqs.push_back({phi_id[u], p.phi_polys[u], 0});
        reqs.push_back({phi_id[u], p.phi_polys[u], 1});
        reqs.push_back({m_id[u], p.m_polys[u], 0});
    }
    const size_t n_written = reqs.size();
    reqs.push_back({h_id, h_poly, 0});  // needed by SHPLONK, not written
    // batch by rotation
    std::map<int64_t, std::vector<size_t>> by_rot;
    for (size_t i = 0; i < reqs.size(); ++i) by_rot[reqs[i].rot].push_back(i);
    std::vector<Fr> evals(reqs.size());
    for (auto &kv : by_rot) {
        const Fr pt = fp_mul(p.x, fr_pow_i64(pk->omega, pk->omega_inv, kv.first));
        p.point_of[kv.first] = pt;
        std::vector<Fr *> ptrs;
        for (size_t i : kv.second) ptrs.push_back(const_cast<Fr *>(reqs[i].poly));
        Fr **d_p = nullptr;
        ZKB_TRY(upload_table(p.pool, ptrs, &d_p, st));
        // multi-GPU: the polynomials of a rotation are dealt, the 32-byte results all-gathered
        const Deal de(p.ctx, ptrs.size());
        std::vector<Fr> res(std::max<size_t>(1, de.padded()));
        const size_t lo = de.first(), hi = std::min(ptrs.size(), lo + de.blk);
        if (hi > lo) ZKB_TRY(poly_eval_device(p.ctx, d_p + lo, (uint32_t)(hi - lo), n, pt, res.data() + lo, st));
        ZKB_TRY(deal_gather_host(p.ctx, de, res.data(), sizeof(Fr), st));
        for (size_t t = 0; t < kv.second.size(); ++t) evals[kv.second[t]] = res[t];
    }
    for (size_t i = 0; i < n_written; ++i) p.s->tr.write_scalar(evals[i]);
    for (size_t i = 0; i < reqs.size(); ++i) p.eval_of[{reqs[i].poly_id, reqs[i].rot}] = evals[i];

    // (2) multiopen queries in prover.rs order: per circuit [advice; z at x, omega x per set, then z at omega^last x for the sets
    // in reverse, skipping the last; lookups], then fixed, sigma, h, random
    auto push_q = [&](int id, const Fr *poly, int64_t rot) { p.queries.push_back({id, poly, rot, p.point_of[rot], p.eval_of[{id, rot}]}); };
    for (uint32_t c = 0; c < nc; ++c) {
        for (auto &q : cs.advq) push_q(adv_id[c * na + q[0]], p.adv_polys[c * na + q[0]], q[1]);
        const uint32_t z0 = c * ns;
        for (uint32_t i = z0; i < z0 + ns; ++i) { push_q(z_id[i], p.z_polys[i], 0); push_q(z_id[i], p.z_polys[i], 1); }
        for (int i = (int)ns - 2; i >= 0; --i) push_q(z_id[z0 + i], p.z_polys[z0 + i], rot_last);
        for (size_t l = c * nl; l < (c + 1) * nl; ++l) { push_q(phi_id[l], p.phi_polys[l], 0); push_q(phi_id[l], p.phi_polys[l], 1); push_q(m_id[l], p.m_polys[l], 0); }
    }
    for (auto &q : cs.fixq) push_q(fix_id[q[0]], pk->fixed_polys[q[0]], q[1]);
    for (size_t i = 0; i < cs.perm.size(); ++i) push_q(sig_id[i], pk->sigma_polys[i], 0);
    push_q(h_id, h_poly, 0);
    push_q(rand_id, p.random_poly, 0);
    return ZKB_OK;
}

// low-degree interpolant through (points, evals): coefficients, low to high
static std::vector<Fr> interpolate(const std::vector<Fr> &pts, const std::vector<Fr> &evs) {
    const size_t m = pts.size();
    std::vector<Fr> coeffs(m, Fr::zero());
    for (size_t j = 0; j < m; ++j) {
        std::vector<Fr> num{Fr::one()};
        Fr den = Fr::one();
        for (size_t t = 0; t < m; ++t) {
            if (t == j) continue;
            std::vector<Fr> nx(num.size() + 1, Fr::zero());
            for (size_t i = 0; i < num.size(); ++i) {
                nx[i + 1] = fp_add(nx[i + 1], num[i]);
                nx[i] = fp_sub(nx[i], fp_mul(pts[t], num[i]));
            }
            num.swap(nx);
            den = fp_mul(den, fp_sub(pts[j], pts[t]));
        }
        const Fr sc = fp_mul(evs[j], fp_inv(den));
        for (size_t i = 0; i < m; ++i) coeffs[i] = fp_add(coeffs[i], fp_mul(num[i], sc));
    }
    return coeffs;
}
static Fr horner_host(const std::vector<Fr> &c, const Fr &at) {
    Fr acc = Fr::zero();
    for (size_t i = c.size(); i-- > 0;) acc = fp_add(fp_mul(acc, at), c[i]);
    return acc;
}

// multiopen/shplonk/prover.rs up to the commitment of h_x: construct_intermediate_sets, then per rotation set
// Q_i = (sum_j y^j (P_ij - R_ij)) / Z_i and h_x = sum_i v^i Q_i
static int32_t shplonk_commit_h(ProofState &p) {
    zkb_session *s = p.s;
    const uint64_t n = p.n;
    cudaStream_t st = p.st;
    const Fr one = Fr::one();
    // construct_intermediate_sets: points sorted by canonical value, commitments and sets by first appearance
    std::vector<ShplonkCommit> &cmap = p.sh_commits;
    for (auto &q : p.queries) {
        if (std::find(p.super_rots.begin(), p.super_rots.end(), q.rot) == p.super_rots.end()) p.super_rots.push_back(q.rot);
        auto it = std::find_if(cmap.begin(), cmap.end(), [&](const ShplonkCommit &c) { return c.id == q.poly_id; });
        if (it == cmap.end()) cmap.push_back({q.poly_id, q.poly, {q.rot}});
        else if (std::find(it->rots.begin(), it->rots.end(), q.rot) == it->rots.end()) it->rots.push_back(q.rot);
    }
    auto sort_rots = [&](std::vector<int64_t> &r) { std::sort(r.begin(), r.end(), [&](int64_t a, int64_t b) { return fr_less(p.point_of[a], p.point_of[b]); }); };
    sort_rots(p.super_rots);
    for (auto &c : cmap) sort_rots(c.rots);
    for (auto &c : cmap) {
        auto it = std::find_if(p.rsets.begin(), p.rsets.end(), [&](const RotationSet &r) { return r.rots == c.rots; });
        if (it == p.rsets.end()) p.rsets.push_back({c.rots, {&c}, {}, {}});
        else it->comms.push_back(&c);
    }
    ZKB_TRY(p.pool.fr(n, &p.hx));
    ZKB_TRY(p.pool.fr(n, &p.work));
    ZKB_TRY(p.pool.fr(n, &p.work2));
    ZKB_TRY(p.pool.fr(256, &p.d_small));
    ZKB_CUDA(cudaMemsetAsync(p.hx, 0, n * sizeof(Fr), st));
    Fr vpow = one;
    for (RotationSet &rs : p.rsets) {
        for (int64_t r : rs.rots) rs.pts.push_back(p.point_of[r]);
        ZKB_ARG(rs.pts.size() <= 256);   // Keccak's hot cell column is opened at 56 rotations (keccak_packed_multi.rs:59-68)
        // N_i(X) = sum_j y^j (P_ij(X) - R_ij(X))
        std::vector<Fr *> ptrs;
        std::vector<Fr> cf;
        std::vector<Fr> rsum(rs.pts.size(), Fr::zero());
        Fr ypow = one;
        for (const ShplonkCommit *c : rs.comms) {
            std::vector<Fr> evs;
            for (int64_t r : rs.rots) evs.push_back(p.eval_of[{c->id, r}]);
            rs.r_coeffs.push_back(interpolate(rs.pts, evs));
            for (size_t i = 0; i < rs.pts.size(); ++i) rsum[i] = fp_add(rsum[i], fp_mul(rs.r_coeffs.back()[i], ypow));
            ptrs.push_back(const_cast<Fr *>(c->poly));
            cf.push_back(ypow);
            ypow = fp_mul(ypow, p.sy);
        }
        ZKB_TRY(lincomb(s, ptrs, cf, p.work, false, st));
        ZKB_CUDA(cudaMemcpyAsync(p.d_small, rsum.data(), rsum.size() * sizeof(Fr), cudaMemcpyHostToDevice, st));
        sub_low_kernel<<<1, 256, 0, st>>>(p.work, p.d_small, (uint32_t)rsum.size());
        p.ctx->launches++;
        ZKB_CUDA(cudaStreamSynchronize(st));
        // divide by the vanishing polynomial of the set, one root at a time
        Fr *src = p.work, *dst = p.work2;
        for (const Fr &pt : rs.pts) {
            ZKB_TRY(kate_division_device(p.ctx, src, n, pt, dst, st));
            std::swap(src, dst);
        }
        // h_x += v^i * Q_i
        const std::vector<Fr> vcoef{vpow};
        ZKB_TRY(lincomb(s, {src}, vcoef, p.hx, true, st));
        ZKB_CUDA(cudaStreamSynchronize(st));
        vpow = fp_mul(vpow, p.sv);
    }
    return commit_write(s, BASIS_G, {p.hx}, st);
}

// multiopen/shplonk/prover.rs after u: L(X) = sum_i v^i z_i sum_j y^j (P_ij(X) - r_ij(u)) - zt h_x(X), scaled by 1/z_0, divided by
// (X - u), committed with g
static int32_t shplonk_open(ProofState &p) {
    const Fr one = Fr::one();
    cudaStream_t st = p.st;
    const std::vector<RotationSet> &rsets = p.rsets;
    std::vector<Fr> super_pts;
    for (int64_t r : p.super_rots) super_pts.push_back(p.point_of[r]);
    std::vector<Fr> zdiff(rsets.size());
    for (size_t si = 0; si < rsets.size(); ++si) {
        Fr z = one;
        for (size_t t = 0; t < p.super_rots.size(); ++t) {
            if (std::find(rsets[si].rots.begin(), rsets[si].rots.end(), p.super_rots[t]) == rsets[si].rots.end()) z = fp_mul(z, fp_sub(p.su, super_pts[t]));
        }
        zdiff[si] = z;
    }
    Fr zt = one;
    for (auto &pt : super_pts) zt = fp_mul(zt, fp_sub(p.su, pt));
    const Fr z0inv = fp_inv(zdiff[0]);
    std::vector<Fr *> ptrs;
    std::vector<Fr> cf;
    Fr const_term = Fr::zero();
    Fr vpow = one;
    for (size_t si = 0; si < rsets.size(); ++si) {
        Fr ypow = one;
        for (size_t ci = 0; ci < rsets[si].comms.size(); ++ci) {
            const Fr w = fp_mul(fp_mul(fp_mul(vpow, zdiff[si]), ypow), z0inv);
            ptrs.push_back(const_cast<Fr *>(rsets[si].comms[ci]->poly));
            cf.push_back(w);
            const_term = fp_add(const_term, fp_mul(w, horner_host(rsets[si].r_coeffs[ci], p.su)));
            ypow = fp_mul(ypow, p.sy);
        }
        vpow = fp_mul(vpow, p.sv);
    }
    ptrs.push_back(p.hx);
    cf.push_back(fp_neg(fp_mul(zt, z0inv)));
    ZKB_TRY(lincomb(p.s, ptrs, cf, p.work, false, st));
    ZKB_CUDA(cudaMemcpyAsync(p.d_small, &const_term, sizeof(Fr), cudaMemcpyHostToDevice, st));
    sub_low_kernel<<<1, 256, 0, st>>>(p.work, p.d_small, 1);
    p.ctx->launches++;
    ZKB_CUDA(cudaStreamSynchronize(st));
    ZKB_TRY(kate_division_device(p.ctx, p.work, p.n, p.su, p.work2, st));
    return commit_write(p.s, BASIS_G, {p.work2}, st);
}

// create_proof after the advice phases.  Every transcript squeeze happens here, so this function reads as the transcript order.
static int32_t prove_finish_impl(zkb_session *s, const uint64_t *z_blinds, const uint64_t *phi_blinds, const uint64_t *random_poly_host) {
    ProofState p(s);
    Transcript &tr = s->tr;
    StageTrace trace(p.st);
    p.theta = tr.squeeze();
    ZKB_TRY(lookups_prepare(p));
    trace.mark("lookups: compress + m + commit");
    p.beta = tr.squeeze();
    p.gamma = tr.squeeze();
    ZKB_TRY(permutation_commit(p, z_blinds));
    trace.mark("permutation z + commit");
    ZKB_TRY(lookups_commit_sums(p, phi_blinds));
    trace.mark("lookup phi + commit");
    ZKB_TRY(vanishing_commit_random(p, random_poly_host));
    p.y = tr.squeeze();
    trace.mark("random poly commit");
    ZKB_TRY(to_coefficients(p));
    trace.mark("lagrange_to_coeff (all columns)");
    ZKB_TRY(quotient_program(p));
    trace.mark("quotient program build+upload");
    ZKB_TRY(quotient_evaluate(p));
    trace.mark("quotient: coset NTTs + fused eval");
    ZKB_TRY(quotient_commit(p));
    p.x = tr.squeeze();
    trace.mark("extended iNTT + h commits");
    ZKB_TRY(evaluate(p));
    trace.mark("evaluations");
    p.sy = tr.squeeze();
    p.sv = tr.squeeze();
    ZKB_TRY(shplonk_commit_h(p));
    p.su = tr.squeeze();
    ZKB_TRY(shplonk_open(p));
    trace.mark("shplonk");
    ZKB_TRY(tr.status());
    s->finished = true;
    return ZKB_OK;
}

}  // namespace zkb

extern "C" int32_t zkb_prove_finish(zkb_session *s, const uint64_t *z_blinds, const uint64_t *phi_blinds, const uint64_t *random_poly,
                                    uint8_t *proof_out, uint64_t proof_cap, uint64_t *proof_len) {
    ZKB_ARG(s && proof_len);
    zkb_pk *pk = s->pk;
    if (!s->finished) {
        // first call: run the proof.  The bytes stay in the session, so a query call (proof_out == NULL) or a call with a short
        // buffer loses nothing: call again with a buffer of *proof_len bytes.
        ZKB_ARG(random_poly != nullptr);
        if (s->next_phase != pk->cs.nphases) { set_error("zkb_prove_finish: advice phases incomplete"); return ZKB_ERR_STATE; }
        ZKB_ARG((pk->nsets == 0 || z_blinds) && (pk->cs.lookups.empty() || phi_blinds));
        ZKB_CUDA(cudaSetDevice(pk->ctx->device));
        ZKB_TRY(prove_finish_impl(s, z_blinds, phi_blinds, random_poly));
    }
    const std::vector<uint8_t> &proof = s->tr.proof;
    *proof_len = proof.size();
    if (proof_out) {
        if (proof_cap < proof.size()) { set_error("zkb_prove_finish: buffer of %llu bytes, proof has %llu (kept in the session: call again)",
                                                  (unsigned long long)proof_cap, (unsigned long long)proof.size()); return ZKB_ERR_ARG; }
        memcpy(proof_out, proof.data(), proof.size());
    }
    return ZKB_OK;
}
