/*
 * zkb200.h -- C ABI of libzkb200.so, the B200 (sm_100a) Halo2/KZG proving backend.
 *
 * This is the boundary a fork-shaped `halo2_proofs` crate binds to (SURVEY.md section 8b): the reference swaps its
 * prover backend at crate level (docker/testool/gpu/Dockerfile:7, cargo `paths` override of halo2_proofs), and the
 * bodies of the upstream functions named below call these entry points instead of their rayon loops.  The
 * reference-side call sites that reach them: circuit-benchmarks/src/super_circuit.rs:117-132 (create_proof),
 * prover/src/common/prover/utils.rs:31 (gen_snark_shplonk), prover/src/common/prover/utils.rs:55 (keygen_pk2).
 *
 * Conventions (precedent: geth-utils/src/lib.rs:9-14 -- plain C types, explicit ownership):
 *   - every function returns int32_t: 0 = ok, negative = error; zkb_last_error() gives a thread-local message.
 *   - field elements / points are caller-owned buffers in halo2curves' in-memory layout (halo2curves 0.1.0 @ a495a7b):
 *       Fr, Fq   : 4 x u64 little-endian limbs, Montgomery form (a * 2^256 mod p), fully reduced, 32 B
 *       G1Affine : x || y, 64 B, identity = (0, 0)          G1 (projective) : x || y || z Jacobian, 96 B, identity z = 0
 *     so Rust passes `slice.as_ptr()` with no conversion.
 *   - `*_host` entry points take HOST pointers and include the H2D / D2H copies; `*_dev` take DEVICE pointers and a
 *     CUDA stream (as void*, NULL = the context's stream) and never synchronise unless stated.
 *   - opaque handles are created / destroyed explicitly; one proving session at a time per context (the reference serialises
 *     proving behind a Mutex<Prover>: prover/src/test/inner.rs:20-30); one session may prove several circuits
 *     (zkb_prove_begin_multi).
 *   - There is NO CPU fallback: without a CUDA device every compute entry point fails with ZKB_ERR_CUDA.
 */
#ifndef ZKB200_H
#define ZKB200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define ZKB_API __attribute__((visibility("default")))
#else
#define ZKB_API
#endif

#define ZKB_OK 0
#define ZKB_ERR_CUDA (-1)    /* CUDA runtime failure or no device */
#define ZKB_ERR_ARG (-2)     /* invalid argument */
#define ZKB_ERR_ALLOC (-3)   /* device memory exhausted */
#define ZKB_ERR_STATE (-4)   /* call sequence violated */

typedef struct zkb_ctx zkb_ctx;

/* ---- context ------------------------------------------------------------------------------------------- */
/* Create a context on CUDA device `device` (one context per GPU / per process rank). */
ZKB_API int32_t zkb_init(int32_t device, zkb_ctx **out);
ZKB_API int32_t zkb_destroy(zkb_ctx *ctx);
ZKB_API const char *zkb_last_error(void);
/* ABI version of this header: major << 16 | minor */
ZKB_API uint32_t zkb_version(void);
/* Number of kernel launches issued through this context so far (bench.py's `gpu_launches`). */
ZKB_API uint64_t zkb_launch_count(const zkb_ctx *ctx);
ZKB_API int32_t zkb_sync(zkb_ctx *ctx);
/* Device time per kernel class, measured with CUDA event pairs on the launching stream (off by default).  cls: 0 ntt_tile_kernel,
 * 1 msm_acc_chunk_kernel, 2 expr_kernel.  zkb_prof_read synchronises on the recorded events; reset != 0 clears the counters. */
ZKB_API int32_t zkb_prof_enable(zkb_ctx *ctx, int32_t on);
ZKB_API int32_t zkb_prof_read(zkb_ctx *ctx, int32_t cls, uint64_t *launches, double *ms, int32_t reset);
/* Stream the context launches on (cudaStream_t as void*), for event timing by the caller. */
ZKB_API void *zkb_stream(zkb_ctx *ctx);

/* ---- device memory (thin wrappers so a non-CUDA host language can own device buffers) --------------------- */
ZKB_API int32_t zkb_malloc(zkb_ctx *ctx, uint64_t bytes, void **dptr);
ZKB_API int32_t zkb_free(zkb_ctx *ctx, void *dptr);
ZKB_API int32_t zkb_h2d(zkb_ctx *ctx, void *dst_dev, const void *src_host, uint64_t bytes);
ZKB_API int32_t zkb_d2h(zkb_ctx *ctx, void *dst_host, const void *src_dev, uint64_t bytes);

/* ---- NTT over Fr ------------------------------------------------------------------------------------------
 * Replaces halo2_proofs::arithmetic::best_fft(a: &mut [Fr], omega: Fr, log_n: u32)   (halo2_proofs 1.1.0 @ e5ddf67
 * src/arithmetic.rs) : in place, natural order in and out, a'[k] = sum_j a[j] * omega^(j k).  omega must have
 * order exactly 2^log_n.  If `scale` is non-NULL every output is additionally multiplied by *scale (Montgomery Fr) --
 * this fuses EvaluationDomain::ifft's `ifft_divisor` (src/poly/domain.rs `lagrange_to_coeff`, `extended_to_coeff`).
 * If `coset_zeta` != 0 the input coefficient i is first multiplied by ZETA^(i mod 3) (coset_zeta = 1) or
 * ZETA^(-(i mod 3)) applied to the OUTPUT (coset_zeta = 2), fusing `distribute_powers_zeta` of coeff_to_extended /
 * extended_to_coeff.                                                                                         */
ZKB_API int32_t zkb_ntt_fr_host(zkb_ctx *ctx, uint64_t *data_host, uint32_t log_n, const uint64_t omega[4],
                        const uint64_t *scale /* 4 limbs or NULL */, int32_t coset_zeta);
ZKB_API int32_t zkb_ntt_fr_dev(zkb_ctx *ctx, uint64_t *data_dev, uint32_t log_n, const uint64_t omega[4],
                       const uint64_t *scale /* HOST pointer, 4 limbs or NULL */, int32_t coset_zeta, void *stream);
/* `count` in-place transforms of one size through ONE kernel launch per pass (all columns of a prover stage): cols_dev is a HOST
 * array of `count` device pointers.                                                                                              */
ZKB_API int32_t zkb_ntt_fr_batch_dev(zkb_ctx *ctx, uint64_t *const *cols_dev, uint32_t count, uint32_t log_n, const uint64_t omega[4],
                                     const uint64_t *scale /* HOST pointer or NULL */, int32_t coset_zeta, void *stream);
/* omega_k = Fr::ROOT_OF_UNITY^(2^(28-k)) and its inverse (EvaluationDomain::new); host-side helper. */
ZKB_API int32_t zkb_fr_root_of_unity(uint32_t k, uint64_t omega[4], uint64_t omega_inv[4]);

/* ---- MSM over G1 -------------------------------------------------------------------------------------------
 * Replaces halo2_proofs::arithmetic::best_multiexp(coeffs: &[Fr], bases: &[G1Affine]) -> G1, the body of
 * ParamsKZG::commit / commit_lagrange (src/poly/kzg/commitment.rs).  out = sum_i coeffs[i] * bases[i].
 * The result is returned normalised: out_affine (64 B) and, if non-NULL, out_jacobian (96 B, z = 1 or identity) and
 * out_compressed (32 B, G1Affine::to_bytes: LE x with (y & 1) << 6 in byte 31; identity = zeros).               */
ZKB_API int32_t zkb_msm_g1_host(zkb_ctx *ctx, const uint64_t *scalars_host, const uint64_t *bases_host, uint64_t n,
                        uint64_t out_affine[8], uint64_t *out_jacobian, uint8_t *out_compressed);
ZKB_API int32_t zkb_msm_g1_dev(zkb_ctx *ctx, const uint64_t *scalars_dev, const uint64_t *bases_dev, uint64_t n,
                       uint64_t out_affine[8], uint64_t *out_jacobian, uint8_t *out_compressed, void *stream);
/* `batch` MSMs over the SAME bases in one pass (all advice columns of a phase are committed this way): scalar_cols_dev is a
 * HOST array of `batch` device pointers (n scalars each); out_affine receives batch x 8 limbs.                              */
ZKB_API int32_t zkb_msm_g1_batch_dev(zkb_ctx *ctx, const uint64_t *const *scalar_cols_dev, uint32_t batch,
                                     const uint64_t *bases_dev, uint64_t n, uint64_t *out_affine, void *stream);
/* Number of bucket additions + reduction additions the last MSM on this context performed (G1-adds metric). */
ZKB_API uint64_t zkb_msm_last_adds(const zkb_ctx *ctx);
/* Bucket-reduction levels beyond the first that the last MSM actually executed (decided on the device, no host round trip). */
ZKB_API uint32_t zkb_msm_last_levels(const zkb_ctx *ctx);

/* out[i] = [scalars[i]] * base, affine outputs (device buffers).  Used for ParamsKZG::setup / unsafe_setup_with_s
 * (g[i] = [s^i] G) and to synthesise distinct benchmark bases.                                                  */
ZKB_API int32_t zkb_g1_fixed_base_mul_dev(zkb_ctx *ctx, const uint64_t base_affine_host[8], const uint64_t *scalars_dev,
                                  uint64_t n, uint64_t *out_affine_dev, void *stream);

/* ---- SRS handle: ParamsKZG<Bn256> resident on the device ---------------------------------------------------------------
 * Replaces the prover-facing part of halo2_proofs::poly::kzg::commitment::ParamsKZG (src/poly/kzg/commitment.rs): the
 * reference loads one params file per degree (prover/src/utils.rs load_params, prover/src/common/prover.rs:37-57) and
 * `downsize`s it for smaller circuits (prover/src/common/prover.rs:54-55, aggregator/src/recursion/util.rs:156).
 * zkb_srs_load       upload g / g_lagrange (2^k x 64 B each, halo2curves G1Affine layout) ONCE per context; g_lagrange may be
 *                    NULL: it is then derived on the device by the inverse FFT over G1 (`g_to_lagrange`).  Memory permitting
 *                    (ZKB_MSM_SHIFT_GB, default 24) the window-shifted copies 2^(c w) P_i of both bases are built, which turns
 *                    every commitment into ONE bucket set with no Horner pass (msm.cu).
 * zkb_srs_downsize   ParamsKZG::downsize(new_k): g truncated to 2^new_k, g_lagrange recomputed; the source handle stays valid.
 * zkb_srs_commit_*   ParamsKZG::commit (basis 0, coefficients against g) / commit_lagrange (basis 1, values against g_lagrange);
 *                    n <= 2^k scalars; the result is normalised like zkb_msm_g1_*.
 * zkb_srs_read       copy one basis back to the host (tests, writing a downsized params file).                                    */
typedef struct zkb_srs zkb_srs;
ZKB_API int32_t zkb_srs_load(zkb_ctx *ctx, uint32_t k, const uint64_t *g_host, const uint64_t *g_lagrange_host, zkb_srs **out);
ZKB_API int32_t zkb_srs_load_dev(zkb_ctx *ctx, uint32_t k, const uint64_t *g_dev, const uint64_t *g_lagrange_dev, zkb_srs **out);
ZKB_API int32_t zkb_srs_destroy(zkb_srs *srs);
ZKB_API uint32_t zkb_srs_k(const zkb_srs *srs);
ZKB_API int32_t zkb_srs_downsize(zkb_srs *srs, uint32_t new_k, zkb_srs **out);
ZKB_API int32_t zkb_srs_read(zkb_srs *srs, int32_t basis, uint64_t *out_host);
ZKB_API int32_t zkb_srs_commit_dev(zkb_srs *srs, int32_t basis, const uint64_t *scalars_dev, uint64_t n, uint64_t out_affine[8],
                                   uint8_t *out_compressed, void *stream);
ZKB_API int32_t zkb_srs_commit_host(zkb_srs *srs, int32_t basis, const uint64_t *scalars_host, uint64_t n, uint64_t out_affine[8],
                                    uint8_t *out_compressed);
ZKB_API int32_t zkb_srs_commit_batch_dev(zkb_srs *srs, int32_t basis, const uint64_t *const *scalar_cols_dev, uint32_t batch, uint64_t n,
                                         uint64_t *out_affine, void *stream);

/* ---- element-wise field kernels (device buffers); field: 0 = Fr, 1 = Fq ------------------------------------
 * op: 0 add, 1 sub, 2 mul (binary);  unary op: 0 invert (0 -> 0), 1 canonical->Montgomery, 2 Montgomery->canonical,
 * 3 square, 4 negate.  These back Polynomial +,-,* and the unit tests of the device arithmetic.                  */
ZKB_API int32_t zkb_field_binop_dev(zkb_ctx *ctx, int32_t field, int32_t op, const uint64_t *a, const uint64_t *b,
                            uint64_t *out, uint64_t n, void *stream);
ZKB_API int32_t zkb_field_unop_dev(zkb_ctx *ctx, int32_t field, int32_t op, const uint64_t *a, uint64_t *out, uint64_t n,
                           void *stream);
/* Montgomery batch inversion (halo2 `BatchInvert` / batch_invert_assigned): out[i] = a[i]^-1, zeros stay zero. */
ZKB_API int32_t zkb_fr_batch_invert_dev(zkb_ctx *ctx, const uint64_t *a, uint64_t *out, uint64_t n, void *stream);

/* ---- polynomial utilities around MSM/NTT (device buffers) ----------------------------------------------------
 * zkb_fr_powers_dev        out[i] = base^i
 * zkb_poly_eval_dev        halo2_proofs::arithmetic::eval_polynomial for `num_polys` polynomials (host array of device
 *                          pointers, n coefficients each) at one point x; results (Montgomery) to out_host; synchronises.
 * zkb_fr_prefix_product_dev / _sum_dev   out[0] = init, out[i+1] = out[i] (*|+) in[i]  (n outputs; the running product z of
 *                          permutation/prover.rs and the running sum phi of mv_lookup/prover.rs)
 * zkb_kate_division_dev    halo2_proofs::arithmetic::kate_division: q = (a(X) - a(u)) / (X - u); q has n entries, q[n-1] = 0 */
ZKB_API int32_t zkb_fr_powers_dev(zkb_ctx *ctx, const uint64_t base[4], uint64_t n, uint64_t *out_dev, void *stream);
ZKB_API int32_t zkb_poly_eval_dev(zkb_ctx *ctx, const uint64_t *const *polys_dev, uint32_t num_polys, uint64_t n,
                                  const uint64_t x[4], uint64_t *out_host, void *stream);
ZKB_API int32_t zkb_fr_prefix_product_dev(zkb_ctx *ctx, const uint64_t *in_dev, uint64_t n, const uint64_t init[4],
                                          uint64_t *out_dev, void *stream);
ZKB_API int32_t zkb_fr_prefix_sum_dev(zkb_ctx *ctx, const uint64_t *in_dev, uint64_t n, const uint64_t init[4],
                                      uint64_t *out_dev, void *stream);
ZKB_API int32_t zkb_kate_division_dev(zkb_ctx *ctx, const uint64_t *a_dev, uint64_t n, const uint64_t u[4],
                                      uint64_t *q_dev, void *stream);

/* ---- multi-GPU building blocks (one process per GPU; collectives are issued by the host layer over NCCL) -----------------
 * zkb_ntt_cross_dev       size-p transform across ranks after the all-to-all of a domain-sharded NTT:
 *                         out[k][t] = sum_j in[j][t] * omega_p^(j k), in/out are p x len row-major, p in {1,2,4,8,16}
 * zkb_g1_sum_affine_host  sum of per-rank MSM partial results (host buffers, 64 B each); host-only, needs no device   */
ZKB_API int32_t zkb_ntt_cross_dev(zkb_ctx *ctx, const uint64_t *in_dev, uint64_t *out_dev, uint32_t p, uint64_t len,
                                  const uint64_t omega_p[4], void *stream);
ZKB_API int32_t zkb_g1_sum_affine_host(const uint64_t *points, uint64_t count, uint64_t out_affine[8], uint8_t *out_compressed);

/* zkb_ntt_fr_sharded_dev   ONE transform of size 2^log_n spread over the ranks of the communicator (north_star: "the k >= 26 domain
 *                          shards across the 8 GPUs"; zkb_comm_init first; COLLECTIVE).  n = P * M.  direction 0: in = this rank's
 *                          cyclic subsequence x[rank + P t] (M elements), out = the strip layout (row k1 * M/P + t holds
 *                          X[k1 M + rank M/P + t]); direction 1: strips in, cyclic out -- so forward (0) followed by the inverse root
 *                          and 1/n scale (1) is a round trip with no re-layout.  The twiddle multiply and the all-to-all are fused
 *                          into the store phase of the transform kernels: results go straight into the owner's window over NVLink
 *                          peer memory (cudaIpc-mapped); ZKB_SHARDED_EXCHANGE=nccl selects the ncclSend/ncclRecv baseline.
 * zkb_msm_g1_sharded_dev   point-range sharded MSM (aggregator/configs/compression_thin.config: 2^26 points over 8 GPUs): every rank
 *                          reduces its own slice, the 64-byte partial sums are all-gathered and added; same result on every rank. */
ZKB_API int32_t zkb_ntt_fr_sharded_dev(zkb_ctx *ctx, const uint64_t *in_dev, uint64_t *out_dev, uint32_t log_n, const uint64_t omega[4],
                                       const uint64_t *scale /* HOST pointer or NULL */, int32_t direction, void *stream);
ZKB_API int32_t zkb_msm_g1_sharded_dev(zkb_ctx *ctx, const uint64_t *scalars_shard_dev, const uint64_t *bases_shard_dev, uint64_t n_local,
                                       uint64_t out_affine[8], uint8_t *out_compressed, void *stream);

/* zkb_comm_*   NCCL communicator of a context for the multi-GPU create_proof (one process per GPU).  Rank 0 creates a
 * 128-byte unique id, the host layer broadcasts it, every rank calls zkb_comm_init.  With a communicator the proving session
 * stays replicated (identical transcript and proof bytes on every rank) while commitment batches (column i -> rank i mod P) and
 * the quotient's coset parts (part j -> rank j mod P) are dealt across the ranks and exchanged by one all-reduce each.        */
ZKB_API int32_t zkb_comm_unique_id(uint8_t out[128]);
ZKB_API int32_t zkb_comm_init(zkb_ctx *ctx, const uint8_t unique_id[128], int32_t rank, int32_t nranks);
ZKB_API int32_t zkb_comm_destroy(zkb_ctx *ctx);

/* ---- create_proof: device-resident proving session --------------------------------------------------------------
 * Replaces the body of halo2_proofs::plonk::create_proof::<KZGCommitmentScheme<Bn256>, ProverSHPLONK, Challenge255, R,
 * Blake2bWrite, C> (plonk/prover.rs; called at circuit-benchmarks/src/super_circuit.rs:117-132 and, through
 * snark_verifier_sdk::gen_snark_shplonk, at prover/src/common/prover/utils.rs:31).  `Circuit::synthesize`, the RNG and
 * vk.transcript_repr stay on the caller's side: advice columns arrive phase by phase already blinded (rows >= n - (bf+1)
 * random), blinding scalars for z / phi and the vanishing argument's random polynomial are passed in.
 *
 * CSF blob (little-endian u32 words) -- the flattened plonk::ConstraintSystem after selector compression and
 * chunk_lookups():  [0] magic 'ZSF1' 0x3146535a [1] k [2] num_fixed [3] num_advice [4] num_instance [5] num_challenges
 *   [6] blinding_factors [7] cs.degree() [8] num_phases [9] n_nodes [10] n_consts [11] n_gates [12] n_lookups
 *   [13] n_permutation_columns [14] n_advice_queries [15] n_fixed_queries [16] n_instance_queries [17] reserved, then
 *   advice_phase[num_advice], challenge_phase[num_challenges], nodes[n_nodes] x (op, a, b), consts[n_consts] x 8 (Fr,
 *   Montgomery), gates[n_gates] (node ids), per lookup: (n_input_sets, width, input node ids..., table node ids),
 *   permutation columns x (type, index), advice / fixed / instance queries x (column, rotation as i32).
 *   node ops: 0 CONST(a = const idx) 1 FIXED(a = col, b = rot) 2 ADVICE 3 INSTANCE 4 CHALLENGE(a = idx) 5 NEG(a)
 *   6 ADD(a, b) 7 MUL(a, b) 8 SCALED(a = node, b = const idx); children precede parents; column type codes 1/2/3.
 * zkb_pk_create      ProvingKey material: fixed and permutation-sigma column VALUES (host pointers, n x Fr each), SRS
 *                    g / g_lagrange (n x G1Affine); polynomial forms, l_0 / l_last / l_blind are derived on the device.
 * zkb_prove_begin    absorbs vk.transcript_repr and the instance values (KZG: QUERY_INSTANCE = false)
 * zkb_prove_advice_phase   commits the advice columns of `phase` (pointers of other phases are ignored), returns the
 *                    challenges squeezed after that phase in challenges_out[num_challenges][4] (Montgomery Fr)
 * zkb_prove_finish   lookups -> permutation -> vanishing -> quotient -> evaluations -> SHPLONK; z_blinds
 *                    [n_sets][bf], phi_blinds [n_lookups][bf], random_poly [n] are Montgomery Fr arrays on the host.
 *                    The first call runs the proof and keeps its bytes in the session: proof_out may be NULL (query the length) or
 *                    too short (ZKB_ERR_ARG, *proof_len set) -- call again with a buffer of *proof_len bytes; later calls only copy.
 *                    Multi-GPU sessions (zkb_comm_init): every zkb_pk_* / zkb_prove_* call, zkb_pk_vk_bytes included, is a COLLECTIVE
 *                    over the communicator and must be issued by all ranks in the same order; a rank-local failure (allocation, CUDA
 *                    error) leaves the other ranks inside a collective, so abort the job on any non-zero return.
 * zkb_prove_begin_multi  create_proof's `circuits: &[C]`: one proof of C >= 1 circuits under one proving key.  They share the
 *                    challenges, one quotient h (every circuit's constraints continue the same Horner chain in y), the random
 *                    polynomial and one SHPLONK opening.  Everything per circuit is CIRCUIT-MAJOR: instance_values / instance_lens hold
 *                    C * num_instance columns (circuit c's column i at c * num_instance + i); zkb_prove_advice_phase takes C * num_advice
 *                    pointers (circuit c's column j at c * num_advice + j); zkb_prove_upload_advice takes that same index; zkb_prove_finish
 *                    takes z_blinds [C][n_sets][bf], phi_blinds [C][n_lookups][bf] and ONE random_poly [n].  transcript_kind 0, 1, 2 as
 *                    zkb_prove_begin_ex (vt must be NULL), 3 = the caller's transcript through vt as zkb_prove_begin_cb.  num_circuits = 0
 *                    is ZKB_ERR_ARG; running out of device memory at any stage is ZKB_ERR_ALLOC.  The other zkb_prove_begin* entry
 *                    points are C = 1 and C = 1 here gives the same bytes as they do.                                                */
typedef struct zkb_pk zkb_pk;
typedef struct zkb_session zkb_session;
ZKB_API int32_t zkb_pk_create(zkb_ctx *ctx, const uint32_t *csf, uint64_t csf_words, const uint64_t *const *fixed_values,
                              const uint64_t *const *sigma_values, const uint64_t *g, const uint64_t *g_lagrange, zkb_pk **out);
/* Same against a loaded SRS handle (shared by every pk of the context; srs->k must equal the circuit's k: downsize first). */
ZKB_API int32_t zkb_pk_create_with_srs(zkb_ctx *ctx, const uint32_t *csf, uint64_t csf_words, const uint64_t *const *fixed_values,
                                       const uint64_t *const *sigma_values, zkb_srs *srs, zkb_pk **out);
/* keygen_pk2 / keygen_vk + keygen_pk (halo2_proofs plonk/keygen.rs; reference call site prover/src/common/prover/utils.rs:43-61,
 * :55): the caller runs Circuit::synthesize in keygen mode and hands over the fixed column values and the COPY CONSTRAINTS
 * (n_copies x 4 u32: left column, left row, right column, right row; columns index the CSF's permutation column list).  The
 * permutation Assembly (cycle merging, permutation/keygen.rs) runs on the host, the sigma columns delta^col * omega^row, every
 * polynomial / coset form and the vk commitments (zkb_pk_vk_bytes) are produced on the device.                                   */
ZKB_API int32_t zkb_keygen_pk(zkb_ctx *ctx, const uint32_t *csf, uint64_t csf_words, const uint64_t *const *fixed_values,
                              const uint32_t *copies, uint64_t n_copies, zkb_srs *srs, zkb_pk **out);
/* sigma column `column` of a proving key (Lagrange values, 2^k x 32 B) back to the host. */
ZKB_API int32_t zkb_pk_sigma_read(zkb_pk *pk, uint32_t column, uint64_t *out_host);
ZKB_API int32_t zkb_pk_destroy(zkb_pk *pk);
/* VerifyingKey bytes in SerdeFormat::Processed layout (u32 BE k || u32 BE num_fixed || fixed || permutation commitments,
 * compressed points; the layout of the reference fixture's vk).  out may be NULL to query the length.                     */
ZKB_API int32_t zkb_pk_vk_bytes(zkb_pk *pk, uint8_t *out, uint64_t cap, uint64_t *len);
/* Host-only structural validation of a CSF blob (no CUDA device needed); zkb_pk_create runs it first.                       */
ZKB_API int32_t zkb_csf_validate(const uint32_t *csf, uint64_t csf_words);
ZKB_API int32_t zkb_prove_begin(zkb_pk *pk, const uint64_t transcript_repr[4], const uint64_t *const *instance_values,
                                const uint32_t *instance_lens, zkb_session **out);
/* Same with a choice of transcript: 0 = Blake2bWrite/Challenge255 (the reference's benches, circuit-benchmarks/src/super_circuit.rs:112),
 * 1 = snark-verifier-sdk PoseidonTranscript<NativeLoader> (gen_snark_shplonk, prover/src/common/prover/utils.rs:31): Poseidon T=5,
 * RATE=4, R_F=8, R_P=60 over Fr; points absorbed as (x mod r, y mod r).  The Poseidon restatement is pinned by the reference's own
 * chunk proof (tests/test_fixture_proof.py);
 * 2 = snark-verifier EvmTranscript<G1Affine, NativeLoader> over Keccak-256 (gen_evm_proof_shplonk, prover/src/common/prover/evm.rs:67):
 * points absorbed AND written uncompressed as x || y big-endian (64 B), scalars 32 B big-endian, challenge = keccak256(buffer) mod r.   */
ZKB_API int32_t zkb_prove_begin_ex(zkb_pk *pk, int32_t transcript_kind, const uint64_t transcript_repr[4],
                                   const uint64_t *const *instance_values, const uint32_t *instance_lens, zkb_session **out);
/* 3 = THE CALLER'S transcript: create_proof is generic over `T: TranscriptWrite<G1Affine, Challenge255<G1Affine>>` (and the SDK
 * instantiates it with Blake2b, Poseidon and Keccak transcripts), and a generic type cannot cross a C ABI -- but its four
 * operations can.  The shim passes a table of extern "C" trampolines around the `&mut T` it was handed; the session then calls
 * exactly the sequence halo2's prover would (common_scalar for vk.transcript_repr and the instances, write_point per commitment,
 * squeeze_challenge, write_scalar per evaluation), so ANY transcript -- including ones this library has never seen -- produces its
 * own proof bytes on the Rust side and the RNG-free session needs no replay.  Scalars are Fr in halo2curves' Montgomery layout,
 * points G1Affine x || y; a callback returns 0 or an error code that aborts the session (ZKB_ERR_STATE).  In this mode
 * zkb_prove_finish reports proof_len = 0: the bytes live in the caller's writer.                                                */
typedef struct zkb_transcript_vtable {
    void *user;
    int32_t (*common_scalar)(void *user, const uint64_t scalar[4]);
    int32_t (*write_scalar)(void *user, const uint64_t scalar[4]);
    int32_t (*write_point)(void *user, const uint64_t point_xy[8]);
    int32_t (*squeeze_challenge)(void *user, uint64_t challenge_out[4]);
} zkb_transcript_vtable;
ZKB_API int32_t zkb_prove_begin_cb(zkb_pk *pk, const zkb_transcript_vtable *vt, const uint64_t transcript_repr[4],
                                   const uint64_t *const *instance_values, const uint32_t *instance_lens, zkb_session **out);
/* num_circuits circuits in one proof; see "zkb_prove_begin_multi" above zkb_pk_create.  (ABI 1.2) */
ZKB_API int32_t zkb_prove_begin_multi(zkb_pk *pk, int32_t transcript_kind, const zkb_transcript_vtable *vt,
                                      const uint64_t transcript_repr[4], uint32_t num_circuits,
                                      const uint64_t *const *instance_values, const uint32_t *instance_lens, zkb_session **out);
/* Host-only transcript primitives (no CUDA device needed; used by the CPU test-suite to pin the session's hashers):
 * zkb_poseidon_hash_host        absorb n Fr (Montgomery) into a fresh PoseidonTranscript sponge, squeeze one challenge
 * zkb_blake2b_challenge_host    feed bytes to a fresh Blake2b("Halo2-Transcript") state, squeeze one Challenge255 (mod r)
 * zkb_keccak256_host            Keccak-256 of a byte string (the EvmTranscript hash; eth-types KECCAK_CODE_HASH_EMPTY is its "" digest)
 * zkb_transcript_script_host    replay ops (0 common_scalar, 1 write_scalar, 2 write_point, 3 squeeze) through the session's transcript
 *                               code of `kind`; operands in order (scalar 4 limbs, point 8 limbs, Montgomery); returns the proof bytes
 *                               written and the squeezed challenges (4 limbs each); proof may be NULL to query the length          */
ZKB_API int32_t zkb_poseidon_hash_host(const uint64_t *inputs, uint64_t n, uint64_t out[4]);
ZKB_API int32_t zkb_blake2b_challenge_host(const uint8_t *bytes, uint64_t len, uint64_t out[4]);
ZKB_API int32_t zkb_keccak256_host(const uint8_t *bytes, uint64_t len, uint8_t out[32]);
ZKB_API int32_t zkb_transcript_script_host(int32_t kind, const uint8_t *ops, uint64_t n_ops, const uint64_t *operands, uint8_t *proof,
                                           uint64_t cap, uint64_t *proof_len, uint64_t *challenges);
ZKB_API int32_t zkb_prove_advice_phase(zkb_session *s, uint32_t phase, const uint64_t *const *advice_columns,
                                       uint64_t *challenges_out);
/* Witness-side overlap (SURVEY 8f row 4; zkevm-circuits/src/super_circuit.rs:714-806 assigns sub-circuit after sub-circuit): hand a
 * finished, blinded advice column over BEFORE its phase is submitted.  The H2D copy runs on the copy stream while the caller keeps
 * synthesising; zkb_prove_advice_phase then accepts NULL for that column.  The buffer must stay valid until the phase call.       */
ZKB_API int32_t zkb_prove_upload_advice(zkb_session *s, uint32_t column, const uint64_t *values);
ZKB_API int32_t zkb_prove_finish(zkb_session *s, const uint64_t *z_blinds, const uint64_t *phi_blinds,
                                 const uint64_t *random_poly, uint8_t *proof_out, uint64_t proof_cap, uint64_t *proof_len);
ZKB_API int32_t zkb_session_destroy(zkb_session *s);

#ifdef __cplusplus
}
#endif
#endif
