//! Raw bindings of include/zkb200.h (ABI version 1.1).  Field elements and points cross as `*const u64` / `*mut u64`:
//! halo2curves' `Fr`, `Fq` are `#[repr(transparent)]` over `[u64; 4]` (Montgomery form) and `G1Affine` is `{ x: Fq, y: Fq }`, so
//! `slice.as_ptr() as *const u64` needs no conversion (layout checked against the reference fixture in tests/test_oracle_golden.py).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_void};

#[repr(C)] pub struct zkb_ctx { _p: [u8; 0] }
#[repr(C)] pub struct zkb_srs { _p: [u8; 0] }
#[repr(C)] pub struct zkb_pk { _p: [u8; 0] }
#[repr(C)] pub struct zkb_session { _p: [u8; 0] }

/// create_proof's generic `T: TranscriptWrite` as four C callbacks (see gpu/transcript.rs)
#[repr(C)]
pub struct zkb_transcript_vtable {
    pub user: *mut c_void,
    pub common_scalar: unsafe extern "C" fn(user: *mut c_void, scalar: *const u64) -> i32,
    pub write_scalar: unsafe extern "C" fn(user: *mut c_void, scalar: *const u64) -> i32,
    pub write_point: unsafe extern "C" fn(user: *mut c_void, point_xy: *const u64) -> i32,
    pub squeeze_challenge: unsafe extern "C" fn(user: *mut c_void, challenge_out: *mut u64) -> i32,
}

extern "C" {
    // context
    pub fn zkb_init(device: i32, out: *mut *mut zkb_ctx) -> i32;
    pub fn zkb_destroy(ctx: *mut zkb_ctx) -> i32;
    pub fn zkb_last_error() -> *const c_char;
    pub fn zkb_version() -> u32;
    pub fn zkb_sync(ctx: *mut zkb_ctx) -> i32;
    // arithmetic::best_fft / best_multiexp
    pub fn zkb_ntt_fr_host(ctx: *mut zkb_ctx, data: *mut u64, log_n: u32, omega: *const u64, scale: *const u64, coset_zeta: i32) -> i32;
    pub fn zkb_msm_g1_host(ctx: *mut zkb_ctx, scalars: *const u64, bases: *const u64, n: u64, out_affine: *mut u64, out_jacobian: *mut u64,
                           out_compressed: *mut u8) -> i32;
    // ParamsKZG
    pub fn zkb_srs_load(ctx: *mut zkb_ctx, k: u32, g: *const u64, g_lagrange: *const u64, out: *mut *mut zkb_srs) -> i32;
    pub fn zkb_srs_downsize(srs: *mut zkb_srs, new_k: u32, out: *mut *mut zkb_srs) -> i32;
    pub fn zkb_srs_read(srs: *mut zkb_srs, basis: i32, out_host: *mut u64) -> i32;
    pub fn zkb_srs_commit_host(srs: *mut zkb_srs, basis: i32, scalars: *const u64, n: u64, out_affine: *mut u64, out_compressed: *mut u8) -> i32;
    pub fn zkb_srs_destroy(srs: *mut zkb_srs) -> i32;
    // keygen / proving key
    pub fn zkb_csf_validate(csf: *const u32, csf_words: u64) -> i32;
    pub fn zkb_keygen_pk(ctx: *mut zkb_ctx, csf: *const u32, csf_words: u64, fixed: *const *const u64, copies: *const u32, n_copies: u64,
                         srs: *mut zkb_srs, out: *mut *mut zkb_pk) -> i32;
    pub fn zkb_pk_create_with_srs(ctx: *mut zkb_ctx, csf: *const u32, csf_words: u64, fixed: *const *const u64, sigma: *const *const u64,
                                  srs: *mut zkb_srs, out: *mut *mut zkb_pk) -> i32;
    pub fn zkb_pk_vk_bytes(pk: *mut zkb_pk, out: *mut u8, cap: u64, len: *mut u64) -> i32;
    pub fn zkb_pk_destroy(pk: *mut zkb_pk) -> i32;
    // create_proof
    pub fn zkb_prove_begin_ex(pk: *mut zkb_pk, kind: i32, transcript_repr: *const u64, instances: *const *const u64, lens: *const u32,
                              out: *mut *mut zkb_session) -> i32;
    pub fn zkb_prove_begin_cb(pk: *mut zkb_pk, vt: *const zkb_transcript_vtable, transcript_repr: *const u64, instances: *const *const u64,
                              lens: *const u32, out: *mut *mut zkb_session) -> i32;
    pub fn zkb_prove_begin_multi(pk: *mut zkb_pk, kind: i32, vt: *const zkb_transcript_vtable, transcript_repr: *const u64, num_circuits: u32,
                                 instances: *const *const u64, lens: *const u32, out: *mut *mut zkb_session) -> i32;
    pub fn zkb_prove_advice_phase(s: *mut zkb_session, phase: u32, advice: *const *const u64, challenges_out: *mut u64) -> i32;
    pub fn zkb_prove_finish(s: *mut zkb_session, z_blinds: *const u64, phi_blinds: *const u64, random_poly: *const u64, proof_out: *mut u8,
                            cap: u64, len: *mut u64) -> i32;
    pub fn zkb_session_destroy(s: *mut zkb_session) -> i32;
    // multi-GPU (one process per GPU)
    pub fn zkb_comm_unique_id(out: *mut u8) -> i32;
    pub fn zkb_comm_init(ctx: *mut zkb_ctx, unique_id: *const u8, rank: i32, nranks: i32) -> i32;
    pub fn zkb_ntt_fr_sharded_dev(ctx: *mut zkb_ctx, in_dev: *const u64, out_dev: *mut u64, log_n: u32, omega: *const u64, scale: *const u64,
                                  direction: i32, stream: *mut c_void) -> i32;
    pub fn zkb_msm_g1_sharded_dev(ctx: *mut zkb_ctx, scalars_dev: *const u64, bases_dev: *const u64, n_local: u64, out_affine: *mut u64,
                                  out_compressed: *mut u8, stream: *mut c_void) -> i32;
}
