//! Raw bindings of include/kzg_bn254_b200.h (hand-written; bindgen would produce the same).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
pub struct kzgb_ctx {
    _private: [u8; 0],
}

#[repr(C)]
pub struct kzgb_group {
    _private: [u8; 0],
}

pub const KZGB_OK: c_int = 0;
pub const KZGB_ERR_GENERIC: c_int = -1;
pub const KZGB_ERR_SRS_CAPACITY: c_int = -2;
pub const KZGB_ERR_SERIALIZATION: c_int = -3;
pub const KZGB_ERR_FFT: c_int = -4;
pub const KZGB_ERR_NOT_ON_CURVE: c_int = -5;
pub const KZGB_ERR_MSM: c_int = -6;
pub const KZGB_ERR_INVALID_INPUT_LENGTH: c_int = -7;
pub const KZGB_ERR_DESERIALIZATION: c_int = -8;
pub const KZGB_ERR_INVALID_FIELD_ELEMENT: c_int = -9;
pub const KZGB_ERR_DEVICE: c_int = -100;

extern "C" {
    pub fn kzgb_ctx_create(out: *mut *mut kzgb_ctx, device: c_int, stream: *mut c_void) -> c_int;
    pub fn kzgb_ctx_destroy(ctx: *mut kzgb_ctx);
    pub fn kzgb_last_error(ctx: *const kzgb_ctx) -> *const c_char;
    pub fn kzgb_srs_load_file(ctx: *mut kzgb_ctx, path: *const c_char, order: u32, points_to_load: u32) -> c_int;
    pub fn kzgb_srs_save_cache(ctx: *mut kzgb_ctx, path: *const c_char) -> c_int;
    pub fn kzgb_srs_load_cache(ctx: *mut kzgb_ctx, path: *const c_char, points_to_load: u32) -> c_int;
    pub fn kzgb_srs_precompute(ctx: *mut kzgb_ctx, max_n: usize, window_bits: c_int) -> c_int;
    pub fn kzgb_srs_prepare_lagrange(ctx: *mut kzgb_ctx, n: usize) -> c_int;
    pub fn kzgb_srs_prepare_all_roots(ctx: *mut kzgb_ctx, n: usize) -> c_int;
    pub fn kzgb_srs_load_affine_mont(ctx: *mut kzgb_ctx, xy: *const u64, inf: *const u8, n: usize) -> c_int;
    pub fn kzgb_srs_len(ctx: *const kzgb_ctx) -> usize;
    pub fn kzgb_srs_get_affine_mont(ctx: *mut kzgb_ctx, start: usize, count: usize, out_xy: *mut u64, out_inf: *mut u8) -> c_int;
    pub fn kzgb_msm_var(ctx: *mut kzgb_ctx, bases_xy: *const u64, bases_inf: *const u8, scalars: *const u64, m: usize,
                        out_xy: *mut u64, out_inf: *mut u8) -> c_int;
    pub fn kzgb_roots_of_unity(ctx: *mut kzgb_ctx, length_of_data_after_padding: u64, out: *mut u64, out_capacity: usize, n_out: *mut usize) -> c_int;
    pub fn kzgb_ntt_fr(ctx: *mut kzgb_ctx, inout: *mut u64, n: usize, inverse: c_int) -> c_int;
    pub fn kzgb_commit_eval(ctx: *mut kzgb_ctx, evals: *const u64, n: usize, out_xy: *mut u64, out_inf: *mut u8) -> c_int;
    pub fn kzgb_commit_coeff(ctx: *mut kzgb_ctx, coeffs: *const u64, n: usize, out_xy: *mut u64, out_inf: *mut u8) -> c_int;
    pub fn kzgb_commit_blob(ctx: *mut kzgb_ctx, blob: *const u8, len: usize, out_xy: *mut u64, out_inf: *mut u8) -> c_int;
    pub fn kzgb_g1_ifft(ctx: *mut kzgb_ctx, n: usize, out_xy: *mut u64, out_inf: *mut u8) -> c_int;
    pub fn kzgb_compute_proof(ctx: *mut kzgb_ctx, evals: *const u64, n: usize, z: *const u64, out_xy: *mut u64,
                              out_inf: *mut u8, y_out: *mut u64) -> c_int;
    pub fn kzgb_compute_proofs_all_roots(ctx: *mut kzgb_ctx, evals: *const u64, n: usize, out_xy: *mut u64,
                                         out_inf: *mut u8) -> c_int;
    pub fn kzgb_compute_blob_proof(ctx: *mut kzgb_ctx, blob: *const u8, len: usize, c_xy: *const u64, c_inf: u8,
                                   out_xy: *mut u64, out_inf: *mut u8) -> c_int;
    pub fn kzgb_commit_and_prove_blobs(ctx: *mut kzgb_ctx, blobs: *const *const u8, lens: *const usize, count: usize,
                                       commitments32: *mut u8, proofs32: *mut u8) -> c_int;
    pub fn kzgb_commit_blobs(ctx: *mut kzgb_ctx, blobs: *const *const u8, lens: *const usize, count: usize, out_xy: *mut u64,
                             out_inf: *mut u8) -> c_int;
    pub fn kzgb_commit_blobs_dev(ctx: *mut kzgb_ctx, blobs_dev: *const *const u8, lens: *const usize, count: usize,
                                 out_xy: *mut u64, out_inf: *mut u8) -> c_int;
    pub fn kzgb_verify_proof_g1(ctx: *mut kzgb_ctx, c_xy: *const u64, c_inf: u8, proof_xy: *const u64, proof_inf: u8, y: *const u64,
                                out_xy: *mut u64, out_inf: *mut u8) -> c_int;
    pub fn kzgb_verify_blob_proof_g1(ctx: *mut kzgb_ctx, blob: *const u8, len: usize, c_xy: *const u64, c_inf: u8, proof_xy: *const u64,
                                     proof_inf: u8, out_xy: *mut u64, out_inf: *mut u8, z_out: *mut u64, y_out: *mut u64) -> c_int;
    // multi-GPU group (one handle over several GPUs of the box)
    pub fn kzgb_group_create(out: *mut *mut kzgb_group, devices: *const c_int, n_devices: c_int) -> c_int;
    pub fn kzgb_group_destroy(group: *mut kzgb_group);
    pub fn kzgb_group_size(group: *const kzgb_group) -> c_int;
    pub fn kzgb_group_ctx(group: *mut kzgb_group, member: c_int) -> *mut kzgb_ctx;
    pub fn kzgb_group_last_error(group: *const kzgb_group) -> *const c_char;
    pub fn kzgb_group_srs_load_file(group: *mut kzgb_group, path: *const c_char, order: u32, points_to_load: u32) -> c_int;
    pub fn kzgb_group_srs_load_affine_mont(group: *mut kzgb_group, xy: *const u64, inf: *const u8, n: usize) -> c_int;
    pub fn kzgb_group_srs_prepare_lagrange(group: *mut kzgb_group, n: usize) -> c_int;
    pub fn kzgb_group_srs_precompute_ranges(group: *mut kzgb_group, n: usize, window_bits: c_int) -> c_int;
    pub fn kzgb_group_commit_and_prove_blobs(group: *mut kzgb_group, blobs: *const *const u8, lens: *const usize, count: usize,
                                             commitments32: *mut u8, proofs32: *mut u8) -> c_int;
    pub fn kzgb_group_commit_blobs(group: *mut kzgb_group, blobs: *const *const u8, lens: *const usize, count: usize,
                                   out_xy: *mut u64, out_inf: *mut u8) -> c_int;
    pub fn kzgb_group_compute_blob_proofs(group: *mut kzgb_group, blobs: *const *const u8, lens: *const usize, count: usize,
                                          commitments_xy: *const u64, commitments_inf: *const u8, out_xy: *mut u64,
                                          out_inf: *mut u8) -> c_int;
    pub fn kzgb_group_compute_proofs(group: *mut kzgb_group, evals: *const *const u64, ns: *const usize, count: usize,
                                     zs_mont: *const u64, out_xy: *mut u64, out_inf: *mut u8, ys_mont: *mut u64) -> c_int;
    pub fn kzgb_group_commit_evals(group: *mut kzgb_group, evals: *const *const u64, ns: *const usize, count: usize,
                                   out_xy: *mut u64, out_inf: *mut u8) -> c_int;
    pub fn kzgb_group_commit_coeffs(group: *mut kzgb_group, coeffs: *const *const u64, ns: *const usize, count: usize,
                                    out_xy: *mut u64, out_inf: *mut u8) -> c_int;
    pub fn kzgb_group_verify_blob_proofs_g1(group: *mut kzgb_group, blobs: *const *const u8, lens: *const usize, count: usize,
                                            commitments_xy: *const u64, commitments_inf: *const u8, proofs_xy: *const u64,
                                            proofs_inf: *const u8, out_xy: *mut u64, out_inf: *mut u8, z_out: *mut u64,
                                            y_out: *mut u64) -> c_int;
    pub fn kzgb_set_g2_tau(ctx: *mut kzgb_ctx, xy: *const u64) -> c_int;
    pub fn kzgb_group_set_g2_tau(group: *mut kzgb_group, xy: *const u64) -> c_int;
    pub fn kzgb_verify_proofs(ctx: *mut kzgb_ctx, count: usize, commitments_xy: *const u64, commitments_inf: *const u8,
                              proofs_xy: *const u64, proofs_inf: *const u8, zs_mont: *const u64, ys_mont: *const u64,
                              ok: *mut u8) -> c_int;
    pub fn kzgb_verify_blob_proofs(ctx: *mut kzgb_ctx, blobs: *const *const u8, lens: *const usize, count: usize,
                                   commitments_xy: *const u64, commitments_inf: *const u8, proofs_xy: *const u64,
                                   proofs_inf: *const u8, ok: *mut u8) -> c_int;
    pub fn kzgb_verify_blob_proofs_dev(ctx: *mut kzgb_ctx, blobs_dev: *const *const u8, blobs_host: *const *const u8,
                                       lens: *const usize, count: usize, commitments_xy: *const u64,
                                       commitments_inf: *const u8, proofs_xy: *const u64, proofs_inf: *const u8,
                                       ok: *mut u8) -> c_int;
    pub fn kzgb_group_verify_blob_proofs(group: *mut kzgb_group, blobs: *const *const u8, lens: *const usize, count: usize,
                                         commitments_xy: *const u64, commitments_inf: *const u8, proofs_xy: *const u64,
                                         proofs_inf: *const u8, ok: *mut u8) -> c_int;
    pub fn kzgb_group_msm_srs(group: *mut kzgb_group, scalars: *const u64, n: usize, out_xy: *mut u64, out_inf: *mut u8) -> c_int;
    pub fn kzgb_verify_batch_rlc(ctx: *mut kzgb_ctx, blobs: *const *const u8, lens: *const usize, count: usize,
                                 commitments_xy: *const u64, commitments_inf: *const u8, proofs_xy: *const u64,
                                 proofs_inf: *const u8, lhs_xy: *mut u64, lhs_inf: *mut u8, rhs_xy: *mut u64,
                                 rhs_inf: *mut u8) -> c_int;
    pub fn kzgb_verify_batch_rlc_dev(ctx: *mut kzgb_ctx, blobs_dev: *const *const u8, blobs_host: *const *const u8,
                                     lens: *const usize, count: usize, commitments_xy: *const u64, commitments_inf: *const u8,
                                     proofs_xy: *const u64, proofs_inf: *const u8, lhs_xy: *mut u64, lhs_inf: *mut u8,
                                     rhs_xy: *mut u64, rhs_inf: *mut u8) -> c_int;
    pub fn kzgb_verify_kzg_proof_batch_rlc(ctx: *mut kzgb_ctx, count: usize, commitments_xy: *const u64,
                                           commitments_inf: *const u8, proofs_xy: *const u64, proofs_inf: *const u8,
                                           zs_mont: *const u64, ys_mont: *const u64, poly_lens: *const u64,
                                           lhs_xy: *mut u64, lhs_inf: *mut u8, rhs_xy: *mut u64, rhs_inf: *mut u8) -> c_int;
    pub fn kzgb_group_verify_batch_rlc(group: *mut kzgb_group, blobs: *const *const u8, lens: *const usize, count: usize,
                                       commitments_xy: *const u64, commitments_inf: *const u8, proofs_xy: *const u64,
                                       proofs_inf: *const u8, lhs_xy: *mut u64, lhs_inf: *mut u8, rhs_xy: *mut u64,
                                       rhs_inf: *mut u8) -> c_int;
}
