/*
 * kzg_bn254_b200 -- C ABI of the B200-native engine for the commitment hot path of
 * Layr-Labs/rust-kzg-bn254 (BN254 G1 MSM over the SRS, Fr (I)NTT, and the Fr glue of
 * KZG::commit_* / compute_blob_proof / the RLC step of verify_blob_kzg_proof_batch).
 *
 * The reference has no FFI of its own (pure Rust on arkworks); each entry point below cites
 * the reference interface it replaces (paths relative to the reference repo).  A Rust shim
 * (INTEGRATION.md) binds these with `extern "C"` and keeps the crates' public API.
 *
 * Conventions
 *  - Fr / Fq : 4 x u64 little-endian limbs in MONTGOMERY form (R = 2^256) -- the in-memory
 *    layout of arkworks' Fp<MontBackend<_,4>,4>, so `&[Fr]` passes as `*const u64`.
 *  - G1 affine : x || y (8 x u64, Montgomery), identity = all-zero words (the shim maps
 *    arkworks' `infinity: bool` to/from this).
 *  - Compressed G1 in SRS files: gnark big-endian 32 B (primitives/src/helpers.rs:175-226).
 *  - All host buffers are caller-owned; the library copies in/out and never keeps a host
 *    pointer after return.  `_dev` variants take CUDA device pointers instead.
 *  - Return value: KZGB_OK (0) or a negative kzgb_status that maps 1:1 onto the reference's
 *    KzgError variants (primitives/src/errors.rs:32-86); kzgb_last_error() has the message
 *    text the reference uses.
 *  - A context is bound to one CUDA device; calls on one context are serialised internally.
 *    There is no CPU fallback: every call fails with KZGB_ERR_DEVICE if the GPU is unusable.
 */
#ifndef KZG_BN254_B200_H
#define KZG_BN254_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct kzgb_ctx kzgb_ctx;
typedef struct kzgb_group kzgb_group; /* several GPUs of one box behind one handle, see "multi-GPU" below */

typedef enum kzgb_status {
    KZGB_OK = 0,
    KZGB_ERR_GENERIC = -1,               /* KzgError::GenericError(String) */
    KZGB_ERR_SRS_CAPACITY = -2,          /* KzgError::SrsCapacityExceeded { polynomial_len, srs_len } (kzg.rs:89-94) */
    KZGB_ERR_SERIALIZATION = -3,         /* KzgError::SerializationError (kzg.rs:112-116) */
    KZGB_ERR_FFT = -4,                   /* KzgError::FFTError (kzg.rs:265-269) */
    KZGB_ERR_NOT_ON_CURVE = -5,          /* KzgError::NotOnCurveError (helpers.rs:694-708, :204-209) */
    KZGB_ERR_MSM = -6,                   /* KzgError::MsmError / CommitError (helpers.rs:332, kzg.rs:102) */
    KZGB_ERR_INVALID_INPUT_LENGTH = -7,  /* KzgError::InvalidInputLength (helpers.rs:485-487) */
    KZGB_ERR_DESERIALIZATION = -8,       /* KzgError::DeserializationError (helpers.rs:176-195) */
    KZGB_ERR_INVALID_FIELD_ELEMENT = -9, /* KzgError::InvalidFieldElement (helpers.rs:784-811) */
    KZGB_ERR_DEVICE = -100               /* CUDA failure -> KzgError::GenericError(<cuda string>) */
} kzgb_status;

/* ---- context ------------------------------------------------------------------------- */
/* device: CUDA ordinal.  stream: optional cudaStream_t to run on (NULL = the context creates its own). */
int kzgb_ctx_create(kzgb_ctx** out, int device, void* stream);
void kzgb_ctx_destroy(kzgb_ctx* ctx);
const char* kzgb_last_error(const kzgb_ctx* ctx);
/* Block until all work queued by this context has finished. */
int kzgb_sync(kzgb_ctx* ctx);

/* ---- SRS (prover/src/srs.rs:11-49 `SRS`, `SRS::new`) ------------------------------------ */
/* Load the first `points_to_load` points of a g1.point file (32 B gnark-BE each).  Replaces
 * SRS::new(path, order, points_to_load) (srs.rs:35-49) incl. its `points_to_load > order` error.
 * Streamed: chunks of 2^22 points are read into pinned memory while the previous chunk is copied and
 * decompressed on the GPU (the reference reads 32 bytes per syscall, srs.rs:154-188). */
int kzgb_srs_load_file(kzgb_ctx* ctx, const char* path, uint32_t order, uint32_t points_to_load);
/* On-disk cache of the DECOMPRESSED points (64-byte header + 64 B x||y Montgomery per point): written
 * from the resident SRS, loaded without the per-point square root (each point is still checked to be on
 * the curve on the GPU).  points_to_load = 0 loads the whole cache; more than the cache holds is the
 * same error as SRS::new's order check. */
int kzgb_srs_save_cache(kzgb_ctx* ctx, const char* path);
int kzgb_srs_load_cache(kzgb_ctx* ctx, const char* path, uint32_t points_to_load);
/* Same from memory (replaces parallel_read_g1_points + read_g1_point_from_bytes_be, srs.rs:81-138). */
int kzgb_srs_load_gnark_be(kzgb_ctx* ctx, const uint8_t* bytes, size_t n_points);
/* From an existing `SRS.g1` slice: n x (x||y) Montgomery words; inf[i] != 0 marks the identity (may be NULL). */
int kzgb_srs_load_affine_mont(kzgb_ctx* ctx, const uint64_t* xy, const uint8_t* inf, size_t n_points);
/* Synthetic SRS_i = tau^i * G generated on the GPU (benches/tests; tau: 4 words Montgomery). */
int kzgb_srs_load_synthetic(kzgb_ctx* ctx, const uint64_t tau_mont[4], size_t n_points);
/* Point range of the same synthetic SRS: local point i is tau^(first+i) * G (point-range sharding of one
 * large MSM across GPUs: each rank holds only its own range). */
int kzgb_srs_load_synthetic_range(kzgb_ctx* ctx, const uint64_t tau_mont[4], size_t first, size_t n_points);
/* Number of monomial points resident (== SRS.g1.len()). */
size_t kzgb_srs_len(const kzgb_ctx* ctx);
/* Read back decompressed points [start, start+count) to fill `SRS.g1` (pub field, srs.rs:13). */
int kzgb_srs_get_affine_mont(kzgb_ctx* ctx, size_t start, size_t count, uint64_t* out_xy, uint8_t* out_inf);
/* Build the fixed-base window tables (2^(c*w) * P_i) for MSMs of up to `max_n` points.  Called lazily
 * by the first commit if the caller does not; window_bits = 0 picks c from max_n. */
int kzgb_srs_precompute(kzgb_ctx* ctx, size_t max_n, int window_bits);
/* The same over SRS points [first, first + count) only: the table of one member's share of a point-range-sharded
 * MSM (kzgb_group_srs_precompute_ranges).  A context holds one monomial window table at a time. */
int kzgb_srs_precompute_range(kzgb_ctx* ctx, size_t first, size_t count, int window_bits);
/* dst gets a copy of src's resident SRS points, device to device (a peer copy over NVLink when the contexts sit
 * on different GPUs).  src must not be reloaded while the call runs. */
int kzgb_srs_clone(kzgb_ctx* dst, kzgb_ctx* src);
/* Build the Lagrange-basis window table for evaluation-form polynomials of exactly n = 2^k elements:
 * L = IFFT_G1(SRS[..n]) -- the points KZG::commit_eval_form recomputes with g1_ifft on EVERY call
 * (kzg.rs:98) -- computed once per size on the GPU and kept resident with their window shifts, so that
 * commit_eval_form / commit_blob / compute_proof* are one MSM on the evaluations themselves with no
 * Fr NTT on the path.  Policy when the caller does not call this: the table of a size is built by the k-th
 * evaluation-form commitment / proof of that size (option "lagrange_after", default 2; a batch of b blobs counts
 * b) -- a one-off commit of a new size is not charged a G1 NTT (12 ms at n = 64, 0.5 s at 2^19); tables are kept
 * within a memory budget (option "lagrange_budget_mib", default half of the device memory), least recently used
 * dropped first; domains above 2^22 never get one.  Without the table the same group element comes from
 * Fr-IFFT + the monomial table.  Err KZGB_ERR_FFT / KZGB_ERR_SRS_CAPACITY as kzgb_g1_ifft; KZGB_ERR_DEVICE if the
 * table cannot be built (switched off, above 2^22, over the budget). */
int kzgb_srs_prepare_lagrange(kzgb_ctx* ctx, size_t n);
/* Build the per-size table of kzgb_compute_proofs_all_roots ahead of the first call: s_hat = DFT_2n of SRS[..n-1]
 * reversed and zero-padded (2n x 64 B, 64 MiB at n = 2^19; one forward G1 NTT of 2n points).  Kept until the SRS
 * changes; the first call of a size builds it when the caller does not.  Errors as kzgb_compute_proofs_all_roots;
 * KZGB_ERR_GENERIC for n > 2^22, where nothing is kept and every call builds its own. */
int kzgb_srs_prepare_all_roots(kzgb_ctx* ctx, size_t n);

/* ---- MSM (ark-ec VariableBaseMSM::msm call sites) ---------------------------------------- */
/* sum scalars[i] * SRS[i], i < n.  Replaces G1Projective::msm(&srs.g1[..n], coeffs) in
 * KZG::commit_coeff_form (prover/src/kzg.rs:107-125). */
int kzgb_msm_srs(kzgb_ctx* ctx, const uint64_t* scalars_mont, size_t n, uint64_t out_xy[8], uint8_t* out_inf);
/* Same over a point range [first, first+n) of the SRS (point-range sharding of a large MSM). */
int kzgb_msm_srs_range(kzgb_ctx* ctx, const uint64_t* scalars_mont, size_t first, size_t n, uint64_t out_xy[8],
                       uint8_t* out_inf);
/* Same with the scalars already resident in device memory (n x 4 words, Montgomery). */
int kzgb_msm_srs_range_dev(kzgb_ctx* ctx, const uint64_t* scalars_dev, size_t first, size_t n, uint64_t out_xy[8],
                           uint8_t* out_inf);
/* out_dev[i] = base^(first_exponent + i), Montgomery, written to DEVICE memory (helpers::compute_powers,
 * primitives/src/helpers.rs:298-314; also the synthetic scalars of the MSM benchmark). */
int kzgb_fr_powers_dev(kzgb_ctx* ctx, const uint64_t base_mont[4], size_t first_exponent, size_t n, uint64_t* out_dev);
/* Variable-base MSM.  Replaces helpers::g1_lincomb (primitives/src/helpers.rs:328-337). */
int kzgb_msm_var(kzgb_ctx* ctx, const uint64_t* bases_xy, const uint8_t* bases_inf, const uint64_t* scalars_mont,
                 size_t m, uint64_t out_xy[8], uint8_t* out_inf);
/* Adds two affine points on the host side of the library (partial-sum reduction of sharded MSMs). */
int kzgb_g1_add(const uint64_t a_xy[8], uint8_t a_inf, const uint64_t b_xy[8], uint8_t b_inf, uint64_t out_xy[8],
                uint8_t* out_inf);

/* ---- roots of unity (helpers::calculate_roots_of_unity, primitives/src/helpers.rs:553-610; KZG::calculate_and_store_roots_of_unity,
 * prover/src/kzg.rs:65-72) ---- */
/* w^0 .. w^(n-1), Montgomery, n = next_pow2(ceil(length_of_data_after_padding / 32)); *n_out = n.  out == NULL only queries n.
 * Errors (GenericError) with the reference's texts: "Length of data after padding is 0", "the length of data after padding is
 * not valid with respect to the SRS". */
int kzgb_roots_of_unity(kzgb_ctx* ctx, uint64_t length_of_data_after_padding, uint64_t* out_mont, size_t out_capacity,
                        size_t* n_out);

/* ---- Fr (I)NTT (ark-poly fft/ifft at primitives/src/polynomial.rs:131-135, 242-246) -------- */
/* In place, natural order in and out; n must be a power of two (<= 2^28). inverse != 0 -> ifft (with 1/n). */
int kzgb_ntt_fr(kzgb_ctx* ctx, uint64_t* inout_mont, size_t n, int inverse);

/* ---- bytes <-> Fr (primitives/src/helpers.rs:40-57 to_fr_array, :80-119 to_byte_array) ----- */
/* out has ceil(len/32) elements */
int kzgb_to_fr_array(kzgb_ctx* ctx, const uint8_t* bytes, size_t len, uint64_t* out_mont);
int kzgb_to_byte_array(kzgb_ctx* ctx, const uint64_t* fr_mont, size_t n, uint8_t* out_be);

/* ---- commitments (prover/src/kzg.rs) ------------------------------------------------------ */
/* KZG::commit_eval_form (kzg.rs:84-104): n evaluations (power of two).  Err KZGB_ERR_SRS_CAPACITY if n > srs_len. */
int kzgb_commit_eval(kzgb_ctx* ctx, const uint64_t* evals_mont, size_t n, uint64_t out_xy[8], uint8_t* out_inf);
/* KZG::commit_coeff_form (kzg.rs:107-125).  Err KZGB_ERR_SERIALIZATION if n > srs_len. */
int kzgb_commit_coeff(kzgb_ctx* ctx, const uint64_t* coeffs_mont, size_t n, uint64_t out_xy[8], uint8_t* out_inf);
/* KZG::commit_eval_form (kzg.rs:84-104) for `count` polynomials in one pipelined call.  Polynomial i is ns[i] evaluations
 * (Montgomery) at evals_mont[i], HOST memory.  out_xy: count x 8 words (x||y Montgomery); out_inf: count flags, may be NULL.
 * Entry i is exactly what kzgb_commit_eval(evals_mont[i], ns[i], ...) returns.  Checks, entry by entry in index order, in
 * kzgb_commit_eval's order: ns[i] <= srs_len (KZGB_ERR_SRS_CAPACITY), then ns[i] a power of two (KZGB_ERR_FFT "length
 * provided is not a power of 2").  The error of the lowest failing entry is returned before any work starts and the outputs
 * are left untouched.  The evaluation words are not validated, as in kzgb_commit_eval.  count == 0 writes nothing.
 * Polynomials of up to 2^17 values are committed in groups of one size, whatever their order in the batch (one batched
 * launch set per group); larger ones one per lane, as kzgb_commit_eval commits them. */
int kzgb_commit_evals(kzgb_ctx* ctx, const uint64_t* const* evals_mont, const size_t* ns, size_t count,
                      uint64_t* out_xy, uint8_t* out_inf);
/* Same with the evaluations in device memory (evals_dev[i]: ns[i] x 4 words), read in place; the outputs and the checks as
 * kzgb_commit_evals. */
int kzgb_commit_evals_dev(kzgb_ctx* ctx, const uint64_t* const* evals_dev, const size_t* ns, size_t count,
                          uint64_t* out_xy, uint8_t* out_inf);
/* KZG::commit_coeff_form (kzg.rs:107-125) for `count` polynomials in one pipelined call.  Polynomial i is ns[i]
 * coefficients (Montgomery) at coeffs_mont[i], HOST memory, of any length (no power of two needed; ns[i] == 0 commits to
 * the identity).  out_xy / out_inf as kzgb_commit_evals.  Entry i is exactly what kzgb_commit_coeff(coeffs_mont[i], ns[i],
 * ...) returns.  Check, entry by entry in index order: ns[i] <= srs_len, else KZGB_ERR_SERIALIZATION "polynomial length is
 * not correct"; the lowest failing entry's error is returned before any work starts, outputs untouched.  The coefficient
 * words are not validated, as in kzgb_commit_coeff.  count == 0 writes nothing.  Polynomials whose next power of two N is at
 * most 2^17 and srs_len are committed in groups of one N (zero-padded to N): one batched MSM over the monomial window
 * table, or one batched forward Fr NTT and one batched MSM over the Lagrange table of size N when that table is resident
 * and has the narrower window; the others one per lane over SRS[0, ns[i]), as kzgb_commit_coeff commits them. */
int kzgb_commit_coeffs(kzgb_ctx* ctx, const uint64_t* const* coeffs_mont, const size_t* ns, size_t count,
                       uint64_t* out_xy, uint8_t* out_inf);
/* Same with the coefficients in device memory (coeffs_dev[i]: ns[i] x 4 words), read in place; the outputs and the checks
 * as kzgb_commit_coeffs. */
int kzgb_commit_coeffs_dev(kzgb_ctx* ctx, const uint64_t* const* coeffs_dev, const size_t* ns, size_t count,
                           uint64_t* out_xy, uint8_t* out_inf);
/* KZG::commit_blob (kzg.rs:182-185): blob.data() bytes (32 B big-endian elements). */
int kzgb_commit_blob(kzgb_ctx* ctx, const uint8_t* blob, size_t len, uint64_t out_xy[8], uint8_t* out_inf);
/* KZG::g1_ifft (kzg.rs:263-285): Lagrange-basis SRS of size n (natural order).  Err KZGB_ERR_FFT if n is not 2^k. */
int kzgb_g1_ifft(kzgb_ctx* ctx, size_t n, uint64_t* out_xy, uint8_t* out_inf);

/* ---- proofs ------------------------------------------------------------------------------- */
/* KZG::compute_proof / compute_proof_impl (kzg.rs:128-178, 215-234): evaluation-form polynomial,
 * caller-supplied z (Montgomery).  Optionally returns y = p(z) (Montgomery) if y_out != NULL. */
int kzgb_compute_proof(kzgb_ctx* ctx, const uint64_t* evals_mont, size_t n, const uint64_t z_mont[4],
                       uint64_t out_xy[8], uint8_t* out_inf, uint64_t y_out[4]);
/* KZG::compute_proof / compute_proof_impl / compute_proof_with_known_z_fr_index (kzg.rs:128-178, 187-234) for `count`
 * polynomials, each at a point the caller chooses, in one pipelined call.  Polynomial i is ns[i] evaluations (Montgomery)
 * at evals_mont[i], HOST memory; z_i is the 4 words at zs_mont + 4 i (Montgomery, host memory).  out_xy: count x 8 words
 * (x||y Montgomery); out_inf: count flags, may be NULL; ys_mont: count x 4 words, y_i = p_i(z_i) (Montgomery), may be
 * NULL.  Entry i is exactly what kzgb_compute_proof(evals_mont[i], ns[i], z_i, ..., y_out) returns, for z_i inside the
 * domain (the quotient of compute_quotient_eval_on_domain, kzg.rs:237-260) and outside it.  Checks, entry by entry in
 * index order: ns[i] a power of two (KZGB_ERR_FFT "length provided is not a power of 2"), ns[i] <= srs_len
 * (KZGB_ERR_SRS_CAPACITY), z_i a reduced Montgomery word, below r (KZGB_ERR_INVALID_FIELD_ELEMENT, the message names i; the
 * single call does not check this, kzgb_verify_proofs demands it of the same z).  The error of the lowest failing entry is
 * returned before any work starts and the outputs are left untouched.  The evaluation words are not validated, as in
 * kzgb_compute_proof.  count == 0 writes nothing.  The batch has no per-instance roots of unity, so the reference's
 * roots-length check (kzg.rs:135-139) is not made. */
int kzgb_compute_proofs(kzgb_ctx* ctx, const uint64_t* const* evals_mont, const size_t* ns, size_t count,
                        const uint64_t* zs_mont, uint64_t* out_xy, uint8_t* out_inf, uint64_t* ys_mont);
/* Same with the evaluations in device memory (evals_dev[i]: ns[i] x 4 words), read in place; z, the outputs and the checks
 * as kzgb_compute_proofs. */
int kzgb_compute_proofs_dev(kzgb_ctx* ctx, const uint64_t* const* evals_dev, const size_t* ns, size_t count,
                            const uint64_t* zs_mont, uint64_t* out_xy, uint8_t* out_inf, uint64_t* ys_mont);
/* KZG::compute_proof_with_known_z_fr_index (kzg.rs:187-207) at EVERY index: out proof i (x||y Montgomery, n x 8 words;
 * out_inf n flags, may be NULL) is the point kzgb_compute_proof(evals, n, w^i) returns.  FK20: one Toeplitz product in G1
 * (two G1 FFTs + 2n scalar multiplications) instead of n MSMs.  Errors and their order as kzgb_compute_proof: KZGB_ERR_FFT
 * (n not 2^k), KZGB_ERR_SRS_CAPACITY (n > srs_len), GenericError "power must be <= 28" (2n > 2^28), KZGB_ERR_DEVICE. */
int kzgb_compute_proofs_all_roots(kzgb_ctx* ctx, const uint64_t* evals_mont, size_t n, uint64_t* out_xy, uint8_t* out_inf);
/* helpers::evaluate_polynomial_in_evaluation_form (primitives/src/helpers.rs:475-535). */
int kzgb_evaluate_polynomial(kzgb_ctx* ctx, const uint64_t* evals_mont, size_t n, const uint64_t z_mont[4],
                             uint64_t y_out[4]);
/* helpers::compute_challenge (helpers.rs:411-472): Fiat-Shamir z for (blob, commitment). */
int kzgb_compute_challenge(kzgb_ctx* ctx, const uint8_t* blob, size_t len, const uint64_t c_xy[8], uint8_t c_inf,
                           uint64_t z_out_mont[4]);
/* KZG::compute_blob_proof (kzg.rs:288-309): validates the commitment, derives z, proves. */
int kzgb_compute_blob_proof(kzgb_ctx* ctx, const uint8_t* blob, size_t len, const uint64_t c_xy[8], uint8_t c_inf,
                            uint64_t out_xy[8], uint8_t* out_inf);

/* ---- batches (blob-sharded hot path) ------------------------------------------------------ */
/* commit_blob + compute_blob_proof for `count` blobs, pipelined (H2D, GPU, host SHA-256 overlap).  The batch has no
 * per-instance roots of unity, so the reference's roots-length check (kzg.rs:135-139) is not made.
 * commitments / proofs: count x 32 B arkworks `serialize_compressed` bytes (the encoding the
 * reference feeds to its transcripts, helpers.rs:457-461).  Blob pointers are HOST memory. */
int kzgb_commit_and_prove_blobs(kzgb_ctx* ctx, const uint8_t* const* blobs, const size_t* lens, size_t count,
                                uint8_t* commitments32, uint8_t* proofs32);
/* Same with blob bytes already resident in device memory (host copies are still needed for the
 * SHA-256 transcript; pass them in `blobs_host`). */
int kzgb_commit_and_prove_blobs_dev(kzgb_ctx* ctx, const uint8_t* const* blobs_dev, const uint8_t* const* blobs_host,
                                    const size_t* lens, size_t count, uint8_t* commitments32, uint8_t* proofs32);
/* KZG::commit_blob (kzg.rs:182-185) for `count` blobs, pipelined; no proofs, no transcripts.  out_xy: count x 8 words
 * (x||y Montgomery), out_inf: count flags (may be NULL).  Blob i's point and every error are those of kzgb_commit_blob
 * on blob i alone; all blobs are checked before any work starts.  count == 0 writes nothing. */
int kzgb_commit_blobs(kzgb_ctx* ctx, const uint8_t* const* blobs, const size_t* lens, size_t count,
                      uint64_t* out_xy, uint8_t* out_inf);
/* Same with the blob bytes in device memory (no host copy needed: nothing is hashed). */
int kzgb_commit_blobs_dev(kzgb_ctx* ctx, const uint8_t* const* blobs_dev, const size_t* lens, size_t count,
                          uint64_t* out_xy, uint8_t* out_inf);
/* KZG::compute_blob_proof (kzg.rs:288-309) for `count` blobs with caller-supplied commitments, pipelined (H2D, GPU, host
 * SHA-256 overlap); no commitment is computed.  commitments_xy: count x 8 words (x||y Montgomery), commitments_inf: count
 * flags (may be NULL).  out_xy / out_inf as kzgb_commit_blobs.  Proof i and every error are those of
 * kzgb_compute_blob_proof on (blob i, commitment i) alone: blob by blob in index order, the commitment on the curve
 * (KZGB_ERR_NOT_ON_CURVE; the identity is valid), the length not 0 (GenericError "Length of data after padding is 0"),
 * the SRS large enough (KZGB_ERR_SRS_CAPACITY); the error of the lowest-index blob that fails is returned before any
 * work starts and the outputs are left untouched.  count == 0 writes nothing.  Like kzgb_commit_and_prove_blobs, the
 * batch has no per-instance roots of unity, so the reference's roots-length check (kzg.rs:135-139) is not made. */
int kzgb_compute_blob_proofs(kzgb_ctx* ctx, const uint8_t* const* blobs, const size_t* lens, size_t count,
                             const uint64_t* commitments_xy, const uint8_t* commitments_inf,
                             uint64_t* out_xy, uint8_t* out_inf);
/* Same with the blob bytes in device memory; host copies are still needed for the SHA-256 transcripts (pass them in
 * `blobs_host`, as for kzgb_commit_and_prove_blobs_dev). */
int kzgb_compute_blob_proofs_dev(kzgb_ctx* ctx, const uint8_t* const* blobs_dev, const uint8_t* const* blobs_host,
                                 const size_t* lens, size_t count, const uint64_t* commitments_xy,
                                 const uint8_t* commitments_inf, uint64_t* out_xy, uint8_t* out_inf);

/* ---- batch verification, everything before the pairing (verifier/src/batch.rs:16-249) ------ */
/* Per-blob challenge z_i and evaluation y_i (helpers.rs:613-662), RLC scalar r and its powers
 * (batch.rs:76-168), and the three linear combinations (batch.rs:225-249).  Outputs the two G1
 * inputs of the final pairing check e(lhs, [tau]G2) == e(rhs, G2) (batch.rs:253-254), which stays
 * in the reference's code.  Points in/out: x||y Montgomery + identity flags. */
int kzgb_verify_batch_rlc(kzgb_ctx* ctx, const uint8_t* const* blobs, const size_t* lens, size_t count,
                          const uint64_t* commitments_xy, const uint8_t* commitments_inf, const uint64_t* proofs_xy,
                          const uint8_t* proofs_inf, uint64_t lhs_xy[8], uint8_t* lhs_inf, uint64_t rhs_xy[8],
                          uint8_t* rhs_inf);
/* Same with the blob bytes in device memory, read in place.  Host copies are still needed for the SHA-256 transcripts
 * (blobs_host), as for kzgb_verify_blob_proofs_g1_dev.  Checks, their order, errors and outputs are the host form's. */
int kzgb_verify_batch_rlc_dev(kzgb_ctx* ctx, const uint8_t* const* blobs_dev, const uint8_t* const* blobs_host,
                              const size_t* lens, size_t count, const uint64_t* commitments_xy, const uint8_t* commitments_inf,
                              const uint64_t* proofs_xy, const uint8_t* proofs_inf, uint64_t lhs_xy[8], uint8_t* lhs_inf,
                              uint64_t rhs_xy[8], uint8_t* rhs_inf);
/* verify_kzg_proof_batch (batch.rs:185-249) up to the pairing: the random linear combination of kzgb_verify_batch_rlc
 * over `count` openings the caller has already evaluated (z_i, y_i = p_i(z_i)), with no blob and no per-blob hashing.
 * zs_mont / ys_mont: count x 4 words Montgomery each, as kzgb_verify_blob_proofs_g1 returns them.  poly_lens[i]: the
 * padded polynomial length n_i that the transcript hashes (batch.rs:48-54), hashed as given -- for a blob of len bytes,
 * next_pow2(ceil(len / 32)).  lhs / rhs: as kzgb_verify_batch_rlc defines them.  Checks, all before any work: the 2m
 * points on the curve as kzgb_verify_batch_rlc checks them (KZGB_ERR_NOT_ON_CURVE), then every z_i and y_i below r
 * (KZGB_ERR_INVALID_FIELD_ELEMENT: an arkworks Fr always is, and a larger word would hash other bytes than the
 * reference's).  count == 0 writes the identity to both outputs.  commitments_inf / proofs_inf may be NULL. */
int kzgb_verify_kzg_proof_batch_rlc(kzgb_ctx* ctx, size_t count, const uint64_t* commitments_xy,
                                    const uint8_t* commitments_inf, const uint64_t* proofs_xy, const uint8_t* proofs_inf,
                                    const uint64_t* zs_mont, const uint64_t* ys_mont, const uint64_t* poly_lens,
                                    uint64_t lhs_xy[8], uint8_t* lhs_inf, uint64_t rhs_xy[8], uint8_t* rhs_inf);

/* ---- point codecs (host) ------------------------------------------------------------------ */
/* arkworks CanonicalSerialize::serialize_compressed of a G1Affine (helpers.rs:458-460). */
int kzgb_g1_serialize_compressed(const uint64_t xy[8], uint8_t inf, uint8_t out32[32]);
/* gnark big-endian compressed (the g1.point format). */
int kzgb_g1_to_gnark_be(const uint64_t xy[8], uint8_t inf, uint8_t out32[32]);
/* helpers::validate_g1_point (helpers.rs:694-708) for `n` points on the GPU. */
int kzgb_validate_g1_points(kzgb_ctx* ctx, const uint64_t* xy, const uint8_t* inf, size_t n);

/* Process-wide switches that never change results, only which exact code path produces them:
 *   "fs_device"            -1 auto (default), 0 host SHA-256 pool, 1 device kernel for the per-blob
 *                          Fiat-Shamir challenges of kzgb_verify_batch_rlc and kzgb_verify_blob_proofs_g1{,_dev}
 *                          (auto: >= 256 blobs of <= 2^13 Fr)
 *   "acc_waves"            waves of bucket-accumulation blocks the sorted list is cut into (default 4; any value >= 1
 *                          gives the same result -- tests use it to move the chunk boundaries)
 *   "fs_force_generic"     1: the device-hashed challenges of kzgb_verify_batch_rlc are all flagged "in the domain", so the
 *                          per-polynomial choice made on the device takes the generic inverses everywhere (tests)
 *   "eval_structured"      1 (default): for z outside the domain the barycentric denominators 1/(z - w_i) come from
 *                          the factorisation of z^n - 1 (~3 multiplications each); 0: generic prefix/suffix products
 *   "srs_chunk_points"     points per chunk of the streamed SRS ingest (0 = default 2^22)
 *   "group"                -1 (default): kzgb_commit_and_prove_blobs processes runs of equal-size blobs of
 *                          <= 2^17 Fr as groups (one batched launch set per phase and group, sized so a group
 *                          holds <= 2^21 Fr and <= 64 blobs); 0: one blob at a time; k > 0: k blobs per group
 *   "lagrange"             1 (default): evaluation-form commits/proofs build and use the Lagrange-basis
 *                          table of their size (kzgb_srs_prepare_lagrange); 0: Fr-IFFT + monomial table
 *   "lagrange_after", "lagrange_budget_mib"   the table policy described at kzgb_srs_prepare_lagrange
 *   "lanes"                lanes (host thread + streams) of the blob-batch pipelines, 0 = the library's choice
 *   "hash_threads"         host SHA-256 pool threads of a batch call, 0 = the library's choice
 *   "lane_wait"            how a lane thread waits for its MSM: 0 spins on the stream, 1 polls an event with short sleeps, 2 sleeps on a
 *                          blocking event; -1 (default): deep large-blob batches (>= 32 blobs, or >= 4 when cores are plentiful) run 6
 *                          lanes in mode 2, everything else spins -- or polls when the lane threads of the ranks on this host
 *                          outnumber half of its hardware threads
 *   "stream_priority"      1 (default): bucket accumulation runs on a low-priority stream of its lane
 *   "l2_fetch_64"          1 (default): contexts that own their stream set the device's L2 fetch granularity to 64 B
 *                          (random 64-byte gathers) and restore it when the last of them is destroyed
 *   "batch_keep_mib"       blob staging memory kept between batch calls (default 4096)
 *   "pipelined_upload"     1 (default): kzgb_msm_srs / kzgb_msm_srs_range calls of >= 2^22 points over a window table upload
 *                          their host scalars in 4 or 8 chunks, each chunk's sort + bucket accumulation overlapping the next
 *                          chunk's copy (bucket sums folded, one reduction); 0: one copy, then one MSM
 *   "ntt_kernel"           Fr (I)NTT implementation: 0 passes through shared-memory tiles, 1 warp-resident passes (registers, warp
 *                          shuffles, bulk asynchronous tile loads), -1 (default) by shape (1 for large batches of transforms of
 *                          <= 2^13, where it is 27 % faster; 0 elsewhere, where it is up to 12 % faster) -- same results
 *   "hash_mb"              -1 (default): kzgb_commit_and_prove_blobs (and kzgb_compute_blob_proofs, where the groups the batch forms
 *                          also hash faster than the pool, behind a single-stream head) hashes the transcripts of a large-blob batch sixteen at a time on
 *                          AVX-512 (multi-buffer SHA-256: ~2x the bytes per second of a core's SHA-NI, the 16 digests arrive together)
 *                          when the single-stream pool of this context's share of the host is slower than the GPU and >= 32 blobs
 *                          of exactly 32 * 2^j bytes are in the batch; 0: never; 1: whenever a group of >= 8 forms
 *   "hash_nice"            1 (default): the SHA-256 pool threads of a batch call run at nice 19, so a waking lane thread preempts them
 *   "hash_trace"           1: every multi-buffer group reports its wall and CPU time on stderr
 *   "device_hash"          -1 (default): kzgb_commit_and_prove_blobs / kzgb_compute_blob_proofs decide how many transcripts of a large-blob batch are
 *                          hashed on the device next to the host pool (none unless the host cannot keep up even with "hash_mb" and
 *                          the batch is several hundred blobs deep); 0: none; k > 0: the last k eligible blobs
 *   "device_hash_lanes"    device kernel for those: 0 one warp per transcript (0.45 s, 16 % of a blob's MSM work each), 1 one lane per
 *                          transcript (0.9 s, 0.5 %), -1 (default): whichever the batch's depth favours
 *   "fs_quad"              1 (default): four lanes per blob in the device-side Fiat-Shamir hashing
 * The library reads NO environment variables of its own (torchrun's LOCAL_WORLD_SIZE is consulted for the "lane_wait" and "hash_mb"
 * auto decisions: how many ranks share this host's hardware threads).
 * Unknown names return KZGB_ERR_GENERIC. */
int kzgb_set_option(const char* name, long value);
/* ---- single-proof verification up to the pairing (verifier/src/verify.rs) ---------------------------------------------
 * verify_proof (verify.rs:10-75), the G1 side: commitment and proof validated (validate_g1_point, :18-22; BN254 G1 has
 * cofactor 1, so on-curve is the subgroup check), out = C - [y] G1 (:37-42).  The caller's reference code computes
 * [tau - z] G2 and runs pairings_verify(out, G2, proof, [tau - z] G2) (:44-74).  Err KZGB_ERR_NOT_ON_CURVE. */
int kzgb_verify_proof_g1(kzgb_ctx* ctx, const uint64_t c_xy[8], uint8_t c_inf, const uint64_t proof_xy[8], uint8_t proof_inf,
                         const uint64_t y_mont[4], uint64_t out_xy[8], uint8_t* out_inf);
/* verify_blob_kzg_proof (verify.rs:77-115) up to the pairing: validation, z = compute_challenge(blob, C), y = p(z)
 * (barycentric evaluation on the GPU), then kzgb_verify_proof_g1.  z_out / y_out (Montgomery, may be NULL) are what the
 * caller needs for [tau - z] G2. */
int kzgb_verify_blob_proof_g1(kzgb_ctx* ctx, const uint8_t* blob, size_t len, const uint64_t c_xy[8], uint8_t c_inf,
                              const uint64_t proof_xy[8], uint8_t proof_inf, uint64_t out_xy[8], uint8_t* out_inf,
                              uint64_t z_out[4], uint64_t y_out[4]);
/* verify_blob_kzg_proof (verify.rs:77-115) up to the pairing for `count` blobs.  out i / z i / y i are what
 * kzgb_verify_blob_proof_g1 returns for (blob i, commitment i, proof i) alone: out = C_i - [y_i] G1 (count x 8 words,
 * x||y Montgomery; out_inf count flags, may be NULL), z_i = compute_challenge(blob i, C_i), y_i = p_i(z_i) (count x 4
 * words Montgomery each, either may be NULL).  Checks, blob by blob in index order: C_i and proof_i on the curve
 * (KZGB_ERR_NOT_ON_CURVE; the identity is valid), length not 0 (GenericError "Length of data after padding is 0"),
 * polynomial length <= 2^28 (GenericError "Input size exceeds maximum polynomial size").  The error of the lowest-index
 * blob that fails is returned before any work starts, and the outputs are left untouched.  count == 0 writes nothing.
 * No SRS is needed.  commitments_inf / proofs_inf may be NULL (no identity among them).  The challenges are hashed as
 * kzgb_verify_batch_rlc hashes them (option "fs_device"); C_i - [y_i] G1 is one GPU thread per blob.  out_xy may be NULL
 * (then out_inf is ignored): only z and y are computed, which is what the RLC over the openings needs
 * (kzgb_verify_kzg_proof_batch_rlc); checks and errors are the same. */
int kzgb_verify_blob_proofs_g1(kzgb_ctx* ctx, const uint8_t* const* blobs, const size_t* lens, size_t count,
                               const uint64_t* commitments_xy, const uint8_t* commitments_inf,
                               const uint64_t* proofs_xy, const uint8_t* proofs_inf,
                               uint64_t* out_xy, uint8_t* out_inf, uint64_t* z_out, uint64_t* y_out);
/* Same with the blob bytes in device memory.  Host copies are still needed for the SHA-256 transcripts (blobs_host),
 * as for kzgb_compute_blob_proofs_dev. */
int kzgb_verify_blob_proofs_g1_dev(kzgb_ctx* ctx, const uint8_t* const* blobs_dev, const uint8_t* const* blobs_host,
                                   const size_t* lens, size_t count, const uint64_t* commitments_xy,
                                   const uint8_t* commitments_inf, const uint64_t* proofs_xy, const uint8_t* proofs_inf,
                                   uint64_t* out_xy, uint8_t* out_inf, uint64_t* z_out, uint64_t* y_out);

/* ---- per-opening verification through the pairing (verifier/src/verify.rs:10-115) ---------------------------------
 * Each opening (C, pi, z, y) is checked as e(C - [y]G1 + [z]pi, G2) * e(-pi, [tau]G2) == 1 -- by bilinearity the bool of
 * the reference's e(C - [y]G1, G2) == e(pi, [tau - z]G2) -- on the GPU, one thread per opening: the lines of the Miller
 * loop of both fixed G2 points are precomputed on the host once per context, the final exponentiation runs per opening.
 * ok[i] is the bool verify_proof / verify_blob_kzg_proof returns for entry i alone, under this context's [tau]G2.
 * If [z_i]G2 == [tau]G2 for some i (the reference's check of [tau - z]G2 = O, verify.rs:55-59), the call returns
 * KZGB_ERR_GENERIC "Evaluation point equals trusted setup secret" for the lowest such i.  On any error `ok` is left
 * untouched.  count == 0 writes nothing; commitments_inf / proofs_inf may be NULL (no identity among them).  No SRS is
 * needed.  The single final pairing of verify_blob_kzg_proof_batch (kzgb_verify_batch_rlc) is not one of these: it
 * stays in the reference's code. */
/* [tau]G2 of this context's pairing checks: x.c0, x.c1, y.c0, y.c1 (4 words each, Montgomery; Fq2 = c0 + c1 u,
 * u^2 = -1 -- the memory layout of arkworks' G2Affine without its flag).  NULL restores the default, the reference's
 * G2_TAU (primitives/src/consts.rs:55-64).  Off the twist, the identity, or outside the order-r subgroup:
 * KZGB_ERR_NOT_ON_CURVE "Invalid trusted setup: G2_TAU not on curve"; the setting is unchanged.  Loading an SRS does
 * not change it. */
int kzgb_set_g2_tau(kzgb_ctx* ctx, const uint64_t xy[16]);
/* verify_proof (verify.rs:10-75) for `count` openings: ok[i] = 1 if the pairing check of (C_i, pi_i, z_i, y_i) holds,
 * else 0.  zs_mont / ys_mont: count x 4 words Montgomery each.  Checks, all before any work: the 2m points on the curve
 * as kzgb_verify_kzg_proof_batch_rlc checks them (KZGB_ERR_NOT_ON_CURVE), then every z_i and y_i below r
 * (KZGB_ERR_INVALID_FIELD_ELEMENT). */
int kzgb_verify_proofs(kzgb_ctx* ctx, size_t count, const uint64_t* commitments_xy, const uint8_t* commitments_inf,
                       const uint64_t* proofs_xy, const uint8_t* proofs_inf, const uint64_t* zs_mont,
                       const uint64_t* ys_mont, uint8_t* ok);
/* verify_blob_kzg_proof (verify.rs:77-115) for `count` blobs, through the pairing: z_i and y_i as
 * kzgb_verify_blob_proofs_g1 computes them (hashing as option "fs_device" says), then the pairing check of each opening
 * while z and y are still on the device.  Checks, their order, codes and messages: those of kzgb_verify_blob_proofs_g1
 * (points on the curve, length not 0, polynomial length <= 2^28, the lowest failing index first). */
int kzgb_verify_blob_proofs(kzgb_ctx* ctx, const uint8_t* const* blobs, const size_t* lens, size_t count,
                            const uint64_t* commitments_xy, const uint8_t* commitments_inf,
                            const uint64_t* proofs_xy, const uint8_t* proofs_inf, uint8_t* ok);
/* Same with the blob bytes in device memory, read in place; host copies feed the SHA-256 transcripts (blobs_host). */
int kzgb_verify_blob_proofs_dev(kzgb_ctx* ctx, const uint8_t* const* blobs_dev, const uint8_t* const* blobs_host,
                                const size_t* lens, size_t count, const uint64_t* commitments_xy,
                                const uint8_t* commitments_inf, const uint64_t* proofs_xy, const uint8_t* proofs_inf,
                                uint8_t* ok);

/* ---- multi-GPU: one handle over several GPUs of one box (SURVEY.md 8e) ------------------------------------
 * The path shards by blob (batches) and by point range (one large MSM) and has no exchange step besides adding
 * G partial sums of 64 bytes, which happens on the host: one process, one host thread per GPU for the duration of
 * a call, no collective library needed.  A caller of KZG::commit_blob in a loop (prover/src/kzg.rs:182-185) or of a
 * 2^26-coefficient KZG::commit_coeff_form (kzg.rs:107-125) reaches every GPU of the box through these.
 * devices == NULL or n_devices <= 0: every visible device.  A device may be listed more than once (independent
 * contexts on one GPU).  The SRS is decompressed ONCE (member 0) and replicated device to device. */
int kzgb_group_create(kzgb_group** out, const int* devices, int n_devices);
void kzgb_group_destroy(kzgb_group* group);
int kzgb_group_size(const kzgb_group* group);
/* Member context (owned by the group): for per-GPU calls such as kzgb_msm_config or kzgb_stats. */
kzgb_ctx* kzgb_group_ctx(kzgb_group* group, int member);
const char* kzgb_group_last_error(const kzgb_group* group);
int kzgb_group_sync(kzgb_group* group);
/* SRS::new and friends, as the kzgb_srs_load_* of a context. */
int kzgb_group_srs_load_file(kzgb_group* group, const char* path, uint32_t order, uint32_t points_to_load);
int kzgb_group_srs_load_cache(kzgb_group* group, const char* path, uint32_t points_to_load);
int kzgb_group_srs_load_gnark_be(kzgb_group* group, const uint8_t* bytes, size_t n_points);
int kzgb_group_srs_load_affine_mont(kzgb_group* group, const uint64_t* xy, const uint8_t* inf, size_t n_points);
int kzgb_group_srs_load_synthetic(kzgb_group* group, const uint64_t tau_mont[4], size_t n_points);
/* kzgb_srs_prepare_lagrange on every member. */
int kzgb_group_srs_prepare_lagrange(kzgb_group* group, size_t n);
/* Fixed-base window tables for kzgb_group_msm_srs calls of n points: member i over its own share of the points
 * (1/G of the table memory per GPU). */
int kzgb_group_srs_precompute_ranges(kzgb_group* group, size_t n, int window_bits);
/* kzgb_commit_and_prove_blobs with the batch cut into contiguous shares of about equal bytes, one per member;
 * byte-identical to the single-context call. */
int kzgb_group_commit_and_prove_blobs(kzgb_group* group, const uint8_t* const* blobs, const size_t* lens, size_t count,
                                      uint8_t* commitments32, uint8_t* proofs32);
/* kzgb_commit_blobs cut into contiguous shares of about equal bytes, one per member; identical to the one-context call.
 * Each member checks its own share before it starts. */
int kzgb_group_commit_blobs(kzgb_group* group, const uint8_t* const* blobs, const size_t* lens, size_t count,
                            uint64_t* out_xy, uint8_t* out_inf);
/* kzgb_compute_blob_proofs cut into contiguous shares of about equal bytes, one per member; identical to the one-context
 * call.  Each member checks its own share before it starts (so on an error, members with valid shares may have written
 * their proofs). */
int kzgb_group_compute_blob_proofs(kzgb_group* group, const uint8_t* const* blobs, const size_t* lens, size_t count,
                                   const uint64_t* commitments_xy, const uint8_t* commitments_inf,
                                   uint64_t* out_xy, uint8_t* out_inf);
/* kzgb_compute_proofs (KZG::compute_proof, kzg.rs:128-178, 187-234) cut into contiguous shares of about equal evaluation
 * bytes (32 ns[i] per polynomial), one per member; identical to the one-context call.  Each member checks its own share
 * before it starts (so on an error, members with valid shares may have written their outputs). */
int kzgb_group_compute_proofs(kzgb_group* group, const uint64_t* const* evals_mont, const size_t* ns, size_t count,
                              const uint64_t* zs_mont, uint64_t* out_xy, uint8_t* out_inf, uint64_t* ys_mont);
/* kzgb_commit_evals (KZG::commit_eval_form, kzg.rs:84-104) and kzgb_commit_coeffs (KZG::commit_coeff_form, kzg.rs:107-125)
 * cut into contiguous shares of about equal bytes (32 ns[i] per polynomial), one per member; identical to the one-context
 * call.  Each member checks its own share before it starts (so on an error, members with valid shares may have written
 * their outputs). */
int kzgb_group_commit_evals(kzgb_group* group, const uint64_t* const* evals_mont, const size_t* ns, size_t count,
                            uint64_t* out_xy, uint8_t* out_inf);
int kzgb_group_commit_coeffs(kzgb_group* group, const uint64_t* const* coeffs_mont, const size_t* ns, size_t count,
                             uint64_t* out_xy, uint8_t* out_inf);
/* kzgb_verify_blob_proofs_g1 cut into contiguous shares of about equal bytes, one per member; identical to the one-context
 * call.  Each member checks its own share before it starts (so on an error, members with valid shares may have written
 * their outputs). */
int kzgb_group_verify_blob_proofs_g1(kzgb_group* group, const uint8_t* const* blobs, const size_t* lens, size_t count,
                                     const uint64_t* commitments_xy, const uint8_t* commitments_inf,
                                     const uint64_t* proofs_xy, const uint8_t* proofs_inf,
                                     uint64_t* out_xy, uint8_t* out_inf, uint64_t* z_out, uint64_t* y_out);
/* kzgb_verify_blob_proofs cut as kzgb_group_verify_blob_proofs_g1 cuts the batch; identical to the one-context call.  Each
 * member checks its own share before it starts (so on an error, members with valid shares may have written their
 * entries of ok). */
int kzgb_group_verify_blob_proofs(kzgb_group* group, const uint8_t* const* blobs, const size_t* lens, size_t count,
                                  const uint64_t* commitments_xy, const uint8_t* commitments_inf,
                                  const uint64_t* proofs_xy, const uint8_t* proofs_inf, uint8_t* ok);
/* kzgb_set_g2_tau on every member; on an error no member's setting changes. */
int kzgb_group_set_g2_tau(kzgb_group* group, const uint64_t xy[16]);
/* kzgb_verify_batch_rlc on the group, with the same output words as the one-context call.  The 2m points are checked on
 * member 0, then the lengths, with the one-context call's order, codes and messages, before any member starts.  Then
 * each member computes z_i and y_i for its share of the blobs (cut as kzgb_group_verify_blob_proofs_g1 cuts them), and
 * member 0 combines all m openings (kzgb_verify_kzg_proof_batch_rlc with n_i = next_pow2(ceil(len_i / 32))).  An error
 * raised inside a member (a device failure) is reported as "member i (device d): <message>"; the outputs are written
 * only on success. */
int kzgb_group_verify_batch_rlc(kzgb_group* group, const uint8_t* const* blobs, const size_t* lens, size_t count,
                                const uint64_t* commitments_xy, const uint8_t* commitments_inf, const uint64_t* proofs_xy,
                                const uint8_t* proofs_inf, uint64_t lhs_xy[8], uint8_t* lhs_inf, uint64_t rhs_xy[8],
                                uint8_t* rhs_inf);
/* kzgb_msm_srs with the points cut into G contiguous ranges; the partial sums are added on the host. */
int kzgb_group_msm_srs(kzgb_group* group, const uint64_t* scalars_mont, size_t n, uint64_t out_xy[8], uint8_t* out_inf);

/* Fixed-base table in use: window bits c, windows W, points covered (0 = none). */
int kzgb_msm_config(const kzgb_ctx* ctx, int* window_bits, int* windows, size_t* table_points);

#ifdef __cplusplus
}
#endif
#endif /* KZG_BN254_B200_H */
