//! Drop-in for `rust_kzg_bn254_prover::{kzg::KZG, srs::SRS}` backed by the B200 engine.
//! SOURCE ONLY (never compiled: no Rust toolchain in the build image).  Signatures follow
//! prover/src/kzg.rs:25-309 and prover/src/srs.rs:10-49 of the reference line by line.
//!
//! `KZG` derives PartialEq + Clone over `expanded_roots_of_unity` and `SRS` has pub fields in the
//! reference, so no device handle can be stored inside them.  The GPU side of an `SRS` -- a `kzgb_group` over every
//! visible GPU, holding the decompressed points, window tables and Lagrange tables -- lives in a process-global
//! registry instead:
//!   * the key is the (address, length) of the `SRS.g1` slice, the value carries a CONTENT fingerprint (length and 64
//!     sampled points) that is checked on every hit, so an allocation reused by a different SRS never resolves to
//!     the old tables;
//!   * `impl Drop for SRS` removes the entry, which frees the group (HBM tables included) when the last call using it
//!     returns; the registry also holds at most `MAX_RESIDENT_SRS` groups, least recently used evicted first;
//!   * the registry lock is held only for the lookup -- calls on different SRS run concurrently, calls on one SRS are
//!     serialised inside the library;
//!   * every return code of context creation and SRS upload is checked and surfaces as `KzgError`.
mod ffi;

use ark_bn254::{Fq, Fr, G1Affine};
use ark_ec::AffineRepr;
use ark_ff::Zero;
use rust_kzg_bn254_primitives::{
    blob::Blob,
    errors::KzgError,
    helpers,
    polynomial::{PolynomialCoeffForm, PolynomialEvalForm},
};
use std::{
    borrow::Cow,
    collections::HashMap,
    ffi::CStr,
    ffi::CString,
    sync::{Arc, Mutex},
};

const _: () = assert!(core::mem::size_of::<Fr>() == 32 && core::mem::size_of::<Fq>() == 32);

/// Groups kept resident at once (each holds an SRS plus its tables on every GPU).
const MAX_RESIDENT_SRS: usize = 4;
/// Polynomials at least this long are committed over all GPUs of the group (point-range sharding).
const GROUP_MSM_MIN_LEN: usize = 1 << 22;

/// One `kzgb_group` (all visible GPUs).  Single-polynomial calls run on member 0; blob batches and very large
/// coefficient-form commitments are spread over the members by the library.
struct Gpu {
    group: *mut ffi::kzgb_group,
    fingerprint: u64,
}
unsafe impl Send for Gpu {}
unsafe impl Sync for Gpu {} // every entry point of the library locks its context / group internally
impl Drop for Gpu {
    fn drop(&mut self) {
        unsafe { ffi::kzgb_group_destroy(self.group) }
    }
}
impl Gpu {
    fn ctx0(&self) -> *mut ffi::kzgb_ctx {
        unsafe { ffi::kzgb_group_ctx(self.group, 0) }
    }
    fn members(&self) -> usize {
        unsafe { ffi::kzgb_group_size(self.group) as usize }
    }
}

struct Entry {
    gpu: Arc<Gpu>,
    last_use: u64,
}
struct Registry {
    map: HashMap<(usize, usize), Entry>,
    clock: u64,
}
static REGISTRY: Mutex<Option<Registry>> = Mutex::new(None);

/// Length and 64 evenly spaced points (x and y limbs) folded with FNV-1a: cheap enough for every call, and enough to
/// tell two SRS of equal length apart (they differ in every point beyond the generator).
fn fingerprint(g1: &[G1Affine]) -> u64 {
    let mut h: u64 = 0xcbf29ce484222325 ^ g1.len() as u64;
    let mut mix = |w: u64| {
        h ^= w;
        h = h.wrapping_mul(0x100000001b3);
    };
    if g1.is_empty() {
        return h;
    }
    for k in 0..64usize {
        let p = &g1[(k * (g1.len() - 1)) / 63];
        if p.is_zero() {
            mix(u64::MAX);
        } else {
            for w in p.x.0 .0.iter().chain(p.y.0 .0.iter()) {
                mix(*w);
            }
        }
    }
    h
}

fn group_err(group: *mut ffi::kzgb_group, rc: i32) -> KzgError {
    let msg = unsafe { CStr::from_ptr(ffi::kzgb_group_last_error(group)) }.to_string_lossy().into_owned();
    match rc {
        ffi::KZGB_ERR_SRS_CAPACITY => KzgError::GenericError(msg),
        ffi::KZGB_ERR_SERIALIZATION => KzgError::SerializationError(msg),
        ffi::KZGB_ERR_NOT_ON_CURVE => KzgError::NotOnCurveError(msg),
        ffi::KZGB_ERR_DESERIALIZATION => KzgError::DeserializationError(msg),
        _ => KzgError::GenericError(msg),
    }
}

/// A group over every visible GPU; the caller loads an SRS into it.
fn new_group() -> Result<*mut ffi::kzgb_group, KzgError> {
    let mut group = std::ptr::null_mut();
    let rc = unsafe { ffi::kzgb_group_create(&mut group, std::ptr::null(), 0) };
    if rc != 0 || group.is_null() {
        return Err(KzgError::GenericError(format!("no usable CUDA device (kzgb_group_create: {rc})")));
    }
    Ok(group)
}

/// Registers `gpu` for the slice `g1`, evicting the least recently used group beyond `MAX_RESIDENT_SRS`.
fn register(g1: &[G1Affine], gpu: Arc<Gpu>) {
    let mut guard = REGISTRY.lock().unwrap();
    let reg = guard.get_or_insert_with(|| Registry { map: HashMap::new(), clock: 0 });
    reg.clock += 1;
    let now = reg.clock;
    reg.map.insert((g1.as_ptr() as usize, g1.len()), Entry { gpu, last_use: now });
    while reg.map.len() > MAX_RESIDENT_SRS {
        let oldest = *reg.map.iter().min_by_key(|(_, e)| e.last_use).map(|(k, _)| k).unwrap();
        reg.map.remove(&oldest); // the group itself is freed when the last Arc (a call in flight) goes
    }
}

fn to_err(ctx: *mut ffi::kzgb_ctx, rc: i32, poly_len: usize, srs_len: usize) -> KzgError {
    let msg = unsafe { CStr::from_ptr(ffi::kzgb_last_error(ctx)) }.to_string_lossy().into_owned();
    match rc {
        ffi::KZGB_ERR_SRS_CAPACITY => KzgError::SrsCapacityExceeded { polynomial_len: poly_len, srs_len },
        ffi::KZGB_ERR_SERIALIZATION => KzgError::SerializationError(msg),
        ffi::KZGB_ERR_FFT => KzgError::FFTError(msg),
        ffi::KZGB_ERR_NOT_ON_CURVE => KzgError::NotOnCurveError(msg),
        ffi::KZGB_ERR_MSM => KzgError::MsmError(msg),
        ffi::KZGB_ERR_INVALID_INPUT_LENGTH => KzgError::InvalidInputLength,
        ffi::KZGB_ERR_DESERIALIZATION => KzgError::DeserializationError(msg),
        ffi::KZGB_ERR_INVALID_FIELD_ELEMENT => KzgError::InvalidFieldElement(msg),
        _ => KzgError::GenericError(msg),
    }
}

/// arkworks `G1Affine {x, y, infinity}` is repr(Rust): repack to the ABI's x||y words + flag.
fn pack_points(pts: &[G1Affine]) -> (Vec<u64>, Vec<u8>) {
    let mut xy = Vec::with_capacity(pts.len() * 8);
    let mut inf = Vec::with_capacity(pts.len());
    for p in pts {
        if p.is_zero() {
            xy.extend_from_slice(&[0u64; 8]);
            inf.push(1);
        } else {
            xy.extend_from_slice(&p.x.0 .0); // Montgomery limbs, as primitives/src/helpers.rs:158 reads them
            xy.extend_from_slice(&p.y.0 .0);
            inf.push(0);
        }
    }
    (xy, inf)
}

fn unpack_point(xy: &[u64; 8], inf: u8) -> G1Affine {
    if inf != 0 {
        return G1Affine::zero();
    }
    let x = Fq::new_unchecked(ark_ff::BigInt([xy[0], xy[1], xy[2], xy[3]]));
    let y = Fq::new_unchecked(ark_ff::BigInt([xy[4], xy[5], xy[6], xy[7]]));
    G1Affine::new_unchecked(x, y)
}

fn fr_words(v: &[Fr]) -> *const u64 {
    v.as_ptr() as *const u64 // Fp<MontBackend<_,4>,4> == [u64; 4], Montgomery form
}

#[derive(Debug, PartialEq)]
pub struct SRS<'a> {
    pub g1: Cow<'a, [G1Affine]>,
    pub order: u32,
}

impl SRS<'_> {
    /// prover/src/srs.rs:35-49: the file is streamed to GPU 0 in chunks and decompressed there, the points are replicated
    /// to the other GPUs device to device, and read back once to fill the reference's `pub g1` field.
    pub fn new(path_to_g1_points: &str, order: u32, points_to_load: u32) -> Result<Self, KzgError> {
        let group = new_group()?;
        let cpath = CString::new(path_to_g1_points).map_err(|_| KzgError::GenericError("path contains a NUL byte".into()))?;
        let rc = unsafe { ffi::kzgb_group_srs_load_file(group, cpath.as_ptr(), order, points_to_load) };
        if rc != 0 {
            let e = group_err(group, rc);
            unsafe { ffi::kzgb_group_destroy(group) };
            return Err(e);
        }
        let ctx0 = unsafe { ffi::kzgb_group_ctx(group, 0) };
        let n = unsafe { ffi::kzgb_srs_len(ctx0) };
        let mut xy = vec![0u64; 8 * n];
        let mut inf = vec![0u8; n];
        let rc = unsafe { ffi::kzgb_srs_get_affine_mont(ctx0, 0, n, xy.as_mut_ptr(), inf.as_mut_ptr()) };
        if rc != 0 {
            let e = to_err(ctx0, rc, 0, n);
            unsafe { ffi::kzgb_group_destroy(group) };
            return Err(e);
        }
        let g1: Vec<G1Affine> = (0..n).map(|i| unpack_point(xy[8 * i..8 * i + 8].try_into().unwrap(), inf[i])).collect();
        register(&g1, Arc::new(Gpu { group, fingerprint: fingerprint(&g1) }));
        Ok(Self { g1: Cow::Owned(g1), order })
    }
}

/// Frees the GPU side with the SRS it belongs to (the key is the slice's address: it must not outlive the slice).
impl Drop for SRS<'_> {
    fn drop(&mut self) {
        if let Ok(mut guard) = REGISTRY.lock() {
            if let Some(reg) = guard.as_mut() {
                reg.map.remove(&(self.g1.as_ptr() as usize, self.g1.len()));
            }
        }
    }
}

/// Additions next to the reference's API (nothing above changes meaning): warm-up and caching hooks.
impl SRS<'_> {
    /// Builds the resident Lagrange-basis window table for evaluation-form polynomials of `n` elements now
    /// instead of on the first commit of that size (the cached form of the `g1_ifft` that
    /// `KZG::commit_eval_form` runs on every call in the reference, prover/src/kzg.rs:98).
    pub fn prepare_lagrange(&self, n: usize) -> Result<(), KzgError> {
        let gpu = gpu_for(self)?;
        let rc = unsafe { ffi::kzgb_group_srs_prepare_lagrange(gpu.group, n) };
        if rc != 0 { Err(group_err(gpu.group, rc)) } else { Ok(()) }
    }
    /// Builds the resident table of `KZG::compute_proofs_at_all_roots` for polynomials of `n` elements (n <= 2^22) now
    /// instead of on the first call of that size.
    pub fn prepare_all_roots(&self, n: usize) -> Result<(), KzgError> {
        with_ctx(self, |ctx| {
            let rc = unsafe { ffi::kzgb_srs_prepare_all_roots(ctx, n) };
            if rc != 0 { Err(to_err(ctx, rc, n, self.g1.len())) } else { Ok(()) }
        })
    }
    /// Writes the decompressed points so that a later process can skip the per-point square root
    /// (`kzgb_srs_load_cache` checks every point to be on the curve instead).
    pub fn save_cache(&self, path: &str) -> Result<(), KzgError> {
        let cpath = CString::new(path).unwrap();
        with_ctx(self, |ctx| {
            let rc = unsafe { ffi::kzgb_srs_save_cache(ctx, cpath.as_ptr()) };
            if rc != 0 { Err(to_err(ctx, rc, 0, 0)) } else { Ok(()) }
        })
    }
}

/// The GPU side of `srs`: looked up under the registry lock, used WITHOUT it.  A hit whose fingerprint does not match
/// the slice's content (the allocation was reused by another SRS built through the pub fields) is replaced.
fn gpu_for(srs: &SRS) -> Result<Arc<Gpu>, KzgError> {
    let key = (srs.g1.as_ptr() as usize, srs.g1.len());
    let fp = fingerprint(&srs.g1);
    {
        let mut guard = REGISTRY.lock().unwrap();
        let reg = guard.get_or_insert_with(|| Registry { map: HashMap::new(), clock: 0 });
        reg.clock += 1;
        let now = reg.clock;
        match reg.map.get_mut(&key) {
            Some(e) if e.gpu.fingerprint == fp => {
                e.last_use = now;
                return Ok(e.gpu.clone());
            }
            Some(_) => {
                reg.map.remove(&key); // stale: same address and length, different points
            }
            None => {}
        }
    }
    // an SRS built by the caller (pub fields, Cow::Borrowed): upload its points once, outside the lock
    if srs.g1.is_empty() {
        return Err(KzgError::GenericError("empty SRS".into()));
    }
    let group = new_group()?;
    let (xy, inf) = pack_points(&srs.g1);
    let rc = unsafe { ffi::kzgb_group_srs_load_affine_mont(group, xy.as_ptr(), inf.as_ptr(), srs.g1.len()) };
    if rc != 0 {
        let e = group_err(group, rc);
        unsafe { ffi::kzgb_group_destroy(group) };
        return Err(e);
    }
    let gpu = Arc::new(Gpu { group, fingerprint: fp });
    register(&srs.g1, gpu.clone());
    Ok(gpu)
}

type GroupCommitFn = unsafe extern "C" fn(*mut ffi::kzgb_group, *const *const u64, *const usize, usize, *mut u64, *mut u8) -> std::os::raw::c_int;

// One kzgb_group_commit_{evals,coeffs} call over the polynomials at ptrs (lengths ns).  The group's message names the member,
// so on an error the reference's error is rebuilt from the lowest polynomial that `check(len, srs_len)` rejects.
fn commit_polys(
    call: GroupCommitFn, ptrs: &[*const u64], ns: &[usize], srs: &SRS, check: impl Fn(usize, usize) -> Option<KzgError>,
) -> Result<Vec<G1Affine>, KzgError> {
    let m = ptrs.len();
    let mut xy = vec![0u64; 8 * m];
    let mut inf = vec![0u8; m];
    let gpu = gpu_for(srs)?;
    let rc = unsafe { call(gpu.group, ptrs.as_ptr(), ns.as_ptr(), m, xy.as_mut_ptr(), inf.as_mut_ptr()) };
    if rc != 0 {
        let srs_len = srs.g1.len();
        return Err(ns.iter().find_map(|&n| check(n, srs_len)).unwrap_or_else(|| group_err(gpu.group, rc)));
    }
    Ok((0..m).map(|i| unpack_point(xy[8 * i..8 * i + 8].try_into().unwrap(), inf[i])).collect())
}

/// Runs `f` on member 0's context of the SRS's group (single-polynomial entry points).
fn with_ctx<T>(srs: &SRS, f: impl FnOnce(*mut ffi::kzgb_ctx) -> Result<T, KzgError>) -> Result<T, KzgError> {
    let gpu = gpu_for(srs)?;
    f(gpu.ctx0())
}

#[derive(Debug, PartialEq, Clone, Default)]
pub struct KZG {
    expanded_roots_of_unity: Vec<Fr>,
}

impl KZG {
    pub fn new() -> Self {
        Self { expanded_roots_of_unity: vec![] }
    }
    pub fn calculate_and_store_roots_of_unity(&mut self, length_of_data_after_padding: u64) -> Result<(), KzgError> {
        self.expanded_roots_of_unity = helpers::calculate_roots_of_unity(length_of_data_after_padding)?;
        Ok(())
    }
    pub fn get_roots_of_unities(&self) -> Vec<Fr> {
        self.expanded_roots_of_unity.clone()
    }
    pub fn get_nth_root_of_unity(&self, i: usize) -> Option<&Fr> {
        self.expanded_roots_of_unity.get(i)
    }

    pub fn commit_eval_form(&self, polynomial: &PolynomialEvalForm, srs: &SRS) -> Result<G1Affine, KzgError> {
        let (mut xy, mut inf) = ([0u64; 8], 0u8);
        let ev = polynomial.evaluations();
        with_ctx(srs, |ctx| {
            let rc = unsafe { ffi::kzgb_commit_eval(ctx, fr_words(ev), ev.len(), xy.as_mut_ptr(), &mut inf) };
            if rc != 0 { Err(to_err(ctx, rc, ev.len(), srs.g1.len())) } else { Ok(unpack_point(&xy, inf)) }
        })
    }
    pub fn commit_coeff_form(&self, polynomial: &PolynomialCoeffForm, srs: &SRS) -> Result<G1Affine, KzgError> {
        let (mut xy, mut inf) = ([0u64; 8], 0u8);
        let cf = polynomial.coeffs();
        let gpu = gpu_for(srs)?;
        if gpu.members() > 1 && cf.len() >= GROUP_MSM_MIN_LEN {
            // one MSM cut by point range over every GPU, partial sums added on the host (kzg.rs:107-125 at 2^26 coefficients)
            if cf.len() > srs.g1.len() {
                return Err(KzgError::SerializationError("polynomial length is not correct".to_string()));
            }
            let rc = unsafe { ffi::kzgb_group_msm_srs(gpu.group, fr_words(cf), cf.len(), xy.as_mut_ptr(), &mut inf) };
            return if rc != 0 { Err(group_err(gpu.group, rc)) } else { Ok(unpack_point(&xy, inf)) };
        }
        let ctx = gpu.ctx0();
        let rc = unsafe { ffi::kzgb_commit_coeff(ctx, fr_words(cf), cf.len(), xy.as_mut_ptr(), &mut inf) };
        if rc != 0 { Err(to_err(ctx, rc, cf.len(), srs.g1.len())) } else { Ok(unpack_point(&xy, inf)) }
    }
    pub fn commit_blob(&self, blob: &Blob, srs: &SRS) -> Result<G1Affine, KzgError> {
        let (mut xy, mut inf) = ([0u64; 8], 0u8);
        let d = blob.data();
        with_ctx(srs, |ctx| {
            let rc = unsafe { ffi::kzgb_commit_blob(ctx, d.as_ptr(), d.len(), xy.as_mut_ptr(), &mut inf) };
            if rc != 0 { Err(to_err(ctx, rc, d.len().div_ceil(32).next_power_of_two(), srs.g1.len())) } else { Ok(unpack_point(&xy, inf)) }
        })
    }
    /// Addition next to the reference's API: `commit_blob` for every blob in ONE call, for callers that check blobs
    /// against the commitments of their certificates.  The batch is cut by bytes across the GPUs of the box
    /// (`kzgb_group_commit_blobs`) and pipelined on each; no proofs, no transcripts.  Point i is `commit_blob` of blob
    /// i, and an error is the one `commit_blob` reports for the first blob the library rejects.
    pub fn commit_blobs(&self, blobs: &[Blob], srs: &SRS) -> Result<Vec<G1Affine>, KzgError> {
        let ptrs: Vec<*const u8> = blobs.iter().map(|b| b.data().as_ptr()).collect();
        let lens: Vec<usize> = blobs.iter().map(|b| b.data().len()).collect();
        let mut xy = vec![0u64; 8 * blobs.len()];
        let mut inf = vec![0u8; blobs.len()];
        let gpu = gpu_for(srs)?;
        let rc = unsafe {
            ffi::kzgb_group_commit_blobs(gpu.group, ptrs.as_ptr(), lens.as_ptr(), blobs.len(), xy.as_mut_ptr(), inf.as_mut_ptr())
        };
        if rc != 0 {
            let poly_lens = lens.iter().map(|l| l.div_ceil(32).next_power_of_two());
            let srs_len = srs.g1.len();
            return Err(match rc {
                ffi::KZGB_ERR_SRS_CAPACITY => {
                    let polynomial_len = poly_lens.clone().find(|&n| n > srs_len).unwrap_or(0);
                    KzgError::SrsCapacityExceeded { polynomial_len, srs_len }
                }
                // the group's message names the member; commit_blob's does not
                ffi::KZGB_ERR_GENERIC if poly_lens.clone().any(|n| n > 1 << 28) => {
                    KzgError::GenericError("Input size exceeds maximum polynomial size".to_string())
                }
                _ => group_err(gpu.group, rc),
            });
        }
        Ok((0..blobs.len()).map(|i| unpack_point(xy[8 * i..8 * i + 8].try_into().unwrap(), inf[i])).collect())
    }
    pub fn compute_proof(&self, polynomial: &PolynomialEvalForm, z_fr: &Fr, srs: &SRS) -> Result<G1Affine, KzgError> {
        if polynomial.len() != self.expanded_roots_of_unity.len() {
            return Err(KzgError::GenericError("inconsistent length between blob and root of unities".to_string()));
        }
        let (mut xy, mut inf) = ([0u64; 8], 0u8);
        let ev = polynomial.evaluations();
        with_ctx(srs, |ctx| {
            let rc = unsafe {
                ffi::kzgb_compute_proof(ctx, fr_words(ev), ev.len(), z_fr as *const Fr as *const u64, xy.as_mut_ptr(), &mut inf,
                                        std::ptr::null_mut())
            };
            if rc != 0 { Err(to_err(ctx, rc, ev.len(), srs.g1.len())) } else { Ok(unpack_point(&xy, inf)) }
        })
    }
    pub fn compute_proof_with_known_z_fr_index(&self, polynomial: &PolynomialEvalForm, index: u64, srs: &SRS) -> Result<G1Affine, KzgError> {
        let z = self
            .get_nth_root_of_unity(index as usize)
            .ok_or_else(|| KzgError::GenericError("Root of unity not found".to_string()))?;
        self.compute_proof(polynomial, z, srs)
    }
    /// `compute_proof_with_known_z_fr_index` (prover/src/kzg.rs:187-207) at every index 0 .. n-1 in one call (FK20 on
    /// the GPU: two G1 FFTs and 2n scalar multiplications instead of n MSMs); element i is the proof at the i-th root.
    pub fn compute_proofs_at_all_roots(&self, polynomial: &PolynomialEvalForm, srs: &SRS) -> Result<Vec<G1Affine>, KzgError> {
        if polynomial.len() != self.expanded_roots_of_unity.len() {
            return Err(KzgError::GenericError("inconsistent length between blob and root of unities".to_string()));
        }
        let ev = polynomial.evaluations();
        let n = ev.len();
        let mut xy = vec![0u64; 8 * n];
        let mut inf = vec![0u8; n];
        with_ctx(srs, |ctx| {
            let rc = unsafe { ffi::kzgb_compute_proofs_all_roots(ctx, fr_words(ev), n, xy.as_mut_ptr(), inf.as_mut_ptr()) };
            if rc != 0 { return Err(to_err(ctx, rc, n, srs.g1.len())); }
            Ok((0..n).map(|i| unpack_point(xy[8 * i..8 * i + 8].try_into().unwrap(), inf[i])).collect())
        })
    }
    pub fn g1_ifft(&self, length: usize, srs: &SRS) -> Result<Vec<G1Affine>, KzgError> {
        if !length.is_power_of_two() {
            return Err(KzgError::FFTError("length provided is not a power of 2".to_string()));
        }
        let mut xy = vec![0u64; 8 * length];
        let mut inf = vec![0u8; length];
        with_ctx(srs, |ctx| {
            let rc = unsafe { ffi::kzgb_g1_ifft(ctx, length, xy.as_mut_ptr(), inf.as_mut_ptr()) };
            if rc != 0 { return Err(to_err(ctx, rc, length, srs.g1.len())); }
            Ok((0..length).map(|i| unpack_point(xy[8 * i..8 * i + 8].try_into().unwrap(), inf[i])).collect())
        })
    }
    pub fn compute_blob_proof(&self, blob: &Blob, commitment: &G1Affine, srs: &SRS) -> Result<G1Affine, KzgError> {
        helpers::validate_g1_point(commitment)?;
        let n = blob.len().div_ceil(32).next_power_of_two();
        if n != self.expanded_roots_of_unity.len() {
            return Err(KzgError::GenericError("inconsistent length between blob and root of unities".to_string()));
        }
        let (cxy, cinf) = pack_points(std::slice::from_ref(commitment));
        let (mut xy, mut inf) = ([0u64; 8], 0u8);
        let d = blob.data();
        with_ctx(srs, |ctx| {
            let rc = unsafe { ffi::kzgb_compute_blob_proof(ctx, d.as_ptr(), d.len(), cxy.as_ptr(), cinf[0], xy.as_mut_ptr(), &mut inf) };
            if rc != 0 { Err(to_err(ctx, rc, n, srs.g1.len())) } else { Ok(unpack_point(&xy, inf)) }
        })
    }
    /// Addition next to the reference's API: `compute_blob_proof` for every (blob, commitment) pair in ONE call, for
    /// callers that already hold the commitments.  The batch is cut by bytes across the GPUs of the box
    /// (`kzgb_group_compute_blob_proofs`) and pipelined on each; no commitment is computed.  Proof i is
    /// `compute_blob_proof(blob i, commitment i)`, and an error is the one `compute_blob_proof` reports for the first
    /// pair the library rejects (without the per-instance roots-length check, which a batch of sizes has no use for).
    pub fn compute_blob_proofs(&self, blobs: &[Blob], commitments: &[G1Affine], srs: &SRS) -> Result<Vec<G1Affine>, KzgError> {
        if blobs.len() != commitments.len() {
            return Err(KzgError::GenericError("length's of the input are not the same".to_string()));
        }
        let ptrs: Vec<*const u8> = blobs.iter().map(|b| b.data().as_ptr()).collect();
        let lens: Vec<usize> = blobs.iter().map(|b| b.data().len()).collect();
        let (cxy, cinf) = pack_points(commitments);
        let mut xy = vec![0u64; 8 * blobs.len()];
        let mut inf = vec![0u8; blobs.len()];
        let gpu = gpu_for(srs)?;
        let rc = unsafe {
            ffi::kzgb_group_compute_blob_proofs(gpu.group, ptrs.as_ptr(), lens.as_ptr(), blobs.len(), cxy.as_ptr(), cinf.as_ptr(),
                                                xy.as_mut_ptr(), inf.as_mut_ptr())
        };
        if rc != 0 {
            // the library fails on the lowest-index pair that does not pass compute_blob_proof's checks; the group's
            // message names the member, so the error is rebuilt from that pair as compute_blob_proof reports it
            let srs_len = srs.g1.len();
            for (len, commitment) in lens.iter().zip(commitments) {
                helpers::validate_g1_point(commitment)?;
                if *len == 0 {
                    return Err(KzgError::GenericError("Length of data after padding is 0".to_string()));
                }
                let polynomial_len = len.div_ceil(32).next_power_of_two();
                if polynomial_len > srs_len {
                    return Err(KzgError::SrsCapacityExceeded { polynomial_len, srs_len });
                }
            }
            return Err(group_err(gpu.group, rc));
        }
        Ok((0..blobs.len()).map(|i| unpack_point(xy[8 * i..8 * i + 8].try_into().unwrap(), inf[i])).collect())
    }
    /// Addition next to the reference's API: `compute_proof` (prover/src/kzg.rs:128-178, 187-234) of polynomial i at
    /// zs[i] for every i in ONE call, returning each proof with its value y_i = p_i(zs[i]) -- the openings a caller of
    /// `compute_proof` or `compute_proof_with_known_z_fr_index` makes in a loop, and that `verify_proof` checks.  The
    /// batch is cut by evaluation bytes across the GPUs of the box (`kzgb_group_compute_proofs`).  Entry i is
    /// `compute_proof(polynomial i, zs[i])` without the per-instance roots-length check, which a batch of sizes has no use
    /// for; an error is the one `compute_proof` reports for the first polynomial the library rejects.  Source only, like
    /// the rest of this crate: it has not been compiled, because the build image has no Rust toolchain.
    pub fn compute_proofs(&self, polynomials: &[PolynomialEvalForm], zs: &[Fr], srs: &SRS) -> Result<Vec<(G1Affine, Fr)>, KzgError> {
        if polynomials.len() != zs.len() {
            return Err(KzgError::GenericError("length's of the input are not the same".to_string()));
        }
        let m = polynomials.len();
        let ptrs: Vec<*const u64> = polynomials.iter().map(|p| fr_words(p.evaluations())).collect();
        let ns: Vec<usize> = polynomials.iter().map(|p| p.evaluations().len()).collect();
        let mut xy = vec![0u64; 8 * m];
        let mut inf = vec![0u8; m];
        let mut ys = vec![0u64; 4 * m];
        let gpu = gpu_for(srs)?;
        let rc = unsafe {
            ffi::kzgb_group_compute_proofs(gpu.group, ptrs.as_ptr(), ns.as_ptr(), m, fr_words(zs), xy.as_mut_ptr(),
                                           inf.as_mut_ptr(), ys.as_mut_ptr())
        };
        if rc != 0 {
            // the library fails on the lowest-index polynomial that does not pass compute_proof's checks (an Fr is always
            // reduced, so its z passes); the group's message names the member, so the error is rebuilt from that polynomial
            let srs_len = srs.g1.len();
            for &polynomial_len in &ns {
                if !polynomial_len.is_power_of_two() {
                    return Err(KzgError::FFTError("length provided is not a power of 2".to_string()));
                }
                if polynomial_len > srs_len {
                    return Err(KzgError::SrsCapacityExceeded { polynomial_len, srs_len });
                }
            }
            return Err(group_err(gpu.group, rc));
        }
        Ok((0..m)
            .map(|i| {
                let y = Fr::new_unchecked(ark_ff::BigInt([ys[4 * i], ys[4 * i + 1], ys[4 * i + 2], ys[4 * i + 3]]));
                (unpack_point(xy[8 * i..8 * i + 8].try_into().unwrap(), inf[i]), y)  // y: Montgomery limbs, as fr_words passes them
            })
            .collect())
    }
    /// Addition next to the reference's API: `commit_eval_form` (prover/src/kzg.rs:84-104) of every polynomial in ONE
    /// call.  The batch is cut by evaluation bytes across the GPUs of the box (`kzgb_group_commit_evals`) and pipelined on
    /// each.  Point i is `commit_eval_form(polynomial i)`; an error is the one `commit_eval_form` reports for the first
    /// polynomial the library rejects.  Source only, like the rest of this crate: it has not been compiled, because the
    /// build image has no Rust toolchain.
    pub fn commit_eval_forms(&self, polynomials: &[PolynomialEvalForm], srs: &SRS) -> Result<Vec<G1Affine>, KzgError> {
        let ptrs: Vec<*const u64> = polynomials.iter().map(|p| fr_words(p.evaluations())).collect();
        let ns: Vec<usize> = polynomials.iter().map(|p| p.evaluations().len()).collect();
        commit_polys(ffi::kzgb_group_commit_evals, &ptrs, &ns, srs, |polynomial_len, srs_len| {
            // commit_eval_form's order: SRS capacity (kzg.rs:89-94), then the power of two of its G1 IFFT (kzg.rs:265-269)
            if polynomial_len > srs_len {
                Some(KzgError::SrsCapacityExceeded { polynomial_len, srs_len })
            } else if !polynomial_len.is_power_of_two() {
                Some(KzgError::FFTError("length provided is not a power of 2".to_string()))
            } else {
                None
            }
        })
    }
    /// Addition next to the reference's API: `commit_coeff_form` (prover/src/kzg.rs:107-125) of every polynomial in ONE
    /// call, for callers with many polynomials (the reference's own commit benchmark commits blobs of 10 000 to 50 000
    /// bytes in coefficient form).  The batch is cut by coefficient bytes across the GPUs of the box
    /// (`kzgb_group_commit_coeffs`).  Point i is `commit_coeff_form(polynomial i)`; an error is the one `commit_coeff_form`
    /// reports for the first polynomial the library rejects.  Source only, not compiled (no Rust toolchain in the build
    /// image).
    pub fn commit_coeff_forms(&self, polynomials: &[PolynomialCoeffForm], srs: &SRS) -> Result<Vec<G1Affine>, KzgError> {
        let ptrs: Vec<*const u64> = polynomials.iter().map(|p| fr_words(p.coeffs())).collect();
        let ns: Vec<usize> = polynomials.iter().map(|p| p.coeffs().len()).collect();
        commit_polys(ffi::kzgb_group_commit_coeffs, &ptrs, &ns, srs, |polynomial_len, srs_len| {
            (polynomial_len > srs_len).then(|| KzgError::SerializationError("polynomial length is not correct".to_string()))
        })
    }
}

impl KZG {
    /// prover/src/kzg.rs:237-260: the quotient's evaluation at the domain point z = w_m itself,
    /// q_m = sum_{i != m} (f_i - y) w_i / (z (z - w_i)).  Host-side (the GPU computes the same value inside
    /// `kzgb_compute_proof`; this stays callable on its own as in the reference): ONE batched inversion for all
    /// denominators instead of the reference's n separate ones.
    pub fn compute_quotient_eval_on_domain(&self, z_fr: &Fr, eval_fr: &[Fr], value_fr: &Fr) -> Fr {
        use ark_ff::{batch_inversion, One};
        let roots = &self.expanded_roots_of_unity;
        let mut denominators: Vec<Fr> = roots.iter().map(|w| if w == z_fr { Fr::one() } else { *z_fr * (*z_fr - *w) }).collect();
        batch_inversion(&mut denominators);
        let mut quotient = Fr::zero();
        for ((w, f), d_inv) in roots.iter().zip(eval_fr.iter()).zip(denominators.iter()) {
            if w == z_fr {
                continue;
            }
            quotient += (*f - *value_fr) * *w * *d_inv;
        }
        quotient
    }

    /// Addition next to the reference's API (BASELINE config 3): commit_blob + compute_blob_proof for a batch of
    /// blobs in ONE call -- the pipelined / grouped path of `kzgb_commit_and_prove_blobs`.  Returns the arkworks
    /// compressed bytes of (commitment, proof) per blob, the encoding the reference's transcripts use.
    pub fn commit_and_prove_blobs(&self, blobs: &[Blob], srs: &SRS) -> Result<Vec<([u8; 32], [u8; 32])>, KzgError> {
        let ptrs: Vec<*const u8> = blobs.iter().map(|b| b.data().as_ptr()).collect();
        let lens: Vec<usize> = blobs.iter().map(|b| b.data().len()).collect();
        let mut commitments = vec![0u8; 32 * blobs.len()];
        let mut proofs = vec![0u8; 32 * blobs.len()];
        let gpu = gpu_for(srs)?;
        // contiguous shares of the batch, one per GPU of the box (kzgb_group_commit_and_prove_blobs)
        let rc = unsafe {
            ffi::kzgb_group_commit_and_prove_blobs(gpu.group, ptrs.as_ptr(), lens.as_ptr(), blobs.len(), commitments.as_mut_ptr(),
                                                   proofs.as_mut_ptr())
        };
        if rc != 0 {
            return Err(group_err(gpu.group, rc));
        }
        Ok((0..blobs.len())
            .map(|i| (commitments[32 * i..32 * i + 32].try_into().unwrap(), proofs[32 * i..32 * i + 32].try_into().unwrap()))
            .collect())
    }
}

/// Entry points of `primitives` / `verifier` that sit on the path but need no SRS: they run on a default context
/// (device 0, created on first use).  The reference crates call these from the bodies named in each doc comment;
/// `primitives` cannot depend on this crate, so the two-line patches go behind a `gpu` feature there
/// (INTEGRATION.md 4).
pub mod backend {
    use super::*;

    struct Ctx(*mut ffi::kzgb_ctx);
    unsafe impl Send for Ctx {}
    impl Drop for Ctx {
        fn drop(&mut self) {
            unsafe { ffi::kzgb_ctx_destroy(self.0) }
        }
    }
    static DEFAULT_CTX: Mutex<Option<Ctx>> = Mutex::new(None);

    struct Grp(*mut ffi::kzgb_group);
    unsafe impl Send for Grp {}
    impl Drop for Grp {
        fn drop(&mut self) {
            unsafe { ffi::kzgb_group_destroy(self.0) }
        }
    }
    /// Every visible GPU (created on first use) for the per-blob verification of a batch, which needs no SRS.
    static DEFAULT_GROUP: Mutex<Option<Grp>> = Mutex::new(None);

    fn with_default_group<T>(f: impl FnOnce(*mut ffi::kzgb_group) -> T) -> Result<T, KzgError> {
        let mut guard = DEFAULT_GROUP.lock().unwrap();
        if guard.is_none() {
            *guard = Some(Grp(new_group()?));
        }
        Ok(f(guard.as_ref().unwrap().0))
    }

    /// `verify_proof`'s pairing (verifier/src/verify.rs:44-74) on the library's `commit_minus_value` = C - [y] G1:
    /// e(C - [y] G1, G2) == e(proof, [tau - z] G2).
    fn pairing_check(commit_minus_value: G1Affine, proof: G1Affine, z: Fr) -> bool {
        use ark_ec::CurveGroup;
        let x_minus_z = (G2_TAU.into_group() - G2Affine::generator() * z).into_affine();
        helpers::pairings_verify(commit_minus_value, G2Affine::generator(), proof, x_minus_z)
    }

    use ark_bn254::G2Affine;
    use rust_kzg_bn254_primitives::consts::G2_TAU;

    fn fr_from_words(w: &[u64]) -> Fr {
        Fr::new_unchecked(ark_ff::BigInt([w[0], w[1], w[2], w[3]])) // Montgomery limbs, as fr_words passes them
    }

    /// `verifier::verify::verify_blob_kzg_proof` (verifier/src/verify.rs:77-115): validation, challenge, evaluation and
    /// C - [y] G1 are one `kzgb_verify_blob_proof_g1` call; the pairing stays the reference's code.
    pub fn verify_blob_kzg_proof(blob: &Blob, commitment: &G1Affine, proof: &G1Affine) -> Result<bool, KzgError> {
        let (cxy, cinf) = pack_points(std::slice::from_ref(commitment));
        let (pxy, pinf) = pack_points(std::slice::from_ref(proof));
        let (mut out, mut out_inf, mut z) = ([0u64; 8], 0u8, [0u64; 4]);
        let data = blob.data();
        let commit_minus_value = with_default_ctx(|ctx| {
            let rc = unsafe {
                ffi::kzgb_verify_blob_proof_g1(ctx, data.as_ptr(), data.len(), cxy.as_ptr(), cinf[0], pxy.as_ptr(), pinf[0],
                                               out.as_mut_ptr(), &mut out_inf, z.as_mut_ptr(), std::ptr::null_mut())
            };
            if rc != 0 { Err(to_err(ctx, rc, 0, 0)) } else { Ok(unpack_point(&out, out_inf)) }
        })??;
        Ok(pairing_check(commit_minus_value, *proof, fr_from_words(&z)))
    }

    /// Addition next to the reference's API: `verify_blob_kzg_proof` for every (blob, commitment, proof) triple in ONE
    /// call, one bool per blob -- what a verifier needs when `verify_blob_kzg_proof_batch` fails and it must find the bad
    /// blobs.  The batch is cut by bytes across the GPUs of the box (`kzgb_group_verify_blob_proofs`), and each blob's
    /// pairing check runs there too, under the library's default [tau]G2, which is this crate's `G2_TAU`.  An error is the
    /// one `verify_blob_kzg_proof` reports for the first triple the library rejects.
    pub fn verify_blob_kzg_proofs(blobs: &[Blob], commitments: &[G1Affine], proofs: &[G1Affine]) -> Result<Vec<bool>, KzgError> {
        if !(commitments.len() == blobs.len() && proofs.len() == blobs.len()) {
            return Err(KzgError::GenericError("length's of the input are not the same".to_string()));
        }
        let m = blobs.len();
        let ptrs: Vec<*const u8> = blobs.iter().map(|b| b.data().as_ptr()).collect();
        let lens: Vec<usize> = blobs.iter().map(|b| b.data().len()).collect();
        let (cxy, cinf) = pack_points(commitments);
        let (pxy, pinf) = pack_points(proofs);
        let mut ok = vec![0u8; m];
        with_default_group(|group| {
            let rc = unsafe {
                ffi::kzgb_group_verify_blob_proofs(group, ptrs.as_ptr(), lens.as_ptr(), m, cxy.as_ptr(), cinf.as_ptr(),
                                                   pxy.as_ptr(), pinf.as_ptr(), ok.as_mut_ptr())
            };
            if rc == 0 {
                return Ok(());
            }
            // the group's message names the member: the error is rebuilt from the first failing triple as the
            // single-blob call reports it
            for (len, (c, p)) in lens.iter().zip(commitments.iter().zip(proofs)) {
                helpers::validate_g1_point(c)?;
                helpers::validate_g1_point(p)?;
                if *len == 0 {
                    return Err(KzgError::GenericError("Length of data after padding is 0".to_string()));
                }
                if len.div_ceil(32).next_power_of_two() > 1 << 28 {
                    return Err(KzgError::GenericError("Input size exceeds maximum polynomial size".to_string()));
                }
            }
            let err = group_err(group, rc);
            match &err {
                KzgError::GenericError(msg) if msg.ends_with("Evaluation point equals trusted setup secret") => {
                    Err(KzgError::GenericError("Evaluation point equals trusted setup secret".to_string()))
                }
                _ => Err(err),
            }
        })??;
        Ok(ok.into_iter().map(|b| b != 0).collect())
    }

    fn with_default_ctx<T>(f: impl FnOnce(*mut ffi::kzgb_ctx) -> T) -> Result<T, KzgError> {
        let mut guard = DEFAULT_CTX.lock().unwrap();
        if guard.is_none() {
            let mut ctx = std::ptr::null_mut();
            if unsafe { ffi::kzgb_ctx_create(&mut ctx, 0, std::ptr::null_mut()) } != 0 || ctx.is_null() {
                return Err(KzgError::GenericError("no usable CUDA device".into()));
            }
            *guard = Some(Ctx(ctx));
        }
        Ok(f(guard.as_ref().unwrap().0))
    }

    /// Body of `PolynomialEvalForm::to_coeff_form` (inverse = true) / `PolynomialCoeffForm::to_eval_form`
    /// (primitives/src/polynomial.rs:130-140, :241-251): natural order in and out, in place.
    pub fn ntt_fr_in_place(data: &mut [Fr], inverse: bool) -> Result<(), KzgError> {
        let n = data.len();
        with_default_ctx(|ctx| {
            let rc = unsafe { ffi::kzgb_ntt_fr(ctx, data.as_mut_ptr() as *mut u64, n, inverse as i32) };
            if rc != 0 { Err(to_err(ctx, rc, n, 0)) } else { Ok(()) }
        })?
    }

    /// `helpers::g1_lincomb` (primitives/src/helpers.rs:328-337): variable-base MSM, result in affine form.
    pub fn g1_lincomb(points: &[G1Affine], scalars: &[Fr]) -> Result<G1Affine, KzgError> {
        if points.len() != scalars.len() {
            return Err(KzgError::MsmError(format!("bases and scalars differ in length: {} vs {}", points.len(), scalars.len())));
        }
        let (xy, inf) = pack_points(points);
        let (mut out, mut out_inf) = ([0u64; 8], 0u8);
        with_default_ctx(|ctx| {
            let rc = unsafe { ffi::kzgb_msm_var(ctx, xy.as_ptr(), inf.as_ptr(), fr_words(scalars), points.len(), out.as_mut_ptr(), &mut out_inf) };
            if rc != 0 { Err(to_err(ctx, rc, points.len(), 0)) } else { Ok(unpack_point(&out, out_inf)) }
        })?
    }

    /// `verifier::batch::verify_blob_kzg_proof_batch` (verifier/src/batch.rs:16-255): the input checks and the final
    /// pairing stay the reference's code; per-blob challenges and evaluations, the RLC scalar and the three linear
    /// combinations (batch.rs:40-249) are one `kzgb_group_verify_batch_rlc` call, whose per-blob half is cut by bytes
    /// across the GPUs of the box.
    pub fn verify_blob_kzg_proof_batch(blobs: &[Blob], commitments: &[G1Affine], proofs: &[G1Affine]) -> Result<bool, KzgError> {
        if !(commitments.len() == blobs.len() && proofs.len() == blobs.len()) {
            return Err(KzgError::GenericError("length's of the input are not the same".to_string()));
        }
        for c in commitments.iter() {
            helpers::validate_g1_point(c)?;
        }
        for p in proofs.iter() {
            helpers::validate_g1_point(p)?;
        }
        let ptrs: Vec<*const u8> = blobs.iter().map(|b| b.data().as_ptr()).collect();
        let lens: Vec<usize> = blobs.iter().map(|b| b.data().len()).collect();
        let (cxy, cinf) = pack_points(commitments);
        let (pxy, pinf) = pack_points(proofs);
        let (mut lhs, mut lhs_inf, mut rhs, mut rhs_inf) = ([0u64; 8], 0u8, [0u64; 8], 0u8);
        let (proof_lincomb, rhs_g1) = with_default_group(|group| {
            let rc = unsafe {
                ffi::kzgb_group_verify_batch_rlc(group, ptrs.as_ptr(), lens.as_ptr(), blobs.len(), cxy.as_ptr(), cinf.as_ptr(),
                                                 pxy.as_ptr(), pinf.as_ptr(), lhs.as_mut_ptr(), &mut lhs_inf, rhs.as_mut_ptr(),
                                                 &mut rhs_inf)
            };
            if rc == 0 {
                return Ok((unpack_point(&lhs, lhs_inf), unpack_point(&rhs, rhs_inf)));
            }
            // the points were validated above; what is left is the one-context call's length check, reported as it
            // reports it, or a device failure, whose group message names the member
            if lens.contains(&0) {
                return Err(KzgError::GenericError("Length of data after padding is 0".to_string()));
            }
            Err(group_err(group, rc))
        })??;
        // e(sum r^i proof_i, [tau]G2) == e(sum r^i (C_i - [y_i]) + sum r^i z_i proof_i, G2)   (batch.rs:253-254)
        Ok(helpers::pairings_verify(proof_lincomb, G2_TAU, rhs_g1, G2Affine::generator()))
    }

    /// Addition next to the reference's API: `verifier::batch::verify_kzg_proof_batch` (verifier/src/batch.rs:185-255)
    /// over openings the caller has already evaluated, for instance the z and y of `verify_blob_kzg_proofs`' G1 call.  No
    /// blob is hashed.  `poly_lens[i]` is the padded polynomial length n_i the RLC transcript hashes (batch.rs:48-54).  The
    /// random linear combination is one `kzgb_verify_kzg_proof_batch_rlc` call; the pairing stays the reference's code.
    pub fn verify_kzg_proof_batch(commitments: &[G1Affine], zs: &[Fr], ys: &[Fr], proofs: &[G1Affine], poly_lens: &[u64])
                                  -> Result<bool, KzgError> {
        let m = commitments.len();
        if !(zs.len() == m && ys.len() == m && proofs.len() == m && poly_lens.len() == m) {
            return Err(KzgError::GenericError("length's of the input are not the same".to_string()));
        }
        for c in commitments.iter() {
            helpers::validate_g1_point(c)?;
        }
        for p in proofs.iter() {
            helpers::validate_g1_point(p)?;
        }
        let (cxy, cinf) = pack_points(commitments);
        let (pxy, pinf) = pack_points(proofs);
        let (mut lhs, mut lhs_inf, mut rhs, mut rhs_inf) = ([0u64; 8], 0u8, [0u64; 8], 0u8);
        let (proof_lincomb, rhs_g1) = with_default_ctx(|ctx| {
            let rc = unsafe {
                ffi::kzgb_verify_kzg_proof_batch_rlc(ctx, m, cxy.as_ptr(), cinf.as_ptr(), pxy.as_ptr(), pinf.as_ptr(), fr_words(zs),
                                                     fr_words(ys), poly_lens.as_ptr(), lhs.as_mut_ptr(), &mut lhs_inf,
                                                     rhs.as_mut_ptr(), &mut rhs_inf)
            };
            if rc != 0 { Err(to_err(ctx, rc, 0, 0)) } else { Ok((unpack_point(&lhs, lhs_inf), unpack_point(&rhs, rhs_inf))) }
        })??;
        Ok(helpers::pairings_verify(proof_lincomb, G2_TAU, rhs_g1, G2Affine::generator()))
    }
}
