// Internal launcher interface between the host orchestration (capi.cu, batch.cu) and the kernel
// translation units.  Everything here takes DEVICE pointers and a stream; nothing blocks.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include <atomic>
#include "ec.cuh"

namespace kzgb {

// kernels launched by this library since load (every launcher bumps it)
extern std::atomic<uint64_t> g_launch_count;

// ---- MSM plan -------------------------------------------------------------------
// Signed-digit Pippenger.  Scalars are cut into W = ceil(255/c) signed c-bit digits.
// With a fixed-base table (precomputed 2^(c*w) * P_i for every window w) all windows
// share ONE bucket set; without it (variable bases) every window has its own set and
// the host finishes with a Horner combine.
inline int window_count(int c) { return (255 + c - 1) / c; }  // W of a c-bit plan or window table
struct MsmPlan {
    int c;             // window bits
    int W;             // number of windows
    int sets;          // 1 (fixed-base table), W (variable base) or the number of batched fixed-base MSMs
    uint32_t batch_n;  // batched fixed-base MSMs: scalars per MSM (scalar i belongs to MSM i / batch_n); 0 = not batched
    uint32_t nbuckets; // sets * 2^(c-1)
    uint32_t n;        // points in this launch
    uint32_t table_stride;  // points per window in the table (0 when sets == W)
    uint32_t base_offset;   // first point of this launch inside the table (point-range sharding)
    uint32_t acc_threads;   // threads of the accumulate kernel (fixed-size chunks)
    uint32_t chunk;         // sorted entries per accumulate thread
    // bucket matrix of one set for the 2-D reduction: 2^(c-1) buckets = 2^h_bits rows x 2^a_bits columns
    int a_bits, h_bits;
    int ngroups;            // bit groups of the weighted sums (= c - 1, or a_bits + 1 when h_bits == 0)
};

struct MsmWorkspace {
    Fr* canon;          // n canonical scalars
    uint32_t* hist;     // nbuckets + 1 (counts, then exclusive offsets)
    uint32_t* cursor;   // nbuckets
    uint32_t* sorted;   // n * W point refs grouped by bucket
    XYZZ* buckets;      // nbuckets
    XYZZ* partial;      // 2 * acc_threads
    XYZZ* line_sums;    // sets * (2^h_bits + 2^a_bits): row sums, then column sums of every set
    XYZZ* group_sums;   // sets * ngroups
    XYZZ* set_sums;     // sets (device), copied to host by the caller
    uint32_t* tile_tot; // scan tile totals (<= 1024)
    uint32_t* long_list; // [0] counter, [1..] buckets spanning many accumulate chunks (k_bucket_fix_long)
};

size_t msm_workspace_bytes(const MsmPlan& p);
void msm_workspace_carve(const MsmPlan& p, void* base, MsmWorkspace* ws);
// batch > 0 (fixed base only): n = batch * (n / batch) scalars of `batch` independent MSMs over the same
// table points [base_offset, base_offset + n / batch); set_sums[k] is the result of MSM k.
MsmPlan msm_make_plan(uint32_t n, int c, bool fixed_base, uint32_t table_stride, uint32_t base_offset, uint32_t batch = 0);
// waves of accumulate blocks (4 blocks of 128 threads per SM and wave) the sorted list is cut into; default 4
void msm_set_acc_waves(int waves);
void msm_set_debug_sync(int on);
void msm_set_experiment(int acc_regs, int sort_block);

// scalars: n Fr (Montgomery unless scalars_canonical).  Result: ws.set_sums[0..sets) on the device.
// The optional events bracket the bucket-accumulation kernel (roofline timing).
void msm_launch(const MsmPlan& p, const MsmWorkspace& ws, const Fr* scalars, bool scalars_canonical,
                const Affine* table, cudaStream_t st, cudaEvent_t ev_acc_begin = nullptr,
                cudaEvent_t ev_acc_end = nullptr, cudaStream_t st_acc = nullptr, cudaEvent_t ev_fork = nullptr,
                cudaEvent_t ev_join = nullptr);
// st_acc (optional): a second, lower-priority stream for the bucket accumulation, fenced against `st`
// with ev_fork / ev_join.
// The two halves of msm_launch: sort + accumulate + stitch (ws.buckets = the sum of every bucket), and the
// bucket reduction of any bucket array of the plan's shape.  Large MSMs whose scalars arrive from the host in
// chunks run the first half per chunk, fold the bucket sums together (msm_merge_buckets) and reduce once.
void msm_launch_buckets(const MsmPlan& p, const MsmWorkspace& ws, const Fr* scalars, bool scalars_canonical,
                        const Affine* table, cudaStream_t st, cudaEvent_t ev_acc_begin = nullptr,
                        cudaEvent_t ev_acc_end = nullptr, cudaStream_t st_acc = nullptr, cudaEvent_t ev_fork = nullptr,
                        cudaEvent_t ev_join = nullptr);
void msm_launch_reduce(const MsmPlan& p, const MsmWorkspace& ws, const XYZZ* buckets, cudaStream_t st);
void msm_merge_buckets(XYZZ* dst, const XYZZ* src, uint32_t nbuckets, cudaStream_t st);
// msm_launch with the scalars read from blob bytes (blob_element below, reduced mod r) by the first sort pass: for
// commitments over a Lagrange table, where the evaluations of the blob are the scalars and nothing needs their
// Montgomery form.  A batched plan reads blob k at blob + 32 * batch_n * k.
void msm_launch_blob(const MsmPlan& p, const MsmWorkspace& ws, const uint8_t* blob, uint64_t len_bytes,
                     const Affine* table, cudaStream_t st, cudaEvent_t ev_acc_begin = nullptr,
                     cudaEvent_t ev_acc_end = nullptr, cudaStream_t st_acc = nullptr, cudaEvent_t ev_fork = nullptr,
                     cudaEvent_t ev_join = nullptr);

// Element i of blob bytes (primitives/src/helpers.rs:40-57): the 32 big-endian bytes at offset 32 i as a 256-bit
// integer, the last partial chunk right-padded with zeros, zero past len.  Not reduced mod r.
__device__ __forceinline__ Fr blob_element(const uint8_t* __restrict__ in, uint64_t len, uint32_t i) {
    const uint64_t off = (uint64_t)i * 32;
    Fr v;
    if (off >= len) { fe_zero(v); return v; }
    uint32_t be[8];
    if (off + 32 <= len && ((uintptr_t)in & 15) == 0) {
        const uint4* q = reinterpret_cast<const uint4*>(in + off);
        uint4 a = __ldg(q), b = __ldg(q + 1);
        be[0] = a.x; be[1] = a.y; be[2] = a.z; be[3] = a.w;
        be[4] = b.x; be[5] = b.y; be[6] = b.z; be[7] = b.w;
    } else {
        for (int k = 0; k < 8; k++) {
            uint32_t w = 0;
            for (int j = 0; j < 4; j++) {
                uint64_t p = off + 4 * k + j;
                uint32_t byte = p < len ? in[p] : 0u;
                w |= byte << (8 * j);
            }
            be[k] = w;
        }
    }
    for (int k = 0; k < 8; k++) v.l[7 - k] = __byte_perm(be[k], 0, 0x0123);
    return v;
}

// ---- SRS ------------------------------------------------------------------------
// gnark big-endian compressed points -> affine Montgomery (n < 2^30 per launch).  err[0] must be preset to
// 0xffffffff; afterwards err[0] = ((1 + index of the lowest bad point) << 2) | kind (0xffffffff = none),
// kind 1 = not on curve, 2 = infinity not coded properly.
void srs_decompress_launch(const uint8_t* in_be, uint32_t n, Affine* out, uint32_t* err, cudaStream_t st);
// table[w * stride + i] = 2^(c*w) * table[i] for w = 1..W-1 (window 0 must already be there)
void srs_precompute_launch(Affine* table, uint32_t n, uint32_t stride, int c, int W, XYZZ* scratch,
                           uint32_t batch, cudaStream_t st);
size_t srs_precompute_scratch_bytes(uint32_t batch, int W);
// point validation (on curve or identity): err[0] preset 0xffffffff -> 1 + lowest offending index
void g1_validate_launch(const Affine* pts, uint32_t n, uint32_t* err, cudaStream_t st);
// SRS_i = tau^(first + i) * G (synthetic SRS for benches/tests; tau in Montgomery form)
void srs_synthetic_launch(Affine* out, uint32_t n, const Fr* tau_mont_host, uint32_t first, cudaStream_t st);

// ---- Fr NTT ---------------------------------------------------------------------
// tw: omega_N^j for j < N/2 (Montgomery), N = 2^logN >= n.
void ntt_twiddles_launch(Fr* tw, int logN, const Fr* omega_mont_host, cudaStream_t st);
// in-place on data (natural order in and out).  inverse scales by 1/n.  batch transforms of size 2^logn
// laid out back to back.
void ntt_launch(Fr* data, int logn, uint32_t batch, bool inverse, const Fr* tw, int logN, const Fr* ninv_mont_host,
                Fr* scratch, cudaStream_t st);

// 0: shared-memory tile passes (default), 1: warp-resident passes (registers + shuffles + bulk copy)
void ntt_set_kernel(int which);

// ---- G1 inverse NTT (KZG::g1_ifft, prover/src/kzg.rs:263-285) --------------------------
// srs: 2^logn affine points; work: 2^logn XYZZ scratch; out: 2^logn affine points (natural order).
// ninv_canon_host: 1/n as a CANONICAL (non-Montgomery) scalar.
void g1_intt_launch(const Affine* srs, int logn, XYZZ* work, Affine* out, const Fr* tw, int logN,
                    const Fr* ninv_canon_host, cudaStream_t st);

// ---- polynomial glue ------------------------------------------------------------
// bytes (big-endian 32 B chunks, last chunk zero-right-padded) -> n Fr Montgomery (zero padded to n)
void bytes_to_fr_launch(const uint8_t* in, uint64_t len_bytes, Fr* out, uint32_t n, cudaStream_t st);
// n Fr Montgomery -> 32 B big-endian canonical
void fr_to_bytes_launch(const Fr* in, uint8_t* out, uint32_t n, cudaStream_t st);
// y = p(z) and quotient q_i = (f_i - y)/(w_i - z), including z = w_m (reference
// prover/src/kzg.rs:141-174,237-260; primitives/src/helpers.rs:475-535).
// scratch: n Fr (inverses) + 2 * 1024 Fr partials.  y_out: 1 Fr (Montgomery, device).
// Batched: `batch` polynomials of n evaluations back to back, z_mont_dev[batch] on the device;
// q_out may be NULL (evaluation only).  y_out: batch Fr (Montgomery, device).
// tinv_mont_dev[batch]: 1/(z^n - 1), or z/n when z^n == 1 (one host inversion per polynomial).
void eval_quotient_launch(const Fr* evals, uint32_t n, int logn, uint32_t batch, const Fr* z_mont_dev,
                          const Fr* tinv_mont_dev, const Fr* tw, int logN, const Fr* ninv_mont_host, Fr* scratch,
                          Fr* q_out, Fr* y_out, cudaStream_t st, bool z_outside_domain = false,
                          const uint32_t* in_domain_dev = nullptr);
// in_domain_dev (device, batch words, e.g. from fs_challenges_launch): per-polynomial choice made ON THE DEVICE --
// polynomials with flag 0 take the structured inverses, flagged ones the generic form (both kernel sets are
// launched; blocks of the wrong kind exit at once).
// z_outside_domain: the caller knows that no z of the batch is a root of the domain (z^n != 1); the
// inverses then come from the factorisation of z^n - 1 (~3 instead of ~10 multiplications per element).
size_t eval_quotient_scratch_elems(uint32_t n, uint32_t batch);
// 0: always the generic prefix/suffix-product inverses (tests compare the two forms)
void eval_set_structured(int on);
// Fiat-Shamir challenges of `batch` blobs of n evaluations each on the device (fs.cu; reference
// primitives/src/helpers.rs:411-472): z_out[k] (Montgomery) and tinv_out[k] = 1/(z^n - 1) (or z/n in the
// domain).  commit32_dev: batch x 32 bytes, arkworks-compressed commitments.
void fs_set_force_flag(int on);
void fs_set_quad(int on);
void fs_set_midstate_lanes(int on);  // 1: one lane per long transcript, 0: one warp per transcript, -1 (default): by the batch's depth
int fs_midstate_lanes();
// Midstates of `count` long Fiat-Shamir transcripts on the device, one warp (or, lanes = true, one lane) per message, from resident blob BYTES:
// state[8k..8k+8) = SHA-256 state after tag || u64_be(n) || chunks 0..n-2 of blob k (exactly 32 n bytes, n = ns[k] = 2^j >= 4).
// state / done / cancel are device-visible pointers to MAPPED pinned host memory: done[k] becomes 1 when state k is final,
// a non-zero *cancel stops the kernel early.
void fs_midstate_long_launch(const uint8_t* const* blobs_dev, const uint32_t* ns_dev, uint32_t count, uint32_t* state_mapped,
                             uint32_t* done_mapped, const uint32_t* cancel_mapped, bool lanes, cudaStream_t st);
// in_domain_out (optional, batch words): 1 where z_k turned out to be a root of the domain.
void fs_challenges_launch(const Fr* evals, uint32_t n, int logn, uint32_t batch, const uint8_t* commit32_dev,
                          const Fr* ninv_mont_host, Fr* z_out, Fr* tinv_out, cudaStream_t st, uint32_t* in_domain_out = nullptr);
// out[i] = base^(first + i) (Montgomery), i < n
void fr_powers_launch(Fr* out, uint32_t n, const Fr* base_mont_host, cudaStream_t st, uint32_t first = 0);
// out[i] = a[i] * b[i]
void fr_mul_vec_launch(Fr* out, const Fr* a, const Fr* b, uint32_t n, cudaStream_t st);
// out[0] = sum a[i]*b[i]   (single block; n small: verifier batch)
void fr_dot_launch(Fr* out, const Fr* a, const Fr* b, uint32_t n, cudaStream_t st);

// ---- microbenchmarks (integer-pipe roof) ------------------------------------------
void imad_peak_launch(uint32_t* sink, int iters, int mode, int blocks, int threads, cudaStream_t st);
void fqmul_peak_launch(uint32_t* sink, int iters, int blocks, int threads, cudaStream_t st);

}  // namespace kzgb
