// The context (one GPU) and the host functions shared by the single-call entry points (capi.cu) and the
// blob-batch pipelines (batch.cu).  The functions declared here are defined in capi.cu.
#pragma once
#include <atomic>
#include <chrono>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/kzg_bn254_b200.h"
#include "kzgb_internal.hpp"

namespace kzgb {

constexpr int MAX_LANES = 8;
constexpr int MAX_SETS = 96;

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        size_t want = (bytes + (1u << 20) - 1) & ~(size_t)((1u << 20) - 1);
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

struct Lane {
    cudaStream_t st = nullptr;      // everything but the bucket accumulation (high priority when owned)
    cudaStream_t st_acc = nullptr;  // bucket accumulation: low priority, so other lanes' short kernels
                                    // slip in between its blocks instead of queueing behind the whole grid
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    bool own_stream = false;
    DevBuf bytes, evals, work, ntt_scratch, eval_scratch, msm_ws, small, bases, bucket_total;
    XYZZ* h_sets = nullptr;   // pinned
    uint32_t* h_entries = nullptr;  // pinned: length of the sorted list of the MSM in flight (= its point additions)
    Fr* h_fr = nullptr;       // pinned, 16 elements
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_done = nullptr, ev_block = nullptr;
    bool ev_pending = false;
    double acc_ms = 0;        // summed duration of bucket-accumulation kernels
    uint64_t acc_launches = 0;
    uint64_t acc_adds = 0;    // sorted-list entries those kernels consumed (every entry is one point addition or install)
};

}  // namespace kzgb

struct kzgb_ctx {
    int device = 0;
    std::mutex mu;
    std::string err;
    kzgb::Lane lanes[kzgb::MAX_LANES];
    int n_lanes = 0;
    // SRS
    kzgb::Affine* srs = nullptr;
    size_t srs_n = 0;
    kzgb::Affine* wtable = nullptr;   // fixed-base window table over SRS points [wt_first, wt_first + wt_n)
    size_t wt_first = 0, wt_n = 0;
    int wt_c = 0, wt_W = 0;
    bool auto_precompute = true;
    std::atomic<bool> lanes_running{false};  // a batch pipeline is driving the lanes: tables are read-only
    bool set_l2_limit = false;
    // Lagrange-basis tables, one per domain size 2^k: window table over L = IFFT_G1(SRS[..2^k]) so that
    // evaluation-form commitments are ONE MSM on the evaluations themselves (no Fr NTT on the path)
    struct LagTable { kzgb::Affine* table = nullptr; size_t n = 0; int c = 0, W = 0; uint64_t last_use = 0; uint32_t calls = 0; } lag[29];
    uint64_t lag_clock = 0;
    kzgb::DevBuf batch_bytes;  // blob bytes of the batch in flight (commit_and_prove_blobs)
    // twiddles
    kzgb::Fr* tw = nullptr;
    int logN = 0;
    // timer
    cudaEvent_t t0 = nullptr, t1 = nullptr;
    // device-side hashing of long Fiat-Shamir transcripts (fs.cu k_fs_midstate_long): its stream, the mapped host block the
    // kernel reports through ([state 8 x cap | done cap | cancel 1] words) and the device-side argument arrays
    cudaStream_t hash_st = nullptr;
    cudaEvent_t ev_hash_uploaded = nullptr;
    uint32_t* fsl_host = nullptr;
    std::atomic<bool> lanes_block{false};  // lanes of the running large-blob batch sleep on a blocking event (lane_wait)
    kzgb::DevBuf fsl_args;
    // upload stream + double-buffer fences of msm_srs_host_pipelined
    cudaStream_t copy_st = nullptr;
    cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_consumed[2] = {nullptr, nullptr};
    // timeline trace (kzgb_trace_begin / kzgb_trace_end, include/kzg_bn254_b200_bench.h): device events and host time
    // stamps of every MSM of every lane, for reading pipeline stalls without a system profiler
    struct TraceRec { int lane, kind; cudaEvent_t ev; double host_ms; };
    std::atomic<bool> trace_on{false};
    std::mutex trace_mu;
    std::vector<TraceRec> trace;
    cudaEvent_t trace_base = nullptr;
    std::chrono::steady_clock::time_point trace_host0;
};

namespace kzgb {

// ---- options (kzgb_set_option; 0 / -1 = the library's own choice)
// -1: choose per call, 0: host SHA-256 pool, 1: device kernel (verify_batch_rlc challenges)
inline std::atomic<int> g_fs_device{-1};
// -1: auto, 0: one blob at a time, > 0: blobs per group in the small-blob batch path
inline std::atomic<int> g_group{-1};
// points per chunk of the streamed SRS ingest (0 = 2^22); tests shrink it to cross chunk boundaries
inline std::atomic<long> g_srs_chunk{0};
inline std::atomic<int> g_group_members{1};  // largest kzgb_group alive in this process
// 1: evaluation-form commitments use a Lagrange-basis window table (built on first use per size), 0: Fr-IFFT + monomial table
inline std::atomic<int> g_lagrange{1};
inline std::atomic<int> g_lagrange_after{2};       // build the Lagrange table of a size at its k-th evaluation-form use
inline std::atomic<long> g_lagrange_budget_mib{0}; // 0 = half of the device memory
inline std::atomic<int> g_lanes{0};            // lanes of the blob-batch pipelines
inline std::atomic<int> g_hash_threads{0};     // host SHA-256 pool threads per batch call
inline std::atomic<int> g_lane_wait{-1};       // -1 auto, 0 spin on the stream, 1 poll with short sleeps
inline std::atomic<int> g_stream_priority{1};  // 1: bucket accumulation on a low-priority stream of its own
inline std::atomic<int> g_l2_fetch_64{1};      // 1: contexts that own their stream set the L2 fetch granularity to 64 B
inline std::atomic<int> g_device_hash{-1};        // blobs of a large-blob batch whose transcript is hashed on the device: -1 auto, 0 none, k > 0 the last k
inline std::atomic<int> g_hash_trace{0};         // option "hash_trace": 1 = every multi-buffer group reports its wall and CPU time on stderr
inline std::atomic<int> g_hash_nice{1};          // 1: the SHA-256 pool threads of a batch call run at the lowest nice level
inline std::atomic<int> g_hash_mb{-1};            // AVX-512 multi-buffer SHA-256 for deep large-blob batches: -1 auto, 0 never, 1 whenever a group of 16 forms
inline std::atomic<int> g_pipelined_upload{1};   // 1: host scalars of MSMs of >= 2^22 points over a window table are uploaded in overlapped chunks
inline std::atomic<long> g_batch_keep_mib{4096};  // blob staging buffer of kzgb_commit_and_prove_blobs kept between calls up to this size

// ---- errors
int fail(kzgb_ctx* c, int code, const std::string& msg);
#define CK(ctx, call)                                                                              \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(ctx, KZGB_ERR_DEVICE, std::string("CUDA error: ") + cudaGetErrorString(e_) + " at " #call); \
    } while (0)
// KZGB_ERR_SRS_CAPACITY unless a polynomial of n coefficients fits the loaded SRS (kzg.rs:89-94)
int check_srs_capacity(kzgb_ctx* c, size_t n);

// Holds the context's lock and makes its device current for the length of an entry point.
struct Guard {
    kzgb_ctx* c;
    int prev = -1;
    std::unique_lock<std::mutex> lk;
    explicit Guard(kzgb_ctx* ctx) : c(ctx), lk(ctx->mu) { cudaGetDevice(&prev); cudaSetDevice(ctx->device); }
    ~Guard() { if (prev >= 0) cudaSetDevice(prev); }
};

// ---- host helpers
int log2_exact(size_t n);
size_t next_pow2(size_t n);
size_t blob_poly_len(size_t len);
Fr ninv_mont(int logn);
Fr eval_tinv(const Fr& z, int logn, bool* in_domain = nullptr);
void affine_to_abi(const Affine& a, uint64_t out_xy[8], uint8_t* out_inf);
Affine affine_from_abi(const uint64_t xy[8], uint8_t inf);

// ---- lanes and tables
int ensure_lanes(kzgb_ctx* c, int want);
int ensure_twiddles(kzgb_ctx* c, int logn);
int ensure_lagrange(kzgb_ctx* c, int logn, uint32_t weight = 1, bool force = false);
int do_precompute(kzgb_ctx* c, size_t first, size_t count, int window_bits);
bool lane_wait_polls();

// ---- MSM and polynomial pieces (enqueue on the lane, finish waits for it)
struct MsmJob {
    MsmPlan plan;
    bool active = false;
};
int msm_finish(kzgb_ctx* c, Lane& L, const MsmJob& job, Affine* out);
int msm_blocking(kzgb_ctx* c, Lane& L, const Fr* d_scalars, bool canonical, size_t first, size_t n,
                 const Affine* var_bases, Affine* out);
int msm_enqueue_batched(kzgb_ctx* c, Lane& L, const Fr* d_scalars, size_t n_per, size_t batch,
                        const kzgb_ctx::LagTable* lag, MsmJob* job);
int msm_finish_batched(kzgb_ctx* c, Lane& L, const MsmJob& job, size_t batch, Affine* outs);
int commit_evals_enqueue(kzgb_ctx* c, Lane& L, const Fr* d_evals, size_t n, MsmJob* job);
int proof_enqueue(kzgb_ctx* c, Lane& L, const Fr* d_evals, size_t n, const Fr& z_mont, MsmJob* job);
int blob_to_evals(kzgb_ctx* c, Lane& L, const uint8_t* blob_host, const uint8_t* blob_dev, size_t len, size_t n);

}  // namespace kzgb
