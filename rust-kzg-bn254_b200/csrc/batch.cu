// The blob-batch pipelines: kzgb_commit_and_prove_blobs{,_dev} -- commitment and proof of many blobs on several lanes
// while a hashing stage produces the Fiat-Shamir transcripts --, kzgb_commit_blobs{,_dev} -- the commitments alone, on
// the same plan and lanes --, kzgb_compute_blob_proofs{,_dev} -- the proofs alone, against the caller's commitments --,
// kzgb_compute_proofs{,_dev} -- proofs of evaluation-form polynomials at the caller's points, on the same plan and lanes --
// and the verifier's calls, kzgb_verify_blob_proofs{,_g1}{,_dev} and kzgb_verify_batch_rlc{,_dev}, over one per-blob stage,
// kzgb_verify_kzg_proof_batch_rlc, the random linear combination alone over openings the caller has evaluated, and
// kzgb_verify_proofs, the pairing check of each such opening.
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <ctime>
#include <mutex>
#include <string>
#include <thread>
#include <utility>
#include <vector>
#include <sys/resource.h>
#include <sys/syscall.h>
#include <unistd.h>

#include "../../include/kzg_bn254_b200.h"
#include "ctx.hpp"
#include "sha256.hpp"
#include "transcript.hpp"

using namespace kzgb;

namespace {

// Host threads for the SHA-256 pool of one context.  One transcript hash is sequential (~9 ms per 16 MiB
// with SHA-NI).  Measured on the 8-GPU box (32 hardware threads): one thread per blob, even
// oversubscribed, beats a pool sized to this rank's share of the cores (1545 vs 1222 blobs/s) -- at
// 8 GPUs the job is bound by the host's aggregate SHA-256 rate (2.1 GB of transcripts per step).
size_t hash_pool_threads() {
    if (int v = g_hash_threads.load()) return (size_t)v;
    unsigned hw = std::thread::hardware_concurrency();
    if (hw == 0) hw = 8;
    size_t pool = std::min<size_t>(hw > 4 ? hw - 2 : 2, 32);
    // the members of a kzgb_group hash at the same time: share the cores (ranks of a torchrun job are separate
    // processes; measured there, one thread per blob even oversubscribed beats a share of the cores)
    size_t members = (size_t)std::max(1, g_group_members.load());
    return std::max<size_t>(2, pool / members);
}

constexpr size_t FSL_CAP = 4096;  // transcripts one batch call can hand to the device
// Who hashes the Fiat-Shamir transcripts of a large-blob batch (everything but the commitment: challenge_midstate).
//  * single stream: one SHA-NI thread per blob, ~9 ms per 16 MiB, the first challenges ready after 9 ms -- the default
//    whenever the pool keeps up with the GPU (16 spare cores next to one GPU: 29 GB/s against 6 GB/s of blobs);
//  * multi-buffer: groups of 16 equal-size blobs hashed in lockstep on AVX-512 (sha256_mb16_blocks), about twice the bytes
//    per second of a core, the 16 midstates arrive together (71-80 ms for 16 MiB blobs) -- for deep batches on a host
//    whose single-stream pool is slower than the GPU (8 ranks on 32 hardware threads: 36 GB/s against 49 GB/s;
//    profiles/r02_scale8.txt: 2184 -> 2857 blobs/s);
//  * device: the last k blobs on the GPU next to the MSMs, one warp (0.45 s, 16 % of a blob's MSM work in issue slots) or
//    one lane (0.9 s: a warp instruction occupies the 16-wide integer ALU for two cycles and the lane does schedule and
//    rounds alone; half a percent) per transcript -- only a batch several hundred blobs deep hides that latency.
struct HashPlan {
    bool mb = false;        // multi-buffer groups on the host
    size_t mb_threads = 0;  // host threads in multi-buffer mode
    size_t head = 0;        // multi-buffer mode: blobs [0, head) are hashed single-stream before the first group
    size_t dev_k = 0;       // transcripts hashed on the device (the last dev_k blobs)
    bool dev_lanes = false; // k_fs_midstate_lanes instead of k_fs_midstate_long
};
// proof_only (kzgb_compute_blob_proofs): no commit phase hides the first transcripts, and a blob's whole GPU work follows
// its transcript.
HashPlan hash_plan(const size_t* lens, size_t count, bool device_possible, bool proof_only) {
    HashPlan hp;
    if (count < 2) return hp;
    double bytes = 0;
    for (size_t i = 0; i < count; i++) bytes += (double)lens[i];
    const double per_blob = bytes / (double)count;
    unsigned hw = std::thread::hardware_concurrency();
    if (hw == 0) hw = 8;
    int procs = g_group_members.load();
    if (const char* w = getenv("LOCAL_WORLD_SIZE")) { int v = atoi(w); if (v > procs) procs = v; }
    const double share = std::max(1.0, (double)hw / procs);                                          // hardware threads of this context
    const double rate_ni = 1.2e9 * std::max(1.0, std::min<double>((double)hash_pool_threads(), share));  // B/s, HT siblings both hashing
    // GPU time of one blob: commit + proof, or (proof_only) the proof alone: 1.6e-3 s = 1 / 622 blobs/s, the rate of
    // kzgb_compute_blob_proofs_dev at 64 x 2^19 Fr with the single-stream pool keeping up (scripts/blob_proofs_bench.py,
    // B200 at 1000 W, 16 hardware threads; the ~9 ms to the first transcript included)
    const double t_gpu = (proof_only ? 1.6e-3 : 2.75e-3) * per_blob / (double)(16u << 20);
    const double after_hash = proof_only ? 1.0 : 0.5;  // the share of t_gpu that waits for the blob's transcript
    // eligible blobs: exactly 32 * 2^j bytes, j >= 10 (the multi-buffer and device kernels hash whole 64-byte blocks)
    size_t eligible_total = 0, eligible_tail = 0;
    for (size_t i = 0; i < count; i++) eligible_total += hash_mb_eligible(lens[i]);
    while (eligible_tail < count && eligible_tail < FSL_CAP && hash_mb_eligible(lens[count - 1 - eligible_tail])) eligible_tail++;
    const int mb_opt = g_hash_mb.load();
    // "keeps up" = the single-stream pool needs at most half of this context's hardware threads for the duration of the GPU work:
    // the other half belongs to the lanes and the driver (measured on 4 hardware threads per rank: 291 blobs/s single stream, 367 multi-buffer)
    const bool ni_keeps_up = bytes / rate_ni <= 0.5 * count * t_gpu;
    const int ht = g_hash_threads.load();
    const size_t mb_threads = (size_t)std::max(1.0, ht > 0 ? (double)ht : share - 1.0);  // one hardware thread of the share stays with the lanes
    // proof_only: multi-buffer only where the groups the batch forms hash faster than the pool (64 blobs are 4 groups,
    // 4 threads: 418 blobs/s against 622 single-stream on 16 hardware threads)
    const bool mb_faster = !proof_only || 2.4e9 * (double)std::min(mb_threads, eligible_total / 16) > rate_ni;
    if (sha256_has_mb16() && mb_opt != 0 && eligible_total >= 16 && (mb_opt == 1 || (!ni_keeps_up && mb_faster && eligible_total >= 32))) {
        hp.mb = true;
        hp.mb_threads = mb_threads;
        // the 16 midstates of a group arrive together after 71-80 ms (16 MiB blobs): without a commit phase the lanes would
        // idle that long, so every hashing thread first hashes one blob of the head single-stream (~9 ms)
        if (proof_only) hp.head = std::min(count, hp.mb_threads);
    }
    const int dev_opt = device_possible ? g_device_hash.load() : 0;
    if (dev_opt > 0) { hp.dev_k = std::min<size_t>((size_t)dev_opt, eligible_tail); hp.dev_lanes = fs_midstate_lanes() != 0; return hp; }
    if (dev_opt == 0 || !eligible_tail) return hp;
    const double rate_host = hp.mb ? 2.4e9 * (double)hp.mb_threads : rate_ni;
    double best = std::max(count * t_gpu, bytes / rate_host);
    for (int lanes = 0; lanes < 2; lanes++) {
        if (fs_midstate_lanes() >= 0 && lanes != fs_midstate_lanes()) continue;
        const double t_dev = (lanes ? 0.95 : 0.45) * per_blob / (double)(16u << 20), dev_cost = lanes ? 0.006 : 0.16;
        for (size_t k = 1; k <= eligible_tail; k++) {
            // GPU busy time; host time for the front of the batch; the device's share lands at t_dev and its proofs follow
            const double t = std::max({(count + dev_cost * k) * t_gpu, (double)(count - k) * per_blob / rate_host, t_dev + k * t_gpu * after_hash});
            if (t < best * 0.97) { best = t; hp.dev_k = k; hp.dev_lanes = lanes != 0; }
        }
    }
    return hp;
}

// ---------------------------------------------------------------- planning
// What a batch computes: kzgb_commit_and_prove_blobs{,_dev}, kzgb_commit_blobs{,_dev} (commitments, no transcripts),
// kzgb_compute_blob_proofs{,_dev} (proofs against the caller's commitments, no commit phase) or kzgb_compute_proofs{,_dev}
// (proofs of the caller's Montgomery evaluations at the caller's points: no blob bytes, no transcripts, no commitments) or
// kzgb_commit_evals{,_dev} / kzgb_commit_coeffs{,_dev} (commitments of the caller's polynomials, in evaluation or
// coefficient form: no blob bytes, no transcripts, no proofs).
enum class Job { CommitAndProve, Commit, Prove, ProveAt, CommitPolys };

// One batch call: its arguments and the plan made for them.  The entry points set their job's outputs by name.
struct Batch {
    Batch(kzgb_ctx* c, Job job, const uint8_t* const* blobs_dev, const uint8_t* const* blobs_host, const size_t* lens,
          size_t count)
        : c(c), job(job), blobs_dev(blobs_dev), blobs_host(blobs_host), lens(lens), count(count) {}
    kzgb_ctx* c;
    Job job;
    const uint8_t* const* blobs_dev;   // nullptr: the blobs are only on the host
    const uint8_t* const* blobs_host;  // the transcripts are hashed from these (Commit with blobs_dev: nullptr)
    const size_t* lens;
    size_t count;
    uint8_t* commitments32 = nullptr;  // CommitAndProve: compressed points
    uint8_t* proofs32 = nullptr;
    uint64_t* out_xy = nullptr;        // Commit, Prove: the affine ABI, out_inf optional
    uint8_t* out_inf = nullptr;
    const uint64_t* commitments_xy = nullptr;  // Prove: the caller's commitments in the ABI ...
    const uint8_t* commitments_inf = nullptr;
    std::vector<Affine> commits;               // ... read and checked by plan_batch
    // ProveAt: polynomial i is ns[i] Montgomery evaluations at evals[i] (device memory when evals_on_device), opened at the
    // 4 words zs_mont + 4 i; its y goes to ys_mont + 4 i (optional).  lens[i] = 32 ns[i], so that the plan groups the
    // polynomials as it groups blobs of that many bytes.
    const uint64_t* const* evals = nullptr;
    bool evals_on_device = false;
    const size_t* ns = nullptr;
    const uint64_t* zs_mont = nullptr;
    uint64_t* ys_mont = nullptr;
    // CommitPolys: polynomial i is ns[i] Montgomery values at evals[i] (as ProveAt), coefficients when `coeff`, and
    // lens[i] = 32 N_i for its domain N_i (ns[i], or next_pow2(ns[i]) for coefficients).  plan_batch sorts the entries
    // stably by N_i: from then on evals, ns and lens are in that order, and entry k of the batch is the caller's order[k].
    bool coeff = false;
    std::vector<size_t> order;
    std::vector<const uint64_t*> sorted_evals;
    std::vector<size_t> sorted_ns, sorted_lens;
    size_t max_n = 0;
    std::vector<std::pair<size_t, size_t>> groups;  // small blobs: (first blob, blobs); empty: one blob per task
    int n_lanes = 0;
    bool deep = false;              // the lanes sleep on a blocking event while they wait (lane_wait)
    std::vector<size_t> byte_off;   // resident: offset of every blob in c->batch_bytes
    bool resident = false;
};

// the 4 little-endian words at w hold a value below r
bool fr_words_reduced(const uint64_t* w) {
    uint32_t r[8];
    FeConst<FR>::mod(r);
    for (int k = 7; k >= 0; k--) {
        const uint32_t x = (uint32_t)(w[k / 2] >> (32 * (k & 1)));
        if (x != r[k]) return x < r[k];
    }
    return false;
}

// Validation, groups, lanes and the tables every size of the batch needs.  A commit-only batch checks every blob as
// kzgb_commit_blob does (a blob of length 0 commits the zero polynomial of size 1); with proofs, length 0 is
// compute_blob_proof's error, and a proof-only batch checks each commitment first, as kzgb_compute_blob_proof does.
// Proofs at the caller's points check each polynomial as kzgb_compute_proof does, then its z.  Commitments of the
// caller's polynomials check each one as kzgb_commit_eval or kzgb_commit_coeff does.
int plan_batch(Batch& b) {
    kzgb_ctx* c = b.c;
    const size_t* lens = b.lens;
    const size_t count = b.count;
    for (size_t i = 0; i < count; i++) {
        if (b.job == Job::CommitPolys) {
            const size_t n = b.ns[i];
            if (b.coeff) {
                if (n > c->srs_n) return fail(c, KZGB_ERR_SERIALIZATION, "polynomial length is not correct");
            } else {
                if (int rc = check_srs_capacity(c, n)) return rc;
                if (n == 0 || (n & (n - 1))) return fail(c, KZGB_ERR_FFT, "length provided is not a power of 2");
            }
        } else if (b.job == Job::ProveAt) {
            const size_t n = b.ns[i];
            if (n == 0 || (n & (n - 1))) return fail(c, KZGB_ERR_FFT, "length provided is not a power of 2");
            if (int rc = check_srs_capacity(c, n)) return rc;
            if (!fr_words_reduced(b.zs_mont + 4 * i))
                return fail(c, KZGB_ERR_INVALID_FIELD_ELEMENT, "z of opening " + std::to_string(i) + " is not a reduced field element");
        } else if (b.job == Job::Commit) {
            if (int rc = check_commit_blob_len(c, blob_poly_len(lens[i]))) return rc;
        } else {
            if (b.job == Job::Prove) {
                b.commits.push_back(affine_from_abi(b.commitments_xy + 8 * i, b.commitments_inf ? b.commitments_inf[i] : 0));
                if (!aff_on_curve(b.commits[i])) return fail(c, KZGB_ERR_NOT_ON_CURVE, "G1 point not on curve");
            }
            if (lens[i] == 0) return fail(c, KZGB_ERR_GENERIC, "Length of data after padding is 0");
            if (int rc = check_srs_capacity(c, blob_poly_len(lens[i]))) return rc;
        }
        b.max_n = std::max(b.max_n, blob_poly_len(lens[i]));
    }
    // A commitment batch gathers every polynomial of a group anyway (group_evals), so its groups are cut from the entries
    // sorted by size rather than from adjacent runs: polynomials of mixed sizes in any order still form full groups, and
    // device polynomials of one size that are back to back stay so.
    if (b.job == Job::CommitPolys) {
        b.order.resize(count);
        for (size_t i = 0; i < count; i++) b.order[i] = i;
        std::stable_sort(b.order.begin(), b.order.end(), [&](size_t x, size_t y) { return b.lens[x] < b.lens[y]; });
        for (size_t k = 0; k < count; k++) {
            b.sorted_evals.push_back(b.evals[b.order[k]]);
            b.sorted_ns.push_back(b.ns[b.order[k]]);
            b.sorted_lens.push_back(b.lens[b.order[k]]);
        }
        b.evals = b.sorted_evals.data();
        b.ns = b.sorted_ns.data();
        b.lens = lens = b.sorted_lens.data();
    }
    // Small blobs (<= 2^17 Fr): runs of equal-size blobs are processed as groups, every kernel of a phase
    // launched ONCE for the whole group (batched conversion, evaluation/quotient and MSM with one bucket set
    // per blob) -- one blob at a time they are latency-bound (bucket-reduction tail, host hand-off per MSM).
    const int group_opt = g_group.load();
    if (group_opt != 0 && count >= 2 && b.max_n <= ((size_t)1 << 17) && c->auto_precompute && c->srs_n <= ((size_t)1 << 22)) {
        for (size_t i = 0; i < count;) {
            size_t n = blob_poly_len(lens[i]);
            size_t cap = group_opt > 0 ? (size_t)group_opt : std::max<size_t>(1, ((size_t)1 << 21) / n);
            cap = std::min<size_t>(cap, 64);
            size_t j = i + 1;
            while (j < count && j - i < cap && blob_poly_len(lens[j]) == n) j++;
            b.groups.emplace_back(i, j - i);
            i = j;
        }
    }
    // lanes in flight: 3 keep the GPU full on 16 MiB blobs; small blobs are latency-bound per lane
    // (bucket reduction, host hand-offs), so they get more
    // Large-blob batches: 6 lanes whose threads SLEEP on a blocking event while their MSM runs (measured against 4 spinning
    // lanes: 342 -> 353 blobs/s e2e with 16 hardware threads, and the only form that leaves a rank of the 8-GPU box -- 4
    // hardware threads -- its cores for hashing: profiles/r02_host_hashing.txt, r02_scale8.txt).  The wake-up latency of a blocking event (~0.1-0.3 ms) hides
    // behind the other lanes; single calls and the latency-bound small-blob groups keep spinning.
    const int lanes_env = g_lanes.load();
    // (a rank short of cores -- lane_wait auto = poll -- with a shallow batch is the exception: 4 polling lanes, measured 316
    // against 288 blobs/s at 16 blobs per step on 4 hardware threads)
    b.deep = b.groups.empty() && count >= 4 && (count >= 32 || !lane_wait_polls());
    int want_lanes = lanes_env > 0 ? lanes_env : (b.deep ? 6 : (b.max_n >= ((size_t)1 << 18) ? 4 : 6));
    if (!b.groups.empty() && lanes_env <= 0) want_lanes = 3;
    b.n_lanes = (int)std::min<size_t>(b.groups.empty() ? count : b.groups.size(), (size_t)std::min(want_lanes, MAX_LANES));
    int rc = ensure_lanes(c, b.n_lanes);
    if (rc) return rc;
    rc = ensure_twiddles(c, log2_exact(b.max_n));
    if (rc) return rc;
    bool all_lagrange = true;
    for (size_t i = 0; i < count; i++) {
        int logn = log2_exact(blob_poly_len(lens[i]));
        rc = ensure_lagrange(c, logn);
        if (rc) return rc;
        if (!lagrange_table(c, logn)) all_lagrange = false;
    }
    // built here: the lanes only read the tables (coefficient tasks always run over the monomial one)
    rc = all_lagrange && !b.coeff ? KZGB_OK : ensure_window_table(c, 0, std::min(b.max_n, c->srs_n));
    if (rc) return rc;
    for (size_t gi = 0; gi < b.groups.size(); gi++) {  // the batched MSM needs a window table for every size
        size_t n = blob_poly_len(lens[b.groups[gi].first]);
        if (!lagrange_table(c, log2_exact(n)) && !wtable_covers(c, 0, n)) { b.groups.clear(); break; }
    }
    return KZGB_OK;
}

// Blob bytes stay resident on the device between a blob's commit and its proof (one H2D per blob).
void stage_blob_bytes(Batch& b) {
    if (b.blobs_dev || !b.groups.empty()) return;
    b.byte_off.assign(b.count, 0);
    size_t total = 0;
    for (size_t i = 0; i < b.count; i++) { b.byte_off[i] = total; total += (b.lens[i] + 255) & ~(size_t)255; }
    if (total <= ((size_t)16 << 30) && b.c->batch_bytes.reserve(total) == cudaSuccess) b.resident = true;
    else cudaGetLastError();
}

// ---------------------------------------------------------------- hashing stage
// What the lanes of one batch share: a lane that fails stops the others.  The hashing stage and the large-blob task
// queue keep their state under the same lock and signal on the same condition.
struct LaneSync {
    std::mutex mu;
    std::condition_variable cv;
    std::atomic<bool> failed{false};  // set under mu, so that a wait on cv sees it
    void fail() {
        std::lock_guard<std::mutex> lk(mu);
        failed = true;
        cv.notify_all();
    }
};

// Transcript midstates (everything but the commitment): a pool of host threads from the front of the batch and, when
// the host cannot keep up with the GPU, one warp per transcript on the device for the blobs at its end
// (device_hash_share).  Whoever delivers a midstate first installs it; the lanes take proofs as they become ready.
class HashStage {
public:
    LaneSync& sync;
    std::vector<Sha256> mid;   // midstate of blob i, once ready[i]
    std::vector<uint8_t> ready;
    const size_t dev_first;    // blobs [dev_first, count) are the device's share

    HashStage(const Batch& batch, const HashPlan& hp, LaneSync& sync);
    // The one teardown, on every exit path: stop the device hashing and wait for it (it reads the blob bytes), then
    // for the pool.
    ~HashStage();
    // Waits for the midstates of blobs [first, first + n); false: a lane failed.
    bool wait_ready(size_t first, size_t n) {
        std::unique_lock<std::mutex> lk(sync.mu);
        for (size_t k = 0; k < n; k++) sync.cv.wait(lk, [&] { return ready[first + k] != 0 || sync.failed.load(); });
        return !sync.failed.load();
    }
    // blob i went up to c->batch_bytes on the hashing stream (ev_hash_uploaded)
    bool uploaded_here(size_t i) const { return i >= dev_first && !dev_failed.load(); }

private:
    struct Task { size_t first, members; };  // one blob on a single stream, or up to 16 equal-size blobs in lockstep
    const Batch& b;
    kzgb_ctx* const c;
    const size_t dev_k;
    std::atomic<bool> dev_failed{false};  // the device share did not start: the pool hashes it
    std::atomic<bool> dev_stop{false};
    uint32_t* fsl_state = nullptr;
    volatile uint32_t* fsl_done = nullptr;
    volatile uint32_t* fsl_cancel = nullptr;
    std::thread poller;
    std::vector<Task> tasks;
    std::atomic<size_t> next_task{0};
    std::vector<std::thread> pool;

    cudaError_t start_device(bool lanes);
    void poll_device();
    void hash_tasks();
    void install(size_t i, const Sha256& sh) {
        std::lock_guard<std::mutex> lk(sync.mu);
        if (!ready[i]) { mid[i] = sh; ready[i] = 1; }
    }
};

HashStage::HashStage(const Batch& batch, const HashPlan& hp, LaneSync& sync)
    : sync(sync), mid(batch.count), ready(batch.count, 0), dev_first(batch.count - hp.dev_k), b(batch), c(batch.c), dev_k(hp.dev_k) {
    if (dev_k && start_device(hp.dev_lanes) != cudaSuccess) { cudaGetLastError(); dev_failed.store(true); }  // the host pool takes the whole batch
    if (dev_k && !dev_failed.load()) poller = std::thread(&HashStage::poll_device, this);
    for (size_t i = 0; i < b.count;) {
        size_t j = i + 1;
        if (hp.mb && i >= hp.head && i < dev_first && hash_mb_eligible(b.lens[i])) {
            while (j < dev_first && j - i < 16 && b.lens[j] == b.lens[i]) j++;
            if (j - i < 8) j = i + 1;  // a group under half full hashes no faster than its members one by one
        }
        tasks.push_back({i, j - i});
        i = j;
    }
    size_t n_hash = std::max<size_t>(1, std::min<size_t>(tasks.size(), hp.mb ? hp.mb_threads : hash_pool_threads()));
    for (size_t t = 0; t < n_hash; t++) pool.emplace_back(&HashStage::hash_tasks, this);
}

HashStage::~HashStage() {
    { std::lock_guard<std::mutex> lk(sync.mu); dev_stop.store(true); }
    if (fsl_cancel) *fsl_cancel = 1;
    next_task.store(tasks.size());
    sync.cv.notify_all();
    if (poller.joinable()) poller.join();
    for (auto& t : pool) t.join();
    if (dev_k && c->hash_st) cudaStreamSynchronize(c->hash_st.get());
}

// The device's share: host blobs go up on the hashing stream, then one kernel hashes all of it.
cudaError_t HashStage::start_device(bool lanes) {
    cudaError_t e = cudaSuccess;
    if (!c->hash_st) {  // the stream, its event and the mapped block go into the context together or not at all
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        StreamPtr st;
        EventPtr uploaded;
        HostPtr<uint32_t[]> host;
        e = stream_create(st, hi);  // its few blocks must become resident at once
        if (e == cudaSuccess) e = event_create(uploaded, cudaEventDisableTiming);
        if (e == cudaSuccess) e = host_alloc(host, (9 * FSL_CAP + 16) * 4, cudaHostAllocMapped);
        if (e != cudaSuccess) return e;
        c->hash_st = std::move(st); c->ev_hash_uploaded = std::move(uploaded); c->fsl_host = std::move(host);
    }
    e = c->fsl_args.reserve(FSL_CAP * 16);
    if (e != cudaSuccess) return e;
    fsl_state = c->fsl_host.get();
    fsl_done = fsl_state + 8 * FSL_CAP;
    fsl_cancel = fsl_state + 9 * FSL_CAP;
    for (size_t j = 0; j < dev_k; j++) fsl_done[j] = 0;
    *fsl_cancel = 0;
    std::vector<const uint8_t*> ptrs(dev_k);
    std::vector<uint32_t> ns(dev_k);
    for (size_t j = 0; j < dev_k && e == cudaSuccess; j++) {
        const size_t i = dev_first + j;
        ns[j] = (uint32_t)(b.lens[i] / 32);
        if (b.blobs_dev) ptrs[j] = b.blobs_dev[i];
        else {
            uint8_t* slot = (uint8_t*)c->batch_bytes.p + b.byte_off[i];
            e = cudaMemcpyAsync(slot, b.blobs_host[i], b.lens[i], cudaMemcpyHostToDevice, c->hash_st.get());
            ptrs[j] = slot;
        }
    }
    const uint8_t** d_ptrs = (const uint8_t**)c->fsl_args.p;
    uint32_t* d_ns = (uint32_t*)((char*)c->fsl_args.p + FSL_CAP * 8);
    if (e == cudaSuccess) e = cudaEventRecord(c->ev_hash_uploaded.get(), c->hash_st.get());
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_ptrs, ptrs.data(), dev_k * 8, cudaMemcpyHostToDevice, c->hash_st.get());
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_ns, ns.data(), dev_k * 4, cudaMemcpyHostToDevice, c->hash_st.get());
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->hash_st.get());  // the argument vectors die with this scope
    if (e != cudaSuccess) return e;
    fs_midstate_long_launch(d_ptrs, d_ns, (uint32_t)dev_k, fsl_state, (uint32_t*)fsl_done, (const uint32_t*)fsl_cancel, lanes, c->hash_st.get());
    return cudaGetLastError();
}

// Installs the device's midstates as their completion flags appear in mapped memory.
void HashStage::poll_device() {
    std::vector<uint8_t> seen(dev_k, 0);
    size_t remaining = dev_k;
    while (remaining && !dev_stop.load()) {
        bool any = false;
        for (size_t j = 0; j < dev_k; j++) {
            if (seen[j] || !fsl_done[j]) continue;
            std::atomic_thread_fence(std::memory_order_acquire);
            uint32_t st[8];
            for (int w = 0; w < 8; w++) st[w] = fsl_state[8 * j + w];
            const size_t i = dev_first + j;
            install(i, challenge_midstate_resume(st, b.blobs_host[i], b.lens[i] / 32));
            seen[j] = 1; remaining--; any = true;
        }
        if (any) sync.cv.notify_all();
        else { struct timespec ts = {0, 100000}; nanosleep(&ts, nullptr); }
    }
}

// One thread of the pool: takes hash tasks in blob order.
void HashStage::hash_tasks() {
    // The pool is pure throughput work; the lane threads next to it are latency work (every microsecond a lane
    // wakes up late is a microsecond its stream may run dry).  Where both share a few cores (8 ranks on 32
    // hardware threads) the hashers yield to them: lowest nice level for this thread only.
    if (g_hash_nice.load()) setpriority(PRIO_PROCESS, (id_t)syscall(SYS_gettid), 19);
    for (;;) {
        size_t ti = next_task.fetch_add(1);
        if (ti >= tasks.size()) return;
        const size_t i = tasks[ti].first, members = tasks[ti].members;
        if (members > 1) {
            uint32_t st[16][8];
            struct timespec w0, w1, c0, c1;
            const bool trace = g_hash_trace.load() != 0;
            if (trace) { clock_gettime(CLOCK_MONOTONIC, &w0); clock_gettime(CLOCK_THREAD_CPUTIME_ID, &c0); }
            challenge_midstates_mb16(b.blobs_host + i, members, b.lens[i] / 32, st);
            if (trace) {  // option "hash_trace": wall and CPU time of the group -- tells a descheduled pool from a slow one
                clock_gettime(CLOCK_MONOTONIC, &w1); clock_gettime(CLOCK_THREAD_CPUTIME_ID, &c1);
                fprintf(stderr, "[hash] group at blob %zu (%zu members): wall %.1f ms, cpu %.1f ms\n", i, members,
                        (w1.tv_sec - w0.tv_sec) * 1e3 + (w1.tv_nsec - w0.tv_nsec) * 1e-6, (c1.tv_sec - c0.tv_sec) * 1e3 + (c1.tv_nsec - c0.tv_nsec) * 1e-6);
            }
            for (size_t m = 0; m < members; m++) install(i + m, challenge_midstate_resume(st[m], b.blobs_host[i + m], b.lens[i + m] / 32));
            sync.cv.notify_all();
            continue;
        }
        if (i >= dev_first) {  // the device's share: only if the device path failed
            std::unique_lock<std::mutex> lk(sync.mu);
            sync.cv.wait(lk, [&] { return ready[i] != 0 || sync.failed.load() || dev_failed.load() || dev_stop.load(); });
            if (ready[i] || sync.failed.load() || dev_stop.load()) continue;
        }
        Sha256 sh;
        challenge_midstate(sh, b.blobs_host[i], b.lens[i], blob_poly_len(b.lens[i]));
        install(i, sh);
        sync.cv.notify_all();
    }
}

// ---------------------------------------------------------------- lanes
// lane_main(li) for every lane of the batch: lanes 1 .. n-1 on threads of their own, lane 0 on the calling thread.
// While they run, the lane threads only READ the context's tables (msm_enqueue builds none).  Returns the error of the
// first lane that failed, in lane order.
template <class F>
int run_lanes(const Batch& b, F lane_main) {
    kzgb_ctx* c = b.c;
    c->lanes_block.store(b.deep);
    c->lanes_running.store(true);
    std::vector<int> rc(b.n_lanes, KZGB_OK);
    auto run = [&](int li) { cudaSetDevice(c->device); rc[li] = lane_main(li); };
    std::vector<std::thread> threads;
    for (int li = 1; li < b.n_lanes; li++) threads.emplace_back(run, li);
    run(0);
    for (auto& t : threads) t.join();
    c->lanes_running.store(false);
    c->lanes_block.store(false);
    for (int r : rc) if (r) return r;
    return KZGB_OK;
}

// Where commitment i and proof i go: arkworks-compressed bytes (CommitAndProve), or the affine ABI (the other jobs); the
// commitment of a CommitPolys entry goes to the caller's index of it.
void put_commitment(const Batch& b, size_t i, const Affine& p) {
    if (!b.order.empty()) i = b.order[i];
    if (b.job == Job::CommitAndProve) serialize_compressed(p, b.commitments32 + 32 * i);
    else affine_to_abi(p, b.out_xy + 8 * i, b.out_inf ? b.out_inf + i : nullptr);
}
void put_proof(const Batch& b, size_t i, const Affine& p) {
    if (b.job == Job::CommitAndProve) serialize_compressed(p, b.proofs32 + 32 * i);
    else affine_to_abi(p, b.out_xy + 8 * i, b.out_inf ? b.out_inf + i : nullptr);
}

// The bytes of the bn blobs from blob i0 (all of n elements) at a stride of 32 n with zero-filled tails, so that one launch
// covers the group: device blobs that already are back to back and full are read in place, the others are gathered
// into L.bytes.
int group_bytes(const Batch& b, Lane& L, size_t i0, size_t bn, const uint8_t** src) {
    kzgb_ctx* c = b.c;
    const uint8_t* const* blobs_dev = b.blobs_dev;
    const size_t n = blob_poly_len(b.lens[i0]);
    bool dev_run = blobs_dev != nullptr;
    for (size_t k = 0; k < bn && dev_run; k++) dev_run = b.lens[i0 + k] == n * 32 && blobs_dev[i0 + k] == blobs_dev[i0] + k * n * 32;
    if (dev_run) { *src = blobs_dev[i0]; return KZGB_OK; }
    CK(c, L.bytes.reserve(bn * n * 32));
    for (size_t k = 0; k < bn; k++) {
        uint8_t* dst = (uint8_t*)L.bytes.p + k * n * 32;
        const size_t len = b.lens[i0 + k];
        if (len && blobs_dev) CK(c, cudaMemcpyAsync(dst, blobs_dev[i0 + k], len, cudaMemcpyDeviceToDevice, L.st));
        else if (len) CK(c, cudaMemcpyAsync(dst, b.blobs_host[i0 + k], len, cudaMemcpyHostToDevice, L.st));
        if (len < n * 32) CK(c, cudaMemsetAsync(dst + len, 0, n * 32 - len, L.st));
    }
    *src = (const uint8_t*)L.bytes.p;
    return KZGB_OK;
}

// The commitment phase of one group: bn blobs of one size n from blob i0, ONE batched launch set; pts[k] is the
// commitment of blob i0 + k.  With proofs to follow, or without a Lagrange table, the blob bytes become Montgomery
// evaluations in L.evals (which the proof phase reads).  A commit-only group over a Lagrange table hands the bytes to
// the MSM's first pass instead (group_bytes).
int group_commit(const Batch& b, Lane& L, size_t i0, size_t bn, Affine* pts) {
    kzgb_ctx* c = b.c;
    const uint8_t* const* blobs_dev = b.blobs_dev;
    const size_t* lens = b.lens;
    const size_t n = blob_poly_len(lens[i0]);
    const int logn = log2_exact(n);
    const kzgb_ctx::LagTable* lag = lagrange_table(c, logn);
    MsmJob job;
    if (b.job == Job::Commit && lag) {
        const uint8_t* src = nullptr;
        int r = group_bytes(b, L, i0, bn, &src);
        if (!r) r = msm_enqueue(c, L, {nullptr, src, (uint64_t)bn * n * 32}, n, bn, lag, nullptr, 0, &job);
        if (!r) r = msm_finish(c, L, job, pts);
        return r;
    }
    int r = KZGB_OK;
    auto ck = [&](cudaError_t e, const char* what) {
        if (!r && e != cudaSuccess) r = fail(c, KZGB_ERR_DEVICE, std::string("CUDA error: ") + cudaGetErrorString(e) + " at " + what);
    };
    bool full = true;  // every blob fills its polynomial: one conversion launch for the group
    for (size_t k = 0; k < bn; k++) full = full && lens[i0 + k] == n * 32;
    bool dev_run = blobs_dev && full;  // device blobs back to back: one conversion launch too
    for (size_t k = 0; k < bn && dev_run; k++) dev_run = blobs_dev[i0 + k] == blobs_dev[i0] + k * n * 32;
    ck(L.evals.reserve(bn * n * sizeof(Fr)), "evals");
    if (!blobs_dev) ck(L.bytes.reserve(bn * n * 32), "bytes");
    if (dev_run) bytes_to_fr_launch(blobs_dev[i0], (uint64_t)bn * n * 32, (Fr*)L.evals.p, (uint32_t)(bn * n), L.st);
    for (size_t k = 0; k < bn && !r && !dev_run; k++) {
        const uint8_t* src = blobs_dev ? blobs_dev[i0 + k] : nullptr;
        if (!src) {
            uint8_t* dst = (uint8_t*)L.bytes.p + k * n * 32;
            ck(cudaMemcpyAsync(dst, b.blobs_host[i0 + k], lens[i0 + k], cudaMemcpyHostToDevice, L.st), "H2D copy of a blob");
            src = dst;
        }
        if (!full || blobs_dev) bytes_to_fr_launch(src, lens[i0 + k], (Fr*)L.evals.p + k * n, (uint32_t)n, L.st);
    }
    if (!r && full && !blobs_dev) bytes_to_fr_launch((const uint8_t*)L.bytes.p, (uint64_t)bn * n * 32, (Fr*)L.evals.p, (uint32_t)(bn * n), L.st);
    if (!r) r = commit_evals_enqueue(c, L, (const Fr*)L.evals.p, n, &job, bn);
    if (!r) r = msm_finish(c, L, job, pts);
    return r;
}

// The points of a blob group whose transcript midstates are ready: the challenges of blobs i0 .. i0 + bn - 1 against the
// commitments cs[0 .. bn) and their tinv (eval_tinv) up to L.small as group_prove reads them.  *outside: no challenge is a
// root of the domain.
int group_challenges(const Batch& b, const HashStage& hs, Lane& L, size_t i0, size_t bn, const Affine* cs, bool* outside) {
    kzgb_ctx* c = b.c;
    const int logn = log2_exact(blob_poly_len(b.lens[i0]));
    CK(c, L.small.reserve((3 * bn + 8) * sizeof(Fr)));
    std::vector<Fr> zt(2 * bn);
    bool any_in_domain = false;
    for (size_t k = 0; k < bn; k++) {
        zt[k] = challenge_finish(hs.mid[i0 + k], cs[k]);
        zt[bn + k] = eval_tinv(zt[k], logn, &any_in_domain);
    }
    CK(c, cudaMemcpyAsync(L.small.p, zt.data(), 2 * bn * sizeof(Fr), cudaMemcpyHostToDevice, L.st));
    *outside = !any_in_domain;
    return KZGB_OK;
}

// The points of a group of proofs at the caller's points, entries i0 .. i0 + bn - 1: the caller's z up to L.small, then
// their tinv and in-domain flags on the device (eval_points_launch), laid out as group_prove reads them; the flags follow
// the y.
int group_points_at(const Batch& b, Lane& L, size_t i0, size_t bn, const uint32_t** in_domain) {
    kzgb_ctx* c = b.c;
    const int logn = log2_exact(b.ns[i0]);
    CK(c, L.small.reserve((4 * bn + 8) * sizeof(Fr)));
    Fr* d_z = (Fr*)L.small.p;
    uint32_t* d_flags = (uint32_t*)(d_z + 3 * bn);
    CK(c, cudaMemcpyAsync(d_z, b.zs_mont + 4 * i0, bn * sizeof(Fr), cudaMemcpyHostToDevice, L.st));
    const Fr ninv = ninv_mont(logn);
    eval_points_launch(d_z, logn, (uint32_t)bn, &ninv, d_z + bn, d_flags, L.st);
    *in_domain = d_flags;
    return KZGB_OK;
}

// The values of the polynomials i0 .. i0 + bn - 1 of a ProveAt or CommitPolys group (domain n = blob_poly_len(lens[i0]))
// back to back on the device at a stride of n, zero-filled past ns[i]: device polynomials of n values that already are
// back to back are read in place, the others are gathered into L.evals, one copy per run of polynomials of n values that
// are adjacent in the caller's memory.
int group_evals(const Batch& b, Lane& L, size_t i0, size_t bn, const Fr** evals) {
    kzgb_ctx* c = b.c;
    const uint64_t* const* src = b.evals + i0;
    const size_t* ns = b.ns + i0;
    const size_t n = blob_poly_len(b.lens[i0]);
    auto adjacent = [&](size_t k, size_t run) { return ns[k] == n && ns[k + run] == n && src[k + run] == src[k] + run * 4 * n; };
    size_t run = 1;
    while (run < bn && adjacent(0, run)) run++;
    if (b.evals_on_device && run == bn && ns[0] == n) { *evals = (const Fr*)src[0]; return KZGB_OK; }
    CK(c, L.evals.reserve(bn * n * sizeof(Fr)));
    const cudaMemcpyKind kind = b.evals_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    for (size_t k = 0; k < bn; k += run) {
        run = 1;
        while (k + run < bn && adjacent(k, run)) run++;
        Fr* dst = (Fr*)L.evals.p + k * n;
        const size_t len = run > 1 ? run * n : ns[k];
        if (len) CK(c, cudaMemcpyAsync(dst, src[k], len * sizeof(Fr), kind, L.st));
        if (len < n) CK(c, cudaMemsetAsync(dst + len, 0, (n - len) * sizeof(Fr), L.st));  // zero coefficients add nothing
    }
    *evals = (const Fr*)L.evals.p;
    return KZGB_OK;
}

// The commitments of a CommitPolys group of bn polynomials of domain n at `values` (stride n, on the device), ONE batched
// launch set.  Evaluations: commit_evals_enqueue.  Coefficients: the scalars of one batched MSM over the monomial window
// table when its window is no wider than that of the Lagrange table of size n, or there is no such table (plan_batch made
// sure a monomial table covers n); else one batched forward Fr NTT into L.work and one batched MSM over the Lagrange table
// (sum c_i [tau^i]G = sum p(w^j) L_j).  A batched plan carries one bucket set of 2^(c-1) buckets per polynomial: a Lagrange
// table has the window of its own size (choose_c_fixed(n)), the monomial table that of the largest polynomial it was built
// for.  Measured on 2048 polynomials of 2^9 .. 2^12 coefficients (DESIGN.md section 4): at equal windows the monomial MSM
// is 0-5 % faster (no transform); with a 2^19 table resident (c = 17) it is 4-10x slower.
int group_commit_polys(const Batch& b, Lane& L, const Fr* values, size_t n, size_t bn, Affine* pts) {
    kzgb_ctx* c = b.c;
    const int logn = log2_exact(n);
    const kzgb_ctx::LagTable* lag = lagrange_table(c, logn);
    MsmJob job;
    int r = KZGB_OK;
    if (b.coeff && (!lag || (wtable_covers(c, 0, n) && c->wt_c <= lag->c))) {
        r = msm_enqueue(c, L, {values}, n, bn, nullptr, nullptr, 0, &job);
    } else {
        if (b.coeff) {
            CK(c, L.work.reserve(bn * n * sizeof(Fr)));
            CK(c, L.ntt_scratch.reserve(bn * n * sizeof(Fr)));
            if ((const void*)values != L.work.p)
                CK(c, cudaMemcpyAsync(L.work.p, values, bn * n * sizeof(Fr), cudaMemcpyDeviceToDevice, L.st));
            const Fr ninv = ninv_mont(logn);  // read by the inverse transform only
            ntt_launch((Fr*)L.work.p, logn, (uint32_t)bn, false, c->tw.get(), c->logN, &ninv, (Fr*)L.ntt_scratch.p, L.st);
            values = (const Fr*)L.work.p;
        }
        r = commit_evals_enqueue(c, L, values, n, &job, bn);
    }
    if (!r) r = msm_finish(c, L, job, pts);
    return r;
}

// The proof phase of one group of bn polynomials of n = blob_poly_len(lens[i0]) evaluations at `evals` (stride n, on the
// device) whose points are in L.small: [z x bn | tinv x bn | y x bn].  ONE batched evaluation / quotient launch set with a
// point per polynomial (outside and in_domain as eval_quotient_launch takes them) and ONE batched MSM of the quotients;
// pts[k] is the proof of polynomial i0 + k.  ys (optional, host) receives the bn y.
int group_prove(const Batch& b, Lane& L, const Fr* evals, size_t i0, size_t bn, bool outside, const uint32_t* in_domain,
                uint64_t* ys, Affine* pts) {
    kzgb_ctx* c = b.c;
    const size_t n = blob_poly_len(b.lens[i0]);
    const int logn = log2_exact(n);
    const kzgb_ctx::LagTable* lag = lagrange_table(c, logn);
    Fr ninv = ninv_mont(logn);
    CK(c, L.eval_scratch.reserve(eval_quotient_scratch_elems((uint32_t)n, (uint32_t)bn) * sizeof(Fr)));
    CK(c, L.work.reserve(bn * n * sizeof(Fr)));
    if (!lag) CK(c, L.ntt_scratch.reserve(bn * n * sizeof(Fr)));
    Fr* d_z = (Fr*)L.small.p;
    eval_quotient_launch(evals, (uint32_t)n, logn, (uint32_t)bn, d_z, d_z + bn, c->tw.get(), c->logN, &ninv,
                         (Fr*)L.eval_scratch.p, (Fr*)L.work.p, d_z + 2 * bn, L.st, outside, in_domain);
    if (!lag) ntt_launch((Fr*)L.work.p, logn, (uint32_t)bn, true, c->tw.get(), c->logN, &ninv, (Fr*)L.ntt_scratch.p, L.st);
    MsmJob job;
    int r = msm_enqueue(c, L, {(const Fr*)L.work.p}, n, bn, lag, nullptr, 0, &job);
    if (!r && ys) CK(c, cudaMemcpyAsync(ys, d_z + 2 * bn, bn * sizeof(Fr), cudaMemcpyDeviceToHost, L.st));
    if (!r) r = msm_finish(c, L, job, pts);
    return r;
}

// Small blobs: groups of equal-size blobs, each phase of a group is ONE batched launch set.  A commit-only group ends
// with its commitment phase (no hashing stage: hs is null).  A proof-only group has no commitment phase: its blob bytes
// (group_bytes) become Montgomery evaluations in one conversion launch and the commitments are the caller's.  A group of
// proofs at the caller's points is its evaluations (group_evals) and its points (group_points_at), then the proof phase.
int group_lane(const Batch& b, LaneSync& sync, HashStage* hs, std::atomic<size_t>& next_group, int li) {
    kzgb_ctx* c = b.c;
    Lane& L = c->lanes[li];
    std::vector<Affine> commits, pts;
    for (;;) {
        size_t gi = next_group.fetch_add(1);
        if (gi >= b.groups.size() || sync.failed.load()) return KZGB_OK;
        const size_t i0 = b.groups[gi].first, bn = b.groups[gi].second;
        const size_t n = blob_poly_len(b.lens[i0]);
        int r = KZGB_OK;
        const Affine* cs = nullptr;
        if (b.job == Job::CommitPolys) {
            const Fr* values = nullptr;
            commits.resize(bn);
            r = group_evals(b, L, i0, bn, &values);
            if (!r) r = group_commit_polys(b, L, values, n, bn, commits.data());
            if (!r) for (size_t k = 0; k < bn; k++) put_commitment(b, i0 + k, commits[k]);
            if (r) { sync.fail(); return r; }
            continue;
        }
        if (b.job == Job::ProveAt) {
            const Fr* evals = nullptr;
            const uint32_t* in_domain = nullptr;
            pts.resize(bn);
            r = group_evals(b, L, i0, bn, &evals);
            if (!r) r = group_points_at(b, L, i0, bn, &in_domain);
            if (!r) r = group_prove(b, L, evals, i0, bn, false, in_domain, b.ys_mont ? b.ys_mont + 4 * i0 : nullptr, pts.data());
            if (!r) for (size_t k = 0; k < bn; k++) put_proof(b, i0 + k, pts[k]);
            if (r) { sync.fail(); return r; }
            continue;
        }
        if (b.job == Job::Prove) {
            const uint8_t* src = nullptr;
            r = group_bytes(b, L, i0, bn, &src);
            if (!r && L.evals.reserve(bn * n * sizeof(Fr)) != cudaSuccess) r = fail(c, KZGB_ERR_DEVICE, "CUDA error: evals");
            if (!r) bytes_to_fr_launch(src, (uint64_t)bn * n * 32, (Fr*)L.evals.p, (uint32_t)(bn * n), L.st);
            cs = b.commits.data() + i0;
        } else {
            commits.resize(bn);
            r = group_commit(b, L, i0, bn, commits.data());
            if (!r) for (size_t k = 0; k < bn; k++) put_commitment(b, i0 + k, commits[k]);
            cs = commits.data();
        }
        if (!r && b.job != Job::Commit) {
            if (!hs->wait_ready(i0, bn)) return KZGB_OK;  // the transcript midstates come from the hashing stage
            pts.resize(bn);
            bool outside = false;
            r = group_challenges(b, *hs, L, i0, bn, cs, &outside);
            if (!r) r = group_prove(b, L, (const Fr*)L.evals.p, i0, bn, outside, nullptr, nullptr, pts.data());
            if (!r) for (size_t k = 0; k < bn; k++) put_proof(b, i0 + k, pts[k]);
        }
        if (r) { sync.fail(); return r; }
    }
}

// Task scheduler.  commit(i) needs nothing; proof(i) needs commit(i) and the transcript midstate of
// blob i (host SHA-256, ~9 ms for 16 MiB).  A lane takes the lowest ready proof, else the next
// commit, so the GPU never idles behind the hashing pool.  The queue lives under the lanes' lock.
struct TaskQueue {
    explicit TaskQueue(size_t count) : commit_done(count, 0), proof_taken(count, 0), commits(count) {}
    std::vector<uint8_t> commit_done, proof_taken;
    std::vector<Affine> commits;
    size_t next_commit = 0, proofs_taken = 0, proof_scan = 0;
};

// false: nothing left for this lane (every proof taken, or a lane failed)
bool take_task(const Batch& b, const HashStage& hs, TaskQueue& q, size_t* task, bool* is_proof) {
    LaneSync& s = hs.sync;
    std::unique_lock<std::mutex> lk(s.mu);
    for (;;) {
        if (s.failed.load()) return false;
        while (q.proof_scan < b.count && q.proof_taken[q.proof_scan]) q.proof_scan++;
        for (size_t k = q.proof_scan; k < b.count && k < q.next_commit; k++) {
            if (q.proof_taken[k] || !q.commit_done[k] || !hs.ready[k]) continue;
            q.proof_taken[k] = 1; q.proofs_taken++;
            *task = k; *is_proof = true;
            if (q.proofs_taken == b.count) s.cv.notify_all();  // lanes with nothing left to take can leave
            return true;
        }
        if (q.next_commit < b.count) { *task = q.next_commit++; *is_proof = false; return true; }
        if (q.proofs_taken == b.count) return false;
        s.cv.wait(lk);
    }
}

// Where blob i's bytes are on the device for a task of lane L: the caller's device blob, the slot of c->batch_bytes the
// hashing stream uploaded it to (with `wait`, L.st first waits for that upload), or nullptr: not on the device yet.
int device_blob(const Batch& b, const HashStage& hs, Lane& L, size_t i, bool wait, const uint8_t** bytes) {
    kzgb_ctx* c = b.c;
    *bytes = b.blobs_dev ? b.blobs_dev[i] : nullptr;
    if (*bytes || !hs.uploaded_here(i)) return KZGB_OK;
    *bytes = (const uint8_t*)c->batch_bytes.p + b.byte_off[i];
    if (wait && cudaStreamWaitEvent(L.st, c->ev_hash_uploaded.get(), 0) != cudaSuccess)
        return fail(c, KZGB_ERR_DEVICE, "CUDA error: cudaStreamWaitEvent failed");
    return KZGB_OK;
}

// Large blobs, commit and prove: the tasks of the queue.  A staged blob goes up into its slot with its commit task (unless
// the hashing stream has put it there) and stays for its proof.
int task_lane(const Batch& b, HashStage& hs, TaskQueue& q, int li) {
    kzgb_ctx* c = b.c;
    Lane& L = c->lanes[li];
    size_t i = 0;
    bool is_proof = false;
    while (take_task(b, hs, q, &i, &is_proof)) {
        size_t len = b.lens[i], n = blob_poly_len(len);
        const uint8_t* dev_bytes = nullptr;
        int r = device_blob(b, hs, L, i, !is_proof, &dev_bytes);
        if (!r && !dev_bytes && b.resident) {
            uint8_t* slot = (uint8_t*)c->batch_bytes.p + b.byte_off[i];
            if (!is_proof && len && cudaMemcpyAsync(slot, b.blobs_host[i], len, cudaMemcpyHostToDevice, L.st) != cudaSuccess)
                r = fail(c, KZGB_ERR_DEVICE, "CUDA error: H2D copy of a blob failed");
            dev_bytes = slot;
        }
        MsmJob job;
        Affine out;
        if (!r) r = blob_to_evals(c, L, b.blobs_host[i], dev_bytes, len, n);
        if (!r && !is_proof) r = commit_evals_enqueue(c, L, (Fr*)L.evals.p, n, &job);
        if (!r && is_proof) {
            Fr z = challenge_finish(hs.mid[i], q.commits[i]);
            r = proof_enqueue(c, L, (Fr*)L.evals.p, n, z, &job);
        }
        if (!r) r = msm_finish(c, L, job, &out);
        if (r) { hs.sync.fail(); return r; }
        if (is_proof) {
            put_proof(b, i, out);
        } else {
            put_commitment(b, i, out);
            { std::lock_guard<std::mutex> lk(hs.sync.mu); q.commits[i] = out; q.commit_done[i] = 1; }
            hs.sync.cv.notify_all();
        }
    }
    return KZGB_OK;
}

// Large blobs, commitments only: every task is "commit blob i", taken in blob order.  A blob is read once, so it goes up
// into the lane's own buffer; over a Lagrange table the MSM reads its bytes, otherwise they are converted,
// inverse-transformed and committed over the monomial table (commit_evals_enqueue).
int commit_task_lane(const Batch& b, LaneSync& sync, std::atomic<size_t>& next, int li) {
    kzgb_ctx* c = b.c;
    Lane& L = c->lanes[li];
    for (;;) {
        const size_t i = next.fetch_add(1);
        if (i >= b.count || sync.failed.load()) return KZGB_OK;
        const size_t len = b.lens[i], n = blob_poly_len(len);
        const kzgb_ctx::LagTable* lag = lagrange_table(c, log2_exact(n));
        const uint8_t* blob_host = b.blobs_dev ? nullptr : b.blobs_host[i];
        const uint8_t* dev_bytes = b.blobs_dev ? b.blobs_dev[i] : nullptr;
        MsmJob job;
        Affine out;
        int r = KZGB_OK;
        if (lag) {
            if (!dev_bytes) {
                r = blob_upload(c, L, blob_host, len);
                dev_bytes = (const uint8_t*)L.bytes.p;
            }
            if (!r) r = msm_enqueue(c, L, {nullptr, dev_bytes, len}, n, 1, lag, nullptr, 0, &job);
        } else {
            r = blob_to_evals(c, L, blob_host, dev_bytes, len, n);
            if (!r) r = commit_evals_enqueue(c, L, (Fr*)L.evals.p, n, &job);
        }
        if (!r) r = msm_finish(c, L, job, &out);
        if (r) { sync.fail(); return r; }
        put_commitment(b, i, out);
    }
}

// Large blobs, proofs only: every task is "prove blob i", taken in blob order.  A blob is read once, so it goes up into
// the lane's own buffer (unless the device's share of the hashing has staged it already) and is converted while its
// transcript is hashed.  Then the challenge with the caller's commitment, the quotient and its MSM.
int prove_task_lane(const Batch& b, HashStage& hs, std::atomic<size_t>& next, int li) {
    kzgb_ctx* c = b.c;
    Lane& L = c->lanes[li];
    for (;;) {
        const size_t i = next.fetch_add(1);
        if (i >= b.count) return KZGB_OK;
        const size_t len = b.lens[i], n = blob_poly_len(len);
        const uint8_t* dev_bytes = nullptr;
        int r = device_blob(b, hs, L, i, true, &dev_bytes);
        if (!r) r = blob_to_evals(c, L, b.blobs_host[i], dev_bytes, len, n);
        if (!r && !hs.wait_ready(i, 1)) return KZGB_OK;
        MsmJob job;
        Affine out;
        if (!r) r = proof_enqueue(c, L, (Fr*)L.evals.p, n, challenge_finish(hs.mid[i], b.commits[i]), &job);
        if (!r) r = msm_finish(c, L, job, &out);
        if (r) { hs.sync.fail(); return r; }
        put_proof(b, i, out);
    }
}

// Large polynomials, and batches without groups, of proofs at the caller's points: every task is "prove polynomial i",
// taken in index order.  The quotient is taken on the caller's device polynomial, or on a copy in the lane's own buffer,
// and y is read as kzgb_compute_proof reads it.
int prove_at_task_lane(const Batch& b, LaneSync& sync, std::atomic<size_t>& next, int li) {
    kzgb_ctx* c = b.c;
    Lane& L = c->lanes[li];
    auto prove = [&](size_t i, Affine* out) {
        const size_t n = b.ns[i];
        const Fr* evals = (const Fr*)b.evals[i];
        if (!b.evals_on_device) {
            CK(c, L.evals.reserve(n * sizeof(Fr)));
            CK(c, cudaMemcpyAsync(L.evals.p, b.evals[i], n * sizeof(Fr), cudaMemcpyHostToDevice, L.st));
            evals = (const Fr*)L.evals.p;
        }
        Fr z;
        memcpy(z.l, b.zs_mont + 4 * i, 32);
        MsmJob job;
        if (int rc = proof_enqueue(c, L, evals, n, z, &job)) return rc;
        if (b.ys_mont) CK(c, cudaMemcpyAsync(&L.h_fr[3], (Fr*)L.small.p + 2, sizeof(Fr), cudaMemcpyDeviceToHost, L.st));
        if (int rc = msm_finish(c, L, job, out)) return rc;
        if (b.ys_mont) memcpy(b.ys_mont + 4 * i, &L.h_fr[3], 32);
        return (int)KZGB_OK;
    };
    for (;;) {
        const size_t i = next.fetch_add(1);
        if (i >= b.count || sync.failed.load()) return KZGB_OK;
        Affine out;
        if (int r = prove(i, &out)) { sync.fail(); return r; }
        put_proof(b, i, out);
    }
}

// Large polynomials, and batches without groups, of commitments to the caller's polynomials: every task is "commit entry
// k", taken in the batch's order.  Host values go up on the lane's stream into its own buffer; device values are read in
// place.  Evaluations are committed as kzgb_commit_eval commits them (commit_evals_enqueue), coefficients by one MSM over
// SRS[0, ns), as kzgb_commit_coeff does (no pipelined upload: its copy stream belongs to the context, not to a lane).
int commit_polys_task_lane(const Batch& b, LaneSync& sync, std::atomic<size_t>& next, int li) {
    kzgb_ctx* c = b.c;
    Lane& L = c->lanes[li];
    auto commit = [&](size_t k, Affine* out) {
        const size_t n = b.ns[k];
        const Fr* values = (const Fr*)b.evals[k];
        if (!b.evals_on_device && n) {  // into L.work, where commit_evals_enqueue transforms without a copy
            CK(c, L.work.reserve(n * sizeof(Fr)));
            CK(c, cudaMemcpyAsync(L.work.p, b.evals[k], n * sizeof(Fr), cudaMemcpyHostToDevice, L.st));
            values = (const Fr*)L.work.p;
        }
        MsmJob job;
        int rc = b.coeff ? msm_enqueue(c, L, {values}, n, 1, nullptr, nullptr, 0, &job) : commit_evals_enqueue(c, L, values, n, &job);
        return rc ? rc : msm_finish(c, L, job, out);
    };
    for (;;) {
        const size_t k = next.fetch_add(1);
        if (k >= b.count || sync.failed.load()) return KZGB_OK;
        Affine out;
        if (int r = commit(k, &out)) { sync.fail(); return r; }
        put_commitment(b, k, out);
    }
}

// ---------------------------------------------------------------- driver
// The plan, then the lanes.  Commit, ProveAt and CommitPolys have no transcripts: no staging, no hashing stage.  CommitAndProve stages
// host blobs (stage_blob_bytes) and may hash on the device what is staged or the caller's; Prove stages host blobs only
// for the device's share of the hashing.  Groups hash on the host pool alone.
int run_batch(Batch& b) {
    if (b.count == 0) return KZGB_OK;
    int rc = plan_batch(b);
    if (rc) return rc;
    LaneSync sync;
    std::atomic<size_t> next{0};  // the next group, or the next blob of a commit-only or proof-only task lane
    if (b.job == Job::Commit)
        return run_lanes(b, [&](int li) {
            return b.groups.empty() ? commit_task_lane(b, sync, next, li) : group_lane(b, sync, nullptr, next, li);
        });
    if (b.job == Job::ProveAt)
        return run_lanes(b, [&](int li) {
            return b.groups.empty() ? prove_at_task_lane(b, sync, next, li) : group_lane(b, sync, nullptr, next, li);
        });
    if (b.job == Job::CommitPolys)
        return run_lanes(b, [&](int li) {
            return b.groups.empty() ? commit_polys_task_lane(b, sync, next, li) : group_lane(b, sync, nullptr, next, li);
        });
    HashPlan hplan;
    if (b.job == Job::CommitAndProve) {
        stage_blob_bytes(b);
        if (b.groups.empty()) hplan = hash_plan(b.lens, b.count, b.blobs_dev || b.resident, false);
    } else if (b.groups.empty()) {
        hplan = hash_plan(b.lens, b.count, true, true);
        if (hplan.dev_k && !b.blobs_dev) {  // the device hashes blobs it holds: stage the host blobs
            stage_blob_bytes(b);
            if (!b.resident) hplan.dev_k = 0;
        }
    }
    {
        HashStage hs(b, hplan, sync);
        TaskQueue q(b.job == Job::CommitAndProve && b.groups.empty() ? b.count : 0);  // task_lane's
        rc = run_lanes(b, [&](int li) {
            if (!b.groups.empty()) return group_lane(b, sync, &hs, next, li);
            return b.job == Job::Prove ? prove_task_lane(b, hs, next, li) : task_lane(b, hs, q, li);
        });
    }
    // bounded residency between calls: only stage_blob_bytes grows the buffer
    if (b.c->batch_bytes.cap > ((size_t)g_batch_keep_mib.load() << 20)) b.c->batch_bytes.release();
    return rc;
}

// ---------------------------------------------------------------- verification
// The per-blob front half of every verification (helpers.rs:613-662) on lane L: zs[i] = compute_challenge(blob i, Cs[i])
// and ys[i] = p_i(zs[i]) for m blobs of ns[i] = blob_poly_len(lens[i]) > 0 elements.  The blobs are evaluated in rounds
// of equal-size runs; after_round(i0, b, d_z, d_y) runs at the end of each round, with z_{i0} .. z_{i0+b-1} resident at
// d_z and y_{i0} .. y_{i0+b-1} at d_y,
// to enqueue more work on L.st before the round's synchronise.  blobs_dev (may be null): the blob bytes on the device,
// read in place; the transcripts are hashed from blobs_host either way.
template <class F>
int blob_evals_stage(kzgb_ctx* c, Lane& L, const uint8_t* const* blobs_dev, const uint8_t* const* blobs_host,
                     const size_t* lens, const std::vector<size_t>& ns, const std::vector<Affine>& Cs, std::vector<Fr>& zs,
                     std::vector<Fr>& ys, F after_round) {
    const size_t m = ns.size();
    const size_t max_n = *std::max_element(ns.begin(), ns.end());
    int rc = ensure_twiddles(c, log2_exact(max_n));
    if (rc) return rc;
    // Thousands of small transcripts: hash them on the GPU, one thread per blob, from the evaluations that
    // are resident anyway (fs.cu).  Otherwise a host SHA-256 pool (one transcript per blob) runs while the
    // blobs are uploaded and converted.
    const int fs_opt = g_fs_device.load();
    const bool fs_device = fs_opt >= 0 ? fs_opt != 0 : (m >= 256 && max_n <= ((size_t)1 << 13));
    std::atomic<size_t> next{fs_device ? m : 0};
    std::vector<std::thread> hashers;
    {
        size_t nt = fs_device ? 0 : std::max<size_t>(1, std::min<size_t>(m, hash_pool_threads() + 1));
        for (size_t t = 0; t < nt; t++)
            hashers.emplace_back([&]() {
                for (;;) {
                    size_t i = next.fetch_add(1);
                    if (i >= m) return;
                    Sha256 sh;
                    challenge_midstate(sh, blobs_host[i], lens[i], ns[i]);
                    zs[i] = challenge_finish(sh, Cs[i]);
                }
            });
    }
    struct Joiner {
        std::vector<std::thread>& t;
        std::atomic<size_t>& next;
        size_t m;
        bool joined = false;
        void join() { if (!joined) { for (auto& x : t) x.join(); joined = true; } }
        ~Joiner() { next.store(m); join(); }  // error paths: stop handing out work, then wait
    } joiner{hashers, next, m};
    const size_t budget_elems = (size_t)1 << 24;  // evaluations resident per GPU batch
    size_t i0 = 0;
    while (i0 < m) {
        size_t n = ns[i0], i1 = i0;
        while (i1 < m && ns[i1] == n && (i1 - i0 + 1) * n <= std::max(budget_elems, n) && i1 - i0 < 65535) i1++;  // b is a gridDim.y
        size_t b = i1 - i0;
        int logn = log2_exact(n);
        CK(c, L.evals.reserve(b * n * sizeof(Fr)));
        if (!blobs_dev) CK(c, L.bytes.reserve(b * n * 32));
        CK(c, L.eval_scratch.reserve(eval_quotient_scratch_elems((uint32_t)n, (uint32_t)b) * sizeof(Fr)));
        CK(c, L.work.reserve(5 * b * sizeof(Fr)));
        bool full = (uint64_t)b * n < 0xffffffffull;  // every blob fills its polynomial: one conversion launch
        for (size_t k = 0; k < b && full; k++) full = lens[i0 + k] == n * 32;
        const uint8_t* const* src = blobs_dev ? blobs_dev : blobs_host;
        for (size_t k = 0; k < b;) {
            size_t run = 1;  // blobs that are adjacent in memory go up in one copy, or are converted in one launch
            while (full && k + run < b && src[i0 + k + run] == src[i0 + k] + run * n * 32) run++;
            size_t bytes = full ? run * n * 32 : lens[i0 + k];
            Fr* evals = (Fr*)L.evals.p + k * n;
            if (blobs_dev) {
                bytes_to_fr_launch(src[i0 + k], bytes, evals, (uint32_t)(full ? run * n : n), L.st);
            } else {
                uint8_t* dst = (uint8_t*)L.bytes.p + k * n * 32;
                CK(c, cudaMemcpyAsync(dst, src[i0 + k], bytes, cudaMemcpyHostToDevice, L.st));
                if (!full) bytes_to_fr_launch(dst, lens[i0 + k], evals, (uint32_t)n, L.st);
            }
            k += run;
        }
        if (full && !blobs_dev) bytes_to_fr_launch((const uint8_t*)L.bytes.p, (uint64_t)b * n * 32, (Fr*)L.evals.p, (uint32_t)(b * n), L.st);
        joiner.join();  // the challenges z_i are needed from here on
        Fr* d_z = (Fr*)L.work.p;
        Fr* d_t = d_z + b;
        Fr* d_y = d_t + b;
        Fr ninv = ninv_mont(logn);
        std::vector<Fr> tinvs;
        std::vector<uint8_t> cbytes;
        bool any_in_domain = false;
        uint32_t* d_in_domain = nullptr;  // challenges hashed on the device: the device says which z are roots of the domain
        if (fs_device) {
            uint8_t* d_c32 = (uint8_t*)(d_y + b);
            cbytes.resize(b * 32);
            for (size_t k = 0; k < b; k++) serialize_compressed(Cs[i0 + k], &cbytes[32 * k]);
            CK(c, cudaMemcpyAsync(d_c32, cbytes.data(), b * 32, cudaMemcpyHostToDevice, L.st));
            d_in_domain = (uint32_t*)(d_c32 + 32 * b);
            fs_challenges_launch((Fr*)L.evals.p, (uint32_t)n, logn, (uint32_t)b, d_c32, &ninv, d_z, d_t, L.st, d_in_domain);
            CK(c, cudaMemcpyAsync(&zs[i0], d_z, b * sizeof(Fr), cudaMemcpyDeviceToHost, L.st));
        } else {
            tinvs.resize(b);
            for (size_t k = 0; k < b; k++) tinvs[k] = eval_tinv(zs[i0 + k], logn, &any_in_domain);
            CK(c, cudaMemcpyAsync(d_z, &zs[i0], b * sizeof(Fr), cudaMemcpyHostToDevice, L.st));
            CK(c, cudaMemcpyAsync(d_t, tinvs.data(), b * sizeof(Fr), cudaMemcpyHostToDevice, L.st));
        }
        eval_quotient_launch((Fr*)L.evals.p, (uint32_t)n, logn, (uint32_t)b, d_z, d_t, c->tw.get(), c->logN, &ninv,
                             (Fr*)L.eval_scratch.p, nullptr, d_y, L.st, !fs_device && !any_in_domain, d_in_domain);
        CK(c, cudaMemcpyAsync(&ys[i0], d_y, b * sizeof(Fr), cudaMemcpyDeviceToHost, L.st));
        rc = after_round(i0, b, (const Fr*)d_z, (const Fr*)d_y);
        if (rc) return rc;
        CK(c, cudaStreamSynchronize(L.st));
        CK(c, cudaGetLastError());
        i0 = i1;
    }
    return KZGB_OK;
}

// generator_window_table() on c's device, uploaded once
int ensure_gen_table(kzgb_ctx* c) {
    if (c->gen_table) return KZGB_OK;
    DevPtr<Affine[]> t;
    CK(c, dev_alloc(t, GEN_TABLE_POINTS * sizeof(Affine)));
    CK(c, cudaMemcpy(t.get(), generator_window_table(), GEN_TABLE_POINTS * sizeof(Affine), cudaMemcpyHostToDevice));
    c->gen_table = std::move(t);
    return KZGB_OK;
}

// verify_blob_kzg_proof (verify.rs:77-115) for `count` blobs on lane 0: every blob checked as kzgb_verify_blob_proof_g1
// checks it, in index order, then the stage and, per round, one k_commit_minus_value launch (out_xy != null: up to the
// pairing) or the pairing check of every opening (ok != null: the bools).  Neither: z and y only.
int verify_blob_proofs(kzgb_ctx* c, const uint8_t* const* blobs_dev, const uint8_t* const* blobs_host, const size_t* lens,
                       size_t count, const uint64_t* commitments_xy, const uint8_t* commitments_inf, const uint64_t* proofs_xy,
                       const uint8_t* proofs_inf, uint64_t* out_xy, uint8_t* out_inf, uint64_t* z_out, uint64_t* y_out,
                       uint8_t* ok = nullptr) {
    if (count == 0) return KZGB_OK;
    std::vector<Affine> Cs(count), Ps(ok ? count : 0);
    std::vector<size_t> ns(count);
    for (size_t i = 0; i < count; i++) {
        Cs[i] = affine_from_abi(commitments_xy + 8 * i, commitments_inf ? commitments_inf[i] : 0);
        const Affine P = affine_from_abi(proofs_xy + 8 * i, proofs_inf ? proofs_inf[i] : 0);
        if (!aff_on_curve(Cs[i]) || !aff_on_curve(P)) return fail(c, KZGB_ERR_NOT_ON_CURVE, "G1 point not on curve");
        if (lens[i] == 0) return fail(c, KZGB_ERR_GENERIC, "Length of data after padding is 0");
        ns[i] = blob_poly_len(lens[i]);
        if (ns[i] > ((size_t)1 << 28)) return fail(c, KZGB_ERR_GENERIC, "Input size exceeds maximum polynomial size");
        if (ok) Ps[i] = P;
    }
    Lane& L = c->lanes[0];
    Affine* d_c = nullptr;  // [C_0 .. C_{count-1} | out_0 .. out_{count-1}], or [C | pi] for the pairing checks
    if (out_xy || ok) {
        if (int rc = ensure_gen_table(c)) return rc;
        if (ok) {
            if (int rc = ensure_pairing_tables(c)) return rc;
            CK(c, L.pairing.reserve(pairing_workspace_bytes((uint32_t)std::min<size_t>(count, 65535))));
        }
        CK(c, L.bases.reserve(2 * count * sizeof(Affine)));
        d_c = (Affine*)L.bases.p;
        CK(c, cudaMemcpyAsync(d_c, Cs.data(), count * sizeof(Affine), cudaMemcpyHostToDevice, L.st));
        if (ok) CK(c, cudaMemcpyAsync(d_c + count, Ps.data(), count * sizeof(Affine), cudaMemcpyHostToDevice, L.st));
    }
    Affine* d_out = d_c ? d_c + count : nullptr;
    std::vector<Fr> zs(count), ys(count);
    std::vector<Affine> outs(out_xy ? count : 0);
    std::vector<uint8_t> flags(ok ? count : 0);
    int rc = blob_evals_stage(c, L, blobs_dev, blobs_host, lens, ns, Cs, zs, ys,
                              [&](size_t i0, size_t b, const Fr* d_z, const Fr* d_y) {
        if (ok) {  // a round holds at most 65 535 blobs
            const uint8_t* d_flags = pairing_check_launch(d_c + i0, d_c + count + i0, d_z, d_y, c->gen_table.get(),
                                                          c->pair_tab.get(), L.pairing.p, (uint32_t)b, L.st);
            CK(c, cudaMemcpyAsync(&flags[i0], d_flags, b, cudaMemcpyDeviceToHost, L.st));
        }
        if (!out_xy) return (int)KZGB_OK;
        commit_minus_value_launch(d_c + i0, d_y, c->gen_table.get(), d_out + i0, (uint32_t)b, L.st);
        CK(c, cudaMemcpyAsync(&outs[i0], d_out + i0, b * sizeof(Affine), cudaMemcpyDeviceToHost, L.st));
        return (int)KZGB_OK;
    });
    if (rc) return rc;
    if (ok) return pairing_finish(c, flags, ok);
    for (size_t i = 0; i < count; i++) {
        if (out_xy) affine_to_abi(outs[i], out_xy + 8 * i, out_inf ? out_inf + i : nullptr);
        if (z_out) memcpy(z_out + 4 * i, zs[i].l, 32);
        if (y_out) memcpy(y_out + 4 * i, ys[i].l, 32);
    }
    return KZGB_OK;
}

// The random linear combination of m validated and evaluated openings (batch.rs:76-249): d_bases holds C_0 .. C_{m-1},
// pi_0 .. pi_{m-1} and room for one more point.
int rlc_combine(kzgb_ctx* c, Lane& L, const std::vector<Affine>& Cs, const std::vector<Affine>& Ps,
                const std::vector<size_t>& ns, const std::vector<Fr>& zs, const std::vector<Fr>& ys, Affine* d_bases,
                Affine* lhs, Affine* rhs) {
    const size_t m = Cs.size();
    // r = SHA-256(transcript) mod r (batch.rs:76-168): bytes 24..32 stay zero, count at 32..40
    std::vector<uint8_t> tr(40 + m * 136, 0);
    memcpy(tr.data(), "EIGENDA_RCKZGBATCH___V1_", 24);
    for (int k = 0; k < 8; k++) tr[32 + k] = (uint8_t)((uint64_t)m >> (56 - 8 * k));
    size_t off = 40;
    for (size_t i = 0; i < m; i++) { for (int k = 0; k < 8; k++) tr[off + k] = (uint8_t)((uint64_t)ns[i] >> (56 - 8 * k)); off += 8; }
    for (size_t i = 0; i < m; i++) {
        serialize_compressed(Cs[i], &tr[off]); off += 32;
        fe_to_be_bytes(zs[i], &tr[off]); off += 32;
        fe_to_be_bytes(ys[i], &tr[off]); off += 32;
        serialize_compressed(Ps[i], &tr[off]); off += 32;
    }
    uint8_t dg[32];
    sha256(tr.data(), tr.size(), dg);
    Fr r = fr_from_be_bytes(dg);

    // scalars on the GPU: [r^i | r^i z_i | -(sum r^i y_i)]
    CK(c, L.work.reserve((4 * m + 8) * sizeof(Fr)));
    Fr* d_sc = (Fr*)L.work.p;          // 2m + 1 scalars
    Fr* d_zy = d_sc + 2 * m + 1;       // z then y (m each)
    Fr* d_dot = d_zy + 2 * m;
    CK(c, cudaMemcpyAsync(d_zy, zs.data(), m * sizeof(Fr), cudaMemcpyHostToDevice, L.st));
    CK(c, cudaMemcpyAsync(d_zy + m, ys.data(), m * sizeof(Fr), cudaMemcpyHostToDevice, L.st));
    fr_powers_launch(d_sc, (uint32_t)m, &r, L.st);                      // helpers.rs:298-314
    fr_mul_vec_launch(d_sc + m, d_sc, d_zy, (uint32_t)m, L.st);         // r^i z_i (batch.rs:239)
    fr_dot_launch(d_dot, d_sc, d_zy + m, (uint32_t)m, L.st);            // sum r^i y_i
    CK(c, cudaMemcpyAsync(&L.h_fr[2], d_dot, sizeof(Fr), cudaMemcpyDeviceToHost, L.st));
    CK(c, cudaStreamSynchronize(L.st));
    fe_neg(L.h_fr[2], L.h_fr[2]);
    CK(c, cudaMemcpyAsync(d_sc + 2 * m, &L.h_fr[2], sizeof(Fr), cudaMemcpyHostToDevice, L.st));
    Affine G;
    fe_one(G.x); fe_dbl(G.y, G.x);
    CK(c, cudaMemcpy(d_bases + 2 * m, &G, sizeof(Affine), cudaMemcpyHostToDevice));
    // lhs = sum r^i pi_i (batch.rs:228); rhs = sum r^i (C_i - y_i G) + sum r^i z_i pi_i (batch.rs:245-249),
    // the m generator multiplications folded into ONE extra base: -(sum r^i y_i) * G  (same group element)
    int rc = msm_blocking(c, L, d_sc, 0, m, d_bases + m, lhs);
    if (rc) return rc;
    return msm_blocking(c, L, d_sc, 0, 2 * m + 1, d_bases, rhs);
}

// The m > 0 openings' points from the ABI into Cs / Ps and onto lane L's d_bases ([C_0..C_{m-1}, pi_0..pi_{m-1}, room for
// G]), then validate_g1_point on all 2m of them (batch.rs:30-37) on the GPU.
int upload_rlc_points(kzgb_ctx* c, Lane& L, size_t m, const uint64_t* commitments_xy, const uint8_t* commitments_inf,
                      const uint64_t* proofs_xy, const uint8_t* proofs_inf, std::vector<Affine>& Cs, std::vector<Affine>& Ps,
                      Affine** d_bases) {
    Cs.resize(m);
    Ps.resize(m);
    for (size_t i = 0; i < m; i++) {
        Cs[i] = affine_from_abi(commitments_xy + 8 * i, commitments_inf ? commitments_inf[i] : 0);
        Ps[i] = affine_from_abi(proofs_xy + 8 * i, proofs_inf ? proofs_inf[i] : 0);
    }
    CK(c, L.bases.reserve((2 * m + 1) * sizeof(Affine)));
    *d_bases = (Affine*)L.bases.p;
    CK(c, cudaMemcpyAsync(*d_bases, Cs.data(), m * sizeof(Affine), cudaMemcpyHostToDevice, L.st));
    CK(c, cudaMemcpyAsync(*d_bases + m, Ps.data(), m * sizeof(Affine), cudaMemcpyHostToDevice, L.st));
    return validate_points_dev(c, L, *d_bases, 2 * m);
}

// The random linear combination on lane 0 of m openings into lhs / rhs in the ABI; m == 0: the identity twice.  The 2m
// points are read and checked first, then openings(L, Cs, ns, zs, ys) checks the rest of the input and fills in the
// polynomial lengths, challenges and evaluations.
template <class F>
int rlc_to_abi(kzgb_ctx* c, size_t m, const uint64_t* commitments_xy, const uint8_t* commitments_inf, const uint64_t* proofs_xy,
               const uint8_t* proofs_inf, uint64_t lhs_xy[8], uint8_t* lhs_inf, uint64_t rhs_xy[8], uint8_t* rhs_inf, F openings) {
    Affine lhs, rhs;
    if (m == 0) {
        aff_set_inf(lhs);
        rhs = lhs;
    } else {
        Lane& L = c->lanes[0];
        std::vector<Affine> Cs, Ps;
        Affine* d_bases = nullptr;
        if (int rc = upload_rlc_points(c, L, m, commitments_xy, commitments_inf, proofs_xy, proofs_inf, Cs, Ps, &d_bases)) return rc;
        std::vector<size_t> ns(m);
        std::vector<Fr> zs(m), ys(m);
        if (int rc = openings(L, Cs, ns, zs, ys)) return rc;
        if (int rc = rlc_combine(c, L, Cs, Ps, ns, zs, ys, d_bases, &lhs, &rhs)) return rc;
    }
    affine_to_abi(lhs, lhs_xy, lhs_inf);
    affine_to_abi(rhs, rhs_xy, rhs_inf);
    return KZGB_OK;
}

// verify_blob_kzg_proof_batch (batch.rs:16-249) up to the pairing on lane 0: the 2m points, then the lengths, then the
// per-blob stage (blobs_dev as blob_evals_stage reads it) and the combination.
int verify_batch_rlc(kzgb_ctx* c, const uint8_t* const* blobs_dev, const uint8_t* const* blobs_host, const size_t* lens,
                     size_t m, const uint64_t* commitments_xy, const uint8_t* commitments_inf, const uint64_t* proofs_xy,
                     const uint8_t* proofs_inf, uint64_t lhs_xy[8], uint8_t* lhs_inf, uint64_t rhs_xy[8], uint8_t* rhs_inf) {
    return rlc_to_abi(c, m, commitments_xy, commitments_inf, proofs_xy, proofs_inf, lhs_xy, lhs_inf, rhs_xy, rhs_inf,
                      [&](Lane& L, const std::vector<Affine>& Cs, std::vector<size_t>& ns, std::vector<Fr>& zs, std::vector<Fr>& ys) {
        for (size_t i = 0; i < m; i++) {
            if (lens[i] == 0) return fail(c, KZGB_ERR_GENERIC, "Length of data after padding is 0");
            ns[i] = blob_poly_len(lens[i]);
        }
        // per-blob challenges and evaluations: the stage the per-blob verification shares
        return blob_evals_stage(c, L, blobs_dev, blobs_host, lens, ns, Cs, zs, ys,
                                [](size_t, size_t, const Fr*, const Fr*) { return (int)KZGB_OK; });
    });
}

// Every z_i and y_i of m openings is a reduced Montgomery value (< r, as an arkworks Fr always is: a larger word would be
// hashed as other bytes than the reference hashes); else KZGB_ERR_INVALID_FIELD_ELEMENT for the first opening that is not.
int check_openings_reduced(kzgb_ctx* c, size_t m, const uint64_t* zs_mont, const uint64_t* ys_mont) {
    for (size_t i = 0; i < m; i++)
        if (!fr_words_reduced(zs_mont + 4 * i) || !fr_words_reduced(ys_mont + 4 * i))
            return fail(c, KZGB_ERR_INVALID_FIELD_ELEMENT,
                        "z or y of opening " + std::to_string(i) + " is not a reduced field element");
    return KZGB_OK;
}

// verify_kzg_proof_batch (batch.rs:185-249) on lane 0 over m openings that are already evaluated: the 2m points, then
// every z_i and y_i reduced, then the combination with the caller's n_i.
int verify_openings_rlc(kzgb_ctx* c, size_t m, const uint64_t* commitments_xy, const uint8_t* commitments_inf,
                        const uint64_t* proofs_xy, const uint8_t* proofs_inf, const uint64_t* zs_mont, const uint64_t* ys_mont,
                        const uint64_t* poly_lens, uint64_t lhs_xy[8], uint8_t* lhs_inf, uint64_t rhs_xy[8], uint8_t* rhs_inf) {
    return rlc_to_abi(c, m, commitments_xy, commitments_inf, proofs_xy, proofs_inf, lhs_xy, lhs_inf, rhs_xy, rhs_inf,
                      [&](Lane&, const std::vector<Affine>&, std::vector<size_t>& ns, std::vector<Fr>& zs, std::vector<Fr>& ys) {
        if (int rc = check_openings_reduced(c, m, zs_mont, ys_mont)) return rc;
        for (size_t i = 0; i < m; i++) {
            memcpy(zs[i].l, zs_mont + 4 * i, 32);
            memcpy(ys[i].l, ys_mont + 4 * i, 32);
            ns[i] = (size_t)poly_lens[i];
        }
        return (int)KZGB_OK;
    });
}

// verify_proof (verify.rs:10-75) on lane 0 for m openings: the 2m points as verify_openings_rlc checks them, then every
// z_i and y_i below r, then the pairing checks (no blob, no hashing, no SRS).
int verify_proofs(kzgb_ctx* c, size_t m, const uint64_t* commitments_xy, const uint8_t* commitments_inf,
                  const uint64_t* proofs_xy, const uint8_t* proofs_inf, const uint64_t* zs_mont, const uint64_t* ys_mont,
                  uint8_t* ok) {
    if (m == 0) return KZGB_OK;
    Lane& L = c->lanes[0];
    std::vector<Affine> Cs, Ps;
    Affine* d_bases = nullptr;
    if (int rc = upload_rlc_points(c, L, m, commitments_xy, commitments_inf, proofs_xy, proofs_inf, Cs, Ps, &d_bases)) return rc;
    if (int rc = check_openings_reduced(c, m, zs_mont, ys_mont)) return rc;
    if (int rc = ensure_gen_table(c)) return rc;
    if (int rc = ensure_pairing_tables(c)) return rc;
    std::vector<uint8_t> flags(m);
    for (size_t i0 = 0; i0 < m; i0 += 65536) {  // bounded workspace
        const size_t b = std::min<size_t>(m - i0, 65536);
        CK(c, L.work.reserve(2 * b * sizeof(Fr)));
        CK(c, L.pairing.reserve(pairing_workspace_bytes((uint32_t)b)));
        Fr* d_zy = (Fr*)L.work.p;  // z then y
        CK(c, cudaMemcpyAsync(d_zy, zs_mont + 4 * i0, b * sizeof(Fr), cudaMemcpyHostToDevice, L.st));
        CK(c, cudaMemcpyAsync(d_zy + b, ys_mont + 4 * i0, b * sizeof(Fr), cudaMemcpyHostToDevice, L.st));
        const uint8_t* d_flags = pairing_check_launch(d_bases + i0, d_bases + m + i0, d_zy, d_zy + b, c->gen_table.get(),
                                                      c->pair_tab.get(), L.pairing.p, (uint32_t)b, L.st);
        CK(c, cudaMemcpyAsync(&flags[i0], d_flags, b, cudaMemcpyDeviceToHost, L.st));
        CK(c, cudaStreamSynchronize(L.st));
        CK(c, cudaGetLastError());
    }
    return pairing_finish(c, flags, ok);
}

// KZG::compute_proof (kzg.rs:128-178, 187-234) for `count` polynomials at the caller's points: the batch driver, with
// polynomial i planned as a blob of 32 ns[i] bytes.  plan_batch checks ns[i] before that length is used.
int compute_proofs(kzgb_ctx* c, const uint64_t* const* evals, bool on_device, const size_t* ns, size_t count,
                   const uint64_t* zs_mont, uint64_t* out_xy, uint8_t* out_inf, uint64_t* ys_mont) {
    std::vector<size_t> lens(count);
    for (size_t i = 0; i < count; i++) lens[i] = 32 * ns[i];
    Batch b(c, Job::ProveAt, nullptr, nullptr, lens.data(), count);
    b.evals = evals;
    b.evals_on_device = on_device;
    b.ns = ns;
    b.zs_mont = zs_mont;
    b.ys_mont = ys_mont;
    b.out_xy = out_xy;
    b.out_inf = out_inf;
    return run_batch(b);
}

// KZG::commit_eval_form / commit_coeff_form (kzg.rs:84-104, 107-125) for `count` polynomials: the batch driver, with
// polynomial i planned as a blob of 32 N_i bytes.  A length no SRS holds is planned as 0 bytes; plan_batch rejects it
// before that length is used.
int commit_polys(kzgb_ctx* c, bool coeff, const uint64_t* const* values, bool on_device, const size_t* ns, size_t count,
                 uint64_t* out_xy, uint8_t* out_inf) {
    std::vector<size_t> lens(count);
    for (size_t i = 0; i < count; i++) lens[i] = ns[i] <= c->srs_n ? 32 * next_pow2(ns[i]) : 0;
    Batch b(c, Job::CommitPolys, nullptr, nullptr, lens.data(), count);
    b.coeff = coeff;
    b.evals = values;
    b.evals_on_device = on_device;
    b.ns = ns;
    b.out_xy = out_xy;
    b.out_inf = out_inf;
    return run_batch(b);
}

}  // namespace

// =====================================================================================
extern "C" {

// kzgb_commit_and_prove_blobs and kzgb_compute_blob_proofs are their _dev forms without device blobs.
int kzgb_commit_and_prove_blobs(kzgb_ctx* c, const uint8_t* const* blobs, const size_t* lens, size_t count,
                                uint8_t* commitments32, uint8_t* proofs32) {
    return kzgb_commit_and_prove_blobs_dev(c, nullptr, blobs, lens, count, commitments32, proofs32);
}
int kzgb_commit_and_prove_blobs_dev(kzgb_ctx* c, const uint8_t* const* blobs_dev, const uint8_t* const* blobs_host,
                                    const size_t* lens, size_t count, uint8_t* commitments32, uint8_t* proofs32) {
    Guard g(c);
    Batch b(c, Job::CommitAndProve, blobs_dev, blobs_host, lens, count);
    b.commitments32 = commitments32;
    b.proofs32 = proofs32;
    return run_batch(b);
}
int kzgb_commit_blobs(kzgb_ctx* c, const uint8_t* const* blobs, const size_t* lens, size_t count, uint64_t* out_xy,
                      uint8_t* out_inf) {
    Guard g(c);
    Batch b(c, Job::Commit, nullptr, blobs, lens, count);
    b.out_xy = out_xy;
    b.out_inf = out_inf;
    return run_batch(b);
}
int kzgb_commit_blobs_dev(kzgb_ctx* c, const uint8_t* const* blobs_dev, const size_t* lens, size_t count,
                          uint64_t* out_xy, uint8_t* out_inf) {
    Guard g(c);
    Batch b(c, Job::Commit, blobs_dev, nullptr, lens, count);
    b.out_xy = out_xy;
    b.out_inf = out_inf;
    return run_batch(b);
}
int kzgb_compute_blob_proofs(kzgb_ctx* c, const uint8_t* const* blobs, const size_t* lens, size_t count,
                             const uint64_t* commitments_xy, const uint8_t* commitments_inf, uint64_t* out_xy, uint8_t* out_inf) {
    return kzgb_compute_blob_proofs_dev(c, nullptr, blobs, lens, count, commitments_xy, commitments_inf, out_xy, out_inf);
}
int kzgb_compute_blob_proofs_dev(kzgb_ctx* c, const uint8_t* const* blobs_dev, const uint8_t* const* blobs_host,
                                 const size_t* lens, size_t count, const uint64_t* commitments_xy,
                                 const uint8_t* commitments_inf, uint64_t* out_xy, uint8_t* out_inf) {
    Guard g(c);
    Batch b(c, Job::Prove, blobs_dev, blobs_host, lens, count);
    b.commitments_xy = commitments_xy;
    b.commitments_inf = commitments_inf;
    b.out_xy = out_xy;
    b.out_inf = out_inf;
    return run_batch(b);
}
// ------------------------------------------------------------------------------- proofs at the caller's points
int kzgb_compute_proofs(kzgb_ctx* c, const uint64_t* const* evals_mont, const size_t* ns, size_t count,
                        const uint64_t* zs_mont, uint64_t* out_xy, uint8_t* out_inf, uint64_t* ys_mont) {
    Guard g(c);
    return compute_proofs(c, evals_mont, false, ns, count, zs_mont, out_xy, out_inf, ys_mont);
}
int kzgb_compute_proofs_dev(kzgb_ctx* c, const uint64_t* const* evals_dev, const size_t* ns, size_t count,
                            const uint64_t* zs_mont, uint64_t* out_xy, uint8_t* out_inf, uint64_t* ys_mont) {
    Guard g(c);
    return compute_proofs(c, evals_dev, true, ns, count, zs_mont, out_xy, out_inf, ys_mont);
}
// ------------------------------------------------------------------------------- commitments of the caller's polynomials
int kzgb_commit_evals(kzgb_ctx* c, const uint64_t* const* evals_mont, const size_t* ns, size_t count, uint64_t* out_xy,
                      uint8_t* out_inf) {
    Guard g(c);
    return commit_polys(c, false, evals_mont, false, ns, count, out_xy, out_inf);
}
int kzgb_commit_evals_dev(kzgb_ctx* c, const uint64_t* const* evals_dev, const size_t* ns, size_t count, uint64_t* out_xy,
                          uint8_t* out_inf) {
    Guard g(c);
    return commit_polys(c, false, evals_dev, true, ns, count, out_xy, out_inf);
}
int kzgb_commit_coeffs(kzgb_ctx* c, const uint64_t* const* coeffs_mont, const size_t* ns, size_t count, uint64_t* out_xy,
                       uint8_t* out_inf) {
    Guard g(c);
    return commit_polys(c, true, coeffs_mont, false, ns, count, out_xy, out_inf);
}
int kzgb_commit_coeffs_dev(kzgb_ctx* c, const uint64_t* const* coeffs_dev, const size_t* ns, size_t count, uint64_t* out_xy,
                           uint8_t* out_inf) {
    Guard g(c);
    return commit_polys(c, true, coeffs_dev, true, ns, count, out_xy, out_inf);
}
// ------------------------------------------------------------------------------- per-blob verification, G1 side
int kzgb_verify_blob_proofs_g1(kzgb_ctx* c, const uint8_t* const* blobs, const size_t* lens, size_t count,
                               const uint64_t* commitments_xy, const uint8_t* commitments_inf, const uint64_t* proofs_xy,
                               const uint8_t* proofs_inf, uint64_t* out_xy, uint8_t* out_inf, uint64_t* z_out, uint64_t* y_out) {
    Guard g(c);
    return verify_blob_proofs(c, nullptr, blobs, lens, count, commitments_xy, commitments_inf, proofs_xy, proofs_inf, out_xy,
                              out_inf, z_out, y_out);
}
int kzgb_verify_blob_proofs_g1_dev(kzgb_ctx* c, const uint8_t* const* blobs_dev, const uint8_t* const* blobs_host,
                                   const size_t* lens, size_t count, const uint64_t* commitments_xy,
                                   const uint8_t* commitments_inf, const uint64_t* proofs_xy, const uint8_t* proofs_inf,
                                   uint64_t* out_xy, uint8_t* out_inf, uint64_t* z_out, uint64_t* y_out) {
    Guard g(c);
    return verify_blob_proofs(c, blobs_dev, blobs_host, lens, count, commitments_xy, commitments_inf, proofs_xy, proofs_inf,
                              out_xy, out_inf, z_out, y_out);
}
// ------------------------------------------------------------------------------- per-blob verification, the bools
int kzgb_verify_proofs(kzgb_ctx* c, size_t count, const uint64_t* commitments_xy, const uint8_t* commitments_inf,
                       const uint64_t* proofs_xy, const uint8_t* proofs_inf, const uint64_t* zs_mont, const uint64_t* ys_mont,
                       uint8_t* ok) {
    Guard g(c);
    return verify_proofs(c, count, commitments_xy, commitments_inf, proofs_xy, proofs_inf, zs_mont, ys_mont, ok);
}
int kzgb_verify_blob_proofs(kzgb_ctx* c, const uint8_t* const* blobs, const size_t* lens, size_t count,
                            const uint64_t* commitments_xy, const uint8_t* commitments_inf, const uint64_t* proofs_xy,
                            const uint8_t* proofs_inf, uint8_t* ok) {
    Guard g(c);
    return verify_blob_proofs(c, nullptr, blobs, lens, count, commitments_xy, commitments_inf, proofs_xy, proofs_inf, nullptr,
                              nullptr, nullptr, nullptr, ok);
}
int kzgb_verify_blob_proofs_dev(kzgb_ctx* c, const uint8_t* const* blobs_dev, const uint8_t* const* blobs_host,
                                const size_t* lens, size_t count, const uint64_t* commitments_xy,
                                const uint8_t* commitments_inf, const uint64_t* proofs_xy, const uint8_t* proofs_inf,
                                uint8_t* ok) {
    Guard g(c);
    return verify_blob_proofs(c, blobs_dev, blobs_host, lens, count, commitments_xy, commitments_inf, proofs_xy, proofs_inf,
                              nullptr, nullptr, nullptr, nullptr, ok);
}
// ------------------------------------------------------------------------------- batch verification (RLC)
int kzgb_verify_batch_rlc(kzgb_ctx* c, const uint8_t* const* blobs, const size_t* lens, size_t count,
                          const uint64_t* commitments_xy, const uint8_t* commitments_inf, const uint64_t* proofs_xy,
                          const uint8_t* proofs_inf, uint64_t lhs_xy[8], uint8_t* lhs_inf, uint64_t rhs_xy[8], uint8_t* rhs_inf) {
    Guard g(c);
    return verify_batch_rlc(c, nullptr, blobs, lens, count, commitments_xy, commitments_inf, proofs_xy, proofs_inf, lhs_xy,
                            lhs_inf, rhs_xy, rhs_inf);
}
int kzgb_verify_batch_rlc_dev(kzgb_ctx* c, const uint8_t* const* blobs_dev, const uint8_t* const* blobs_host,
                              const size_t* lens, size_t count, const uint64_t* commitments_xy, const uint8_t* commitments_inf,
                              const uint64_t* proofs_xy, const uint8_t* proofs_inf, uint64_t lhs_xy[8], uint8_t* lhs_inf,
                              uint64_t rhs_xy[8], uint8_t* rhs_inf) {
    Guard g(c);
    return verify_batch_rlc(c, blobs_dev, blobs_host, lens, count, commitments_xy, commitments_inf, proofs_xy, proofs_inf,
                            lhs_xy, lhs_inf, rhs_xy, rhs_inf);
}
int kzgb_verify_kzg_proof_batch_rlc(kzgb_ctx* c, size_t count, const uint64_t* commitments_xy, const uint8_t* commitments_inf,
                                    const uint64_t* proofs_xy, const uint8_t* proofs_inf, const uint64_t* zs_mont,
                                    const uint64_t* ys_mont, const uint64_t* poly_lens, uint64_t lhs_xy[8], uint8_t* lhs_inf,
                                    uint64_t rhs_xy[8], uint8_t* rhs_inf) {
    Guard g(c);
    return verify_openings_rlc(c, count, commitments_xy, commitments_inf, proofs_xy, proofs_inf, zs_mont, ys_mont, poly_lens,
                               lhs_xy, lhs_inf, rhs_xy, rhs_inf);
}
}  // extern "C"
