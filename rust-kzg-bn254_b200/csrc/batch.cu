// The blob-batch pipelines: kzgb_commit_and_prove_blobs{,_dev} -- commitment and proof of many blobs on several lanes
// while a hashing stage produces the Fiat-Shamir transcripts -- and kzgb_verify_batch_rlc.
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
    size_t dev_k = 0;       // transcripts hashed on the device (the last dev_k blobs)
    bool dev_lanes = false; // k_fs_midstate_lanes instead of k_fs_midstate_long
};
HashPlan hash_plan(const size_t* lens, size_t count, bool device_possible) {
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
    const double t_gpu = 2.75e-3 * per_blob / (double)(16u << 20);  // commit + proof of one blob
    // eligible blobs: exactly 32 * 2^j bytes, j >= 10 (the multi-buffer and device kernels hash whole 64-byte blocks)
    size_t eligible_total = 0, eligible_tail = 0;
    for (size_t i = 0; i < count; i++) eligible_total += hash_mb_eligible(lens[i]);
    while (eligible_tail < count && eligible_tail < FSL_CAP && hash_mb_eligible(lens[count - 1 - eligible_tail])) eligible_tail++;
    const int mb_opt = g_hash_mb.load();
    // "keeps up" = the single-stream pool needs at most half of this context's hardware threads for the duration of the GPU work:
    // the other half belongs to the lanes and the driver (measured on 4 hardware threads per rank: 291 blobs/s single stream, 367 multi-buffer)
    const bool ni_keeps_up = bytes / rate_ni <= 0.5 * count * t_gpu;
    if (sha256_has_mb16() && mb_opt != 0 && eligible_total >= 16 && (mb_opt == 1 || (!ni_keeps_up && eligible_total >= 32))) {
        hp.mb = true;
        const int ht = g_hash_threads.load();
        hp.mb_threads = (size_t)std::max(1.0, ht > 0 ? (double)ht : share - 1.0);  // one hardware thread of the share stays with the lanes
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
            const double t = std::max({(count + dev_cost * k) * t_gpu, (double)(count - k) * per_blob / rate_host, t_dev + k * t_gpu * 0.5});
            if (t < best * 0.97) { best = t; hp.dev_k = k; hp.dev_lanes = lanes != 0; }
        }
    }
    return hp;
}

// ---------------------------------------------------------------- planning
// One kzgb_commit_and_prove_blobs{,_dev} call: its arguments and the plan made for them.
struct Batch {
    kzgb_ctx* c;
    const uint8_t* const* blobs_dev;   // nullptr: the blobs are only on the host
    const uint8_t* const* blobs_host;  // the transcripts are hashed from these
    const size_t* lens;
    size_t count;
    uint8_t* commitments32;
    uint8_t* proofs32;
    size_t max_n = 0;
    std::vector<std::pair<size_t, size_t>> groups;  // small blobs: (first blob, blobs); empty: one blob per task
    int n_lanes = 0;
    bool deep = false;              // the lanes sleep on a blocking event while they wait (lane_wait)
    std::vector<size_t> byte_off;   // resident: offset of every blob in c->batch_bytes
    bool resident = false;
};

// Validation, groups, lanes and the tables every size of the batch needs.
int plan_batch(Batch& b) {
    kzgb_ctx* c = b.c;
    const size_t* lens = b.lens;
    const size_t count = b.count;
    for (size_t i = 0; i < count; i++) {
        if (lens[i] == 0) return fail(c, KZGB_ERR_GENERIC, "Length of data after padding is 0");
        if (int rc = check_srs_capacity(c, blob_poly_len(lens[i]))) return rc;
        b.max_n = std::max(b.max_n, blob_poly_len(lens[i]));
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
        if (!c->lag[logn].table) all_lagrange = false;
    }
    if (!all_lagrange && c->auto_precompute && (!c->wtable || c->wt_first != 0 || b.max_n > c->wt_n) && c->srs_n <= ((size_t)1 << 22)) {
        rc = do_precompute(c, 0, std::min(c->srs_n, next_pow2(b.max_n)), 0);
        if (rc && rc != KZGB_ERR_DEVICE) return rc;
    }
    for (size_t gi = 0; gi < b.groups.size(); gi++) {  // the batched MSM needs a window table for every size
        size_t n = blob_poly_len(lens[b.groups[gi].first]);
        int logn = log2_exact(n);
        bool lag_ok = c->lag[logn].table && g_lagrange.load();
        if (!lag_ok && !(c->wtable && c->wt_first == 0 && n <= c->wt_n)) { b.groups.clear(); break; }
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
// Transcript midstates (everything but the commitment): a pool of host threads from the front of the batch and, when
// the host cannot keep up with the GPU, one warp per transcript on the device for the blobs at its end
// (device_hash_share).  Whoever delivers a midstate first installs it; the lanes take proofs as they become ready.
// The lane schedulers keep their own shared state under the stage's lock as well.
class HashStage {
public:
    std::mutex mu;
    std::condition_variable cv;
    std::vector<Sha256> mid;   // midstate of blob i, once ready[i]
    std::vector<uint8_t> ready;
    bool failed = false;       // a lane failed: everyone stops
    const size_t dev_first;    // blobs [dev_first, count) are the device's share

    HashStage(const Batch& batch, const HashPlan& hp);
    // The one teardown, on every exit path: stop the device hashing and wait for it (it reads the blob bytes), then
    // for the pool.
    ~HashStage();
    void fail() {
        std::lock_guard<std::mutex> lk(mu);
        failed = true;
        cv.notify_all();
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
        std::lock_guard<std::mutex> lk(mu);
        if (!ready[i]) { mid[i] = sh; ready[i] = 1; }
    }
};

HashStage::HashStage(const Batch& batch, const HashPlan& hp)
    : mid(batch.count), ready(batch.count, 0), dev_first(batch.count - hp.dev_k), b(batch), c(batch.c), dev_k(hp.dev_k) {
    if (dev_k && start_device(hp.dev_lanes) != cudaSuccess) { cudaGetLastError(); dev_failed.store(true); }  // the host pool takes the whole batch
    if (dev_k && !dev_failed.load()) poller = std::thread(&HashStage::poll_device, this);
    for (size_t i = 0; i < b.count;) {
        size_t j = i + 1;
        if (hp.mb && i < dev_first && hash_mb_eligible(b.lens[i])) {
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
    { std::lock_guard<std::mutex> lk(mu); dev_stop.store(true); }
    if (fsl_cancel) *fsl_cancel = 1;
    next_task.store(tasks.size());
    cv.notify_all();
    if (poller.joinable()) poller.join();
    for (auto& t : pool) t.join();
    if (dev_k && c->hash_st) cudaStreamSynchronize(c->hash_st);
}

// The device's share: host blobs go up on the hashing stream, then one kernel hashes all of it.
cudaError_t HashStage::start_device(bool lanes) {
    cudaError_t e = cudaSuccess;
    if (!c->hash_st) {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        e = cudaStreamCreateWithPriority(&c->hash_st, cudaStreamNonBlocking, hi);  // its few blocks must become resident at once
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&c->ev_hash_uploaded, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaHostAlloc((void**)&c->fsl_host, (9 * FSL_CAP + 16) * 4, cudaHostAllocMapped);
    }
    if (e == cudaSuccess) e = c->fsl_args.reserve(FSL_CAP * 16);
    if (e != cudaSuccess) return e;
    fsl_state = c->fsl_host;
    fsl_done = c->fsl_host + 8 * FSL_CAP;
    fsl_cancel = c->fsl_host + 9 * FSL_CAP;
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
            e = cudaMemcpyAsync(slot, b.blobs_host[i], b.lens[i], cudaMemcpyHostToDevice, c->hash_st);
            ptrs[j] = slot;
        }
    }
    const uint8_t** d_ptrs = (const uint8_t**)c->fsl_args.p;
    uint32_t* d_ns = (uint32_t*)((char*)c->fsl_args.p + FSL_CAP * 8);
    if (e == cudaSuccess) e = cudaEventRecord(c->ev_hash_uploaded, c->hash_st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_ptrs, ptrs.data(), dev_k * 8, cudaMemcpyHostToDevice, c->hash_st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_ns, ns.data(), dev_k * 4, cudaMemcpyHostToDevice, c->hash_st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->hash_st);  // the argument vectors die with this scope
    if (e != cudaSuccess) return e;
    fs_midstate_long_launch(d_ptrs, d_ns, (uint32_t)dev_k, fsl_state, (uint32_t*)fsl_done, (const uint32_t*)fsl_cancel, lanes, c->hash_st);
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
        if (any) cv.notify_all();
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
            cv.notify_all();
            continue;
        }
        if (i >= dev_first) {  // the device's share: only if the device path failed
            std::unique_lock<std::mutex> lk(mu);
            cv.wait(lk, [&] { return ready[i] != 0 || failed || dev_failed.load() || dev_stop.load(); });
            if (ready[i] || failed || dev_stop.load()) continue;
        }
        Sha256 sh;
        challenge_midstate(sh, b.blobs_host[i], b.lens[i], blob_poly_len(b.lens[i]));
        install(i, sh);
        cv.notify_all();
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

// Small blobs: groups of equal-size blobs, each phase of a group is ONE batched launch set.
int group_lane(const Batch& b, HashStage& hs, std::atomic<size_t>& next_group, int li) {
    kzgb_ctx* c = b.c;
    const uint8_t* const* blobs_dev = b.blobs_dev;
    const size_t* lens = b.lens;
    Lane& L = c->lanes[li];
    std::vector<Affine> pts;
    std::vector<Fr> zt;
    for (;;) {
        size_t gi = next_group.fetch_add(1);
        if (gi >= b.groups.size()) return KZGB_OK;
        { std::lock_guard<std::mutex> lk(hs.mu); if (hs.failed) return KZGB_OK; }
        const size_t i0 = b.groups[gi].first, bn = b.groups[gi].second;
        const size_t n = blob_poly_len(lens[i0]);
        const int logn = log2_exact(n);
        const kzgb_ctx::LagTable* lag = (c->lag[logn].table && g_lagrange.load()) ? &c->lag[logn] : nullptr;
        Fr ninv = ninv_mont(logn);
        int r = KZGB_OK;
        auto ck = [&](cudaError_t e, const char* what) {
            if (!r && e != cudaSuccess) r = fail(c, KZGB_ERR_DEVICE, std::string("CUDA error: ") + cudaGetErrorString(e) + " at " + what);
        };
        ck(L.evals.reserve(bn * n * sizeof(Fr)), "evals");
        ck(L.work.reserve(bn * n * sizeof(Fr)), "work");
        ck(L.small.reserve((3 * bn + 8) * sizeof(Fr)), "small");
        ck(L.eval_scratch.reserve(eval_quotient_scratch_elems((uint32_t)n, (uint32_t)bn) * sizeof(Fr)), "eval scratch");
        if (!lag) ck(L.ntt_scratch.reserve(bn * n * sizeof(Fr)), "ntt scratch");
        if (!blobs_dev) ck(L.bytes.reserve(bn * n * 32), "bytes");
        bool full = true;  // every blob fills its polynomial: one conversion launch for the group
        for (size_t k = 0; k < bn; k++) full = full && lens[i0 + k] == n * 32;
        bool dev_run = blobs_dev && full;  // device blobs back to back: one conversion launch too
        for (size_t k = 0; k < bn && dev_run; k++) dev_run = blobs_dev[i0 + k] == blobs_dev[i0] + k * n * 32;
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
        // commitments
        MsmJob job;
        pts.resize(bn);
        if (!r) {
            const Fr* sc = (const Fr*)L.evals.p;
            if (!lag) {
                ck(cudaMemcpyAsync(L.work.p, L.evals.p, bn * n * sizeof(Fr), cudaMemcpyDeviceToDevice, L.st), "copy");
                ntt_launch((Fr*)L.work.p, logn, (uint32_t)bn, true, c->tw, c->logN, &ninv, (Fr*)L.ntt_scratch.p, L.st);
                sc = (const Fr*)L.work.p;
            }
            if (!r) r = msm_enqueue_batched(c, L, sc, n, bn, lag, &job);
        }
        if (!r) r = msm_finish_batched(c, L, job, bn, pts.data());
        if (!r) {
            for (size_t k = 0; k < bn; k++) serialize_compressed(pts[k], b.commitments32 + 32 * (i0 + k));
            // challenges: the transcript midstates come from the hashing stage
            zt.resize(2 * bn);
            {
                std::unique_lock<std::mutex> lk(hs.mu);
                for (size_t k = 0; k < bn; k++) hs.cv.wait(lk, [&] { return hs.ready[i0 + k] != 0 || hs.failed; });
                if (hs.failed) return KZGB_OK;
            }
            bool any_in_domain = false;
            for (size_t k = 0; k < bn; k++) {
                zt[k] = challenge_finish(hs.mid[i0 + k], pts[k]);
                zt[bn + k] = eval_tinv(zt[k], logn, &any_in_domain);
            }
            Fr* d_z = (Fr*)L.small.p;  // [z x bn | tinv x bn | y x bn]
            ck(cudaMemcpyAsync(d_z, zt.data(), 2 * bn * sizeof(Fr), cudaMemcpyHostToDevice, L.st), "H2D of the challenges");
            eval_quotient_launch((Fr*)L.evals.p, (uint32_t)n, logn, (uint32_t)bn, d_z, d_z + bn, c->tw, c->logN, &ninv,
                                 (Fr*)L.eval_scratch.p, (Fr*)L.work.p, d_z + 2 * bn, L.st, !any_in_domain);
            if (!lag) ntt_launch((Fr*)L.work.p, logn, (uint32_t)bn, true, c->tw, c->logN, &ninv, (Fr*)L.ntt_scratch.p, L.st);
            if (!r) r = msm_enqueue_batched(c, L, (const Fr*)L.work.p, n, bn, lag, &job);
            if (!r) r = msm_finish_batched(c, L, job, bn, pts.data());
        }
        if (r) { hs.fail(); return r; }
        for (size_t k = 0; k < bn; k++) serialize_compressed(pts[k], b.proofs32 + 32 * (i0 + k));
    }
}

int run_groups(const Batch& b, HashStage& hs) {
    std::atomic<size_t> next_group{0};
    return run_lanes(b, [&](int li) { return group_lane(b, hs, next_group, li); });
}

// Task scheduler.  commit(i) needs nothing; proof(i) needs commit(i) and the transcript midstate of
// blob i (host SHA-256, ~9 ms for 16 MiB).  A lane takes the lowest ready proof, else the next
// commit, so the GPU never idles behind the hashing pool.  The queue lives under the hashing stage's lock.
struct TaskQueue {
    std::vector<uint8_t> commit_done, proof_taken;
    std::vector<Affine> commits;
    size_t next_commit = 0, proofs_taken = 0, proof_scan = 0;
};

// false: nothing left for this lane (every proof taken, or a lane failed)
bool take_task(const Batch& b, HashStage& hs, TaskQueue& q, size_t* task, bool* is_proof) {
    std::unique_lock<std::mutex> lk(hs.mu);
    for (;;) {
        if (hs.failed) return false;
        while (q.proof_scan < b.count && q.proof_taken[q.proof_scan]) q.proof_scan++;
        for (size_t k = q.proof_scan; k < b.count && k < q.next_commit; k++) {
            if (q.proof_taken[k] || !q.commit_done[k] || !hs.ready[k]) continue;
            q.proof_taken[k] = 1; q.proofs_taken++;
            *task = k; *is_proof = true;
            if (q.proofs_taken == b.count) hs.cv.notify_all();  // lanes with nothing left to take can leave
            return true;
        }
        if (q.next_commit < b.count) { *task = q.next_commit++; *is_proof = false; return true; }
        if (q.proofs_taken == b.count) return false;
        hs.cv.wait(lk);
    }
}

int task_lane(const Batch& b, HashStage& hs, TaskQueue& q, int li) {
    kzgb_ctx* c = b.c;
    Lane& L = c->lanes[li];
    size_t i = 0;
    bool is_proof = false;
    while (take_task(b, hs, q, &i, &is_proof)) {
        size_t len = b.lens[i], n = blob_poly_len(len);
        const uint8_t* dev_bytes = b.blobs_dev ? b.blobs_dev[i] : nullptr;
        int r = KZGB_OK;
        if (!dev_bytes && b.resident) {
            uint8_t* slot = (uint8_t*)c->batch_bytes.p + b.byte_off[i];
            if (hs.uploaded_here(i)) {
                if (!is_proof && cudaStreamWaitEvent(L.st, c->ev_hash_uploaded, 0) != cudaSuccess)
                    r = fail(c, KZGB_ERR_DEVICE, "CUDA error: cudaStreamWaitEvent failed");
            } else if (!is_proof && len) {
                if (cudaMemcpyAsync(slot, b.blobs_host[i], len, cudaMemcpyHostToDevice, L.st) != cudaSuccess)
                    r = fail(c, KZGB_ERR_DEVICE, "CUDA error: H2D copy of a blob failed");
            }
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
        if (r) { hs.fail(); return r; }
        if (is_proof) {
            serialize_compressed(out, b.proofs32 + 32 * i);
        } else {
            serialize_compressed(out, b.commitments32 + 32 * i);
            { std::lock_guard<std::mutex> lk(hs.mu); q.commits[i] = out; q.commit_done[i] = 1; }
            hs.cv.notify_all();
        }
    }
    return KZGB_OK;
}

int run_tasks(const Batch& b, HashStage& hs) {
    TaskQueue q{std::vector<uint8_t>(b.count, 0), std::vector<uint8_t>(b.count, 0), std::vector<Affine>(b.count)};
    return run_lanes(b, [&](int li) { return task_lane(b, hs, q, li); });
}

int commit_and_prove(kzgb_ctx* c, const uint8_t* const* blobs_dev, const uint8_t* const* blobs_host, const size_t* lens,
                     size_t count, uint8_t* commitments32, uint8_t* proofs32) {
    if (count == 0) return KZGB_OK;
    Batch b{c, blobs_dev, blobs_host, lens, count, commitments32, proofs32};
    int rc = plan_batch(b);
    if (rc) return rc;
    stage_blob_bytes(b);
    const HashPlan hplan = b.groups.empty() ? hash_plan(lens, count, blobs_dev || b.resident) : HashPlan();
    {
        HashStage hs(b, hplan);
        rc = b.groups.empty() ? run_tasks(b, hs) : run_groups(b, hs);
    }
    if (b.groups.empty() && c->batch_bytes.cap > ((size_t)g_batch_keep_mib.load() << 20)) c->batch_bytes.release();  // bounded residency between calls
    return rc;
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
    int rc = msm_blocking(c, L, d_sc, false, 0, m, d_bases + m, lhs);
    if (rc) return rc;
    return msm_blocking(c, L, d_sc, false, 0, 2 * m + 1, d_bases, rhs);
}

}  // namespace

// =====================================================================================
extern "C" {

int kzgb_commit_and_prove_blobs(kzgb_ctx* c, const uint8_t* const* blobs, const size_t* lens, size_t count,
                                uint8_t* commitments32, uint8_t* proofs32) {
    Guard g(c);
    return commit_and_prove(c, nullptr, blobs, lens, count, commitments32, proofs32);
}
int kzgb_commit_and_prove_blobs_dev(kzgb_ctx* c, const uint8_t* const* blobs_dev, const uint8_t* const* blobs_host,
                                    const size_t* lens, size_t count, uint8_t* commitments32, uint8_t* proofs32) {
    Guard g(c);
    return commit_and_prove(c, blobs_dev, blobs_host, lens, count, commitments32, proofs32);
}
// ------------------------------------------------------------------------------- batch verification (RLC)
int kzgb_verify_batch_rlc(kzgb_ctx* c, const uint8_t* const* blobs, const size_t* lens, size_t count,
                          const uint64_t* commitments_xy, const uint8_t* commitments_inf, const uint64_t* proofs_xy,
                          const uint8_t* proofs_inf, uint64_t lhs_xy[8], uint8_t* lhs_inf, uint64_t rhs_xy[8], uint8_t* rhs_inf) {
    Guard g(c);
    Lane& L = c->lanes[0];
    const size_t m = count;
    Affine inf_pt; aff_set_inf(inf_pt);
    if (m == 0) { affine_to_abi(inf_pt, lhs_xy, lhs_inf); affine_to_abi(inf_pt, rhs_xy, rhs_inf); return KZGB_OK; }
    std::vector<Affine> Cs(m), Ps(m);
    for (size_t i = 0; i < m; i++) {
        Cs[i] = affine_from_abi(commitments_xy + 8 * i, commitments_inf ? commitments_inf[i] : 0);
        Ps[i] = affine_from_abi(proofs_xy + 8 * i, proofs_inf ? proofs_inf[i] : 0);
    }
    // validate_g1_point on all 2m points (batch.rs:30-37) -- on the GPU
    CK(c, L.bases.reserve((2 * m + 1) * sizeof(Affine)));
    CK(c, L.small.reserve(64 * sizeof(Fr)));
    Affine* d_bases = (Affine*)L.bases.p;  // [C_0..C_{m-1}, pi_0..pi_{m-1}, G]
    CK(c, cudaMemcpyAsync(d_bases, Cs.data(), m * sizeof(Affine), cudaMemcpyHostToDevice, L.st));
    CK(c, cudaMemcpyAsync(d_bases + m, Ps.data(), m * sizeof(Affine), cudaMemcpyHostToDevice, L.st));
    uint32_t* d_err = (uint32_t*)((Fr*)L.small.p + 32);
    CK(c, cudaMemsetAsync(d_err, 0xff, 32, L.st));
    g1_validate_launch(d_bases, (uint32_t)(2 * m), d_err, L.st);
    uint32_t herr = 0;
    CK(c, cudaMemcpyAsync(&herr, d_err, 4, cudaMemcpyDeviceToHost, L.st));
    CK(c, cudaStreamSynchronize(L.st));
    if (herr != 0xffffffffu) return fail(c, KZGB_ERR_NOT_ON_CURVE, "G1 point not on curve");

    // per-blob challenge (host SHA pool) and evaluation (GPU, batched over blobs of equal length)
    std::vector<size_t> ns(m);
    size_t max_n = 0;
    for (size_t i = 0; i < m; i++) {
        if (lens[i] == 0) return fail(c, KZGB_ERR_GENERIC, "Length of data after padding is 0");
        ns[i] = blob_poly_len(lens[i]);
        max_n = std::max(max_n, ns[i]);
    }
    int rc = ensure_twiddles(c, log2_exact(max_n));
    if (rc) return rc;
    std::vector<Fr> zs(m), ys(m);
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
                    challenge_midstate(sh, blobs[i], lens[i], ns[i]);
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
        CK(c, L.bytes.reserve(b * n * 32));
        CK(c, L.eval_scratch.reserve(eval_quotient_scratch_elems((uint32_t)n, (uint32_t)b) * sizeof(Fr)));
        CK(c, L.work.reserve(5 * b * sizeof(Fr)));
        bool full = (uint64_t)b * n < 0xffffffffull;  // every blob fills its polynomial: one conversion launch
        for (size_t k = 0; k < b && full; k++) full = lens[i0 + k] == n * 32;
        for (size_t k = 0; k < b;) {
            uint8_t* dst = (uint8_t*)L.bytes.p + k * n * 32;
            size_t run = 1;  // blobs that are adjacent in host memory go up in one copy
            while (full && k + run < b && blobs[i0 + k + run] == blobs[i0 + k] + run * n * 32) run++;
            size_t bytes = full ? run * n * 32 : lens[i0 + k];
            CK(c, cudaMemcpyAsync(dst, blobs[i0 + k], bytes, cudaMemcpyHostToDevice, L.st));
            if (!full) bytes_to_fr_launch(dst, lens[i0 + k], (Fr*)L.evals.p + k * n, (uint32_t)n, L.st);
            k += run;
        }
        if (full) bytes_to_fr_launch((const uint8_t*)L.bytes.p, (uint64_t)b * n * 32, (Fr*)L.evals.p, (uint32_t)(b * n), L.st);
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
        eval_quotient_launch((Fr*)L.evals.p, (uint32_t)n, logn, (uint32_t)b, d_z, d_t, c->tw, c->logN, &ninv,
                             (Fr*)L.eval_scratch.p, nullptr, d_y, L.st, !fs_device && !any_in_domain, d_in_domain);
        CK(c, cudaMemcpyAsync(&ys[i0], d_y, b * sizeof(Fr), cudaMemcpyDeviceToHost, L.st));
        CK(c, cudaStreamSynchronize(L.st));
        CK(c, cudaGetLastError());
        i0 = i1;
    }
    Affine lhs, rhs;
    rc = rlc_combine(c, L, Cs, Ps, ns, zs, ys, d_bases, &lhs, &rhs);
    if (rc) return rc;
    affine_to_abi(lhs, lhs_xy, lhs_inf);
    affine_to_abi(rhs, rhs_xy, rhs_inf);
    return KZGB_OK;
}
}  // extern "C"
