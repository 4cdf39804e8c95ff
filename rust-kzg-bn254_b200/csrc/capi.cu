// Host orchestration and the C ABI (include/kzg_bn254_b200.h): the context, its tables, the MSM plumbing, every
// single-call entry point, the measurement hooks and the option table.  The blob-batch pipelines are in batch.cu.
//
// One context = one GPU.  The context owns the HBM-resident SRS (monomial points plus the
// fixed-base window tables), the omega_N twiddle table, and a small set of "lanes": a lane is a
// CUDA stream with its own device workspace, driven by one host thread.  Single calls use
// lane 0; the blob-batch entry points run several lanes plus a pool of host threads that hash
// the Fiat-Shamir transcripts (SHA-256 of a 16 MiB blob is ~9 ms of inherently serial CPU work,
// several times the GPU time of the same blob, so it must overlap).
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstring>
#include <ctime>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/kzg_bn254_b200.h"
#include "../../include/kzg_bn254_b200_bench.h"
#include "ctx.hpp"
#include "kzgb_internal.hpp"
#include "sha256.hpp"
#include "transcript.hpp"

using namespace kzgb;

namespace kzgb {

std::atomic<uint64_t> g_launch_count{0};

static std::mutex g_err_mu;
int fail(kzgb_ctx* c, int code, const std::string& msg) {
    if (c) { std::lock_guard<std::mutex> lk(g_err_mu); c->err = msg; }
    return code;
}
int check_srs_capacity(kzgb_ctx* c, size_t n) {
    if (n <= c->srs_n) return KZGB_OK;
    char msg[160];
    snprintf(msg, sizeof msg, "SRS capacity exceeded: polynomial_len=%zu srs_len=%zu", n, c->srs_n);
    return fail(c, KZGB_ERR_SRS_CAPACITY, msg);
}
int check_commit_blob_len(kzgb_ctx* c, size_t n) {
    if (n > ((size_t)1 << 28)) return fail(c, KZGB_ERR_GENERIC, "Input size exceeds maximum polynomial size");
    return check_srs_capacity(c, n);
}

// The MSM gathers 64-byte points at random from tables far larger than L2: with the default fetch granularity a
// miss pulls the whole 128-byte line and doubles the DRAM traffic of the accumulation.  The limit is device-wide,
// so only contexts that own their stream touch it (a caller-supplied stream means the caller owns the device's
// configuration), the previous value is put back when the last such context of a device is destroyed, and option
// "l2_fetch_64" = 0 leaves it alone altogether.
struct L2Limit { int refs = 0; size_t prev = 0; };
std::mutex g_l2_mu;
L2Limit g_l2[64];
void l2_limit_acquire(int device) {  // current device == device
    if (device < 0 || device >= 64) return;
    std::lock_guard<std::mutex> lk(g_l2_mu);
    if (g_l2[device].refs++ == 0) {
        if (cudaDeviceGetLimit(&g_l2[device].prev, cudaLimitMaxL2FetchGranularity) != cudaSuccess) g_l2[device].prev = 0;
        cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, 64);
        cudaGetLastError();
    }
}
void l2_limit_release(int device) {
    if (device < 0 || device >= 64) return;
    std::lock_guard<std::mutex> lk(g_l2_mu);
    if (--g_l2[device].refs == 0 && g_l2[device].prev) {
        cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, g_l2[device].prev);
        cudaGetLastError();
    }
}

// ---------------------------------------------------------------- host field helpers
const uint32_t ROOT28_CANON[8] = {0x725b19f0u, 0x9bd61b6eu, 0x41112ed4u, 0x402d111eu,
                                  0x8ef62abcu, 0x00e0a7ebu, 0xa58a7e85u, 0x2a3c09f0u};  // consts.rs:51

Fr root_of_unity_mont(int k) {  // PRIMITIVE_ROOTS_OF_UNITY[k], Montgomery
    Fr w;
    memcpy(w.l, ROOT28_CANON, 32);
    fe_to_mont(w, w);
    for (int i = 28; i > k; i--) fe_sqr(w, w);
    return w;
}
Fr fr_from_u64(uint64_t v) {
    Fr a; fe_zero(a);
    a.l[0] = (uint32_t)v; a.l[1] = (uint32_t)(v >> 32);
    fe_to_mont(a, a);
    return a;
}
Fr ninv_mont(int logn) {
    Fr n = fr_from_u64(1ull << logn), r;
    fe_inv(r, n);
    return r;
}
// 1 / prod_i (z - w_i) with the zero factor (z = w_m) replaced by 1: prod = z^n - 1, or n / z in the domain
Fr eval_tinv(const Fr& z, int logn, bool* in_domain) {
    Fr zn = z, one, r;
    for (int k = 0; k < logn; k++) fe_sqr(zn, zn);
    fe_one(one);
    if (fe_eq(zn, one)) { if (in_domain) *in_domain = true; Fr ni = ninv_mont(logn); fe_mul(r, z, ni); return r; }
    fe_sub(zn, zn, one);
    fe_inv(r, zn);
    return r;
}
int log2_exact(size_t n) {
    int k = 0;
    while (((size_t)1 << k) < n) k++;
    return k;
}
size_t next_pow2(size_t n) { size_t p = 1; while (p < n) p <<= 1; return p; }

void affine_to_abi(const Affine& a, uint64_t out_xy[8], uint8_t* out_inf) {
    memcpy(out_xy, &a, 64);
    if (out_inf) *out_inf = aff_is_inf(a) ? 1 : 0;
}
Affine affine_from_abi(const uint64_t xy[8], uint8_t inf) {
    Affine a;
    if (inf) aff_set_inf(a); else memcpy(&a, xy, 64);
    return a;
}
void to_gnark_be(const Affine& a, uint8_t out[32]) {
    if (aff_is_inf(a)) { memset(out, 0, 32); out[0] = 0x40; return; }
    fe_to_be_bytes(a.x, out);
    out[0] |= fe_lexicographically_largest(a.y) ? 0xC0 : 0x80;
}

// ---------------------------------------------------------------- plan heuristics
int choose_c_var(size_t n) {
    int best = 4; double bc = 1e300;
    for (int c = 4; c <= 20; c++) {
        int W = window_count(c);
        if (W > MAX_SETS) continue;
        double cost = (double)n * W * 10.0 + (double)W * (double)(1u << (c - 1)) * 40.0;
        if (cost < bc) { bc = cost; best = c; }
    }
    return best;
}
int choose_c_fixed(size_t n) {
    int best = 4; double bc = 1e300;
    // measured at n = 2^19: c = 17 beats 16 (1.99 vs 2.08 ms); 18+ lose to the bucket tail.  Point-range shards
    // of a very large MSM (2^22 .. 2^26 points per GPU) amortise a longer tail: up to c = 22 (W = 12, a
    // 51.5 GB table at 2^26 points -- what 180 GB of HBM is for).
    const int c_max = n > ((size_t)1 << 20) ? 22 : 17;
    for (int c = 4; c <= c_max; c++) {
        int W = window_count(c);
        double cost = (double)n * W * 10.0 + (double)(1u << (c - 1)) * 140.0;  // the bucket tail is latency-bound
        if (cost < bc) { bc = cost; best = c; }
    }
    return best;
}

// ---------------------------------------------------------------- lanes
int lane_init(kzgb_ctx* c, Lane& L, cudaStream_t st) {
    if (st) { L.st = st; L.own_stream = false; }
    else {
        int lo = 0, hi = 0;
        CK(c, cudaDeviceGetStreamPriorityRange(&lo, &hi));  // numerically lower = higher priority
        CK(c, cudaStreamCreateWithPriority(&L.st, cudaStreamNonBlocking, hi));
        L.own_stream = true;
        if (g_stream_priority.load() && lo != hi) {
            CK(c, cudaStreamCreateWithPriority(&L.st_acc, cudaStreamNonBlocking, lo));
            CK(c, cudaEventCreateWithFlags(&L.ev_fork, cudaEventDisableTiming));
            CK(c, cudaEventCreateWithFlags(&L.ev_join, cudaEventDisableTiming));
        }
    }
    CK(c, cudaMallocHost((void**)&L.h_sets, sizeof(XYZZ) * MAX_SETS));
    CK(c, cudaMallocHost((void**)&L.h_fr, sizeof(Fr) * 16));
    CK(c, cudaMallocHost((void**)&L.h_entries, 16));
    CK(c, cudaEventCreate(&L.ev0));
    CK(c, cudaEventCreate(&L.ev1));
    CK(c, cudaEventCreateWithFlags(&L.ev_done, cudaEventDisableTiming));
    CK(c, cudaEventCreateWithFlags(&L.ev_block, cudaEventDisableTiming | cudaEventBlockingSync));
    return KZGB_OK;
}
void lane_destroy(Lane& L) {
    L.bytes.release(); L.evals.release(); L.work.release(); L.ntt_scratch.release();
    L.eval_scratch.release(); L.msm_ws.release(); L.small.release(); L.bases.release(); L.bucket_total.release();
    if (L.h_sets) cudaFreeHost(L.h_sets);
    if (L.h_fr) cudaFreeHost(L.h_fr);
    if (L.h_entries) cudaFreeHost(L.h_entries);
    if (L.ev0) cudaEventDestroy(L.ev0);
    if (L.ev1) cudaEventDestroy(L.ev1);
    if (L.ev_done) cudaEventDestroy(L.ev_done);
    if (L.ev_block) cudaEventDestroy(L.ev_block);
    if (L.ev_fork) cudaEventDestroy(L.ev_fork);
    if (L.ev_join) cudaEventDestroy(L.ev_join);
    if (L.st_acc) cudaStreamDestroy(L.st_acc);
    if (L.own_stream && L.st) cudaStreamDestroy(L.st);
    L = Lane();
}
int ensure_lanes(kzgb_ctx* c, int want) {
    if (want > MAX_LANES) want = MAX_LANES;
    while (c->n_lanes < want) {
        int rc = lane_init(c, c->lanes[c->n_lanes], nullptr);
        if (rc) return rc;
        c->n_lanes++;
    }
    return KZGB_OK;
}
cudaError_t drain_lanes(kzgb_ctx* c) {  // waits for every lane's stream, up to the first error
    for (int i = 0; i < c->n_lanes; i++)
        if (cudaError_t e = cudaStreamSynchronize(c->lanes[i].st)) return e;
    return cudaSuccess;
}
// called once the lane's stream has drained: duration of the accumulate kernel and the additions it performed
void lane_collect_acc(Lane& L) {
    if (L.ev_pending) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, L.ev0, L.ev1) == cudaSuccess) { L.acc_ms += ms; L.acc_launches++; L.acc_adds += *L.h_entries; }
        L.ev_pending = false;
    }
}

// ---------------------------------------------------------------- timeline trace
// kinds: 0 sort begins, 1 accumulate begins, 2 accumulate ends, 3 MSM ends (device events on the lane's streams);
//        10 host: MSM enqueued, 11 host: lane woke up with the result, 12 host: result finished (affine, serialised)
int lane_index(kzgb_ctx* c, const Lane& L) { return (int)(&L - &c->lanes[0]); }
cudaEvent_t trace_mark(kzgb_ctx* c, const Lane& L, int kind, cudaStream_t st) {
    if (!c->trace_on.load()) return nullptr;
    cudaEvent_t ev = nullptr;
    if (st) { if (cudaEventCreate(&ev) != cudaSuccess) return nullptr; cudaEventRecord(ev, st); }
    double host = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - c->trace_host0).count();
    std::lock_guard<std::mutex> lk(c->trace_mu);
    c->trace.push_back({lane_index(c, L), kind, ev, host});
    return ev;
}
// an event the caller records itself (accumulate begin / end inside msm_launch)
cudaEvent_t trace_event(kzgb_ctx* c, const Lane& L, int kind) {
    if (!c->trace_on.load()) return nullptr;
    cudaEvent_t ev = nullptr;
    if (cudaEventCreate(&ev) != cudaSuccess) return nullptr;
    std::lock_guard<std::mutex> lk(c->trace_mu);
    c->trace.push_back({lane_index(c, L), kind, ev, -1.0});
    return ev;
}

// ---------------------------------------------------------------- twiddles
int ensure_twiddles(kzgb_ctx* c, int logn) {
    if (c->tw && logn <= c->logN) return KZGB_OK;
    int want = std::max(logn, 1);
    if (c->srs_n) want = std::max(want, log2_exact(next_pow2(c->srs_n)) > 28 ? 28 : log2_exact(next_pow2(c->srs_n)));
    if (want > 28) return fail(c, KZGB_ERR_GENERIC, "power must be <= 28");
    CK(c, drain_lanes(c));
    if (c->tw) { cudaFree(c->tw); c->tw = nullptr; }
    CK(c, cudaMalloc((void**)&c->tw, sizeof(Fr) * ((size_t)1 << (want - 1))));
    Fr w = root_of_unity_mont(want);
    ntt_twiddles_launch(c->tw, want, &w, c->lanes[0].st);
    CK(c, cudaStreamSynchronize(c->lanes[0].st));
    c->logN = want;
    return KZGB_OK;
}

// ---------------------------------------------------------------- SRS tables
// A table of `bytes` fits in the free device memory plus the `reusable` bytes of the one it replaces, 2 GiB to spare.
int check_table_fits(kzgb_ctx* c, size_t bytes, size_t reusable) {
    size_t free_b = 0, total_b = 0;
    CK(c, cudaMemGetInfo(&free_b, &total_b));
    if (bytes + (2ull << 30) > free_b + reusable)
        return fail(c, KZGB_ERR_DEVICE, "not enough device memory for the fixed-base window tables");
    return KZGB_OK;
}
// Window table over `points` (n affine points on the device): table[w*n + i] = 2^(c*w) * points[i].
int build_window_table(kzgb_ctx* c, const Affine* points, size_t n, int cb, Affine** out, int* W_out) {
    if (cb < 2 || cb > 24) return fail(c, KZGB_ERR_GENERIC, "window_bits out of range");
    int W = window_count(cb);
    if ((uint64_t)W * n >= ((uint64_t)1 << 31))  // sorted refs are 31 bits + sign (msm.cu k_scatter)
        return fail(c, KZGB_ERR_GENERIC, "window table too large: windows x points must stay below 2^31 (use more window bits)");
    size_t bytes = (size_t)W * n * sizeof(Affine);
    if (int rc = check_table_fits(c, bytes, 0)) return rc;
    Lane& L = c->lanes[0];
    Affine* table = nullptr;
    CK(c, cudaMalloc((void**)&table, bytes));
    cudaError_t e = cudaMemcpyAsync(table, points, n * sizeof(Affine), cudaMemcpyDeviceToDevice, L.st);
    uint32_t batch = (uint32_t)std::min<size_t>(n, (size_t)1 << 18);
    DevBuf scratch;
    if (e == cudaSuccess) e = scratch.reserve(srs_precompute_scratch_bytes(batch, W));
    if (e == cudaSuccess) {
        srs_precompute_launch(table, (uint32_t)n, (uint32_t)n, cb, W, (XYZZ*)scratch.p, batch, L.st);
        e = cudaStreamSynchronize(L.st);
    }
    scratch.release();
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) { cudaFree(table); CK(c, e); }
    *out = table; *W_out = W;
    return KZGB_OK;
}

// Fixed-base window table over SRS points [first, first + count).  The fit is checked BEFORE the current table
// is given up, so a request that cannot be met leaves the context as it was.
int do_precompute(kzgb_ctx* c, size_t first, size_t count, int window_bits) {
    if (first >= c->srs_n) return KZGB_OK;
    if (count > c->srs_n - first) count = c->srs_n - first;
    if (count == 0) return KZGB_OK;
    int cb = window_bits > 0 ? window_bits : choose_c_fixed(count);
    if (cb < 2 || cb > 24) return fail(c, KZGB_ERR_GENERIC, "window_bits out of range");
    CK(c, drain_lanes(c));
    size_t reusable = c->wtable ? (size_t)c->wt_W * c->wt_n * sizeof(Affine) : 0;
    if (int rc = check_table_fits(c, (size_t)window_count(cb) * count * sizeof(Affine), reusable)) return rc;
    drop_window_table(c);
    Affine* table = nullptr;
    int W = 0;
    int rc = build_window_table(c, c->srs + first, count, cb, &table, &W);
    if (rc) return rc;
    c->wtable = table; c->wt_first = first; c->wt_n = count; c->wt_c = cb; c->wt_W = W;
    return KZGB_OK;
}

void drop_window_table(kzgb_ctx* c) {
    if (c->wtable) { cudaFree(c->wtable); c->wtable = nullptr; c->wt_n = 0; c->wt_first = 0; }
}
bool wtable_covers(const kzgb_ctx* c, size_t first, size_t n) { return c->wtable && first >= c->wt_first && first + n <= c->wt_first + c->wt_n; }
// Lazy build of the monomial window table over [0, next_pow2(first + n)) when none covers [first, first + n); SRS above
// 2^22 points get one only on request.  Short of device memory (KZGB_ERR_DEVICE) the MSMs run on the variable-base plan.
int ensure_window_table(kzgb_ctx* c, size_t first, size_t n) {
    if (!c->auto_precompute || wtable_covers(c, first, n) || c->srs_n > ((size_t)1 << 22)) return KZGB_OK;
    int rc = do_precompute(c, 0, std::min(c->srs_n, next_pow2(first + n)), 0);
    return rc == KZGB_ERR_DEVICE ? KZGB_OK : rc;
}

void lagrange_release(kzgb_ctx* c) {
    for (auto& t : c->lag) { if (t.table) cudaFree(t.table); t = kzgb_ctx::LagTable(); }
}

// Lagrange-basis window table for the domain of size n = 2^logn: L = IFFT_G1(SRS[..n]) (the points
// KZG::commit_eval_form recomputes on every call, kzg.rs:98), then the same window shifts as the
// monomial table.  One G1 inverse NTT per size and context; MSM(L, evals) is the eval-form commitment.
// Policy (kzgb_set_option):
//   "lagrange_after" k (default 2)  the table of a size is built when the k-th evaluation-form commitment / proof of
//                                   that size is requested (`weight` = how many this call stands for: a batch of b
//                                   blobs counts b); until then, and whenever there is no table, the same group element
//                                   comes from the Fr-IFFT + monomial MSM.  kzgb_srs_prepare_lagrange builds at once.
//   "lagrange_budget_mib" (default 0 = half of the device's memory)  bytes of Lagrange tables kept per context; the
//                                   least recently used ones are dropped to make room, a table that cannot fit is not built.
// Domains above 2^22 never get a table (W x 2^23 x 64 B = 6.4 GB and a 40 s G1 NTT per size): they stay on the
// Fr-IFFT + monomial path, documented in include/kzg_bn254_b200.h.
// Returns KZGB_OK with no table (t.table == nullptr) when the policy says "not yet", the feature is off or memory is short.
// Called under the context lock, never while lane threads run.
int ensure_lagrange(kzgb_ctx* c, int logn, uint32_t weight, bool force) {
    if (logn < 1 || logn > 28) return KZGB_OK;
    kzgb_ctx::LagTable& t = c->lag[logn];
    t.last_use = ++c->lag_clock;
    if (t.calls < 0xffff0000u) t.calls += weight;
    if (t.table) return KZGB_OK;
    const size_t n = (size_t)1 << logn;
    if (!g_lagrange.load() || !c->auto_precompute || n > c->srs_n || n > ((size_t)1 << 22)) return KZGB_OK;
    if (!force && t.calls < (uint32_t)std::max(1, g_lagrange_after.load())) return KZGB_OK;
    const int cb_plan = (c->wtable && c->wt_first == 0 && c->wt_n == n) ? c->wt_c : choose_c_fixed(n);
    {   // memory budget: drop least recently used tables until this one fits
        size_t free_b = 0, total_b = 0;
        CK(c, cudaMemGetInfo(&free_b, &total_b));
        size_t budget = g_lagrange_budget_mib.load() > 0 ? (size_t)g_lagrange_budget_mib.load() << 20 : total_b / 2;
        const size_t need = (size_t)window_count(cb_plan) * n * sizeof(Affine);
        if (need > budget) return KZGB_OK;
        for (;;) {
            size_t held = 0;
            kzgb_ctx::LagTable* lru = nullptr;
            for (auto& o : c->lag) {
                if (!o.table) continue;
                held += (size_t)o.W * o.n * sizeof(Affine);
                if (!lru || o.last_use < lru->last_use) lru = &o;
            }
            if (held + need <= budget || !lru) break;
            CK(c, drain_lanes(c));
            cudaFree(lru->table);
            lru->table = nullptr; lru->n = 0; lru->calls = 0;
        }
    }
    int rc = ensure_twiddles(c, logn);
    if (rc) return rc;
    CK(c, drain_lanes(c));
    Lane& L = c->lanes[0];
    DevBuf work, pts;
    if (work.reserve(n * sizeof(XYZZ)) != cudaSuccess || pts.reserve(n * sizeof(Affine)) != cudaSuccess) {
        cudaGetLastError(); work.release(); pts.release();
        return KZGB_OK;
    }
    Fr ninv = ninv_mont(logn), ninv_canon;
    fe_from_mont(ninv_canon, ninv);
    g1_intt_launch(c->srs, logn, (XYZZ*)work.p, (Affine*)pts.p, c->tw, c->logN, &ninv_canon, L.st);
    cudaError_t e = cudaStreamSynchronize(L.st);
    work.release();
    if (e != cudaSuccess) { pts.release(); CK(c, e); }
    Affine* table = nullptr;
    int W = 0, cb = cb_plan;  // an explicit window override of the monomial table carries over
    rc = build_window_table(c, (const Affine*)pts.p, n, cb, &table, &W);
    pts.release();
    if (rc == KZGB_ERR_DEVICE) { cudaGetLastError(); return KZGB_OK; }  // short of memory: stay on the monomial path
    if (rc) return rc;
    t.table = table; t.n = n; t.c = cb; t.W = W;
    return KZGB_OK;
}

// The table that serves evaluation-form MSMs of size 2^logn; none while option "lagrange" is off, even if one is resident.
const kzgb_ctx::LagTable* lagrange_table(const kzgb_ctx* c, int logn) {
    return logn >= 1 && logn <= 28 && c->lag[logn].table && g_lagrange.load() ? &c->lag[logn] : nullptr;
}

int srs_install(kzgb_ctx* c, Affine* dev_points, size_t n) {
    drain_lanes(c);
    if (c->srs) cudaFree(c->srs);
    drop_window_table(c);
    lagrange_release(c);
    c->srs = dev_points;
    c->srs_n = n;
    return KZGB_OK;
}

// ---------------------------------------------------------------- MSM
// Launch plan p on lane L in the lane's workspace and queue the copies of its window sums (and, for the statistics, of
// the length of its sorted list) to the host; msm_finish picks them up.
// d_blob != nullptr: the scalars are read from blob_len bytes of blob data instead (msm_launch_blob).
int msm_enqueue_plan(kzgb_ctx* c, Lane& L, const MsmPlan& p, const Fr* d_scalars, bool canonical, const Affine* table,
                     MsmJob* job, const uint8_t* d_blob = nullptr, uint64_t blob_len = 0) {
    CK(c, L.msm_ws.reserve(msm_workspace_bytes(p)));
    MsmWorkspace ws;
    msm_workspace_carve(p, L.msm_ws.p, &ws);
    lane_collect_acc(L);
    trace_mark(c, L, 0, L.st);
    cudaEvent_t tr1 = trace_event(c, L, 1), tr2 = trace_event(c, L, 2);
    if (d_blob) msm_launch_blob(p, ws, d_blob, blob_len, table, L.st, tr1 ? tr1 : L.ev0, tr2 ? tr2 : L.ev1, L.st_acc, L.ev_fork, L.ev_join);
    else msm_launch(p, ws, d_scalars, canonical, table, L.st, tr1 ? tr1 : L.ev0, tr2 ? tr2 : L.ev1, L.st_acc, L.ev_fork, L.ev_join);
    trace_mark(c, L, 3, L.st);
    trace_mark(c, L, 10, nullptr);
    L.ev_pending = !tr1;
    CK(c, cudaMemcpyAsync(L.h_entries, ws.hist + p.nbuckets, 4, cudaMemcpyDeviceToHost, L.st));
    CK(c, cudaMemcpyAsync(L.h_sets, ws.set_sums, sizeof(XYZZ) * p.sets, cudaMemcpyDeviceToHost, L.st));
    job->plan = p;
    job->active = true;
    return KZGB_OK;
}

// Enqueue an MSM on lane L.  bases == nullptr: over the SRS range [first, first+n).
// lag != nullptr: over the Lagrange-basis table of the domain of size n instead.
int msm_enqueue(kzgb_ctx* c, Lane& L, const Fr* d_scalars, bool canonical, size_t first, size_t n,
                const Affine* var_bases, MsmJob* job, const kzgb_ctx::LagTable* lag = nullptr) {
    if (n == 0) { job->active = false; return KZGB_OK; }
    MsmPlan p;
    const Affine* table;
    if (lag) {
        p = msm_make_plan((uint32_t)n, lag->c, true, (uint32_t)lag->n, 0);
        table = lag->table;
    } else if (!var_bases) {
        if (first > c->srs_n || n > c->srs_n - first) return fail(c, KZGB_ERR_GENERIC, "MSM range exceeds the SRS");
        if (!c->lanes_running.load()) {  // never from the lane threads of a running batch (they only read the tables)
            if (int rc = ensure_window_table(c, first, n)) return rc;
        }
        if (wtable_covers(c, first, n)) {
            p = msm_make_plan((uint32_t)n, c->wt_c, true, (uint32_t)c->wt_n, (uint32_t)(first - c->wt_first));
            table = c->wtable;
        } else {
            p = msm_make_plan((uint32_t)n, choose_c_var(n), false, 0, 0);
            table = c->srs + first;
        }
    } else {
        p = msm_make_plan((uint32_t)n, choose_c_var(n), false, 0, 0);
        table = var_bases;
    }
    if ((uint64_t)n * p.W >= 0xfff00000ull) return fail(c, KZGB_ERR_GENERIC, "MSM too large for one launch");
    return msm_enqueue_plan(c, L, p, d_scalars, canonical, table, job);
}

// 0: spin on the stream, 1: poll an event with short sleeps, 2: block on an event (option "lane_wait"; -1 = auto: spin
// unless the lane threads of the ranks on this host outnumber half of its hardware threads, then poll)
int lane_wait_mode() {
    const int opt = g_lane_wait.load();
    if (opt >= 0) return opt;
    static int mode = -1;
    if (mode < 0) {
        unsigned hw = std::thread::hardware_concurrency();
        int local = g_group_members.load();  // GPUs driven by this process (kzgb_group)
        if (const char* w = getenv("LOCAL_WORLD_SIZE")) { int v = atoi(w); if (v > local) local = v; }  // torchrun: ranks on this host
        mode = ((unsigned)local * 4u > hw / 2u) ? 1 : 0;
    }
    return mode;
}
bool lane_wait_polls() { return lane_wait_mode() != 0; }

// Wait for everything queued on the lane.  Spinning by default (a blocking-sync event costs ~0.3 ms per
// MSM in wake-up latency).  When the ranks on this host have more lane threads than spare cores, spinning
// lanes starve the SHA-256 pool (8 GPUs x 4 lanes on 32 cores): poll with short sleeps instead.
int lane_wait(kzgb_ctx* c, Lane& L) {
    const int mode = (g_lane_wait.load() < 0 && c->lanes_block.load()) ? 2 : lane_wait_mode();
    if (mode == 2) {  // sleep in the driver until the GPU's interrupt: no CPU at all while waiting
        CK(c, cudaEventRecord(L.ev_block, L.st));
        CK(c, cudaEventSynchronize(L.ev_block));
    } else if (mode == 1) {
        CK(c, cudaEventRecord(L.ev_done, L.st));
        for (;;) {
            cudaError_t q = cudaEventQuery(L.ev_done);
            if (q == cudaSuccess) break;
            if (q != cudaErrorNotReady) CK(c, q);
            struct timespec ts = {0, 30000};
            nanosleep(&ts, nullptr);
        }
    } else {
        CK(c, cudaStreamSynchronize(L.st));
    }
    CK(c, cudaGetLastError());
    return KZGB_OK;
}
// Wait for the lane and finish on the host: Horner over the window sums, then to affine.
int msm_finish(kzgb_ctx* c, Lane& L, const MsmJob& job, Affine* out) {
    if (!job.active) { aff_set_inf(*out); return KZGB_OK; }
    { int rc = lane_wait(c, L); if (rc) return rc; }
    trace_mark(c, L, 11, nullptr);
    lane_collect_acc(L);
    const MsmPlan& p = job.plan;
    XYZZ acc = L.h_sets[p.sets - 1];
    for (int w = p.sets - 2; w >= 0; w--) {
        for (int k = 0; k < p.c; k++) xyzz_dbl(acc, acc);
        xyzz_add(acc, L.h_sets[w]);
    }
    xyzz_to_affine(*out, acc);
    trace_mark(c, L, 12, nullptr);
    return KZGB_OK;
}

int msm_blocking(kzgb_ctx* c, Lane& L, const Fr* d_scalars, bool canonical, size_t first, size_t n,
                 const Affine* var_bases, Affine* out) {
    MsmJob job;
    int rc = msm_enqueue(c, L, d_scalars, canonical, first, n, var_bases, &job);
    if (rc) return rc;
    return msm_finish(c, L, job, out);
}

// A large fixed-base MSM whose scalars live in HOST memory (KZG::commit_coeff_form on a 2^26-coefficient polynomial,
// prover/src/kzg.rs:107-125): uploading 32 n bytes first and only then sorting leaves the GPU idle for the length of
// the copy (2 GiB at n = 2^26: ~40 ms in front of a 150 ms MSM).  Here the points are cut into S sub-ranges; the upload
// of sub-range k+1 runs on a copy stream while sub-range k is sorted and accumulated (double-buffered staging), the
// bucket sums of the sub-ranges are folded into one array (k_merge_buckets: one XYZZ addition per bucket and
// sub-range) and reduced ONCE.  Only the first sub-range's upload is exposed.
// Returns KZGB_OK with *done = false when the shape does not qualify (no table over the range, or too small to matter).
int msm_srs_host_pipelined(kzgb_ctx* c, Lane& L, const uint64_t* scalars, size_t first, size_t n, Affine* out, bool* done) {
    *done = false;
    if (n < ((size_t)1 << 22) || !g_pipelined_upload.load() || !wtable_covers(c, first, n)) return KZGB_OK;
    const size_t S = n >= ((size_t)1 << 24) ? 8 : 4;
    const size_t per = ((n + S - 1) / S + 31) & ~(size_t)31;
    if ((uint64_t)per * window_count(c->wt_c) >= 0xfff00000ull) return KZGB_OK;
    if (!c->copy_st) {
        CK(c, cudaStreamCreateWithFlags(&c->copy_st, cudaStreamNonBlocking));
        for (int k = 0; k < 2; k++) {
            CK(c, cudaEventCreateWithFlags(&c->ev_copied[k], cudaEventDisableTiming));
            CK(c, cudaEventCreateWithFlags(&c->ev_consumed[k], cudaEventDisableTiming));
        }
    }
    const MsmPlan p0 = msm_make_plan((uint32_t)per, c->wt_c, true, (uint32_t)c->wt_n, (uint32_t)(first - c->wt_first));
    CK(c, L.msm_ws.reserve(msm_workspace_bytes(p0)));
    CK(c, L.work.reserve(2 * per * sizeof(Fr)));
    CK(c, L.bucket_total.reserve((size_t)p0.nbuckets * sizeof(XYZZ)));
    MsmWorkspace ws;
    msm_workspace_carve(p0, L.msm_ws.p, &ws);
    Fr* stage[2] = {(Fr*)L.work.p, (Fr*)L.work.p + per};
    XYZZ* total = (XYZZ*)L.bucket_total.p;
    CK(c, cudaEventRecord(c->ev_consumed[0], L.st));  // the staging buffers are free once earlier work on the lane is done
    CK(c, cudaEventRecord(c->ev_consumed[1], L.st));
    size_t k = 0;
    for (size_t off = 0; off < n; off += per, k++) {
        const size_t cnt = std::min(per, n - off);
        const int b = (int)(k & 1);
        CK(c, cudaStreamWaitEvent(c->copy_st, c->ev_consumed[b], 0));
        CK(c, cudaMemcpyAsync(stage[b], scalars + 4 * off, cnt * sizeof(Fr), cudaMemcpyHostToDevice, c->copy_st));
        CK(c, cudaEventRecord(c->ev_copied[b], c->copy_st));
        CK(c, cudaStreamWaitEvent(L.st, c->ev_copied[b], 0));
        const MsmPlan p = msm_make_plan((uint32_t)cnt, c->wt_c, true, (uint32_t)c->wt_n, (uint32_t)(first + off - c->wt_first));
        msm_launch_buckets(p, ws, stage[b], false, c->wtable, L.st, nullptr, nullptr, L.st_acc, L.ev_fork, L.ev_join);
        CK(c, cudaEventRecord(c->ev_consumed[b], L.st));
        if (k == 0) CK(c, cudaMemcpyAsync(total, ws.buckets, (size_t)p0.nbuckets * sizeof(XYZZ), cudaMemcpyDeviceToDevice, L.st));
        else msm_merge_buckets(total, ws.buckets, p0.nbuckets, L.st);
    }
    msm_launch_reduce(p0, ws, total, L.st);
    CK(c, cudaMemcpyAsync(L.h_sets, ws.set_sums, sizeof(XYZZ), cudaMemcpyDeviceToHost, L.st));
    { int rc = lane_wait(c, L); if (rc) return rc; }
    xyzz_to_affine(*out, L.h_sets[0]);
    *done = true;
    return KZGB_OK;
}

// `batch` independent fixed-base MSMs of n_per scalars each in ONE set of launches (one bucket set per
// MSM): d_scalars holds batch * n_per scalars back to back.  Over the Lagrange-basis table `lag`, or the
// monomial window table when lag == nullptr.  Small polynomials are latency-bound one at a time (bucket
// reduction tail, host hand-off per MSM); batched they fill the GPU.
int msm_enqueue_batched(kzgb_ctx* c, Lane& L, const Fr* d_scalars, size_t n_per, size_t batch,
                        const kzgb_ctx::LagTable* lag, MsmJob* job) {
    if (n_per == 0 || batch == 0) { job->active = false; return KZGB_OK; }
    if (batch > (size_t)MAX_SETS) return fail(c, KZGB_ERR_GENERIC, "too many MSMs in one batch");
    const Affine* table;
    MsmPlan p;
    if (lag) {
        p = msm_make_plan((uint32_t)(n_per * batch), lag->c, true, (uint32_t)lag->n, 0, (uint32_t)batch);
        table = lag->table;
    } else {
        if (!wtable_covers(c, 0, n_per)) return fail(c, KZGB_ERR_GENERIC, "batched MSM needs a fixed-base table");
        p = msm_make_plan((uint32_t)(n_per * batch), c->wt_c, true, (uint32_t)c->wt_n, 0, (uint32_t)batch);
        table = c->wtable;
    }
    if ((uint64_t)n_per * batch * p.W >= 0xfff00000ull) return fail(c, KZGB_ERR_GENERIC, "MSM too large for one launch");
    return msm_enqueue_plan(c, L, p, d_scalars, false, table, job);
}
// Commitments of `batch` blobs over the Lagrange table `lag` of their size n, in ONE MSM whose first pass reads the
// blob bytes (no Montgomery form in between): blob k at d_bytes + 32 n k, len bytes in all, zero past len.  The
// result is read with msm_finish_batched (or msm_finish when batch == 1).
int commit_blob_enqueue(kzgb_ctx* c, Lane& L, const uint8_t* d_bytes, uint64_t len, size_t n, size_t batch,
                        const kzgb_ctx::LagTable* lag, MsmJob* job) {
    if (batch > (size_t)MAX_SETS) return fail(c, KZGB_ERR_GENERIC, "too many MSMs in one batch");
    const MsmPlan p = msm_make_plan((uint32_t)(n * batch), lag->c, true, (uint32_t)lag->n, 0, (uint32_t)batch);
    if ((uint64_t)n * batch * p.W >= 0xfff00000ull) return fail(c, KZGB_ERR_GENERIC, "MSM too large for one launch");
    return msm_enqueue_plan(c, L, p, nullptr, false, lag->table, job, d_bytes, len);
}
int msm_finish_batched(kzgb_ctx* c, Lane& L, const MsmJob& job, size_t batch, Affine* outs) {
    if (!job.active) { for (size_t k = 0; k < batch; k++) aff_set_inf(outs[k]); return KZGB_OK; }
    int rc = lane_wait(c, L);
    if (rc) return rc;
    lane_collect_acc(L);
    for (size_t k = 0; k < batch; k++) xyzz_to_affine(outs[k], L.h_sets[k]);
    return KZGB_OK;
}

// ---------------------------------------------------------------- polynomial pipeline pieces
// d_evals (n Fr, Montgomery) -> commitment.  Uses L.work / L.ntt_scratch.
int commit_evals_enqueue(kzgb_ctx* c, Lane& L, const Fr* d_evals, size_t n, MsmJob* job) {
    int logn = log2_exact(n);
    if (const kzgb_ctx::LagTable* lag = lagrange_table(c, logn))  // the evaluations ARE the scalars
        return msm_enqueue(c, L, d_evals, false, 0, n, nullptr, job, lag);
    int rc = ensure_twiddles(c, logn);
    if (rc) return rc;
    CK(c, L.work.reserve(n * sizeof(Fr)));
    CK(c, L.ntt_scratch.reserve(n * sizeof(Fr)));
    if ((const void*)d_evals != L.work.p)
        CK(c, cudaMemcpyAsync(L.work.p, d_evals, n * sizeof(Fr), cudaMemcpyDeviceToDevice, L.st));
    Fr ninv = ninv_mont(logn);
    ntt_launch((Fr*)L.work.p, logn, 1, true, c->tw, c->logN, &ninv, (Fr*)L.ntt_scratch.p, L.st);
    return msm_enqueue(c, L, (Fr*)L.work.p, false, 0, n, nullptr, job);
}

// y = p(z) into L.small[2] and, unless d_quotient is nullptr, the quotient; the twiddles of size n must be resident.
int eval_enqueue(kzgb_ctx* c, Lane& L, const Fr* d_evals, size_t n, const Fr& z, Fr* d_quotient) {
    const int logn = log2_exact(n);
    CK(c, L.eval_scratch.reserve(eval_quotient_scratch_elems((uint32_t)n, 1) * sizeof(Fr)));
    CK(c, L.small.reserve(64 * sizeof(Fr)));
    Fr* d_z = (Fr*)L.small.p;  // [z, tinv, y]
    L.h_fr[0] = z;
    bool in_domain = false;
    L.h_fr[1] = eval_tinv(z, logn, &in_domain);
    CK(c, cudaMemcpyAsync(d_z, &L.h_fr[0], 2 * sizeof(Fr), cudaMemcpyHostToDevice, L.st));
    Fr ninv = ninv_mont(logn);
    eval_quotient_launch(d_evals, (uint32_t)n, logn, 1, d_z, d_z + 1, c->tw, c->logN, &ninv, (Fr*)L.eval_scratch.p,
                         d_quotient, d_z + 2, L.st, !in_domain);
    return KZGB_OK;
}
// Waits for the lane and returns the y of the last eval_enqueue.
int eval_read_y(kzgb_ctx* c, Lane& L, Fr* y) {
    CK(c, cudaMemcpyAsync(&L.h_fr[3], (Fr*)L.small.p + 2, sizeof(Fr), cudaMemcpyDeviceToHost, L.st));
    CK(c, cudaStreamSynchronize(L.st));
    CK(c, cudaGetLastError());
    *y = L.h_fr[3];
    return KZGB_OK;
}

// quotient of d_evals at z (device, Montgomery) into L.work, then commit it.  y stays in L.small[2].
int proof_enqueue(kzgb_ctx* c, Lane& L, const Fr* d_evals, size_t n, const Fr& z_mont, MsmJob* job) {
    if (int rc = ensure_twiddles(c, log2_exact(n))) return rc;
    CK(c, L.work.reserve(n * sizeof(Fr)));
    CK(c, L.ntt_scratch.reserve(n * sizeof(Fr)));
    if (int rc = eval_enqueue(c, L, d_evals, n, z_mont, (Fr*)L.work.p)) return rc;
    return commit_evals_enqueue(c, L, (Fr*)L.work.p, n, job);  // the quotient is in evaluation form
}


size_t blob_poly_len(size_t len) { return next_pow2((len + 31) / 32); }  // Rust: 0usize.next_power_of_two() == 1

// blob bytes on the host -> L.bytes
int blob_upload(kzgb_ctx* c, Lane& L, const uint8_t* blob_host, size_t len) {
    CK(c, L.bytes.reserve(len ? len : 32));
    if (len) CK(c, cudaMemcpyAsync(L.bytes.p, blob_host, len, cudaMemcpyHostToDevice, L.st));
    return KZGB_OK;
}

// blob bytes on the host -> L.evals (n Fr Montgomery)
int blob_to_evals(kzgb_ctx* c, Lane& L, const uint8_t* blob_host, const uint8_t* blob_dev, size_t len, size_t n) {
    CK(c, L.evals.reserve(n * sizeof(Fr)));
    const uint8_t* src = blob_dev;
    if (!src) {
        if (int rc = blob_upload(c, L, blob_host, len)) return rc;
        src = (const uint8_t*)L.bytes.p;
    }
    bytes_to_fr_launch(src, len, (Fr*)L.evals.p, (uint32_t)n, L.st);
    return KZGB_OK;
}

// KZGB_ERR_NOT_ON_CURVE unless each of the n points at d_pts (device) is on the curve or the identity.  Waits for the lane.
int validate_points_dev(kzgb_ctx* c, Lane& L, const Affine* d_pts, size_t n) {
    CK(c, L.small.reserve(64 * sizeof(Fr)));
    uint32_t* d_err = (uint32_t*)((Fr*)L.small.p + 32);
    CK(c, cudaMemsetAsync(d_err, 0xff, 32, L.st));
    g1_validate_launch(d_pts, (uint32_t)n, d_err, L.st);
    uint32_t herr = 0;
    CK(c, cudaMemcpyAsync(&herr, d_err, 4, cudaMemcpyDeviceToHost, L.st));
    CK(c, cudaStreamSynchronize(L.st));
    if (herr != 0xffffffffu) return fail(c, KZGB_ERR_NOT_ON_CURVE, "G1 point not on curve");
    return KZGB_OK;
}

// Streamed ingest of `n` compressed points: `read(dst, first, count)` fills a pinned staging buffer with
// points [first, first+count); the read of chunk k+1 overlaps the H2D copy and the decompression kernel of
// chunk k (two staging buffers).  The reference does one 32-byte read + one channel send per point
// (srs.rs:154-188) and a sqrt per point on CPU threads ("a few minutes" for the 2^28-point mainnet SRS).
// raw = true: the source already holds 64-byte affine Montgomery points (the table cache); they are only
// checked to be on the curve.
template <class Reader>
int srs_ingest_stream(kzgb_ctx* c, size_t n, bool raw, Reader read) {
    if (n == 0 || n > ((size_t)1 << 28)) return fail(c, KZGB_ERR_GENERIC, "invalid number of SRS points");
    Lane& L = c->lanes[0];
    const size_t unit = raw ? sizeof(Affine) : 32;
    size_t chunk = (size_t)g_srs_chunk.load();
    if (chunk == 0) chunk = (size_t)1 << 22;
    chunk = std::min(chunk, n);
    uint8_t* pin[2] = {nullptr, nullptr};
    cudaEvent_t ev[2] = {nullptr, nullptr};
    DevBuf stage[2], errb;
    Affine* pts = nullptr;
    int rc = KZGB_OK;
    bool pinned = true;
    auto cleanup = [&]() {
        for (int k = 0; k < 2; k++) {
            if (pin[k]) { if (pinned) cudaFreeHost(pin[k]); else free(pin[k]); }
            if (ev[k]) cudaEventDestroy(ev[k]);
            stage[k].release();
        }
        errb.release();
    };
    auto ck = [&](cudaError_t e, const char* what) {
        if (!rc && e != cudaSuccess) rc = fail(c, KZGB_ERR_DEVICE, std::string("CUDA error: ") + cudaGetErrorString(e) + " at " + what);
    };
    const size_t n_chunks = (n + chunk - 1) / chunk;
    pinned = n_chunks > 1;  // a single chunk has nothing to overlap with: skip the (slow) pinned allocation
    ck(cudaMalloc((void**)&pts, n * sizeof(Affine)), "cudaMalloc(SRS points)");
    ck(errb.reserve(4 * n_chunks), "cudaMalloc");
    for (int k = 0; k < (pinned ? 2 : 1) && !rc; k++) {
        if (pinned) ck(cudaMallocHost((void**)&pin[k], chunk * unit), "cudaMallocHost(staging)");
        else if (!(pin[k] = (uint8_t*)malloc(chunk * unit))) rc = fail(c, KZGB_ERR_GENERIC, "out of host memory");
        ck(cudaEventCreateWithFlags(&ev[k], cudaEventDisableTiming), "cudaEventCreate");
        if (!raw) ck(stage[k].reserve(chunk * unit), "cudaMalloc(staging)");
    }
    std::vector<uint32_t> herr(n_chunks, 0xffffffffu);
    uint32_t* d_err = (uint32_t*)errb.p;  // one slot per chunk
    if (!rc) ck(cudaMemsetAsync(d_err, 0xff, 4 * n_chunks, L.st), "memset");
    for (size_t k = 0; k < n_chunks && !rc; k++) {
        const size_t first = k * chunk, count = std::min(chunk, n - first);
        const int b = (int)(k & 1);
        if (k >= 2) ck(cudaEventSynchronize(ev[b]), "cudaEventSynchronize");  // staging buffer free again
        if (rc) break;
        if (!read(pin[b], first, count)) { rc = fail(c, KZGB_ERR_GENERIC, "Failed to read G1 points: file shorter than points_to_load"); break; }
        if (raw) {
            ck(cudaMemcpyAsync(pts + first, pin[b], count * unit, cudaMemcpyHostToDevice, L.st), "H2D copy of SRS points");
            g1_validate_launch(pts + first, (uint32_t)count, d_err + k, L.st);
        } else {
            ck(cudaMemcpyAsync(stage[b].p, pin[b], count * unit, cudaMemcpyHostToDevice, L.st), "H2D copy of SRS points");
            srs_decompress_launch((const uint8_t*)stage[b].p, (uint32_t)count, pts + first, d_err + k, L.st);
        }
        ck(cudaEventRecord(ev[b], L.st), "cudaEventRecord");
    }
    if (!rc) ck(cudaMemcpyAsync(herr.data(), d_err, 4 * n_chunks, cudaMemcpyDeviceToHost, L.st), "D2H");
    ck(cudaStreamSynchronize(L.st), "sync");
    if (!rc) ck(cudaGetLastError(), "SRS ingest kernels");
    for (size_t k = 0; k < n_chunks && !rc; k++) {
        if (herr[k] == 0xffffffffu) continue;
        char msg[128];
        if (raw) {
            snprintf(msg, sizeof msg, "G1 point not on curve (cached point %zu)", k * chunk + herr[k] - 1);
            rc = fail(c, KZGB_ERR_NOT_ON_CURVE, msg);
        } else if ((herr[k] & 3u) == 2u) {
            snprintf(msg, sizeof msg, "point at infinity not coded properly for g1 (point %zu)", k * chunk + (herr[k] >> 2) - 1);
            rc = fail(c, KZGB_ERR_DESERIALIZATION, msg);
        } else {
            snprintf(msg, sizeof msg, "compressed g1 point not on curve (point %zu)", k * chunk + (herr[k] >> 2) - 1);
            rc = fail(c, KZGB_ERR_NOT_ON_CURVE, msg);
        }
    }
    cleanup();
    if (rc) { if (pts) cudaFree(pts); return rc; }
    return srs_install(c, pts, n);
}

}  // namespace

// =====================================================================================
extern "C" {

int kzgb_ctx_create(kzgb_ctx** out, int device, void* stream) {
    if (!out) return KZGB_ERR_GENERIC;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return KZGB_ERR_DEVICE;
    kzgb_ctx* c = new kzgb_ctx();
    c->device = device;
    int prev = 0;
    cudaGetDevice(&prev);
    if (cudaSetDevice(device) != cudaSuccess) { delete c; return KZGB_ERR_DEVICE; }
    int rc = lane_init(c, c->lanes[0], (cudaStream_t)stream);
    if (rc == KZGB_OK && !stream && g_l2_fetch_64.load()) { l2_limit_acquire(device); c->set_l2_limit = true; }
    if (rc == KZGB_OK) {
        c->n_lanes = 1;
        if (cudaEventCreate(&c->t0) != cudaSuccess || cudaEventCreate(&c->t1) != cudaSuccess) rc = KZGB_ERR_DEVICE;
    }
    cudaSetDevice(prev);
    if (rc) { delete c; return rc; }
    *out = c;
    return KZGB_OK;
}

void kzgb_ctx_destroy(kzgb_ctx* c) {
    if (!c) return;
    int prev = 0;
    cudaGetDevice(&prev);
    cudaSetDevice(c->device);
    for (int i = 0; i < c->n_lanes; i++) { cudaStreamSynchronize(c->lanes[i].st); lane_destroy(c->lanes[i]); }
    if (c->srs) cudaFree(c->srs);
    drop_window_table(c);
    lagrange_release(c);
    if (c->tw) cudaFree(c->tw);
    c->batch_bytes.release();
    if (c->t0) cudaEventDestroy(c->t0);
    if (c->t1) cudaEventDestroy(c->t1);
    if (c->copy_st) cudaStreamDestroy(c->copy_st);
    if (c->hash_st) cudaStreamDestroy(c->hash_st);
    if (c->ev_hash_uploaded) cudaEventDestroy(c->ev_hash_uploaded);
    if (c->fsl_host) cudaFreeHost(c->fsl_host);
    c->fsl_args.release();
    for (int k = 0; k < 2; k++) { if (c->ev_copied[k]) cudaEventDestroy(c->ev_copied[k]); if (c->ev_consumed[k]) cudaEventDestroy(c->ev_consumed[k]); }
    if (c->trace_base) cudaEventDestroy(c->trace_base);
    for (auto& r : c->trace) if (r.ev) cudaEventDestroy(r.ev);
    if (c->set_l2_limit) l2_limit_release(c->device);
    cudaSetDevice(prev);
    delete c;
}

const char* kzgb_last_error(const kzgb_ctx* c) { return c ? c->err.c_str() : "null context"; }

int kzgb_sync(kzgb_ctx* c) {
    Guard g(c);
    CK(c, drain_lanes(c));
    return KZGB_OK;
}

uint64_t kzgb_launch_count(const kzgb_ctx*) { return g_launch_count.load(); }

// ------------------------------------------------------------------------------- SRS
int kzgb_srs_load_gnark_be(kzgb_ctx* c, const uint8_t* bytes, size_t n) {
    Guard g(c);
    return srs_ingest_stream(c, n, false, [&](uint8_t* dst, size_t first, size_t count) {
        memcpy(dst, bytes + first * 32, count * 32);
        return true;
    });
}

int kzgb_srs_load_file(kzgb_ctx* c, const char* path, uint32_t order, uint32_t points_to_load) {
    if (points_to_load > order) return fail(c, KZGB_ERR_GENERIC, "Number of points to load exceeds SRS order.");  // srs.rs:36-40
    FILE* f = fopen(path, "rb");
    if (!f) return fail(c, KZGB_ERR_GENERIC, std::string("Failed to read G1 points: cannot open ") + path);
    Guard g(c);
    // bulk sequential reads of whole chunks instead of one 32-byte read per point (srs.rs:173)
    int rc = srs_ingest_stream(c, points_to_load, false, [&](uint8_t* dst, size_t, size_t count) {
        return fread(dst, 32, count, f) == count;
    });
    fclose(f);
    return rc;
}

// ---- on-disk cache of the decompressed points ---------------------------------------------------
// Header (64 bytes): "KZGBSRS1", u64 point count, zero padding; then count x 64 bytes x || y Montgomery
// (identity = all zero).  Loading it skips the per-point square root; every point is still checked to be
// on the curve on the GPU, so a damaged cache fails instead of giving wrong commitments.
static const char SRS_CACHE_MAGIC[8] = {'K', 'Z', 'G', 'B', 'S', 'R', 'S', '1'};

int kzgb_srs_save_cache(kzgb_ctx* c, const char* path) {
    Guard g(c);
    if (!c->srs_n) return fail(c, KZGB_ERR_GENERIC, "no SRS loaded");
    FILE* f = fopen(path, "wb");
    if (!f) return fail(c, KZGB_ERR_GENERIC, std::string("cannot create ") + path);
    uint8_t hdr[64] = {0};
    memcpy(hdr, SRS_CACHE_MAGIC, 8);
    uint64_t n64 = c->srs_n;
    memcpy(hdr + 8, &n64, 8);
    bool ok = fwrite(hdr, 1, 64, f) == 64;
    const size_t chunk = (size_t)1 << 20;
    std::vector<Affine> buf(std::min(chunk, c->srs_n));
    for (size_t first = 0; first < c->srs_n && ok; first += chunk) {
        size_t count = std::min(chunk, c->srs_n - first);
        cudaError_t e = cudaMemcpy(buf.data(), c->srs + first, count * sizeof(Affine), cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) { fclose(f); remove(path); CK(c, e); }
        ok = fwrite(buf.data(), sizeof(Affine), count, f) == count;
    }
    ok = (fclose(f) == 0) && ok;
    if (!ok) { remove(path); return fail(c, KZGB_ERR_GENERIC, std::string("short write to ") + path); }
    return KZGB_OK;
}

int kzgb_srs_load_cache(kzgb_ctx* c, const char* path, uint32_t points_to_load) {
    FILE* f = fopen(path, "rb");
    if (!f) return fail(c, KZGB_ERR_GENERIC, std::string("Failed to read G1 points: cannot open ") + path);
    uint8_t hdr[64];
    uint64_t n64 = 0;
    if (fread(hdr, 1, 64, f) != 64 || memcmp(hdr, SRS_CACHE_MAGIC, 8) != 0) {
        fclose(f);
        return fail(c, KZGB_ERR_DESERIALIZATION, "not an SRS point cache (bad header)");
    }
    memcpy(&n64, hdr + 8, 8);
    if (points_to_load == 0) points_to_load = (uint32_t)std::min<uint64_t>(n64, 0xffffffffu);
    if (points_to_load > n64) {
        fclose(f);
        return fail(c, KZGB_ERR_GENERIC, "Number of points to load exceeds SRS order.");
    }
    Guard g(c);
    int rc = srs_ingest_stream(c, points_to_load, true, [&](uint8_t* dst, size_t, size_t count) {
        return fread(dst, sizeof(Affine), count, f) == count;
    });
    fclose(f);
    return rc;
}

int kzgb_srs_load_affine_mont(kzgb_ctx* c, const uint64_t* xy, const uint8_t* inf, size_t n) {
    Guard g(c);
    if (n == 0) return fail(c, KZGB_ERR_GENERIC, "empty SRS");
    std::vector<Affine> host(n);
    memcpy(host.data(), xy, n * sizeof(Affine));
    if (inf) for (size_t i = 0; i < n; i++) if (inf[i]) aff_set_inf(host[i]);
    Affine* pts = nullptr;
    CK(c, cudaMalloc((void**)&pts, n * sizeof(Affine)));
    cudaError_t e = cudaMemcpy(pts, host.data(), n * sizeof(Affine), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { cudaFree(pts); CK(c, e); }
    return srs_install(c, pts, n);
}

// dst gets a copy of src's SRS points, device to device (peer copy over NVLink when the contexts sit on different
// GPUs): how a kzgb_group replicates an SRS that was decompressed once.
int kzgb_srs_clone(kzgb_ctx* dst, kzgb_ctx* src) {
    if (!dst || !src || dst == src) return KZGB_ERR_GENERIC;
    size_t n = 0;
    const Affine* from = nullptr;
    int src_dev = 0;
    {
        Guard gs(src);
        CK(src, drain_lanes(src));
        n = src->srs_n; from = src->srs; src_dev = src->device;
    }
    Guard g(dst);
    if (n == 0) return fail(dst, KZGB_ERR_GENERIC, "no SRS loaded in the source context");
    Affine* pts = nullptr;
    CK(dst, cudaMalloc((void**)&pts, n * sizeof(Affine)));
    cudaError_t e = (src_dev == dst->device) ? cudaMemcpy(pts, from, n * sizeof(Affine), cudaMemcpyDeviceToDevice)
                                              : cudaMemcpyPeer(pts, dst->device, from, src_dev, n * sizeof(Affine));
    if (e != cudaSuccess) { cudaFree(pts); CK(dst, e); }
    return srs_install(dst, pts, n);
}

int kzgb_srs_load_synthetic_range(kzgb_ctx* c, const uint64_t tau_mont[4], size_t first, size_t n);
int kzgb_srs_load_synthetic(kzgb_ctx* c, const uint64_t tau_mont[4], size_t n) {
    return kzgb_srs_load_synthetic_range(c, tau_mont, 0, n);
}
int kzgb_srs_load_synthetic_range(kzgb_ctx* c, const uint64_t tau_mont[4], size_t first, size_t n) {
    Guard g(c);
    if (n == 0 || n > ((size_t)1 << 28)) return fail(c, KZGB_ERR_GENERIC, "invalid number of SRS points");
    Affine* pts = nullptr;
    CK(c, cudaMalloc((void**)&pts, n * sizeof(Affine)));
    Fr tau;
    memcpy(tau.l, tau_mont, 32);
    srs_synthetic_launch(pts, (uint32_t)n, &tau, (uint32_t)first, c->lanes[0].st);
    cudaError_t e = cudaStreamSynchronize(c->lanes[0].st);
    if (e != cudaSuccess) { cudaFree(pts); CK(c, e); }
    return srs_install(c, pts, n);
}

size_t kzgb_srs_len(const kzgb_ctx* c) { return c ? c->srs_n : 0; }

int kzgb_srs_get_affine_mont(kzgb_ctx* c, size_t start, size_t count, uint64_t* out_xy, uint8_t* out_inf) {
    Guard g(c);
    if (start > c->srs_n || count > c->srs_n - start) return fail(c, KZGB_ERR_GENERIC, "SRS range out of bounds");
    CK(c, cudaMemcpy(out_xy, c->srs + start, count * sizeof(Affine), cudaMemcpyDeviceToHost));
    if (out_inf) {
        const Affine* a = (const Affine*)out_xy;
        for (size_t i = 0; i < count; i++) out_inf[i] = aff_is_inf(a[i]) ? 1 : 0;
    }
    return KZGB_OK;
}

int kzgb_srs_precompute(kzgb_ctx* c, size_t max_n, int window_bits) {
    Guard g(c);
    if (window_bits < 0) {  // disable fixed-base tables (variable-base mode over the monomial points)
        c->auto_precompute = false;
        drain_lanes(c);
        drop_window_table(c);
        lagrange_release(c);
        return KZGB_OK;
    }
    if (!c->srs_n) return fail(c, KZGB_ERR_GENERIC, "no SRS loaded");
    return do_precompute(c, 0, max_n ? max_n : c->srs_n, window_bits);
}

int kzgb_srs_precompute_range(kzgb_ctx* c, size_t first, size_t count, int window_bits) {
    Guard g(c);
    if (!c->srs_n) return fail(c, KZGB_ERR_GENERIC, "no SRS loaded");
    if (first > c->srs_n || count > c->srs_n - first) return fail(c, KZGB_ERR_GENERIC, "SRS range out of bounds");
    return do_precompute(c, first, count, window_bits < 0 ? 0 : window_bits);
}

int kzgb_srs_prepare_lagrange(kzgb_ctx* c, size_t n) {
    Guard g(c);
    if (n == 0 || (n & (n - 1))) return fail(c, KZGB_ERR_FFT, "length provided is not a power of 2");
    if (int rc = check_srs_capacity(c, n)) return rc;
    int logn = log2_exact(n);
    int rc = ensure_lagrange(c, logn, 1, true);
    if (rc) return rc;
    if (logn >= 1 && !c->lag[logn].table) return fail(c, KZGB_ERR_DEVICE, "Lagrange-basis table not built (disabled, above 2^22, or over the memory budget)");
    return KZGB_OK;
}

// ------------------------------------------------------------------------------- MSM
int kzgb_msm_srs_range(kzgb_ctx* c, const uint64_t* scalars, size_t first, size_t n, uint64_t out_xy[8], uint8_t* out_inf) {
    Guard g(c);
    Lane& L = c->lanes[0];
    if (first > c->srs_n || n > c->srs_n - first) return fail(c, KZGB_ERR_SERIALIZATION, "polynomial length is not correct");
    Affine r;
    if (n == 0) { aff_set_inf(r); affine_to_abi(r, out_xy, out_inf); return KZGB_OK; }
    bool done = false;
    int rc = msm_srs_host_pipelined(c, L, scalars, first, n, &r, &done);  // large MSMs over a window table: upload overlapped
    if (rc) return rc;
    if (!done) {
        CK(c, L.work.reserve(n * sizeof(Fr)));
        CK(c, cudaMemcpyAsync(L.work.p, scalars, n * sizeof(Fr), cudaMemcpyHostToDevice, L.st));
        rc = msm_blocking(c, L, (Fr*)L.work.p, false, first, n, nullptr, &r);
    }
    if (rc) return rc;
    affine_to_abi(r, out_xy, out_inf);
    return KZGB_OK;
}
int kzgb_msm_srs_range_dev(kzgb_ctx* c, const uint64_t* scalars_dev, size_t first, size_t n, uint64_t out_xy[8],
                           uint8_t* out_inf) {
    Guard g(c);
    Lane& L = c->lanes[0];
    if (first > c->srs_n || n > c->srs_n - first) return fail(c, KZGB_ERR_SERIALIZATION, "polynomial length is not correct");
    Affine r;
    int rc = msm_blocking(c, L, (const Fr*)scalars_dev, false, first, n, nullptr, &r);
    if (rc) return rc;
    affine_to_abi(r, out_xy, out_inf);
    return KZGB_OK;
}
int kzgb_fr_powers_dev(kzgb_ctx* c, const uint64_t base_mont[4], size_t first_exponent, size_t n, uint64_t* out_dev) {
    Guard g(c);
    if (n > 0xffffffffull || first_exponent > 0xffffffffull - n) return fail(c, KZGB_ERR_GENERIC, "kzgb_fr_powers_dev: exponent range exceeds 32 bits");
    Fr b;
    memcpy(b.l, base_mont, 32);
    fr_powers_launch((Fr*)out_dev, (uint32_t)n, &b, c->lanes[0].st, (uint32_t)first_exponent);
    CK(c, cudaStreamSynchronize(c->lanes[0].st));
    CK(c, cudaGetLastError());
    return KZGB_OK;
}
int kzgb_msm_srs(kzgb_ctx* c, const uint64_t* scalars, size_t n, uint64_t out_xy[8], uint8_t* out_inf) {
    return kzgb_msm_srs_range(c, scalars, 0, n, out_xy, out_inf);
}

int kzgb_msm_var(kzgb_ctx* c, const uint64_t* bases_xy, const uint8_t* bases_inf, const uint64_t* scalars, size_t m,
                 uint64_t out_xy[8], uint8_t* out_inf) {
    Guard g(c);
    Lane& L = c->lanes[0];
    Affine r;
    if (m == 0) { aff_set_inf(r); affine_to_abi(r, out_xy, out_inf); return KZGB_OK; }
    CK(c, L.work.reserve(m * sizeof(Fr)));
    CK(c, L.bases.reserve(m * sizeof(Affine)));
    if (bases_inf) {
        std::vector<Affine> tmp(m);
        memcpy(tmp.data(), bases_xy, m * sizeof(Affine));
        for (size_t i = 0; i < m; i++) if (bases_inf[i]) aff_set_inf(tmp[i]);
        CK(c, cudaMemcpy(L.bases.p, tmp.data(), m * sizeof(Affine), cudaMemcpyHostToDevice));
    } else {
        CK(c, cudaMemcpyAsync(L.bases.p, bases_xy, m * sizeof(Affine), cudaMemcpyHostToDevice, L.st));
    }
    CK(c, cudaMemcpyAsync(L.work.p, scalars, m * sizeof(Fr), cudaMemcpyHostToDevice, L.st));
    int rc = msm_blocking(c, L, (Fr*)L.work.p, false, 0, m, (const Affine*)L.bases.p, &r);
    if (rc) return rc;
    affine_to_abi(r, out_xy, out_inf);
    return KZGB_OK;
}

int kzgb_g1_add(const uint64_t a_xy[8], uint8_t a_inf, const uint64_t b_xy[8], uint8_t b_inf, uint64_t out_xy[8], uint8_t* out_inf) {
    Affine a = affine_from_abi(a_xy, a_inf), b = affine_from_abi(b_xy, b_inf), r;
    XYZZ acc;
    xyzz_from_affine(acc, a);
    xyzz_madd(acc, b);
    xyzz_to_affine(r, acc);
    affine_to_abi(r, out_xy, out_inf);
    return KZGB_OK;
}

// ------------------------------------------------------------------------------- roots of unity
// helpers::calculate_roots_of_unity (primitives/src/helpers.rs:553-589; expand_root_of_unity :592-610): w^0 .. w^(n-1) for
// n = next_pow2(ceil(len / 32)), w = PRIMITIVE_ROOTS_OF_UNITY[log2 n] (consts.rs:22-52).  The reference builds them with n serial
// multiplications (and again inside every evaluation, helpers.rs:482); here one kernel, each power by square-and-multiply.
int kzgb_roots_of_unity(kzgb_ctx* c, uint64_t length_of_data_after_padding, uint64_t* out, size_t out_capacity, size_t* n_out) {
    if (length_of_data_after_padding == 0) return fail(c, KZGB_ERR_GENERIC, "Length of data after padding is 0");
    uint64_t nelem = (length_of_data_after_padding + 31) / 32;
    if (nelem > ((uint64_t)1 << 28))
        return fail(c, KZGB_ERR_GENERIC, "the length of data after padding is not valid with respect to the SRS");
    size_t n = next_pow2((size_t)nelem);
    if (n_out) *n_out = n;
    if (!out) return KZGB_OK;  // size query
    if (out_capacity < n) return fail(c, KZGB_ERR_GENERIC, "output buffer too small for the roots of unity");
    Guard g(c);
    Lane& L = c->lanes[0];
    CK(c, L.work.reserve(n * sizeof(Fr)));
    Fr w = root_of_unity_mont(log2_exact(n));
    fr_powers_launch((Fr*)L.work.p, (uint32_t)n, &w, L.st);
    CK(c, cudaMemcpyAsync(out, L.work.p, n * sizeof(Fr), cudaMemcpyDeviceToHost, L.st));
    CK(c, cudaStreamSynchronize(L.st));
    CK(c, cudaGetLastError());
    return KZGB_OK;
}

// ------------------------------------------------------------------------------- NTT / codecs
int kzgb_ntt_fr(kzgb_ctx* c, uint64_t* inout, size_t n, int inverse) {
    Guard g(c);
    if (n == 0 || (n & (n - 1))) return fail(c, KZGB_ERR_FFT, "length provided is not a power of 2");
    if (n > ((size_t)1 << 28)) return fail(c, KZGB_ERR_GENERIC, "Input size exceeds maximum polynomial size");
    Lane& L = c->lanes[0];
    int logn = log2_exact(n);
    int rc = ensure_twiddles(c, logn);
    if (rc) return rc;
    CK(c, L.work.reserve(n * sizeof(Fr)));
    CK(c, L.ntt_scratch.reserve(n * sizeof(Fr)));
    CK(c, cudaMemcpyAsync(L.work.p, inout, n * sizeof(Fr), cudaMemcpyHostToDevice, L.st));
    Fr ninv = ninv_mont(logn);
    ntt_launch((Fr*)L.work.p, logn, 1, inverse != 0, c->tw, c->logN, &ninv, (Fr*)L.ntt_scratch.p, L.st);
    CK(c, cudaMemcpyAsync(inout, L.work.p, n * sizeof(Fr), cudaMemcpyDeviceToHost, L.st));
    CK(c, cudaStreamSynchronize(L.st));
    CK(c, cudaGetLastError());
    return KZGB_OK;
}

int kzgb_to_fr_array(kzgb_ctx* c, const uint8_t* bytes, size_t len, uint64_t* out) {
    Guard g(c);
    Lane& L = c->lanes[0];
    size_t n = (len + 31) / 32;
    if (!n) return KZGB_OK;
    int rc = blob_to_evals(c, L, bytes, nullptr, len, n);
    if (rc) return rc;
    CK(c, cudaMemcpyAsync(out, L.evals.p, n * sizeof(Fr), cudaMemcpyDeviceToHost, L.st));
    CK(c, cudaStreamSynchronize(L.st));
    CK(c, cudaGetLastError());
    return KZGB_OK;
}

int kzgb_to_byte_array(kzgb_ctx* c, const uint64_t* fr, size_t n, uint8_t* out) {
    Guard g(c);
    Lane& L = c->lanes[0];
    if (!n) return KZGB_OK;
    CK(c, L.evals.reserve(n * sizeof(Fr)));
    CK(c, L.bytes.reserve(n * 32));
    CK(c, cudaMemcpyAsync(L.evals.p, fr, n * sizeof(Fr), cudaMemcpyHostToDevice, L.st));
    fr_to_bytes_launch((Fr*)L.evals.p, (uint8_t*)L.bytes.p, (uint32_t)n, L.st);
    CK(c, cudaMemcpyAsync(out, L.bytes.p, n * 32, cudaMemcpyDeviceToHost, L.st));
    CK(c, cudaStreamSynchronize(L.st));
    CK(c, cudaGetLastError());
    return KZGB_OK;
}

// ------------------------------------------------------------------------------- commitments
static int commit_evals_host(kzgb_ctx* c, const uint64_t* evals, size_t n, uint64_t out_xy[8], uint8_t* out_inf) {
    Lane& L = c->lanes[0];
    CK(c, L.work.reserve(n * sizeof(Fr)));
    CK(c, cudaMemcpyAsync(L.work.p, evals, n * sizeof(Fr), cudaMemcpyHostToDevice, L.st));
    MsmJob job;
    int rc = commit_evals_enqueue(c, L, (Fr*)L.work.p, n, &job);
    if (rc) return rc;
    Affine r;
    rc = msm_finish(c, L, job, &r);
    if (rc) return rc;
    affine_to_abi(r, out_xy, out_inf);
    return KZGB_OK;
}

int kzgb_commit_eval(kzgb_ctx* c, const uint64_t* evals, size_t n, uint64_t out_xy[8], uint8_t* out_inf) {
    Guard g(c);
    if (int rc = check_srs_capacity(c, n)) return rc;  // kzg.rs:89-94
    if (n == 0 || (n & (n - 1))) return fail(c, KZGB_ERR_FFT, "length provided is not a power of 2");  // kzg.rs:265-269
    int rc = ensure_lagrange(c, log2_exact(n));
    if (rc) return rc;
    return commit_evals_host(c, evals, n, out_xy, out_inf);
}

int kzgb_commit_coeff(kzgb_ctx* c, const uint64_t* coeffs, size_t n, uint64_t out_xy[8], uint8_t* out_inf) {
    if (n > kzgb_srs_len(c)) return fail(c, KZGB_ERR_SERIALIZATION, "polynomial length is not correct");  // kzg.rs:112-116
    return kzgb_msm_srs_range(c, coeffs, 0, n, out_xy, out_inf);
}

int kzgb_commit_blob(kzgb_ctx* c, const uint8_t* blob, size_t len, uint64_t out_xy[8], uint8_t* out_inf) {
    Guard g(c);
    Lane& L = c->lanes[0];
    size_t n = blob_poly_len(len);
    if (int rc = check_commit_blob_len(c, n)) return rc;
    int rc = ensure_lagrange(c, log2_exact(n));
    if (rc) return rc;
    rc = blob_to_evals(c, L, blob, nullptr, len, n);
    if (rc) return rc;
    MsmJob job;
    rc = commit_evals_enqueue(c, L, (Fr*)L.evals.p, n, &job);
    if (rc) return rc;
    Affine r;
    rc = msm_finish(c, L, job, &r);
    if (rc) return rc;
    affine_to_abi(r, out_xy, out_inf);
    return KZGB_OK;
}

// KZG::g1_ifft (kzg.rs:263-285): the Lagrange-basis SRS, a G1-point inverse NTT on the GPU (g1ntt.cu).
// The same transform builds the resident Lagrange window tables (ensure_lagrange); this entry point returns
// the points themselves to the caller.
int kzgb_g1_ifft(kzgb_ctx* c, size_t n, uint64_t* out_xy, uint8_t* out_inf) {
    if (n == 0 || (n & (n - 1))) return fail(c, KZGB_ERR_FFT, "length provided is not a power of 2");
    Guard g(c);
    Lane& L = c->lanes[0];
    if (int rc = check_srs_capacity(c, n)) return rc;
    if (n > ((size_t)1 << 28)) return fail(c, KZGB_ERR_GENERIC, "power must be <= 28");
    int logn = log2_exact(n);
    int rc = ensure_twiddles(c, logn);
    if (rc) return rc;
    CK(c, L.work.reserve(n * sizeof(XYZZ)));
    CK(c, L.bases.reserve(n * sizeof(Affine)));
    Fr ninv = ninv_mont(logn), ninv_canon;
    fe_from_mont(ninv_canon, ninv);
    g1_intt_launch(c->srs, logn, (XYZZ*)L.work.p, (Affine*)L.bases.p, c->tw, c->logN, &ninv_canon, L.st);
    std::vector<Affine> host(n);
    CK(c, cudaMemcpyAsync(host.data(), L.bases.p, n * sizeof(Affine), cudaMemcpyDeviceToHost, L.st));
    CK(c, cudaStreamSynchronize(L.st));
    CK(c, cudaGetLastError());
    for (size_t i = 0; i < n; i++) affine_to_abi(host[i], out_xy + 8 * i, out_inf ? out_inf + i : nullptr);
    return KZGB_OK;
}

// ------------------------------------------------------------------------------- proofs
int kzgb_compute_proof(kzgb_ctx* c, const uint64_t* evals, size_t n, const uint64_t z_mont[4], uint64_t out_xy[8],
                       uint8_t* out_inf, uint64_t y_out[4]) {
    Guard g(c);
    Lane& L = c->lanes[0];
    if (n == 0 || (n & (n - 1))) return fail(c, KZGB_ERR_FFT, "length provided is not a power of 2");
    if (int rc = check_srs_capacity(c, n)) return rc;
    int rc = ensure_lagrange(c, log2_exact(n));
    if (rc) return rc;
    CK(c, L.evals.reserve(n * sizeof(Fr)));
    CK(c, cudaMemcpyAsync(L.evals.p, evals, n * sizeof(Fr), cudaMemcpyHostToDevice, L.st));
    Fr z;
    memcpy(z.l, z_mont, 32);
    MsmJob job;
    rc = proof_enqueue(c, L, (Fr*)L.evals.p, n, z, &job);
    if (rc) return rc;
    if (y_out) CK(c, cudaMemcpyAsync(&L.h_fr[3], (Fr*)L.small.p + 2, sizeof(Fr), cudaMemcpyDeviceToHost, L.st));
    Affine r;
    rc = msm_finish(c, L, job, &r);
    if (rc) return rc;
    if (y_out) memcpy(y_out, &L.h_fr[3], 32);
    affine_to_abi(r, out_xy, out_inf);
    return KZGB_OK;
}

int kzgb_evaluate_polynomial(kzgb_ctx* c, const uint64_t* evals, size_t n, const uint64_t z_mont[4], uint64_t y_out[4]) {
    Guard g(c);
    Lane& L = c->lanes[0];
    if (n == 0 || (n & (n - 1))) return fail(c, KZGB_ERR_INVALID_INPUT_LENGTH, "polynomial length must be a power of two");
    int rc = ensure_twiddles(c, log2_exact(n));
    if (rc) return rc;
    CK(c, L.evals.reserve(n * sizeof(Fr)));
    CK(c, cudaMemcpyAsync(L.evals.p, evals, n * sizeof(Fr), cudaMemcpyHostToDevice, L.st));
    Fr z, y;
    memcpy(z.l, z_mont, 32);
    rc = eval_enqueue(c, L, (Fr*)L.evals.p, n, z, nullptr);
    if (!rc) rc = eval_read_y(c, L, &y);
    if (rc) return rc;
    memcpy(y_out, y.l, 32);
    return KZGB_OK;
}

int kzgb_compute_challenge(kzgb_ctx* c, const uint8_t* blob, size_t len, const uint64_t c_xy[8], uint8_t c_inf,
                           uint64_t z_out[4]) {
    Affine C = affine_from_abi(c_xy, c_inf);
    if (!aff_on_curve(C)) return fail(c, KZGB_ERR_NOT_ON_CURVE, "G1 point not on curve");
    size_t n = blob_poly_len(len);
    Sha256 sh;
    challenge_midstate(sh, blob, len, n);
    Fr z = challenge_finish(sh, C);
    memcpy(z_out, z.l, 32);
    return KZGB_OK;
}

int kzgb_compute_blob_proof(kzgb_ctx* c, const uint8_t* blob, size_t len, const uint64_t c_xy[8], uint8_t c_inf,
                            uint64_t out_xy[8], uint8_t* out_inf) {
    Guard g(c);
    Lane& L = c->lanes[0];
    Affine C = affine_from_abi(c_xy, c_inf);
    if (!aff_on_curve(C)) return fail(c, KZGB_ERR_NOT_ON_CURVE, "G1 point not on curve");  // helpers.rs:694-699
    size_t n = blob_poly_len(len);
    if (len == 0) return fail(c, KZGB_ERR_GENERIC, "Length of data after padding is 0");  // helpers.rs:554-558 via :482
    if (int rc = check_srs_capacity(c, n)) return rc;
    int rc = ensure_lagrange(c, log2_exact(n));
    if (rc) return rc;
    rc = blob_to_evals(c, L, blob, nullptr, len, n);  // H2D + conversion run while the host hashes
    if (rc) return rc;
    Sha256 sh;
    challenge_midstate(sh, blob, len, n);
    Fr z = challenge_finish(sh, C);
    MsmJob job;
    rc = proof_enqueue(c, L, (Fr*)L.evals.p, n, z, &job);
    if (rc) return rc;
    Affine r;
    rc = msm_finish(c, L, job, &r);
    if (rc) return rc;
    affine_to_abi(r, out_xy, out_inf);
    return KZGB_OK;
}

// ------------------------------------------------------------------------------- single-proof verification, G1 side
// [k] G on the host (one 254-bit double-and-add on the 4x64 host field: ~0.1 ms, below the latency of any launch)
static void g1_generator_mul(XYZZ& out, const Fr& k_mont) {
    Fr k; fe_from_mont(k, k_mont);
    Affine G;
    fe_one(G.x); fe_dbl(G.y, G.x);
    XYZZ acc; xyzz_set_inf(acc);
    for (int i = 255; i >= 0; i--) {
        xyzz_dbl(acc, acc);
        if ((k.l[i >> 5] >> (i & 31)) & 1u) xyzz_madd(acc, G);
    }
    out = acc;
}
// verify_proof (verifier/src/verify.rs:10-75), everything that lives in G1: both points validated (:18-22), then
// commit_minus_value = C - [y] G1 (:37-42).  [tau - z] G2 and the pairing stay in the reference's code.
int kzgb_verify_proof_g1(kzgb_ctx* c, const uint64_t c_xy[8], uint8_t c_inf, const uint64_t proof_xy[8], uint8_t proof_inf,
                         const uint64_t y_mont[4], uint64_t out_xy[8], uint8_t* out_inf) {
    Affine C = affine_from_abi(c_xy, c_inf), P = affine_from_abi(proof_xy, proof_inf);
    if (!aff_on_curve(C) || !aff_on_curve(P)) return fail(c, KZGB_ERR_NOT_ON_CURVE, "G1 point not on curve");
    Fr y, ny;
    memcpy(y.l, y_mont, 32);
    fe_neg(ny, y);
    XYZZ acc;
    g1_generator_mul(acc, ny);  // -[y] G
    xyzz_madd(acc, C);
    Affine r;
    xyzz_to_affine(r, acc);
    affine_to_abi(r, out_xy, out_inf);
    return KZGB_OK;
}
// verify_blob_kzg_proof (verifier/src/verify.rs:77-115) up to the pairing: validation, z = compute_challenge(blob, C) on the
// host SHA-256 while the blob is uploaded and converted, y = p(z) on the GPU (no quotient), then kzgb_verify_proof_g1.
int kzgb_verify_blob_proof_g1(kzgb_ctx* c, const uint8_t* blob, size_t len, const uint64_t c_xy[8], uint8_t c_inf,
                              const uint64_t proof_xy[8], uint8_t proof_inf, uint64_t out_xy[8], uint8_t* out_inf,
                              uint64_t z_out[4], uint64_t y_out[4]) {
    Affine C = affine_from_abi(c_xy, c_inf), P = affine_from_abi(proof_xy, proof_inf);
    if (!aff_on_curve(C) || !aff_on_curve(P)) return fail(c, KZGB_ERR_NOT_ON_CURVE, "G1 point not on curve");
    if (len == 0) return fail(c, KZGB_ERR_GENERIC, "Length of data after padding is 0");  // helpers.rs:554-558 via :482
    const size_t n = blob_poly_len(len);
    if (n > ((size_t)1 << 28)) return fail(c, KZGB_ERR_GENERIC, "Input size exceeds maximum polynomial size");
    Fr y;
    {
        Guard g(c);
        Lane& L = c->lanes[0];
        int rc = ensure_twiddles(c, log2_exact(n));
        if (rc) return rc;
        rc = blob_to_evals(c, L, blob, nullptr, len, n);
        if (rc) return rc;
        Sha256 sh;
        challenge_midstate(sh, blob, len, n);
        const Fr z = challenge_finish(sh, C);
        rc = eval_enqueue(c, L, (Fr*)L.evals.p, n, z, nullptr);
        if (!rc) rc = eval_read_y(c, L, &y);
        if (rc) return rc;
        if (z_out) memcpy(z_out, z.l, 32);
        if (y_out) memcpy(y_out, y.l, 32);
    }
    return kzgb_verify_proof_g1(c, c_xy, c_inf, proof_xy, proof_inf, (const uint64_t*)y.l, out_xy, out_inf);
}


// ------------------------------------------------------------------------------- codecs / validation
int kzgb_g1_serialize_compressed(const uint64_t xy[8], uint8_t inf, uint8_t out32[32]) {
    serialize_compressed(affine_from_abi(xy, inf), out32);
    return KZGB_OK;
}
int kzgb_g1_to_gnark_be(const uint64_t xy[8], uint8_t inf, uint8_t out32[32]) {
    to_gnark_be(affine_from_abi(xy, inf), out32);
    return KZGB_OK;
}
int kzgb_validate_g1_points(kzgb_ctx* c, const uint64_t* xy, const uint8_t* inf, size_t n) {
    Guard g(c);
    Lane& L = c->lanes[0];
    if (!n) return KZGB_OK;
    std::vector<Affine> pts(n);
    for (size_t i = 0; i < n; i++) pts[i] = affine_from_abi(xy + 8 * i, inf ? inf[i] : 0);
    CK(c, L.bases.reserve(n * sizeof(Affine)));
    CK(c, cudaMemcpyAsync(L.bases.p, pts.data(), n * sizeof(Affine), cudaMemcpyHostToDevice, L.st));
    return validate_points_dev(c, L, (const Affine*)L.bases.p, n);
}

// ------------------------------------------------------------------------------- measurement hooks
int kzgb_microbench(kzgb_ctx* c, int kind, double* ops_per_second) {
    Guard g(c);
    Lane& L = c->lanes[0];
    const int blocks = 148 * 8, threads = 256;
    CK(c, L.work.reserve((size_t)blocks * threads * 4));
    const int iters = (kind == 3) ? 512 : 2048;
    double per_thread = (kind == 3) ? iters * 4.0 : (kind == 2 ? iters * 64.0 : iters * 128.0);
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
        CK(c, cudaEventRecord(c->t0, L.st));
        if (kind == 3) fqmul_peak_launch((uint32_t*)L.work.p, iters, blocks, threads, L.st);
        else imad_peak_launch((uint32_t*)L.work.p, iters, kind, blocks, threads, L.st);
        CK(c, cudaEventRecord(c->t1, L.st));
        CK(c, cudaEventSynchronize(c->t1));
        float ms = 0;
        CK(c, cudaEventElapsedTime(&ms, c->t0, c->t1));
        if (rep > 0 && ms < best) best = ms;
    }
    CK(c, cudaGetLastError());
    *ops_per_second = per_thread * blocks * threads / (best * 1e-3);
    return KZGB_OK;
}

int kzgb_bench_msm(kzgb_ctx* c, size_t n, int reps, double* ms_total, double* ms_accumulate) {
    Guard g(c);
    Lane& L = c->lanes[0];
    if (n == 0 || n > c->srs_n) return fail(c, KZGB_ERR_GENERIC, "bench size exceeds the SRS");
    CK(c, L.evals.reserve(n * sizeof(Fr)));
    // pseudo-random Montgomery scalars: powers of a fixed element
    Fr base = fr_from_u64(0x9e3779b97f4a7c15ull);
    fr_powers_launch((Fr*)L.evals.p, (uint32_t)n, &base, L.st);
    Affine r;
    int rc = msm_blocking(c, L, (Fr*)L.evals.p, false, 0, n, nullptr, &r);  // warm-up (+ lazy table build)
    if (rc) return rc;
    double acc0 = L.acc_ms;
    uint64_t l0 = L.acc_launches;
    CK(c, cudaEventRecord(c->t0, L.st));
    for (int i = 0; i < reps; i++) {
        rc = msm_blocking(c, L, (Fr*)L.evals.p, false, 0, n, nullptr, &r);
        if (rc) return rc;
    }
    CK(c, cudaEventRecord(c->t1, L.st));
    CK(c, cudaEventSynchronize(c->t1));
    float ms = 0;
    CK(c, cudaEventElapsedTime(&ms, c->t0, c->t1));
    *ms_total = ms / reps;
    uint64_t nl = L.acc_launches - l0;
    *ms_accumulate = nl ? (L.acc_ms - acc0) / nl : 0.0;
    return KZGB_OK;
}

int kzgb_bench_ntt(kzgb_ctx* c, int logn, size_t batch, int reps, double* ms_per_call) {
    Guard g(c);
    Lane& L = c->lanes[0];
    if (logn < 1 || logn > 28 || batch == 0 || reps < 1) return fail(c, KZGB_ERR_GENERIC, "bad NTT bench shape");
    int rc = ensure_twiddles(c, logn);
    if (rc) return rc;
    size_t total = batch << logn;
    CK(c, L.work.reserve(total * sizeof(Fr)));
    CK(c, L.ntt_scratch.reserve(total * sizeof(Fr)));
    Fr base = fr_from_u64(0x9e3779b97f4a7c15ull);
    fr_powers_launch((Fr*)L.work.p, (uint32_t)std::min<size_t>(total, 0xffffffffu), &base, L.st);
    Fr ninv = ninv_mont(logn);
    ntt_launch((Fr*)L.work.p, logn, (uint32_t)batch, true, c->tw, c->logN, &ninv, (Fr*)L.ntt_scratch.p, L.st);  // warm-up
    CK(c, cudaEventRecord(c->t0, L.st));
    for (int i = 0; i < reps; i++)
        ntt_launch((Fr*)L.work.p, logn, (uint32_t)batch, (i & 1) == 0, c->tw, c->logN, &ninv, (Fr*)L.ntt_scratch.p, L.st);
    CK(c, cudaEventRecord(c->t1, L.st));
    CK(c, cudaEventSynchronize(c->t1));
    CK(c, cudaGetLastError());
    float ms = 0;
    CK(c, cudaEventElapsedTime(&ms, c->t0, c->t1));
    *ms_per_call = ms / reps;
    return KZGB_OK;
}

// Device-side stopwatch over ALL lanes: everything queued between begin and end is inside [t0, t1].
int kzgb_timer_begin(kzgb_ctx* c) {
    Guard g(c);
    CK(c, cudaEventRecord(c->t0, c->lanes[0].st));
    for (int i = 1; i < c->n_lanes; i++) CK(c, cudaStreamWaitEvent(c->lanes[i].st, c->t0, 0));
    return KZGB_OK;
}
int kzgb_timer_end(kzgb_ctx* c, double* ms_out) {
    Guard g(c);
    for (int i = 1; i < c->n_lanes; i++) {
        CK(c, cudaEventRecord(c->lanes[i].ev_done, c->lanes[i].st));
        CK(c, cudaStreamWaitEvent(c->lanes[0].st, c->lanes[i].ev_done, 0));
    }
    CK(c, cudaEventRecord(c->t1, c->lanes[0].st));
    CK(c, cudaEventSynchronize(c->t1));
    float ms = 0;
    CK(c, cudaEventElapsedTime(&ms, c->t0, c->t1));
    *ms_out = ms;
    return KZGB_OK;
}
int kzgb_trace_begin(kzgb_ctx* c) {
    Guard g(c);
    CK(c, drain_lanes(c));
    for (auto& r : c->trace) if (r.ev) cudaEventDestroy(r.ev);
    c->trace.clear();
    if (!c->trace_base) CK(c, cudaEventCreate(&c->trace_base));
    CK(c, cudaEventRecord(c->trace_base, c->lanes[0].st));
    CK(c, cudaEventSynchronize(c->trace_base));
    c->trace_host0 = std::chrono::steady_clock::now();
    c->trace_on.store(true);
    return KZGB_OK;
}
// out: 4 doubles per record (lane, kind, device ms since begin or -1, host ms since begin or -1)
int kzgb_trace_end(kzgb_ctx* c, double* out, size_t capacity_records, size_t* n_records) {
    Guard g(c);
    c->trace_on.store(false);
    for (int i = 0; i < c->n_lanes; i++) {
        CK(c, cudaStreamSynchronize(c->lanes[i].st));
        if (c->lanes[i].st_acc) CK(c, cudaStreamSynchronize(c->lanes[i].st_acc));
    }
    size_t n = 0;
    for (auto& r : c->trace) {
        float ms = -1.f;
        if (r.ev && cudaEventElapsedTime(&ms, c->trace_base, r.ev) != cudaSuccess) { ms = -1.f; cudaGetLastError(); }
        if (out && n < capacity_records) { out[4 * n] = r.lane; out[4 * n + 1] = r.kind; out[4 * n + 2] = ms; out[4 * n + 3] = r.host_ms; }
        n++;
        if (r.ev) cudaEventDestroy(r.ev);
    }
    c->trace.clear();
    if (n_records) *n_records = n;
    return KZGB_OK;
}
int kzgb_stats(kzgb_ctx* c, double* acc_ms, uint64_t* acc_launches, uint64_t* acc_point_adds, int reset) {
    Guard g(c);
    double ms = 0; uint64_t nl = 0, na = 0;
    for (int i = 0; i < c->n_lanes; i++) {
        Lane& L = c->lanes[i];
        cudaStreamSynchronize(L.st);
        lane_collect_acc(L);
        ms += L.acc_ms; nl += L.acc_launches; na += L.acc_adds;
        if (reset) { L.acc_ms = 0; L.acc_launches = 0; L.acc_adds = 0; }
    }
    if (acc_ms) *acc_ms = ms;
    if (acc_launches) *acc_launches = nl;
    if (acc_point_adds) *acc_point_adds = na;
    return KZGB_OK;
}
int kzgb_set_option(const char* name, long value) {
    if (!name) return KZGB_ERR_GENERIC;
    if (!strcmp(name, "fs_device")) { g_fs_device.store((int)value); return KZGB_OK; }
    if (!strcmp(name, "srs_chunk_points")) { g_srs_chunk.store(value < 0 ? 0 : value); return KZGB_OK; }
    if (!strcmp(name, "fs_force_generic")) { fs_set_force_flag((int)value); return KZGB_OK; }
    if (!strcmp(name, "eval_structured")) { eval_set_structured((int)value); return KZGB_OK; }
    if (!strcmp(name, "group")) { g_group.store((int)value); return KZGB_OK; }
    if (!strcmp(name, "lanes")) { g_lanes.store(value < 0 ? 0 : (int)value); return KZGB_OK; }
    if (!strcmp(name, "hash_threads")) { g_hash_threads.store(value < 0 ? 0 : (int)value); return KZGB_OK; }
    if (!strcmp(name, "lane_wait")) { g_lane_wait.store(value < 0 ? -1 : (value > 2 ? 2 : (int)value)); return KZGB_OK; }
    if (!strcmp(name, "stream_priority")) { g_stream_priority.store(value != 0); return KZGB_OK; }
    if (!strcmp(name, "l2_fetch_64")) { g_l2_fetch_64.store(value != 0); return KZGB_OK; }
    if (!strcmp(name, "device_hash")) { g_device_hash.store(value < 0 ? -1 : (int)value); return KZGB_OK; }
    if (!strcmp(name, "pipelined_upload")) { g_pipelined_upload.store(value != 0); return KZGB_OK; }
    if (!strcmp(name, "batch_keep_mib")) { g_batch_keep_mib.store(value < 0 ? 0 : value); return KZGB_OK; }
    if (!strcmp(name, "ntt_kernel")) { ntt_set_kernel((int)value); return KZGB_OK; }
    if (!strcmp(name, "fs_quad")) { fs_set_quad((int)value); return KZGB_OK; }
    if (!strcmp(name, "device_hash_lanes")) { fs_set_midstate_lanes((int)value); return KZGB_OK; }
    if (!strcmp(name, "hash_trace")) { g_hash_trace.store(value != 0); return KZGB_OK; }
    if (!strcmp(name, "hash_nice")) { g_hash_nice.store(value != 0); return KZGB_OK; }
    if (!strcmp(name, "hash_mb")) { g_hash_mb.store(value < 0 ? -1 : (value ? 1 : 0)); return KZGB_OK; }
    if (!strcmp(name, "group_members")) { g_group_members.store(value < 1 ? 1 : (int)value); return KZGB_OK; }
    if (!strcmp(name, "lagrange")) { g_lagrange.store(value != 0); return KZGB_OK; }
    if (!strcmp(name, "lagrange_after")) { g_lagrange_after.store(value < 1 ? 1 : (int)value); return KZGB_OK; }
    if (!strcmp(name, "lagrange_budget_mib")) { g_lagrange_budget_mib.store(value < 0 ? 0 : value); return KZGB_OK; }
    if (!strcmp(name, "acc_waves")) { msm_set_acc_waves((int)value); return KZGB_OK; }
    if (!strcmp(name, "msm_debug_sync")) { msm_set_debug_sync((int)value); return KZGB_OK; }
    if (!strcmp(name, "acc_regs")) { msm_set_experiment((int)value, -1); return KZGB_OK; }
    if (!strcmp(name, "sort_block")) { msm_set_experiment(-1, (int)value); return KZGB_OK; }
    return KZGB_ERR_GENERIC;
}

int kzgb_msm_config(const kzgb_ctx* c, int* window_bits, int* windows, size_t* table_points) {
    if (window_bits) *window_bits = c->wt_c;
    if (windows) *windows = c->wt_W;
    if (table_points) *table_points = c->wt_n;
    return KZGB_OK;
}

}  // extern "C"
