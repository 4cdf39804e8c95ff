// kzgb_group: several GPUs of one box behind ONE handle (include/kzg_bn254_b200.h, "multi-GPU").
//
// The path shards two ways and needs no collective (SURVEY.md 8e):
//   * batches of blobs by blob    -- every member commits and proves its own contiguous share of the batch
//   * one very large MSM by point range -- member i owns SRS points [i n/G, (i+1) n/G), the G partial sums
//     (64 bytes each) are added on the host
// A group is a set of ordinary contexts, one per member, each driven by its own host thread for the duration of
// a call; the SRS is decompressed once and replicated device to device (peer copies over NVLink).  Everything here
// is written on the public C ABI, so a group behaves exactly like its members called one by one.
// The same device may appear more than once (independent contexts on one GPU): that is how the group paths are
// exercised on a single-GPU box.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/kzg_bn254_b200.h"

struct kzgb_group {
    std::vector<kzgb_ctx*> ctx;
    std::vector<int> dev;
    std::mutex mu;  // one group call at a time
    std::string err;
    // share of member i in the last kzgb_group_srs_precompute_ranges (points)
    size_t ranges_n = 0;
};

namespace {

int gfail(kzgb_group* g, int code, const std::string& msg) {
    if (g) g->err = msg;
    return code;
}

// run fn(i) for every member on its own host thread; first failure wins (its context's message is kept)
template <class F>
int for_members(kzgb_group* g, F fn) {
    const int G = (int)g->ctx.size();
    std::vector<int> rc(G, KZGB_OK);
    std::vector<std::thread> th;
    for (int i = 1; i < G; i++) th.emplace_back([&, i]() { rc[i] = fn(i); });
    rc[0] = fn(0);
    for (auto& t : th) t.join();
    for (int i = 0; i < G; i++)
        if (rc[i]) return gfail(g, rc[i], std::string("member ") + std::to_string(i) + " (device " + std::to_string(g->dev[i]) + "): " + kzgb_last_error(g->ctx[i]));
    return KZGB_OK;
}

// member i's share [first, first + count) of n items, boundaries on multiples of `align`
void share(size_t n, int G, int i, size_t align, size_t* first, size_t* count) {
    size_t per = (n + G - 1) / G;
    per = (per + align - 1) / align * align;
    size_t a = std::min(n, per * (size_t)i), b = std::min(n, per * (size_t)(i + 1));
    *first = a; *count = b - a;
}

// cut points of a blob batch: member i takes blobs [cut[i], cut[i+1]) with about 1/G of the bytes
std::vector<size_t> byte_balanced_cut(const size_t* lens, size_t count, int G) {
    size_t total = 0;
    for (size_t k = 0; k < count; k++) total += lens[k];
    std::vector<size_t> cut(G + 1, count);
    cut[0] = 0;
    size_t acc = 0, k = 0;
    for (int i = 1; i < G; i++) {
        const size_t target = (size_t)((__uint128_t)total * i / G);
        while (k < count && acc + lens[k] / 2 < target) acc += lens[k++];
        cut[i] = k;
    }
    return cut;
}

// fn(ctx, first, n) on every member whose byte-balanced share [first, first + n) of a blob batch is not empty.  The
// caller holds g->mu.
template <class F>
int for_blob_shares(kzgb_group* g, const size_t* lens, size_t count, F fn) {
    if (count == 0) return KZGB_OK;
    const std::vector<size_t> cut = byte_balanced_cut(lens, count, (int)g->ctx.size());
    return for_members(g, [&](int i) {
        const size_t a = cut[i], b = cut[i + 1];
        return a < b ? fn(g->ctx[i], a, b - a) : (int)KZGB_OK;
    });
}

// The weights of the cut of a batch of polynomials, 32 ns[i] bytes each, before any member has checked ns[i]: capped at
// 32 * 2^31, so that a length no SRS holds (which its member rejects) cannot wrap the product or the cut's sum.
std::vector<size_t> poly_bytes(const size_t* ns, size_t count) {
    std::vector<size_t> bytes(count);
    for (size_t i = 0; i < count; i++) bytes[i] = 32 * std::min<size_t>(ns[i], (size_t)1 << 31);
    return bytes;
}

// p + off, or nullptr for an optional array the caller left out
template <class T>
T* at_or_null(T* p, size_t off) { return p ? p + off : nullptr; }

int replicate_from_member0(kzgb_group* g) {
    return for_members(g, [&](int i) { return i == 0 ? KZGB_OK : kzgb_srs_clone(g->ctx[i], g->ctx[0]); });
}

}  // namespace

extern "C" {

int kzgb_group_create(kzgb_group** out, const int* devices, int n_devices) {
    if (!out) return KZGB_ERR_GENERIC;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return KZGB_ERR_DEVICE;
    std::vector<int> devs;
    if (!devices || n_devices <= 0) { for (int d = 0; d < count; d++) devs.push_back(d); }
    else devs.assign(devices, devices + n_devices);
    for (int d : devs) if (d < 0 || d >= count) return KZGB_ERR_DEVICE;
    kzgb_group* g = new kzgb_group();
    for (int d : devs) {
        kzgb_ctx* c = nullptr;
        int rc = kzgb_ctx_create(&c, d, nullptr);
        if (rc) { for (kzgb_ctx* x : g->ctx) kzgb_ctx_destroy(x); delete g; return rc; }
        g->ctx.push_back(c);
        g->dev.push_back(d);
    }
    // peer access between distinct member devices (ignored where unavailable: cudaMemcpyPeer then stages through the host)
    int prev = 0;
    cudaGetDevice(&prev);
    for (size_t a = 0; a < devs.size(); a++)
        for (size_t b = 0; b < devs.size(); b++) {
            if (devs[a] == devs[b]) continue;
            int can = 0;
            if (cudaDeviceCanAccessPeer(&can, devs[a], devs[b]) == cudaSuccess && can) {
                cudaSetDevice(devs[a]);
                cudaError_t e = cudaDeviceEnablePeerAccess(devs[b], 0);
                if (e != cudaSuccess) cudaGetLastError();  // already enabled
            }
        }
    cudaSetDevice(prev);
    kzgb_set_option("group_members", (long)devs.size());
    *out = g;
    return KZGB_OK;
}

void kzgb_group_destroy(kzgb_group* g) {
    if (!g) return;
    for (kzgb_ctx* c : g->ctx) kzgb_ctx_destroy(c);
    kzgb_set_option("group_members", 1);
    delete g;
}

int kzgb_group_size(const kzgb_group* g) { return g ? (int)g->ctx.size() : 0; }
kzgb_ctx* kzgb_group_ctx(kzgb_group* g, int member) { return (g && member >= 0 && member < (int)g->ctx.size()) ? g->ctx[member] : nullptr; }
const char* kzgb_group_last_error(const kzgb_group* g) { return g ? g->err.c_str() : "null group"; }

// ---- SRS: loaded (decompressed, validated) once on member 0, replicated device to device ---------------------
int kzgb_group_srs_load_file(kzgb_group* g, const char* path, uint32_t order, uint32_t points_to_load) {
    std::lock_guard<std::mutex> lk(g->mu);
    int rc = kzgb_srs_load_file(g->ctx[0], path, order, points_to_load);
    if (rc) return gfail(g, rc, kzgb_last_error(g->ctx[0]));
    return replicate_from_member0(g);
}
int kzgb_group_srs_load_cache(kzgb_group* g, const char* path, uint32_t points_to_load) {
    std::lock_guard<std::mutex> lk(g->mu);
    int rc = kzgb_srs_load_cache(g->ctx[0], path, points_to_load);
    if (rc) return gfail(g, rc, kzgb_last_error(g->ctx[0]));
    return replicate_from_member0(g);
}
int kzgb_group_srs_load_gnark_be(kzgb_group* g, const uint8_t* bytes, size_t n) {
    std::lock_guard<std::mutex> lk(g->mu);
    int rc = kzgb_srs_load_gnark_be(g->ctx[0], bytes, n);
    if (rc) return gfail(g, rc, kzgb_last_error(g->ctx[0]));
    return replicate_from_member0(g);
}
int kzgb_group_srs_load_affine_mont(kzgb_group* g, const uint64_t* xy, const uint8_t* inf, size_t n) {
    std::lock_guard<std::mutex> lk(g->mu);
    int rc = kzgb_srs_load_affine_mont(g->ctx[0], xy, inf, n);
    if (rc) return gfail(g, rc, kzgb_last_error(g->ctx[0]));
    return replicate_from_member0(g);
}
int kzgb_group_srs_load_synthetic(kzgb_group* g, const uint64_t tau_mont[4], size_t n) {
    std::lock_guard<std::mutex> lk(g->mu);
    int rc = kzgb_srs_load_synthetic(g->ctx[0], tau_mont, n);
    if (rc) return gfail(g, rc, kzgb_last_error(g->ctx[0]));
    return replicate_from_member0(g);
}

int kzgb_group_srs_prepare_lagrange(kzgb_group* g, size_t n) {
    std::lock_guard<std::mutex> lk(g->mu);
    return for_members(g, [&](int i) { return kzgb_srs_prepare_lagrange(g->ctx[i], n); });
}

// fixed-base window tables for the point-range shares of an n-point MSM: member i over its own share only
int kzgb_group_srs_precompute_ranges(kzgb_group* g, size_t n, int window_bits) {
    std::lock_guard<std::mutex> lk(g->mu);
    const int G = (int)g->ctx.size();
    int rc = for_members(g, [&](int i) {
        size_t first, count;
        share(n, G, i, 32, &first, &count);
        return count ? kzgb_srs_precompute_range(g->ctx[i], first, count, window_bits) : KZGB_OK;
    });
    if (!rc) g->ranges_n = n;
    return rc;
}

// ---- blob batches, sharded by blob ---------------------------------------------------------------------------
// KZG::commit_blob + KZG::compute_blob_proof (prover/src/kzg.rs:182-185,288-309) for `count` blobs: contiguous
// shares balanced by bytes, one host thread and one GPU per share, results written straight into the caller's arrays.
int kzgb_group_commit_and_prove_blobs(kzgb_group* g, const uint8_t* const* blobs, const size_t* lens, size_t count,
                                      uint8_t* commitments32, uint8_t* proofs32) {
    std::lock_guard<std::mutex> lk(g->mu);
    return for_blob_shares(g, lens, count, [&](kzgb_ctx* c, size_t a, size_t n) {
        return kzgb_commit_and_prove_blobs(c, blobs + a, lens + a, n, commitments32 + 32 * a, proofs32 + 32 * a);
    });
}

// KZG::commit_blob (prover/src/kzg.rs:182-185) for `count` blobs, cut as kzgb_group_commit_and_prove_blobs cuts them.
int kzgb_group_commit_blobs(kzgb_group* g, const uint8_t* const* blobs, const size_t* lens, size_t count,
                            uint64_t* out_xy, uint8_t* out_inf) {
    std::lock_guard<std::mutex> lk(g->mu);
    return for_blob_shares(g, lens, count, [&](kzgb_ctx* c, size_t a, size_t n) {
        return kzgb_commit_blobs(c, blobs + a, lens + a, n, out_xy + 8 * a, at_or_null(out_inf, a));
    });
}

// KZG::compute_blob_proof (prover/src/kzg.rs:288-309) for `count` blobs with the caller's commitments, cut as
// kzgb_group_commit_and_prove_blobs cuts them.
int kzgb_group_compute_blob_proofs(kzgb_group* g, const uint8_t* const* blobs, const size_t* lens, size_t count,
                                   const uint64_t* commitments_xy, const uint8_t* commitments_inf, uint64_t* out_xy,
                                   uint8_t* out_inf) {
    std::lock_guard<std::mutex> lk(g->mu);
    return for_blob_shares(g, lens, count, [&](kzgb_ctx* c, size_t a, size_t n) {
        return kzgb_compute_blob_proofs(c, blobs + a, lens + a, n, commitments_xy + 8 * a, at_or_null(commitments_inf, a),
                                        out_xy + 8 * a, at_or_null(out_inf, a));
    });
}

// KZG::compute_proof (prover/src/kzg.rs:128-178, 187-234) for `count` polynomials at the caller's points, cut as
// kzgb_group_commit_and_prove_blobs cuts a batch whose blob i has the 32 ns[i] bytes of polynomial i.
int kzgb_group_compute_proofs(kzgb_group* g, const uint64_t* const* evals_mont, const size_t* ns, size_t count,
                              const uint64_t* zs_mont, uint64_t* out_xy, uint8_t* out_inf, uint64_t* ys_mont) {
    std::lock_guard<std::mutex> lk(g->mu);
    const std::vector<size_t> bytes = poly_bytes(ns, count);
    return for_blob_shares(g, bytes.data(), count, [&](kzgb_ctx* c, size_t a, size_t n) {
        return kzgb_compute_proofs(c, evals_mont + a, ns + a, n, zs_mont + 4 * a, out_xy + 8 * a, at_or_null(out_inf, a),
                                   at_or_null(ys_mont, 4 * a));
    });
}

// KZG::commit_eval_form (prover/src/kzg.rs:84-104) for `count` polynomials, cut as kzgb_group_compute_proofs cuts them.
int kzgb_group_commit_evals(kzgb_group* g, const uint64_t* const* evals_mont, const size_t* ns, size_t count,
                            uint64_t* out_xy, uint8_t* out_inf) {
    std::lock_guard<std::mutex> lk(g->mu);
    const std::vector<size_t> bytes = poly_bytes(ns, count);
    return for_blob_shares(g, bytes.data(), count, [&](kzgb_ctx* c, size_t a, size_t n) {
        return kzgb_commit_evals(c, evals_mont + a, ns + a, n, out_xy + 8 * a, at_or_null(out_inf, a));
    });
}

// KZG::commit_coeff_form (prover/src/kzg.rs:107-125) for `count` polynomials, cut as kzgb_group_compute_proofs cuts them.
int kzgb_group_commit_coeffs(kzgb_group* g, const uint64_t* const* coeffs_mont, const size_t* ns, size_t count,
                             uint64_t* out_xy, uint8_t* out_inf) {
    std::lock_guard<std::mutex> lk(g->mu);
    const std::vector<size_t> bytes = poly_bytes(ns, count);
    return for_blob_shares(g, bytes.data(), count, [&](kzgb_ctx* c, size_t a, size_t n) {
        return kzgb_commit_coeffs(c, coeffs_mont + a, ns + a, n, out_xy + 8 * a, at_or_null(out_inf, a));
    });
}

// verify_blob_kzg_proof (verifier/src/verify.rs:77-115) up to the pairing for `count` blobs, cut as
// kzgb_group_commit_and_prove_blobs cuts them.
int kzgb_group_verify_blob_proofs_g1(kzgb_group* g, const uint8_t* const* blobs, const size_t* lens, size_t count,
                                     const uint64_t* commitments_xy, const uint8_t* commitments_inf,
                                     const uint64_t* proofs_xy, const uint8_t* proofs_inf, uint64_t* out_xy,
                                     uint8_t* out_inf, uint64_t* z_out, uint64_t* y_out) {
    std::lock_guard<std::mutex> lk(g->mu);
    return for_blob_shares(g, lens, count, [&](kzgb_ctx* c, size_t a, size_t n) {
        return kzgb_verify_blob_proofs_g1(c, blobs + a, lens + a, n, commitments_xy + 8 * a, at_or_null(commitments_inf, a),
                                          proofs_xy + 8 * a, at_or_null(proofs_inf, a), at_or_null(out_xy, 8 * a),
                                          at_or_null(out_inf, a), at_or_null(z_out, 4 * a), at_or_null(y_out, 4 * a));
    });
}

// verify_blob_kzg_proof (verifier/src/verify.rs:77-115) through the pairing for `count` blobs, cut as
// kzgb_group_commit_and_prove_blobs cuts them.
int kzgb_group_verify_blob_proofs(kzgb_group* g, const uint8_t* const* blobs, const size_t* lens, size_t count,
                                  const uint64_t* commitments_xy, const uint8_t* commitments_inf, const uint64_t* proofs_xy,
                                  const uint8_t* proofs_inf, uint8_t* ok) {
    std::lock_guard<std::mutex> lk(g->mu);
    return for_blob_shares(g, lens, count, [&](kzgb_ctx* c, size_t a, size_t n) {
        return kzgb_verify_blob_proofs(c, blobs + a, lens + a, n, commitments_xy + 8 * a, at_or_null(commitments_inf, a),
                                       proofs_xy + 8 * a, at_or_null(proofs_inf, a), ok + a);
    });
}

// [tau]G2 of every member: checked on member 0 first, so an invalid point changes no member
int kzgb_group_set_g2_tau(kzgb_group* g, const uint64_t xy[16]) {
    std::lock_guard<std::mutex> lk(g->mu);
    const int rc = kzgb_set_g2_tau(g->ctx[0], xy);
    if (rc) return gfail(g, rc, kzgb_last_error(g->ctx[0]));
    return for_members(g, [&](int i) { return i == 0 ? (int)KZGB_OK : kzgb_set_g2_tau(g->ctx[i], xy); });
}

// verify_blob_kzg_proof_batch (verifier/src/batch.rs:16-249) up to the pairing.  The per-blob challenges and evaluations,
// nearly all of the work, are cut by bytes across the members; the combination (two MSMs of m and 2m + 1 points) runs
// on member 0 over all m openings, so the result is the one-context call's.
int kzgb_group_verify_batch_rlc(kzgb_group* g, const uint8_t* const* blobs, const size_t* lens, size_t count,
                                const uint64_t* commitments_xy, const uint8_t* commitments_inf, const uint64_t* proofs_xy,
                                const uint8_t* proofs_inf, uint64_t lhs_xy[8], uint8_t* lhs_inf, uint64_t rhs_xy[8],
                                uint8_t* rhs_inf) {
    std::lock_guard<std::mutex> lk(g->mu);
    kzgb_ctx* c0 = g->ctx[0];
    const size_t m = count;
    std::vector<uint64_t> zs(4 * m), ys(4 * m), ns(m);
    if (m) {
        // the one-context call's checks, in its order: the 2m points (batch.rs:30-37), then the lengths
        std::vector<uint64_t> xy(16 * m);
        std::vector<uint8_t> inf(2 * m, 0);
        memcpy(xy.data(), commitments_xy, 64 * m);
        memcpy(xy.data() + 8 * m, proofs_xy, 64 * m);
        if (commitments_inf) memcpy(inf.data(), commitments_inf, m);
        if (proofs_inf) memcpy(inf.data() + m, proofs_inf, m);
        int rc = kzgb_validate_g1_points(c0, xy.data(), inf.data(), 2 * m);
        if (rc) return gfail(g, rc, kzgb_last_error(c0));
        for (size_t i = 0; i < m; i++) {
            if (lens[i] == 0) return gfail(g, KZGB_ERR_GENERIC, "Length of data after padding is 0");
            size_t n = 1;
            while (n < (lens[i] + 31) / 32) n <<= 1;
            ns[i] = n;
        }
        rc = for_blob_shares(g, lens, m, [&](kzgb_ctx* c, size_t a, size_t n) {
            return kzgb_verify_blob_proofs_g1(c, blobs + a, lens + a, n, commitments_xy + 8 * a, at_or_null(commitments_inf, a),
                                              proofs_xy + 8 * a, at_or_null(proofs_inf, a), nullptr, nullptr, &zs[4 * a], &ys[4 * a]);
        });
        if (rc) return rc;
    }
    const int rc = kzgb_verify_kzg_proof_batch_rlc(c0, m, commitments_xy, commitments_inf, proofs_xy, proofs_inf, zs.data(),
                                                   ys.data(), ns.data(), lhs_xy, lhs_inf, rhs_xy, rhs_inf);
    if (rc) return gfail(g, rc, std::string("member 0 (device ") + std::to_string(g->dev[0]) + "): " + kzgb_last_error(c0));
    return KZGB_OK;
}

// ---- one large MSM over the SRS, sharded by point range -------------------------------------------------------
// KZG::commit_coeff_form (prover/src/kzg.rs:107-125) for polynomials too large for one GPU's liking: member i
// computes sum_{j in share i} s_j SRS_j (fixed-base over its range table when kzgb_group_srs_precompute_ranges was
// called for this n), the G partial sums are added on the host (G1 addition of 64-byte points: no collective needed
// inside one process).
int kzgb_group_msm_srs(kzgb_group* g, const uint64_t* scalars, size_t n, uint64_t out_xy[8], uint8_t* out_inf) {
    std::lock_guard<std::mutex> lk(g->mu);
    const int G = (int)g->ctx.size();
    if (n > kzgb_srs_len(g->ctx[0])) return gfail(g, KZGB_ERR_SERIALIZATION, "polynomial length is not correct");
    std::vector<uint64_t> part((size_t)G * 8, 0);
    std::vector<uint8_t> pinf(G, 1);
    int rc = for_members(g, [&](int i) {
        size_t first, cnt;
        share(n, G, i, 32, &first, &cnt);
        if (!cnt) return (int)KZGB_OK;
        return kzgb_msm_srs_range(g->ctx[i], scalars + 4 * first, first, cnt, &part[8 * (size_t)i], &pinf[i]);
    });
    if (rc) return rc;
    uint64_t acc[8] = {0};
    uint8_t ainf = 1;
    for (int i = 0; i < G; i++) kzgb_g1_add(acc, ainf, &part[8 * (size_t)i], pinf[i], acc, &ainf);
    memcpy(out_xy, acc, 64);
    if (out_inf) *out_inf = ainf;
    return KZGB_OK;
}

int kzgb_group_sync(kzgb_group* g) {
    std::lock_guard<std::mutex> lk(g->mu);
    return for_members(g, [&](int i) { return kzgb_sync(g->ctx[i]); });
}

}  // extern "C"
