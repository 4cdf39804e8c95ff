// Fr glue around the MSM/NTT: blob bytes <-> field elements, barycentric evaluation and the
// KZG quotient in evaluation form, powers of a challenge.
//   to_fr_array                         reference primitives/src/helpers.rs:40-57
//   evaluate_polynomial_in_evaluation_form   primitives/src/helpers.rs:475-535
//   quotient loop + z-in-domain case    prover/src/kzg.rs:141-174, 237-260
//   compute_powers                      primitives/src/helpers.rs:298-314
// The reference does n separate field inversions (twice); here the n denominators z - w_i are
// inverted with Montgomery's trick: 8 per thread in registers, a product scan across the warp
// with shuffles, ONE Fermat inversion per warp.
#include <cstdlib>
#include "kzgb_internal.hpp"

namespace kzgb {

__device__ __forceinline__ uint32_t bswap32(uint32_t x) { return __byte_perm(x, 0, 0x0123); }

__global__ void __launch_bounds__(256) k_bytes_to_fr(const uint8_t* __restrict__ in, uint64_t len, Fr* __restrict__ out,
                                                      uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fr v = blob_element(in, len, i);
    if ((uint64_t)i * 32 < len) fe_to_mont(v, v);  // also reduces any 256-bit value mod r
    fe_store(&out[i], v);
}

__global__ void __launch_bounds__(256) k_fr_to_bytes(const Fr* __restrict__ in, uint8_t* __restrict__ out, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fr v = fe_load_ro(&in[i]);
    fe_from_mont(v, v);
    uint4* q = reinterpret_cast<uint4*>(out + (size_t)i * 32);
    q[0] = make_uint4(bswap32(v.l[7]), bswap32(v.l[6]), bswap32(v.l[5]), bswap32(v.l[4]));
    q[1] = make_uint4(bswap32(v.l[3]), bswap32(v.l[2]), bswap32(v.l[1]), bswap32(v.l[0]));
}

// w_i = omega_n^i from the omega_N table (i < n)
__device__ __forceinline__ Fr domain_root(const Fr* __restrict__ tw, uint32_t i, int logn, int logN) {
    Fr w;
    if (logn == 0) { fe_one(w); return w; }
    uint32_t half = 1u << (logn - 1);
    if (i < half) return fe_load_ro(&tw[i << (logN - logn)]);
    w = fe_load_ro(&tw[(i - half) << (logN - logn)]);
    fe_neg(w, w);
    return w;
}

__device__ __forceinline__ Fr shfl_fe(const Fr& v, int src) {
    Fr r;
#pragma unroll
    for (int k = 0; k < 8; k++) r.l[k] = __shfl_sync(0xffffffffu, v.l[k], src);
    return r;
}

static constexpr int EVAL_E = 8;        // denominators per thread
static constexpr int EVAL_THREADS = 256;
static constexpr int EVAL_TILE = EVAL_E * EVAL_THREADS;

// block reduction of one Fr per thread into out (thread 0 writes)
__device__ __forceinline__ void block_sum_fr(Fr v, Fr* out) {
    __shared__ uint32_t red[8][EVAL_THREADS / 32];
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int off = 16; off >= 1; off >>= 1) {
        Fr o;
#pragma unroll
        for (int k = 0; k < 8; k++) o.l[k] = __shfl_down_sync(0xffffffffu, v.l[k], off);
        fe_add(v, v, o);
    }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 8; k++) red[k][wid] = v.l[k];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        Fr acc = v;
        for (int w = 1; w < (int)(blockDim.x >> 5); w++) {  // blockDim.x <= EVAL_THREADS
            Fr o;
#pragma unroll
            for (int k = 0; k < 8; k++) o.l[k] = red[k][w];
            fe_add(acc, acc, o);
        }
        fe_store(out, acc);
    }
    __syncthreads();
}

// ---- batched inversion of the n denominators d_i = z - w_i WITHOUT any field inversion on the GPU:
// prod_i d_i = z^n - 1, so T^-1 = 1/(z^n - 1) is one host inversion per polynomial (z = w_m:
// the zero factor is replaced by 1 and the product becomes n / z).  Then
//     1/d_i = T^-1 * prod_{j != i} d_j ,
// assembled from per-thread, per-warp, per-block and grid-level prefix/suffix products.
// Batched over blockIdx.y (one polynomial of n evaluations per batch entry, its own z).

// d[k], running prefix pp[k] for this thread's EVAL_E denominators; returns which k (if any) was zero
__device__ __forceinline__ uint32_t eval_thread_denoms(const Fr& z, const Fr* __restrict__ tw, uint32_t base, uint32_t n,
                                                       int logn, int logN, Fr* d, Fr* pp, uint32_t* zidx) {
    Fr one; fe_one(one);
    uint32_t zero_k = 0xffffffffu;
#pragma unroll
    for (int k = 0; k < EVAL_E; k++) {
        uint32_t i = base + k * EVAL_THREADS;
        if (i < n) {
            Fr w = domain_root(tw, i, logn, logN);
            fe_sub(d[k], z, w);
            if (fe_is_zero(d[k])) { d[k] = one; zero_k = k; if (zidx) zidx[0] = i + 1; }
        } else {
            d[k] = one;
        }
        if (k == 0) pp[0] = d[0]; else fe_mul(pp[k], pp[k - 1], d[k]);
    }
    return zero_k;
}

// inclusive prefix (inc) and suffix (suf) products of v across the warp
__device__ __forceinline__ void warp_scan_products(const Fr& v, uint32_t lane, Fr& inc, Fr& suf) {
    inc = v;
    for (int off = 1; off < 32; off <<= 1) {
        Fr o;
#pragma unroll
        for (int k = 0; k < 8; k++) o.l[k] = __shfl_up_sync(0xffffffffu, inc.l[k], off);
        if ((int)lane >= off) fe_mul(inc, inc, o);
    }
    suf = v;
    for (int off = 1; off < 32; off <<= 1) {
        Fr o;
#pragma unroll
        for (int k = 0; k < 8; k++) o.l[k] = __shfl_down_sync(0xffffffffu, suf.l[k], off);
        if ((int)lane + off < 32) fe_mul(suf, suf, o);
    }
}

// E1: product of each block's 2048 denominators
__global__ void __launch_bounds__(EVAL_THREADS) k_eval_block_products(uint32_t n, int logn, const Fr* __restrict__ z_all,
                                                                      const Fr* __restrict__ tw, int logN,
                                                                      Fr* __restrict__ bprod_all, uint32_t nparts,
                                                                      uint32_t* __restrict__ zidx_all,
                                                                      const uint32_t* __restrict__ only_flagged) {
    __shared__ uint32_t wt[8][EVAL_THREADS / 32];
    const uint32_t bi = blockIdx.y;
    if (only_flagged && !only_flagged[bi]) return;
    const Fr z = fe_load(&z_all[bi]);
    const uint32_t base = blockIdx.x * EVAL_TILE + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    Fr d[EVAL_E], pp[EVAL_E];
    eval_thread_denoms(z, tw, base, n, logn, logN, d, pp, zidx_all + bi);
    Fr v = pp[EVAL_E - 1];
    for (int off = 16; off >= 1; off >>= 1) {
        Fr o;
#pragma unroll
        for (int k = 0; k < 8; k++) o.l[k] = __shfl_down_sync(0xffffffffu, v.l[k], off);
        fe_mul(v, v, o);
    }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 8; k++) wt[k][wid] = v.l[k];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        Fr acc = v;
        for (int w = 1; w < EVAL_THREADS / 32; w++) {
            Fr o;
#pragma unroll
            for (int k = 0; k < 8; k++) o.l[k] = wt[k][w];
            fe_mul(acc, acc, o);
        }
        fe_store(&bprod_all[(size_t)bi * nparts + blockIdx.x], acc);
    }
}

// E2 (one block per polynomial): fac[j] = T^-1 * prod_{k != j} bprod[k]
__global__ void __launch_bounds__(EVAL_THREADS) k_eval_block_factors(const Fr* __restrict__ bprod_all, uint32_t nparts,
                                                                     const Fr* __restrict__ tinv_all, Fr* __restrict__ fac_all,
                                                                     const uint32_t* __restrict__ only_flagged) {
    __shared__ Fr pre[EVAL_THREADS], post[EVAL_THREADS];
    const uint32_t bi = blockIdx.x, tid = threadIdx.x;
    if (only_flagged && !only_flagged[bi]) return;
    const Fr* bprod = bprod_all + (size_t)bi * nparts;
    Fr* fac = fac_all + (size_t)bi * nparts;
    const uint32_t per = (nparts + EVAL_THREADS - 1) / EVAL_THREADS;
    const uint32_t lo = min(tid * per, nparts), hi = min(lo + per, nparts);
    Fr one; fe_one(one);
    Fr prod = one;
    for (uint32_t j = lo; j < hi; j++) { Fr v = fe_load(&bprod[j]); fe_mul(prod, prod, v); }
    pre[tid] = prod;
    post[tid] = prod;
    __syncthreads();
    // Hillis-Steele inclusive scans (prefix in pre, suffix in post)
    for (uint32_t off = 1; off < EVAL_THREADS; off <<= 1) {
        Fr a = pre[tid], b = post[tid];
        bool ha = tid >= off, hb = tid + off < EVAL_THREADS;
        Fr oa = ha ? pre[tid - off] : one, ob = hb ? post[tid + off] : one;
        __syncthreads();
        if (ha) { fe_mul(a, a, oa); pre[tid] = a; }
        if (hb) { fe_mul(b, b, ob); post[tid] = b; }
        __syncthreads();
    }
    Fr before = tid > 0 ? pre[tid - 1] : one;                    // product of all parts owned by lower threads
    Fr after = tid + 1 < EVAL_THREADS ? post[tid + 1] : one;     // ... by higher threads
    Fr tinv = fe_load(&tinv_all[bi]);
    fe_mul(after, after, tinv);
    // forward: fac[j] = before * prod_{lo <= k < j}; backward: times prod_{j < k < hi} * after
    Fr run = before;
    for (uint32_t j = lo; j < hi; j++) { fe_store(&fac[j], run); Fr v = fe_load(&bprod[j]); fe_mul(run, run, v); }
    run = after;
    for (uint32_t j = hi; j-- > lo;) {
        Fr f = fe_load(&fac[j]);
        fe_mul(f, f, run);
        fe_store(&fac[j], f);
        Fr v = fe_load(&bprod[j]);
        fe_mul(run, run, v);
    }
}

// E3: inv[i] = 1/(z - w_i) (1 where z == w_i); partial[block] = sum f_i w_i inv[i]
__global__ void __launch_bounds__(EVAL_THREADS) k_eval_inverses(const Fr* __restrict__ evals_all, uint32_t n, int logn,
                                                                const Fr* __restrict__ z_all, const Fr* __restrict__ tw,
                                                                int logN, const Fr* __restrict__ fac_all,
                                                                Fr* __restrict__ inv_all, Fr* __restrict__ partial_all,
                                                                uint32_t nparts, const uint32_t* __restrict__ only_flagged) {
    __shared__ uint32_t wt[8][EVAL_THREADS / 32];
    const uint32_t bi = blockIdx.y;
    if (only_flagged && !only_flagged[bi]) return;
    const Fr* evals = evals_all + (size_t)bi * n;
    Fr* inv = inv_all + (size_t)bi * n;
    Fr* partial = partial_all + (size_t)bi * nparts;
    const Fr z = fe_load(&z_all[bi]);
    const uint32_t base = blockIdx.x * EVAL_TILE + threadIdx.x;
    const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    Fr d[EVAL_E], pp[EVAL_E];
    Fr one; fe_one(one);
    const uint32_t zero_k = eval_thread_denoms(z, tw, base, n, logn, logN, d, pp, nullptr);
    Fr inc, suf;
    warp_scan_products(pp[EVAL_E - 1], lane, inc, suf);
    if (lane == 31) {
#pragma unroll
        for (int k = 0; k < 8; k++) wt[k][wid] = inc.l[k];
    }
    Fr exc, sufx;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        exc.l[k] = __shfl_up_sync(0xffffffffu, inc.l[k], 1);
        sufx.l[k] = __shfl_down_sync(0xffffffffu, suf.l[k], 1);
    }
    if (lane == 0) exc = one;
    if (lane == 31) sufx = one;
    __syncthreads();
    // product of the other warps of the block, times the grid-level factor of this block
    Fr run = fe_load(&fac_all[(size_t)bi * nparts + blockIdx.x]);
    for (uint32_t w = 0; w < EVAL_THREADS / 32; w++) {
        if (w == wid) continue;
        Fr o;
#pragma unroll
        for (int k = 0; k < 8; k++) o.l[k] = wt[k][w];
        fe_mul(run, run, o);
    }
    fe_mul(run, run, exc);
    fe_mul(run, run, sufx);  // 1 / (product of this thread's denominators)
    Fr sum; fe_zero(sum);
#pragma unroll
    for (int k = EVAL_E - 1; k >= 0; k--) {
        Fr iv;
        if (k > 0) { fe_mul(iv, run, pp[k - 1]); fe_mul(run, run, d[k]); } else iv = run;
        uint32_t i = base + k * EVAL_THREADS;
        if (i < n) {
            fe_store(&inv[i], iv);
            if ((uint32_t)k != zero_k) {
                Fr f = fe_load_ro(&evals[i]);
                Fr w = domain_root(tw, i, logn, logN);
                fe_mul(f, f, w);
                fe_mul(f, f, iv);
                fe_add(sum, sum, f);
            }
        }
    }
    block_sum_fr(sum, &partial[blockIdx.x]);
}

// ---- the same inverses from the STRUCTURE of the domain, for z outside it (the generic case: z is a hash) ----
//     (z - w_i) * prod_{j < k} (z^(2^j) + w_i^(2^j)) = z^n - 1        (n = 2^k)
// so 1/(z - w_i) = T^-1 * prod_j (Z_j + w^((i << j) mod n)), Z_j = z^(2^j), and the factor of level j only
// depends on i mod (n >> j): a thread that owns the 16 elements i = r + t * n/16 shares the k - 4 top factors
// among all of them and the lower ones pairwise -> (k - 3) + 30 multiplications per 16 inverses (2.8 per
// element instead of ~10 for the prefix/suffix products), no block or grid level products at all.
static constexpr int EV2_THREADS = 128;
static std::atomic<int> g_eval_structured{1};
void eval_set_structured(int on) { g_eval_structured.store(on != 0); }
static constexpr int ZP_STRIDE = 32;  // Z_j slots per polynomial

__global__ void __launch_bounds__(64) k_eval_zpowers(const Fr* __restrict__ z_all, int logn, uint32_t batch, Fr* __restrict__ zp_all,
                                                     const uint32_t* __restrict__ skip_flagged) {
    uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= batch) return;
    if (skip_flagged && skip_flagged[b]) return;
    Fr z = fe_load(&z_all[b]);
    for (int j = 0; j < logn; j++) {
        fe_store(&zp_all[(size_t)b * ZP_STRIDE + j], z);
        fe_sqr(z, z);
    }
}

__global__ void __launch_bounds__(EV2_THREADS) k_eval_inverses2(const Fr* __restrict__ evals_all, uint32_t n, int logn,
                                                                 const Fr* __restrict__ tw, int logN,
                                                                 const Fr* __restrict__ tinv_all, const Fr* __restrict__ zp_all,
                                                                 Fr* __restrict__ inv_all, Fr* __restrict__ partial_all,
                                                                 uint32_t nparts, const uint32_t* __restrict__ skip_flagged) {
    __shared__ Fr zs[ZP_STRIDE];
    const uint32_t bi = blockIdx.y;
    if (skip_flagged && skip_flagged[bi]) return;
    if ((int)threadIdx.x < logn) zs[threadIdx.x] = fe_load(&zp_all[(size_t)bi * ZP_STRIDE + threadIdx.x]);
    __syncthreads();
    const Fr* evals = evals_all + (size_t)bi * n;
    Fr* inv = inv_all + (size_t)bi * n;
    const uint32_t q = n >> 4, mask = n - 1;
    const uint32_t r = blockIdx.x * EV2_THREADS + threadIdx.x;
    Fr sum; fe_zero(sum);
    if (r < q) {
        Fr P4 = fe_load(&tinv_all[bi]);  // 1 / (z^n - 1)
#pragma unroll 1
        for (int m = logn - 1; m >= 4; m--) {
            Fr t = domain_root(tw, (r << m) & mask, logn, logN);
            fe_add(t, t, zs[m]);
            fe_mul(P4, P4, t);
        }
#pragma unroll 1
        for (uint32_t a = 0; a < 2; a++) {
            const uint32_t i3 = r + a * q;
            Fr P3 = domain_root(tw, (i3 << 3) & mask, logn, logN);
            fe_add(P3, P3, zs[3]);
            fe_mul(P3, P3, P4);
#pragma unroll 1
            for (uint32_t b = 0; b < 2; b++) {
                const uint32_t i2 = i3 + 2 * b * q;
                Fr P2 = domain_root(tw, (i2 << 2) & mask, logn, logN);
                fe_add(P2, P2, zs[2]);
                fe_mul(P2, P2, P3);
#pragma unroll 1
                for (uint32_t cc = 0; cc < 2; cc++) {
                    const uint32_t i1 = i2 + 4 * cc * q;
                    Fr P1 = domain_root(tw, (i1 << 1) & mask, logn, logN);
                    fe_add(P1, P1, zs[1]);
                    fe_mul(P1, P1, P2);
#pragma unroll 1
                    for (uint32_t d = 0; d < 2; d++) {
                        const uint32_t i0 = i1 + 8 * d * q;
                        Fr w = domain_root(tw, i0, logn, logN);
                        Fr iv;
                        fe_add(iv, w, zs[0]);
                        fe_mul(iv, iv, P1);  // 1 / (z - w_i)
                        fe_store(&inv[i0], iv);
                        Fr f = fe_load_ro(&evals[i0]);
                        fe_mul(f, f, w);
                        fe_mul(f, f, iv);
                        fe_add(sum, sum, f);
                    }
                }
            }
        }
    }
    block_sum_fr(sum, &partial_all[(size_t)bi * nparts + blockIdx.x]);
}

// y = (z^n - 1)/n * sum   or   f_m when z = w_m          (one block per batch entry)
__global__ void __launch_bounds__(EVAL_THREADS) k_eval_finish(const Fr* __restrict__ evals_all, uint32_t n, int logn,
                                                              const Fr* __restrict__ z_all, Fr ninv,
                                                              const Fr* __restrict__ partial_all, uint32_t nparts,
                                                              const uint32_t* __restrict__ zidx_all, Fr* __restrict__ y_all) {
    const uint32_t bi = blockIdx.x;
    const Fr* evals = evals_all + (size_t)bi * n;
    const Fr* partial = partial_all + (size_t)bi * nparts;
    Fr sum; fe_zero(sum);
    for (uint32_t k = threadIdx.x; k < nparts; k += EVAL_THREADS) {
        Fr v = fe_load(&partial[k]);
        fe_add(sum, sum, v);
    }
    __shared__ Fr total;
    block_sum_fr(sum, &total);
    if (threadIdx.x == 0) {
        uint32_t zi = zidx_all[bi];
        Fr y;
        if (zi != 0) {
            y = fe_load(&evals[zi - 1]);
        } else {
            Fr zn = fe_load(&z_all[bi]);
            for (int k = 0; k < logn; k++) fe_sqr(zn, zn);
            Fr one; fe_one(one);
            fe_sub(zn, zn, one);
            Fr t = total;
            fe_mul(y, t, zn);
            fe_mul(y, y, ninv);
        }
        fe_store(&y_all[bi], y);
    }
}

// q_i = (y - f_i) * inv_i ; when z = w_m also partial sums of q_i * w_i (i != m)
__global__ void __launch_bounds__(EVAL_THREADS) k_quotient(const Fr* __restrict__ evals_all, uint32_t n, int logn,
                                                           const Fr* __restrict__ tw, int logN, const Fr* __restrict__ inv_all,
                                                           const Fr* __restrict__ y_all, const uint32_t* __restrict__ zidx_all,
                                                           Fr* __restrict__ q_all, Fr* __restrict__ partial_all, uint32_t nparts) {
    const uint32_t bi = blockIdx.y;
    const Fr* evals = evals_all + (size_t)bi * n;
    const Fr* inv = inv_all + (size_t)bi * n;
    Fr* q = q_all + (size_t)bi * n;
    Fr* partial = partial_all + (size_t)bi * nparts;
    const uint32_t i = blockIdx.x * EVAL_THREADS + threadIdx.x;
    const uint32_t zi = zidx_all[bi];
    Fr y = fe_load(&y_all[bi]);
    Fr term; fe_zero(term);
    if (i < n) {
        Fr f = fe_load_ro(&evals[i]);
        Fr iv = fe_load_ro(&inv[i]);
        Fr qi;
        fe_sub(qi, y, f);
        fe_mul(qi, qi, iv);
        if (zi != 0 && i == zi - 1) fe_zero(qi);  // patched by k_quotient_fix
        fe_store(&q[i], qi);
        if (zi != 0 && i != zi - 1) {
            Fr w = domain_root(tw, i, logn, logN);
            fe_mul(term, qi, w);
        }
    }
    if (zi != 0) block_sum_fr(term, &partial[blockIdx.x]);
}

// q_m = -(1/z) * sum_{i != m} q_i w_i  with 1/z = w_{(n-m) mod n}     (prover/src/kzg.rs:237-260)
__global__ void __launch_bounds__(EVAL_THREADS) k_quotient_fix(uint32_t n, int logn, const Fr* __restrict__ tw, int logN,
                                                               const Fr* __restrict__ partial_all, uint32_t nparts,
                                                               const uint32_t* __restrict__ zidx_all, Fr* __restrict__ q_all) {
    const uint32_t bi = blockIdx.x;
    const uint32_t zi = zidx_all[bi];
    if (zi == 0) return;
    const Fr* partial = partial_all + (size_t)bi * nparts;
    Fr* q = q_all + (size_t)bi * n;
    Fr sum; fe_zero(sum);
    for (uint32_t k = threadIdx.x; k < nparts; k += EVAL_THREADS) {
        Fr v = fe_load(&partial[k]);
        fe_add(sum, sum, v);
    }
    __shared__ Fr total;
    block_sum_fr(sum, &total);
    if (threadIdx.x == 0) {
        uint32_t m = zi - 1;
        Fr zinv = domain_root(tw, (n - m) & (n - 1), logn, logN);
        Fr r;
        Fr t = total;
        fe_mul(r, t, zinv);
        fe_neg(r, r);
        fe_store(&q[m], r);
    }
}

// The points of a batch of openings at caller-given z (kzgb_compute_proofs), one thread per opening: tinv_k = 1/(z^n - 1),
// or z/n when z^n == 1 (eval_tinv's formula), and in_domain_k = 1 in that case.
__global__ void __launch_bounds__(64) k_eval_points(const Fr* __restrict__ z_all, int logn, uint32_t batch, Fr ninv,
                                                    Fr* __restrict__ tinv_out, uint32_t* __restrict__ in_domain_out) {
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= batch) return;
    const Fr z = fe_load(&z_all[k]);
    Fr zn = z, one, t;
    for (int s = 0; s < logn; s++) fe_sqr(zn, zn);
    fe_one(one);
    const bool in_domain = fe_eq(zn, one);
    if (in_domain) fe_mul(t, z, ninv);
    else { fe_sub(zn, zn, one); fe_inv_fast(t, zn); }
    fe_store(&tinv_out[k], t);
    in_domain_out[k] = in_domain ? 1u : 0u;
}

__global__ void __launch_bounds__(256) k_fr_powers(Fr* __restrict__ out, uint32_t n, Fr base, uint32_t first) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t e[8] = {first + i, 0, 0, 0, 0, 0, 0, 0};
    Fr r;
    fe_pow(r, base, e);
    fe_store(&out[i], r);
}

__global__ void __launch_bounds__(256) k_fr_mul_vec(Fr* __restrict__ out, const Fr* __restrict__ a, const Fr* __restrict__ b,
                                                     uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Fr x = fe_load_ro(&a[i]), y = fe_load_ro(&b[i]);
    fe_mul(x, x, y);
    fe_store(&out[i], x);
}

__global__ void __launch_bounds__(EVAL_THREADS) k_fr_dot(Fr* __restrict__ out, const Fr* __restrict__ a,
                                                         const Fr* __restrict__ b, uint32_t n) {
    Fr sum; fe_zero(sum);
    for (uint32_t k = threadIdx.x; k < n; k += EVAL_THREADS) {
        Fr x = fe_load_ro(&a[k]), y = fe_load_ro(&b[k]);
        fe_mul(x, x, y);
        fe_add(sum, sum, x);
    }
    block_sum_fr(sum, out);
}

// ---------------------------------------------------------------------------------
void bytes_to_fr_launch(const uint8_t* in, uint64_t len_bytes, Fr* out, uint32_t n, cudaStream_t st) {
    if (!n) return;
    k_bytes_to_fr<<<(n + 255) / 256, 256, 0, st>>>(in, len_bytes, out, n);
    g_launch_count++;
}
void fr_to_bytes_launch(const Fr* in, uint8_t* out, uint32_t n, cudaStream_t st) {
    if (!n) return;
    k_fr_to_bytes<<<(n + 255) / 256, 256, 0, st>>>(in, out, n);
    g_launch_count++;
}

size_t eval_quotient_scratch_elems(uint32_t n, uint32_t batch) {
    uint32_t parts1 = (n + EVAL_TILE - 1) / EVAL_TILE;
    uint32_t parts2 = (n + EVAL_THREADS - 1) / EVAL_THREADS;
    // inverses, block products, block factors, partial sums (both kernels), zidx words (whole Fr slots)
    return (size_t)batch * ((size_t)n + 3 * (size_t)parts1 + parts2 + ZP_STRIDE) + ((size_t)batch * 4 + 31) / 32 + 1;
}

void eval_quotient_launch(const Fr* evals, uint32_t n, int logn, uint32_t batch, const Fr* z_mont_dev,
                          const Fr* tinv_mont_dev, const Fr* tw, int logN, const Fr* ninv_mont_host, Fr* scratch,
                          Fr* q_out, Fr* y_out, cudaStream_t st, bool z_outside_domain, const uint32_t* in_domain_dev) {
    if (!batch) return;
    uint32_t parts1 = (n + EVAL_TILE - 1) / EVAL_TILE;
    uint32_t parts2 = (n + EVAL_THREADS - 1) / EVAL_THREADS;
    Fr* inv = scratch;
    Fr* bprod = inv + (size_t)batch * n;
    Fr* fac = bprod + (size_t)batch * parts1;
    Fr* partial1 = fac + (size_t)batch * parts1;
    Fr* partial2 = partial1 + (size_t)batch * parts1;
    uint32_t* zidx = reinterpret_cast<uint32_t*>(partial2 + (size_t)batch * parts2);
    Fr* zp = partial2 + (size_t)batch * parts2 + (((size_t)batch * 4 + 31) / 32 + 1);
    cudaMemsetAsync(zidx, 0, (size_t)batch * 4, st);
    const bool can_structure = g_eval_structured.load() && logn >= 6 && logn <= 28;
    const bool per_poly = in_domain_dev != nullptr && can_structure;  // the device decides per polynomial
    if ((z_outside_domain && can_structure) || per_poly) {
        // z outside the domain: inverses from the factorisation of z^n - 1 (EVAL_TILE = 16 * EV2_THREADS,
        // so the per-block partial sums land exactly where k_eval_finish expects them)
        static_assert(16 * EV2_THREADS == EVAL_TILE, "partial-sum layout");
        const uint32_t* skip = per_poly ? in_domain_dev : nullptr;
        k_eval_zpowers<<<(batch + 63) / 64, 64, 0, st>>>(z_mont_dev, logn, batch, zp, skip);
        k_eval_inverses2<<<dim3(parts1, batch), EV2_THREADS, 0, st>>>(evals, n, logn, tw, logN, tinv_mont_dev, zp, inv, partial1, parts1, skip);
        g_launch_count += 2;
    }
    if (!(z_outside_domain && can_structure)) {
        const uint32_t* only = per_poly ? in_domain_dev : nullptr;
        k_eval_block_products<<<dim3(parts1, batch), EVAL_THREADS, 0, st>>>(n, logn, z_mont_dev, tw, logN, bprod, parts1, zidx, only);
        k_eval_block_factors<<<batch, EVAL_THREADS, 0, st>>>(bprod, parts1, tinv_mont_dev, fac, only);
        k_eval_inverses<<<dim3(parts1, batch), EVAL_THREADS, 0, st>>>(evals, n, logn, z_mont_dev, tw, logN, fac, inv, partial1,
                                                                      parts1, only);
        g_launch_count += 3;
    }
    k_eval_finish<<<batch, EVAL_THREADS, 0, st>>>(evals, n, logn, z_mont_dev, *ninv_mont_host, partial1, parts1, zidx, y_out);
    g_launch_count += 1;
    if (q_out) {
        k_quotient<<<dim3(parts2, batch), EVAL_THREADS, 0, st>>>(evals, n, logn, tw, logN, inv, y_out, zidx, q_out,
                                                                 partial2, parts2);
        k_quotient_fix<<<batch, EVAL_THREADS, 0, st>>>(n, logn, tw, logN, partial2, parts2, zidx, q_out);
        g_launch_count += 2;
    }
}

void eval_points_launch(const Fr* z_mont_dev, int logn, uint32_t batch, const Fr* ninv_mont_host, Fr* tinv_out,
                        uint32_t* in_domain_out, cudaStream_t st) {
    if (!batch) return;
    k_eval_points<<<(batch + 63) / 64, 64, 0, st>>>(z_mont_dev, logn, batch, *ninv_mont_host, tinv_out, in_domain_out);
    g_launch_count++;
}

void fr_powers_launch(Fr* out, uint32_t n, const Fr* base_mont_host, cudaStream_t st, uint32_t first) {
    if (!n) return;
    k_fr_powers<<<(n + 255) / 256, 256, 0, st>>>(out, n, *base_mont_host, first);
    g_launch_count++;
}
void fr_mul_vec_launch(Fr* out, const Fr* a, const Fr* b, uint32_t n, cudaStream_t st) {
    if (!n) return;
    k_fr_mul_vec<<<(n + 255) / 256, 256, 0, st>>>(out, a, b, n);
    g_launch_count++;
}
void fr_dot_launch(Fr* out, const Fr* a, const Fr* b, uint32_t n, cudaStream_t st) {
    k_fr_dot<<<1, EVAL_THREADS, 0, st>>>(out, a, b, n);
    g_launch_count++;
}

}  // namespace kzgb
