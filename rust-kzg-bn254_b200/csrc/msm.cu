// BN254 G1 multi-scalar multiplication: signed-digit Pippenger, hand-written for sm_100a.
// Replaces the reference's `G1Projective::msm` call sites (prover/src/kzg.rs:100,121,
// primitives/src/helpers.rs:332).
//
// Pipeline (all on one stream, no host sync):
//   1. k_digits_hist     scalar -> canonical -> W signed c-bit digits; histogram of bucket keys
//                        (k_digits_hist_blob: the same from blob bytes, for commit-only blob batches)
//   2. k_scan            exclusive scan of the histogram (bucket offsets)
//   3. k_scatter         counting-sort scatter: point refs grouped by bucket (order inside a
//                        bucket is irrelevant: group addition is commutative and exact)
//   4. k_accumulate      FIXED-SIZE chunks of the sorted list per thread (perfect balance for any
//                        digit distribution); XYZZ += affine gathers from the HBM-resident table
//   5. k_bucket_fix      stitches buckets that span several chunks, zeroes empty buckets
//   6. k_reduce_lines    2-D bucket reduction, step 1: with bucket index k = A*h + l,
//                            sum_k (k+1) B_k = A * sum_h h R_h + sum_l (l+1) C_l,
//                        R_h / C_l the plain row / column sums of the H x A bucket matrix: 2 additions
//                        per bucket, all of them independent (log-depth trees)
//   7. k_reduce_groups   step 2: the two weighted sums bit by bit -- T_b = sum of the R_h (C_l) whose index
//                        has bit b set, doubled b times
//   8. k_reduce_final    sum of the c - 1 group results -> one XYZZ point per bucket set
// Steps 6-8 run on QUAD-COOPERATIVE point arithmetic (4 lanes per addition, one coordinate each, the
// independent multiplications of an addition side by side): a tree level costs 4 multiplication latencies
// instead of 14, which is what a reduction with no parallel slack left is bound by.
// The caller copies `sets` XYZZ points (128 B each) back and finishes on the host.
// One launch set can also carry `batch` independent fixed-base MSMs over the same table (MsmPlan.batch_n):
// scalar i belongs to MSM i / batch_n, which owns bucket set i / batch_n -- how runs of small blobs are committed.
#include <cstdio>
#include "kzgb_internal.hpp"

namespace kzgb {

static constexpr int SM_COUNT = 148;

__device__ __forceinline__ uint32_t scalar_bits(const uint32_t* l, int pos, int c) {
    int w = pos >> 5, b = pos & 31;
    if (w >= 8) return 0;
    uint64_t v = l[w];
    if (w + 1 < 8) v |= (uint64_t)l[w + 1] << 32;
    return (uint32_t)(v >> b) & ((1u << c) - 1u);
}

// One signed digit step.  Returns magnitude in [0, 2^(c-1)], sets neg, updates carry.
__device__ __forceinline__ uint32_t signed_digit(const uint32_t* l, int w, int c, uint32_t& carry, bool& neg) {
    uint32_t d = scalar_bits(l, w * c, c) + carry;
    uint32_t half = 1u << (c - 1);
    if (d > half) { neg = true; carry = 1; return (1u << c) - d; }
    neg = false; carry = 0;
    return d;
}

// canonical scalar i -> canon[i], and its digits into the bucket histogram
__device__ __forceinline__ void digits_hist(const Fr& s, uint32_t i, const MsmPlan& p, Fr* __restrict__ canon,
                                            uint32_t* __restrict__ hist) {
    fe_store(&canon[i], s);
    uint32_t half = 1u << (p.c - 1);
    uint32_t carry = 0;
    for (int w = 0; w < p.W; w++) {
        bool neg;
        uint32_t mag = signed_digit(s.l, w, p.c, carry, neg);
        if (mag) {
            uint32_t key = (p.batch_n ? (i / p.batch_n) * half : (p.sets == 1 ? 0u : (uint32_t)w * half)) + mag - 1u;
            atomicAdd(&hist[key], 1u);
        }
    }
}

__global__ void __launch_bounds__(256) k_digits_hist(const Fr* __restrict__ scalars, MsmPlan p, Fr* __restrict__ canon,
                                                      uint32_t* __restrict__ hist) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    Fr s = fe_load_ro(&scalars[i]);
    fe_from_mont(s, s);
    digits_hist(s, i, p, canon, hist);
}

// x -= m when x >= m (8 little-endian limbs)
__device__ __forceinline__ void sub_if_geq(uint32_t* x, const uint32_t* m) {
    uint32_t t[8];
    uint32_t borrow = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const uint64_t d = (uint64_t)x[k] - m[k] - borrow;
        t[k] = (uint32_t)d;
        borrow = (uint32_t)(d >> 63);
    }
#pragma unroll
    for (int k = 0; k < 8; k++) x[k] = borrow ? x[k] : t[k];
}

// The first sort pass over blob bytes (MsmScalars::blob): scalar i is blob_element(i) mod r.  Every 256-bit value is
// below 6r, so subtracting 4r, 2r and r where they fit leaves the canonical value.
__global__ void __launch_bounds__(256) k_digits_hist_blob(const uint8_t* __restrict__ blob, uint64_t len, MsmPlan p,
                                                           Fr* __restrict__ canon, uint32_t* __restrict__ hist) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    Fr s = blob_element(blob, len, i);
    uint32_t r[8], r2[8], r4[8];
    FeConst<FR>::mod(r);
#pragma unroll
    for (int k = 0; k < 8; k++) {
        r2[k] = (r[k] << 1) | (k ? r[k - 1] >> 31 : 0u);
        r4[k] = (r[k] << 2) | (k ? r[k - 1] >> 30 : 0u);
    }
    sub_if_geq(s.l, r4);
    sub_if_geq(s.l, r2);
    sub_if_geq(s.l, r);
    digits_hist(s, i, p, canon, hist);
}

// Exclusive scan of the bucket histogram, 32 counters per thread held in registers (8 x 128-bit
// loads in flight), warp-shuffle scan of the thread totals, one smem hop across warps.
// block b scans items [b*SCAN_TILE, (b+1)*SCAN_TILE); block_tot[b] = its total.
static constexpr uint32_t SCAN_PER_THREAD = 32;
static constexpr uint32_t SCAN_THREADS = 1024;
static constexpr uint32_t SCAN_TILE = SCAN_PER_THREAD * SCAN_THREADS;

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_tiles(uint32_t* __restrict__ hist, uint32_t* __restrict__ cursor,
                                                             uint32_t nb, uint32_t* __restrict__ block_tot, bool single) {
    __shared__ uint32_t warp_tot[32];
    const uint32_t tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const uint32_t base = blockIdx.x * SCAN_TILE + tid * SCAN_PER_THREAD;
    uint32_t v[SCAN_PER_THREAD];
    if (base + SCAN_PER_THREAD <= nb) {
        const uint4* q = reinterpret_cast<const uint4*>(hist + base);
#pragma unroll
        for (int k = 0; k < 8; k++) { uint4 t = q[k]; v[4 * k] = t.x; v[4 * k + 1] = t.y; v[4 * k + 2] = t.z; v[4 * k + 3] = t.w; }
    } else {
#pragma unroll
        for (int k = 0; k < (int)SCAN_PER_THREAD; k++) v[k] = (base + k < nb) ? hist[base + k] : 0u;
    }
    uint32_t sum = 0;
#pragma unroll
    for (int k = 0; k < (int)SCAN_PER_THREAD; k++) { uint32_t t = v[k]; v[k] = sum; sum += t; }
    uint32_t inc = sum;
    for (int off = 1; off < 32; off <<= 1) {
        uint32_t o = __shfl_up_sync(0xffffffffu, inc, off);
        if ((int)lane >= off) inc += o;
    }
    if (lane == 31) warp_tot[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        uint32_t w = warp_tot[lane], wi = w;
        for (int off = 1; off < 32; off <<= 1) {
            uint32_t o = __shfl_up_sync(0xffffffffu, wi, off);
            if ((int)lane >= off) wi += o;
        }
        warp_tot[lane] = wi - w;  // exclusive
        if (lane == 31) {
            block_tot[blockIdx.x] = wi;
            if (single) hist[nb] = wi;
        }
    }
    __syncthreads();
    const uint32_t off0 = warp_tot[wid] + (inc - sum);
    if (base + SCAN_PER_THREAD <= nb) {
        uint4* q = reinterpret_cast<uint4*>(hist + base);
        uint4* qc = reinterpret_cast<uint4*>(cursor + base);
#pragma unroll
        for (int k = 0; k < 8; k++) {
            uint4 t = make_uint4(v[4 * k] + off0, v[4 * k + 1] + off0, v[4 * k + 2] + off0, v[4 * k + 3] + off0);
            q[k] = t;
            if (single) qc[k] = t;
        }
    } else {
#pragma unroll
        for (int k = 0; k < (int)SCAN_PER_THREAD; k++)
            if (base + k < nb) { hist[base + k] = v[k] + off0; if (single) cursor[base + k] = v[k] + off0; }
    }
}

// multi-tile case: exclusive scan of the tile totals (<= 1024 tiles), then add them back
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_tile_totals(uint32_t* __restrict__ block_tot, uint32_t ntiles,
                                                                   uint32_t* __restrict__ hist, uint32_t nb) {
    __shared__ uint32_t sm[SCAN_THREADS];
    const uint32_t tid = threadIdx.x;
    uint32_t v = tid < ntiles ? block_tot[tid] : 0u;
    sm[tid] = v;
    __syncthreads();
    for (uint32_t off = 1; off < SCAN_THREADS; off <<= 1) {
        uint32_t o = tid >= off ? sm[tid - off] : 0u;
        __syncthreads();
        sm[tid] += o;
        __syncthreads();
    }
    if (tid < ntiles) block_tot[tid] = sm[tid] - v;
    if (tid == SCAN_THREADS - 1) hist[nb] = sm[tid];
}
__global__ void __launch_bounds__(256) k_scan_add(uint32_t* __restrict__ hist, uint32_t* __restrict__ cursor, uint32_t nb,
                                                   const uint32_t* __restrict__ block_tot) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nb) return;
    uint32_t v = hist[i] + block_tot[i / SCAN_TILE];
    hist[i] = v;
    cursor[i] = v;
}

__global__ void __launch_bounds__(256) k_scatter(const Fr* __restrict__ canon, MsmPlan p, uint32_t* __restrict__ cursor,
                                                  uint32_t* __restrict__ sorted) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    Fr s = fe_load_ro(&canon[i]);
    uint32_t half = 1u << (p.c - 1);
    uint32_t carry = 0;
    for (int w = 0; w < p.W; w++) {
        bool neg;
        uint32_t mag = signed_digit(s.l, w, p.c, carry, neg);
        if (mag) {
            uint32_t key = (p.batch_n ? (i / p.batch_n) * half : (p.sets == 1 ? 0u : (uint32_t)w * half)) + mag - 1u;
            uint32_t pos = atomicAdd(&cursor[key], 1u);
            uint32_t ref = p.batch_n ? ((uint32_t)w * p.table_stride + p.base_offset + i % p.batch_n)
                                     : (p.sets == 1) ? ((uint32_t)w * p.table_stride + p.base_offset + i) : i;
            sorted[pos] = ref | (neg ? 0x80000000u : 0u);
        }
    }
}

// ---------------------------------------------------------------------------------
// Bucket accumulation.  acc += q on RELAXED coordinates (every coordinate of acc in [0, 2p), q canonical;
// ec.cuh explains the range argument): 10 products, 9 Montgomery reductions, no conditional subtraction
// after any product.  The state "accumulator empty" is a flag and the first point of a run is installed on a
// real branch, so the addition itself never tests for the identity; PP = P^2 goes through the dedicated
// squaring (36 instead of 64 wide multiplies in the product), a - b (+ 2p) uses predicated additions, and the
// digit's sign is applied by predicated subtractions instead of a divergent branch.
// This is the winner of the round-2 sweep at 2^19 points (profiles/r02_variant_sweep.txt: 1.166 -> 1.133 ms);
// the variants it beat are kept, unbuilt, under experiments/accumulate_variants/.
// Returns false when the sum is the identity.
// ---------------------------------------------------------------------------------
__device__ __forceinline__ bool xyzz_madd_relaxed_nonempty(XYZZ& acc, const Affine& q) {
    Fq U2, S2, Pp, Rr, PP, PPP, Q, t;
    fq_mulnr_ptx(U2.l, q.x.l, acc.zz.l);
    fq_mulnr_ptx(S2.l, q.y.l, acc.zzz.l);
    fq_sub2pp_ptx(Pp.l, U2.l, acc.x.l);
    fq_sub2pp_ptx(Rr.l, S2.l, acc.y.l);
    if (fq_is_zero_mod(Pp)) {
        if (!fq_is_zero_mod(Rr)) return false;
        xyzz_dbl_affine(acc, q);  // canonical result from the canonical q
        return !xyzz_is_inf(acc);
    }
    fq_sqrnr_ptx(PP.l, Pp.l);
    fq_mulnr_ptx(PPP.l, Pp.l, PP.l);
    fq_mulnr_ptx(Q.l, acc.x.l, PP.l);
    fq_mulnr_ptx(acc.zz.l, acc.zz.l, PP.l);
    fq_mulnr_ptx(acc.zzz.l, acc.zzz.l, PPP.l);
    fq_mulnr_ptx(t.l, Rr.l, Rr.l);
    fq_sub2pp_ptx(t.l, t.l, PPP.l); fq_sub2pp_ptx(t.l, t.l, Q.l); fq_sub2pp_ptx(t.l, t.l, Q.l);  // X3
    fq_sub2pp_ptx(Q.l, Q.l, t.l);
    fq_mul2subnr_ptx(acc.y.l, Rr.l, Q.l, acc.y.l, PPP.l);
    acc.x = t;
    return true;
}

// Thread t owns sorted entries [t*chunk, (t+1)*chunk).  A bucket run that lies entirely inside the chunk is
// written to buckets[b]; the run cut by the chunk's start goes to partial[2t], the one cut by its end to
// partial[2t+1] (k_bucket_fix adds them up).
__global__ void __launch_bounds__(128, 4) k_accumulate(const uint32_t* __restrict__ sorted, const uint32_t* __restrict__ offsets,
                                                        const Affine* __restrict__ table, uint32_t nb, uint32_t acc_threads,
                                                        uint32_t chunk, XYZZ* __restrict__ buckets, XYZZ* __restrict__ partial) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= acc_threads) return;
    const uint32_t M = offsets[nb];
    uint64_t start64 = (uint64_t)t * chunk;
    if (start64 >= M) return;  // k_bucket_fix only reads slots of chunks that hold entries
    uint32_t start = (uint32_t)start64;
    uint32_t end = (uint32_t)min((uint64_t)M, start64 + chunk);
    uint32_t lo = 0, hi = nb;  // invariant: offsets[lo] <= start < offsets[hi] (offsets[nb] = M > start)
    while (hi - lo > 1) {
        uint32_t mid = (lo + hi) >> 1;
        if (offsets[mid] <= start) lo = mid; else hi = mid;
    }
    uint32_t b = lo;
    uint32_t run_begin = offsets[b], next = offsets[b + 1];
    XYZZ acc; xyzz_set_inf(acc);
    bool nonempty = false;
    auto flush = [&](XYZZ* dst) {
        if (nonempty) xyzz_relaxed_normalise(acc); else xyzz_set_inf(acc);
        xyzz_store(dst, acc);
    };
    auto boundary = [&](uint32_t pos) {  // entry `pos` opens a new bucket run: store the finished one
        flush((run_begin >= start) ? &buckets[b] : &partial[2 * t]);
        nonempty = false;
        do { b++; } while (offsets[b + 1] <= pos);
        run_begin = offsets[b]; next = offsets[b + 1];
    };
    for (uint32_t pos = start; pos < end; pos++) {
        const uint32_t ref = sorted[pos];
        Affine q = aff_gather_ro(&table[ref & 0x7fffffffu]);
        if (pos >= next) boundary(pos);
        if (aff_is_inf(q)) continue;  // an identity point in the table (SRS files may hold them)
        fq_cneg_ptx(q.y.l, q.y.l, ref & 0x80000000u);
        if (!nonempty) {
            asm volatile("" ::: "memory");  // keep this path a real branch: nothing of it is worth speculating
            acc.x = q.x; acc.y = q.y; fe_one(acc.zz); fe_one(acc.zzz);
            nonempty = true;
            continue;
        }
        nonempty = xyzz_madd_relaxed_nonempty(acc, q);
    }
    bool complete = (run_begin >= start) && (next <= end);
    flush(complete ? &buckets[b] : (run_begin <= start) ? &partial[2 * t] : &partial[2 * t + 1]);
}

// Buckets whose entries span more than LONG_SPAN chunks (hot buckets: equal scalars, a top window with a
// few possible digits, adversarial blobs) are queued for k_bucket_fix_long instead of being summed by one
// thread: with 4 waves of chunks a single bucket can own thousands of partial sums.
static constexpr uint32_t LONG_SPAN = 48;
static constexpr int LONG_THREADS = 128;
static constexpr uint32_t LONG_BLOCKS = 296;

__global__ void __launch_bounds__(128) k_bucket_fix(const uint32_t* __restrict__ offsets, uint32_t nbuckets, uint32_t chunk,
                                                     XYZZ* __restrict__ buckets, const XYZZ* __restrict__ partial,
                                                     uint32_t* __restrict__ long_count, uint32_t* __restrict__ long_list,
                                                     uint32_t long_cap) {
    uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nbuckets) return;
    uint32_t s = offsets[b], e = offsets[b + 1];
    if (s == e) {
        XYZZ inf; xyzz_set_inf(inf);
        xyzz_store(&buckets[b], inf);
        return;
    }
    uint32_t t_lo = s / chunk, t_hi = (e - 1) / chunk;
    if (t_lo == t_hi) return;  // written directly by k_accumulate
    if (t_hi - t_lo >= LONG_SPAN) {
        uint32_t slot = atomicAdd(long_count, 1u);
        if (slot < long_cap) { long_list[slot] = b; return; }  // (cap = every possible long bucket; never exceeded)
    }
    XYZZ acc; xyzz_set_inf(acc);
    for (uint32_t t = t_lo; t <= t_hi; t++) {
        uint32_t slot = ((uint64_t)s <= (uint64_t)t * chunk) ? 0u : 1u;
        XYZZ v = xyzz_load(&partial[2 * t + slot]);
        xyzz_add(acc, v);
    }
    xyzz_store(&buckets[b], acc);
}

// one block per queued bucket (grid-stride over the queue): strided partial sums per thread, then a
// shared-memory tree
__global__ void __launch_bounds__(LONG_THREADS) k_bucket_fix_long(const uint32_t* __restrict__ offsets, uint32_t chunk,
                                                                   XYZZ* __restrict__ buckets, const XYZZ* __restrict__ partial,
                                                                   const uint32_t* __restrict__ long_count,
                                                                   const uint32_t* __restrict__ long_list, uint32_t long_cap) {
    __shared__ XYZZ sm[LONG_THREADS];
    uint32_t count = *long_count;
    if (count > long_cap) count = long_cap;
    for (uint32_t q = blockIdx.x; q < count; q += gridDim.x) {
        const uint32_t b = long_list[q];
        const uint32_t s = offsets[b], e = offsets[b + 1];
        const uint32_t t_lo = s / chunk, t_hi = (e - 1) / chunk;
        XYZZ acc; xyzz_set_inf(acc);
        for (uint32_t t = t_lo + threadIdx.x; t <= t_hi; t += LONG_THREADS) {
            uint32_t slot = ((uint64_t)s <= (uint64_t)t * chunk) ? 0u : 1u;
            XYZZ v = xyzz_load(&partial[2 * t + slot]);
            xyzz_add(acc, v);
        }
        sm[threadIdx.x] = acc;
        __syncthreads();
        for (uint32_t w = LONG_THREADS / 2; w >= 1; w >>= 1) {
            if (threadIdx.x < w) {
                XYZZ x = sm[threadIdx.x], y = sm[threadIdx.x + w];
                xyzz_add(x, y);
                sm[threadIdx.x] = x;
            }
            __syncthreads();
        }
        if (threadIdx.x == 0) xyzz_store(&buckets[b], sm[0]);
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------
// Quad-cooperative XYZZ arithmetic.  Lane r = lane & 3 of an aligned group of four lanes holds coordinate r
// (0: X, 1: Y, 2: ZZ, 3: ZZZ) of a point.  Every function below must be called by all 32 lanes of the warp
// in convergence (full-mask shuffles); a quad with nothing to add passes the identity (all coordinates 0).
// Exact on all inputs like xyzz_add / xyzz_dbl (ec.cuh), and bit-identical to them: the same formulas, the
// same canonical field results -- only who computes which product differs.  Arguments and results by value
// (registers), the functions out of line: four inlined multiplications each.
// ---------------------------------------------------------------------------------
static constexpr uint32_t FULL = 0xffffffffu;

__device__ __forceinline__ Fq fq_shfl(const Fq& v, int src) {
    Fq r;
#pragma unroll
    for (int i = 0; i < 8; i++) r.l[i] = __shfl_sync(FULL, v.l[i], src);
    return r;
}
__device__ __forceinline__ Fq fq_shfl_xor(const Fq& v, int m) {
    Fq r;
#pragma unroll
    for (int i = 0; i < 8; i++) r.l[i] = __shfl_xor_sync(FULL, v.l[i], m);
    return r;
}
__device__ __forceinline__ Fq fq_sel(bool c, const Fq& a, const Fq& b) {
    Fq r;
#pragma unroll
    for (int i = 0; i < 8; i++) r.l[i] = c ? a.l[i] : b.l[i];
    return r;
}

// a = 2a   (EFD dbl-2008-s-1, a = 0): three multiplication steps
__device__ __noinline__ Fq quad_dbl(Fq a) {
    const int lane = threadIdx.x & 31, r = lane & 3, base = lane & ~3;
    const bool z = fe_is_zero(a);
    // (two statements: `a || b` would let the lanes of an identity quad skip the second full-mask shuffle -- a deadlock)
    const bool zz0 = __shfl_sync(FULL, z, base + 2);
    const bool y0 = __shfl_sync(FULL, z, base + 1);
    const bool inf = zz0 || y0;
    Fq u; fe_dbl(u, a);                                   // lane 1: U = 2Y
    const Fq s1 = fq_sel(r == 1, u, a);
    Fq m1; fe_mul(m1, s1, s1);                            // lane 0: X^2, lane 1: V = U^2
    const Fq v = fq_shfl(m1, base + 1);
    Fq t = fq_shfl(m1, base);                             // X^2 for lane 3
    Fq M; fe_dbl(M, t); fe_add(M, M, t);                  // 3 X^2 (used in lanes 0 and 3)
    const Fq x2 = fq_sel(r == 3, M, s1), y2 = fq_sel(r == 3, M, v);
    Fq m2; fe_mul(m2, x2, y2);                            // lane 0: S = X V, lane 1: W = U V, lane 2: ZZ3 = ZZ V, lane 3: M^2
    const Fq w = fq_shfl(m2, base + 1);
    const Fq mm = fq_shfl(m2, base + 3);
    Fq x3; fe_sub(x3, mm, m2); fe_sub(x3, x3, m2);        // lane 0: X3 = M^2 - 2S
    Fq smx; fe_sub(smx, m2, x3);                          // lane 0: S - X3
    const Fq x4 = fq_sel(r == 0, M, a), y4 = fq_sel(r == 0, smx, w);
    Fq m3; fe_mul(m3, x4, y4);                            // lane 0: M (S - X3), lane 1: Y W, lane 3: ZZZ3 = ZZZ W
    const Fq t1 = fq_shfl(m3, base);
    Fq y3; fe_sub(y3, t1, m3);                            // lane 1: Y3
    Fq res = fq_sel(r == 0, x3, fq_sel(r == 1, y3, fq_sel(r == 2, m2, m3)));
    if (inf) fe_zero(res);
    return res;
}

// a += b   (EFD add-2008-s): four multiplication steps
__device__ __noinline__ Fq quad_add(Fq a, Fq b) {
    const int lane = threadIdx.x & 31, r = lane & 3, base = lane & ~3;
    const bool inf1 = __shfl_sync(FULL, fe_is_zero(a), base + 2);
    const bool inf2 = __shfl_sync(FULL, fe_is_zero(b), base + 2);
    const Fq o2 = fq_shfl_xor(b, 2);                      // lane 0: ZZ2, 1: ZZZ2, 2: X2, 3: Y2
    Fq m1; fe_mul(m1, a, o2);                             // lane 0: U1, 1: S1, 2: U2, 3: S2
    const Fq pt = fq_shfl_xor(m1, 2);
    Fq d; fe_sub(d, fq_sel(r < 2, pt, m1), fq_sel(r < 2, m1, pt));  // lanes 0, 2: P = U2 - U1; lanes 1, 3: R = S2 - S1
    const bool dz = fe_is_zero(d);
    const bool pz = __shfl_sync(FULL, dz, base), rz = __shfl_sync(FULL, dz, base + 1);
    Fq m2; fe_mul(m2, fq_sel(r < 2, d, a), fq_sel(r < 2, d, b));    // lane 0: PP, 1: R^2, 2: ZZ1 ZZ2, 3: ZZZ1 ZZZ2
    const Fq pp = fq_shfl(m2, base);
    const Fq u1 = fq_shfl(m1, base);
    Fq m3; fe_mul(m3, fq_sel(r == 0, d, fq_sel(r == 1, u1, m2)), pp);  // lane 0: PPP, 1: Q = U1 PP, 2: ZZ3
    const Fq ppp = fq_shfl(m3, base);
    Fq x3; fe_sub(x3, m2, ppp); fe_sub(x3, x3, m3); fe_sub(x3, x3, m3);  // lane 1: X3 = R^2 - PPP - 2Q
    Fq qmx; fe_sub(qmx, m3, x3);                                          // lane 1: Q - X3
    const Fq s1 = fq_shfl(m1, base + 1);
    Fq m4; fe_mul(m4, fq_sel(r == 0, s1, fq_sel(r == 1, d, m2)), fq_sel(r == 1, qmx, ppp));  // lane 0: S1 PPP, 1: R (Q - X3), 3: ZZZ3
    const Fq t2 = fq_shfl(m4, base);
    Fq y3; fe_sub(y3, m4, t2);                            // lane 1: Y3
    const Fq x3b = fq_shfl(x3, base + 1);
    Fq res = fq_sel(r == 0, x3b, fq_sel(r == 1, y3, fq_sel(r == 2, m3, m4)));
    const bool same_x = !inf1 && !inf2 && pz;
    if (__any_sync(FULL, same_x && rz)) {                 // P + P somewhere in the warp: the doubling, for everyone
        const Fq dd = quad_dbl(b);
        if (same_x && rz) res = dd;
    }
    if (same_x && !rz) fe_zero(res);                      // P + (-P)
    if (inf2) res = a;
    else if (inf1) res = b;
    return res;
}

__device__ __forceinline__ Fq quad_load(const XYZZ* p) {  // this lane's coordinate
    return fe_load(&p->x + (threadIdx.x & 3));
}
__device__ __forceinline__ void quad_store(XYZZ* p, const Fq& v) { fe_store(&p->x + (threadIdx.x & 3), v); }

// Sum over the whole block of every quad's point; valid in the first quad of warp 0.  smem: one XYZZ per warp.
template <int WARPS>
__device__ __forceinline__ void block_quad_sum(Fq& acc, XYZZ* smem) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll 1
    for (int m = 4; m < 32; m <<= 1) {
        Fq o = fq_shfl_xor(acc, m);
        acc = quad_add(acc, o);
    }
    if (WARPS == 1) return;
    if (lane < 4) fe_store(&smem[wid].x + lane, acc);
    __syncthreads();
    if (wid == 0) {
        const int q = lane >> 2;
        if (q < WARPS) acc = fe_load(&smem[q].x + (lane & 3)); else fe_zero(acc);
#pragma unroll 1
        for (int m = 4; m < 4 * WARPS; m <<= 1) {
            Fq o = fq_shfl_xor(acc, m);
            acc = quad_add(acc, o);
        }
    }
}

// The buckets of one set as a matrix of H = 2^hb rows by A = 2^ab columns (bucket k = A h + l).
// Line L < H is row L, line H + l is column l.  One block of LINE_THREADS per line and set: every quad sums
// the elements q, q + 32, ... of its line, then the 32 quads are summed.  line_sums[set * (H + A) + L].
static constexpr int LINE_THREADS = 128;
__global__ void __launch_bounds__(LINE_THREADS) k_reduce_lines(const XYZZ* __restrict__ buckets, int ab, int hb,
                                                                XYZZ* __restrict__ line_sums) {
    __shared__ XYZZ sm[LINE_THREADS / 32];
    const uint32_t A = 1u << ab, H = 1u << hb;
    const uint32_t L = blockIdx.x, set = blockIdx.y;
    const XYZZ* src = buckets + (size_t)set * ((size_t)A << hb);
    uint32_t len, stride;
    if (L < H) { src += (size_t)L << ab; len = A; stride = 1; }
    else { src += L - H; len = H; stride = A; }
    const uint32_t q = threadIdx.x >> 2;
    Fq acc; fe_zero(acc);
    if (q < len) acc = quad_load(src + (size_t)q * stride);
#pragma unroll 1
    for (uint32_t e0 = LINE_THREADS / 4; e0 < len; e0 += LINE_THREADS / 4) {
        Fq v; fe_zero(v);
        if (e0 + q < len) v = quad_load(src + (size_t)(e0 + q) * stride);
        acc = quad_add(acc, v);
    }
    block_quad_sum<LINE_THREADS / 32>(acc, sm);
    if (threadIdx.x < 4) quad_store(&line_sums[(size_t)set * (H + A) + L], acc);
}

// Group g < ab:  T_g = sum of the column sums C_l, l <= A - 2, with bit g of (l + 1) set      (weight 2^g)
// group ab + j:  T   = sum of the row sums R_h with bit j of h set                             (weight 2^(ab + j))
// and group ab also takes C_{A-1} (l + 1 = A).  sum_k (k + 1) B_k = sum_g 2^g T_g; the block doubles its
// T_g g times.  group_sums[set * ngroups + g].
static constexpr int GROUP_THREADS = 128;
__global__ void __launch_bounds__(GROUP_THREADS) k_reduce_groups(const XYZZ* __restrict__ line_sums, int ab, int hb, int ngroups,
                                                                  XYZZ* __restrict__ group_sums) {
    __shared__ XYZZ sm[GROUP_THREADS / 32];
    const uint32_t A = 1u << ab, H = 1u << hb;
    const uint32_t g = blockIdx.x, set = blockIdx.y;
    const XYZZ* rows = line_sums + (size_t)set * (H + A);
    const XYZZ* cols = rows + H;
    const uint32_t q = threadIdx.x >> 2, Q = GROUP_THREADS / 4;
    Fq acc; fe_zero(acc);
    if ((int)g < ab) {
        // (l + 1) with bit g set, l + 1 < A: the j-th such value is ((j >> g) << (g + 1)) | (1 << g) | (j & ((1 << g) - 1))
        const uint32_t cnt = A >> 1;
#pragma unroll 1
        for (uint32_t j0 = 0; j0 < cnt; j0 += Q) {
            const uint32_t j = j0 + q;
            Fq v; fe_zero(v);
            if (j < cnt) {
                uint32_t m = ((j >> g) << (g + 1)) | (1u << g) | (j & ((1u << g) - 1u));
                v = quad_load(cols + (m - 1));
            }
            acc = quad_add(acc, v);
        }
    } else {
        const uint32_t jb = g - ab;  // bit of h
        const uint32_t cnt = hb > 0 ? (H >> 1) : 0;
#pragma unroll 1
        for (uint32_t j0 = 0; j0 < cnt; j0 += Q) {
            const uint32_t j = j0 + q;
            Fq v; fe_zero(v);
            if (j < cnt) {
                uint32_t h = ((j >> jb) << (jb + 1)) | (1u << jb) | (j & ((1u << jb) - 1u));
                v = quad_load(rows + h);
            }
            acc = quad_add(acc, v);
        }
        if ((int)g == ab) {
            Fq v; fe_zero(v);
            if (q == 0) v = quad_load(cols + (A - 1));
            acc = quad_add(acc, v);
        }
    }
    block_quad_sum<GROUP_THREADS / 32>(acc, sm);
    if (threadIdx.x < 32) {  // warp 0 (uniform): g doublings of the total held by its first quad
#pragma unroll 1
        for (uint32_t i = 0; i < g; i++) acc = quad_dbl(acc);
        if (threadIdx.x < 4) quad_store(&group_sums[(size_t)set * ngroups + g], acc);
    }
}

// one warp per set: out[set] = sum of its ngroups (<= 32) group results
__global__ void __launch_bounds__(32) k_reduce_final(const XYZZ* __restrict__ group_sums, int ngroups, XYZZ* __restrict__ out) {
    const uint32_t set = blockIdx.x, q = threadIdx.x >> 2;
    const XYZZ* src = group_sums + (size_t)set * ngroups;
    Fq acc; fe_zero(acc);
    if ((int)q < ngroups) acc = quad_load(src + q);
#pragma unroll 1
    for (int e0 = 8; e0 < ngroups; e0 += 8) {
        Fq v; fe_zero(v);
        if (e0 + (int)q < ngroups) v = quad_load(src + e0 + q);
        acc = quad_add(acc, v);
    }
    block_quad_sum<1>(acc, nullptr);
    if (threadIdx.x < 4) quad_store(&out[set], acc);
}

// ---------------------------------------------------------------------------------
static std::atomic<int> g_acc_waves{4};
static std::atomic<int> g_debug_sync{0};  // option "msm_debug_sync": synchronise and report after every kernel of an MSM
void msm_set_debug_sync(int on) { g_debug_sync.store(on); }
#define KZ_DBG(name)                                                                                         \
    do {                                                                                                     \
        if (g_debug_sync.load()) {                                                                           \
            cudaError_t e1_ = cudaStreamSynchronize(st), e2_ = cudaStreamSynchronize(sa);                    \
            fprintf(stderr, "[msm] %s: %s / %s\n", name, cudaGetErrorString(e1_), cudaGetErrorString(e2_)); \
        }                                                                                                    \
    } while (0)
void msm_set_acc_waves(int waves) { g_acc_waves.store(waves < 1 ? 1 : (waves > 64 ? 64 : waves)); }

MsmPlan msm_make_plan(uint32_t n, int c, bool fixed_base, uint32_t table_stride, uint32_t base_offset, uint32_t batch) {
    MsmPlan p;
    p.c = c;
    p.W = window_count(c);
    p.batch_n = (fixed_base && batch > 0) ? n / batch : 0;  // `batch` independent MSMs over the same table, one bucket set each
    p.sets = fixed_base ? (p.batch_n ? (int)batch : 1) : p.W;
    p.nbuckets = (uint32_t)p.sets << (c - 1);
    p.n = n;
    p.table_stride = fixed_base ? table_stride : 0;
    p.base_offset = fixed_base ? base_offset : 0;
    uint64_t entries = (uint64_t)n * p.W;
    // Fixed-size chunks of the sorted list, 4 waves of 4 blocks of 128 threads per SM: measured at 2^19 points
    // (profiles/r02_variant_sweep.txt) the kernel itself is fastest at 4 waves (1.133 ms; 2: 1.185, 1: 1.250) and
    // so is the blob pipeline, although fewer waves would leave k_bucket_fix fewer partial sums.
    uint64_t max_threads = (uint64_t)SM_COUNT * 512 * (uint64_t)g_acc_waves.load();
    uint64_t want = (entries + 15) / 16;
    if (want < 1) want = 1;
    p.acc_threads = (uint32_t)(want < max_threads ? want : max_threads);
    p.chunk = (uint32_t)((entries + p.acc_threads - 1) / p.acc_threads);
    if (p.chunk == 0) p.chunk = 1;
    // bucket matrix of one set: 2^(c-1) = H x A, A >= H
    p.a_bits = c / 2;            // ceil((c - 1) / 2)
    p.h_bits = (c - 1) - p.a_bits;
    p.ngroups = p.a_bits + (p.h_bits > 0 ? p.h_bits : 1);
    return p;
}

static size_t align_up(size_t x) { return (x + 255) & ~(size_t)255; }
static size_t lines_per_set(const MsmPlan& p) { return ((size_t)1 << p.a_bits) + ((size_t)1 << p.h_bits); }

size_t msm_workspace_bytes(const MsmPlan& p) {
    size_t b = 0;
    b += align_up((size_t)p.n * sizeof(Fr));
    b += align_up(((size_t)p.nbuckets + 1) * 4);
    b += align_up((size_t)p.nbuckets * 4);
    b += align_up((size_t)p.n * p.W * 4);
    b += align_up((size_t)p.nbuckets * sizeof(XYZZ));
    b += align_up((size_t)2 * p.acc_threads * sizeof(XYZZ));
    b += align_up(lines_per_set(p) * p.sets * sizeof(XYZZ));
    b += align_up((size_t)p.ngroups * p.sets * sizeof(XYZZ));
    b += align_up((size_t)p.sets * sizeof(XYZZ));
    b += align_up(1024 * 4);  // scan tile totals
    b += align_up(((size_t)p.acc_threads / LONG_SPAN + 8) * 4);  // long-bucket queue (+ its counter)
    return b;
}

void msm_workspace_carve(const MsmPlan& p, void* base, MsmWorkspace* ws) {
    char* c = (char*)base;
    ws->canon = (Fr*)c; c += align_up((size_t)p.n * sizeof(Fr));
    ws->hist = (uint32_t*)c; c += align_up(((size_t)p.nbuckets + 1) * 4);
    ws->cursor = (uint32_t*)c; c += align_up((size_t)p.nbuckets * 4);
    ws->sorted = (uint32_t*)c; c += align_up((size_t)p.n * p.W * 4);
    ws->buckets = (XYZZ*)c; c += align_up((size_t)p.nbuckets * sizeof(XYZZ));
    ws->partial = (XYZZ*)c; c += align_up((size_t)2 * p.acc_threads * sizeof(XYZZ));
    ws->line_sums = (XYZZ*)c; c += align_up(lines_per_set(p) * p.sets * sizeof(XYZZ));
    ws->group_sums = (XYZZ*)c; c += align_up((size_t)p.ngroups * p.sets * sizeof(XYZZ));
    ws->set_sums = (XYZZ*)c; c += align_up((size_t)p.sets * sizeof(XYZZ));
    ws->tile_tot = (uint32_t*)c; c += align_up(1024 * 4);
    ws->long_list = (uint32_t*)c;
}

// dst[k] += src[k]: bucket sums of a further point sub-range folded into the running totals (msm_launch_buckets
// of the chunks of one large MSM whose scalars arrive piecewise, capi.cu msm_srs_host_pipelined)
__global__ void __launch_bounds__(128) k_merge_buckets(XYZZ* __restrict__ dst, const XYZZ* __restrict__ src, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    XYZZ b = xyzz_load(&src[i]);
    if (xyzz_is_inf(b)) return;
    XYZZ a = xyzz_load(&dst[i]);
    xyzz_add(a, b);
    xyzz_store(&dst[i], a);
}
void msm_merge_buckets(XYZZ* dst, const XYZZ* src, uint32_t nbuckets, cudaStream_t st) {
    k_merge_buckets<<<(nbuckets + 127) / 128, 128, 0, st>>>(dst, src, nbuckets);
    g_launch_count++;
}

// sort + accumulate + stitch: afterwards ws.buckets holds the sum of every bucket (identity where empty)
void msm_launch_buckets(const MsmPlan& p, const MsmWorkspace& ws, const MsmScalars& scalars, const Affine* table,
                        const MsmStreams& s) {
    const cudaStream_t st = s.st;
    const bool split = s.st_acc && s.fork && s.join;
    const cudaStream_t sa = split ? s.st_acc : st;
    cudaMemsetAsync(ws.hist, 0, ((size_t)p.nbuckets + 1) * 4, st);
    const uint32_t gb = (p.n + 255) / 256;
    if (p.n) {
        if (scalars.blob) k_digits_hist_blob<<<gb, 256, 0, st>>>(scalars.blob, scalars.blob_len, p, ws.canon, ws.hist);
        else k_digits_hist<<<gb, 256, 0, st>>>(scalars.mont, p, ws.canon, ws.hist);
        g_launch_count += 2;
    }
    {
        uint32_t ntiles = (p.nbuckets + SCAN_TILE - 1) / SCAN_TILE;
        k_scan_tiles<<<ntiles, SCAN_THREADS, 0, st>>>(ws.hist, ws.cursor, p.nbuckets, ws.tile_tot, ntiles == 1);
        g_launch_count++;
        if (ntiles > 1) {
            k_scan_tile_totals<<<1, SCAN_THREADS, 0, st>>>(ws.tile_tot, ntiles, ws.hist, p.nbuckets);
            k_scan_add<<<(p.nbuckets + 255) / 256, 256, 0, st>>>(ws.hist, ws.cursor, p.nbuckets, ws.tile_tot);
            g_launch_count += 2;
        }
    }
    if (p.n) k_scatter<<<gb, 256, 0, st>>>(ws.canon, p, ws.cursor, ws.sorted);
    KZ_DBG("sort");
    if (split) { cudaEventRecord(s.fork, st); cudaStreamWaitEvent(sa, s.fork, 0); }
    if (s.acc_begin) cudaEventRecord(s.acc_begin, sa);
    k_accumulate<<<(p.acc_threads + 127) / 128, 128, 0, sa>>>(ws.sorted, ws.hist, table, p.nbuckets, p.acc_threads, p.chunk,
                                                             ws.buckets, ws.partial);
    if (s.acc_end) cudaEventRecord(s.acc_end, sa);
    if (split) { cudaEventRecord(s.join, sa); cudaStreamWaitEvent(st, s.join, 0); }
    KZ_DBG("accumulate");
    {
        const uint32_t long_cap = p.acc_threads / LONG_SPAN + 4;  // a long bucket owns >= LONG_SPAN chunks
        uint32_t* long_count = ws.long_list;                      // [0] = counter, [1..] = queue
        cudaMemsetAsync(long_count, 0, 4, st);
        k_bucket_fix<<<(p.nbuckets + 127) / 128, 128, 0, st>>>(ws.hist, p.nbuckets, p.chunk, ws.buckets, ws.partial,
                                                                long_count, ws.long_list + 1, long_cap);
        k_bucket_fix_long<<<LONG_BLOCKS, LONG_THREADS, 0, st>>>(ws.hist, p.chunk, ws.buckets, ws.partial, long_count,
                                                                  ws.long_list + 1, long_cap);
    }
    KZ_DBG("bucket_fix");
    g_launch_count += 3;  // accumulate, bucket_fix, bucket_fix_long
}

// bucket sums -> ws.set_sums (one XYZZ point per bucket set)
void msm_launch_reduce(const MsmPlan& p, const MsmWorkspace& ws, const XYZZ* buckets, cudaStream_t st) {
    cudaStream_t sa = st;
    k_reduce_lines<<<dim3((unsigned)lines_per_set(p), (unsigned)p.sets), LINE_THREADS, 0, st>>>(buckets, p.a_bits, p.h_bits, ws.line_sums);
    KZ_DBG("reduce_lines");
    k_reduce_groups<<<dim3((unsigned)p.ngroups, (unsigned)p.sets), GROUP_THREADS, 0, st>>>(ws.line_sums, p.a_bits, p.h_bits, p.ngroups,
                                                                                          ws.group_sums);
    KZ_DBG("reduce_groups");
    k_reduce_final<<<p.sets, 32, 0, st>>>(ws.group_sums, p.ngroups, ws.set_sums);
    KZ_DBG("reduce_final");
    g_launch_count += 3;  // reduce_lines, reduce_groups, reduce_final
}

}  // namespace kzgb
