// commit_minus_value = C - [y] G1 (verifier/src/verify.rs:37-42) for a batch of openings: the G1 step of
// kzgb_verify_blob_proofs_g1 after the batched challenges and evaluations.  One thread per opening; the host form is
// kzgb_verify_proof_g1 (capi.cu), and affine coordinates are unique, so both give the same words.
#include <mutex>

#include "kzgb_internal.hpp"

namespace kzgb {

// The signed 4-bit windows of xyzz_mul_scalar_w4 with the generator's window multiples precomputed: k = sum (e_i - 8) 16^i
// over the 64 nibbles e_i of k + 0x88..8, and term i is +-tab[8 i + |e_i - 8| - 1] -- 64 mixed additions, no doubling.
// out[i] = C[i] + [-y[i]] G  (y Montgomery; the identity comes out as (0, 0))
__global__ void __launch_bounds__(64) k_commit_minus_value(const Affine* __restrict__ C, const Fr* __restrict__ y,
                                                           const Affine* __restrict__ gtab, Affine* __restrict__ out,
                                                           uint32_t count) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    Fr k = fe_load_ro(&y[i]);
    fe_neg(k, k);
    fe_from_mont(k, k);  // canonical, < r < 2^254: the nibble sum below cannot carry out of 256 bits
    uint64_t carry = 0;
    XYZZ acc; xyzz_set_inf(acc);
    for (int w = 0; w < 8; w++) {
        carry += (uint64_t)k.l[w] + 0x88888888u;
        const uint32_t K = (uint32_t)carry;
        carry >>= 32;
        for (int q = 0; q < 8; q++) {
            const int v = (int)((K >> (4 * q)) & 15u) - 8;
            if (v == 0) continue;
            Affine t = aff_load_ro(&gtab[8 * (8 * w + q) + (v > 0 ? v : -v) - 1]);
            if (v < 0) fe_neg(t.y, t.y);
            xyzz_madd(acc, t);
        }
    }
    xyzz_madd(acc, aff_load_ro(&C[i]));
    Affine r;
    xyzz_to_affine(r, acc);
    aff_store(&out[i], r);
}

const Affine* generator_window_table() {
    static Affine tab[GEN_TABLE_POINTS];
    static std::once_flag once;
    std::call_once(once, [] {
        XYZZ base;
        Affine g;
        fe_one(g.x); fe_dbl(g.y, g.x);  // G1 generator (1, 2)
        xyzz_from_affine(base, g);
        for (int w = 0; w < 64; w++) {
            XYZZ m = base;
            for (int d = 0; d < 8; d++) {
                if (d) xyzz_add(m, base);
                xyzz_to_affine(tab[8 * w + d], m);
            }
            for (int s = 0; s < 4; s++) xyzz_dbl(base, base);
        }
    });
    return tab;
}

void commit_minus_value_launch(const Affine* C, const Fr* y_mont, const Affine* gen_table, Affine* out, uint32_t count,
                               cudaStream_t st) {
    if (!count) return;
    k_commit_minus_value<<<(count + 63) / 64, 64, 0, st>>>(C, y_mont, gen_table, out, count);
    g_launch_count++;
}

}  // namespace kzgb
