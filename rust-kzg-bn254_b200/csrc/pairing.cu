// The pairing check of verify_proof (verifier/src/verify.rs:10-75) for a batch of openings (C_i, pi_i, z_i, y_i), one
// thread per opening: the bool of kzgb_verify_proofs and kzgb_verify_blob_proofs{,_dev}.
//
// e(C - [y]G1, G2) == e(pi, [tau - z]G2) is, by bilinearity, the same bool as
//   e(C - [y]G1 + [z]pi, G2) e(-pi, [tau]G2) == 1,
// where both G2 arguments are fixed per context.  So the host precomputes the Miller-loop lines of G2 and of [tau]G2
// once (pairing.cuh g2_lines), and the device runs, per opening and with no host round trip:
//   k_pairing_prep   A = C - [y]G1 + [z]pi, B = -pi, and whether [z]G2 == [tau]G2 (the reference's "evaluation point
//                    equals trusted setup secret", verify.rs:55-59), over fixed-base window tables of G1 and G2
//   k_miller         the two-pair Miller loop over the precomputed lines
//   k_final_exp      the final exponentiation and the comparison with 1
#include <memory>
#include <mutex>

#include "ctx.hpp"

namespace kzgb {

namespace {

// term(index into a window table of j 16^w P at [8 w + j - 1], negate) for the 64 signed 4-bit digits of a canonical
// k < 2^254 -- the digits of k + 0x88..8 minus 8, as k_commit_minus_value (verify.cu) reads them
template <class F>
KZ_D void for_w4_digits(const Fr& k, F term) {
    uint64_t carry = 0;
    for (int w = 0; w < 8; w++) {
        carry += (uint64_t)k.l[w] + 0x88888888u;
        const uint32_t K = (uint32_t)carry;
        carry >>= 32;
        for (int q = 0; q < 8; q++) {
            const int v = (int)((K >> (4 * q)) & 15u) - 8;
            if (v) term(8 * (8 * w + q) + (v > 0 ? v : -v) - 1, v < 0);
        }
    }
}

KZ_D Fq2 fq2_load_ro(const Fq2* p) {
    Fq2 r;
    r.c0 = fe_load_ro(&p->c0);
    r.c1 = fe_load_ro(&p->c1);
    return r;
}

// AB[2 i] = C_i - [y_i]G1 + [z_i]pi_i, AB[2 i + 1] = -pi_i (affine, the identity as (0, 0)); flag[i] = 2 if
// [z_i]G2 == [tau]G2, else 0
__global__ void __launch_bounds__(64) k_pairing_prep(const Affine* __restrict__ C, const Affine* __restrict__ Pi,
                                                     const Fr* __restrict__ z, const Fr* __restrict__ y,
                                                     const Affine* __restrict__ gtab, const PairingTables* __restrict__ tab,
                                                     Affine* __restrict__ AB, uint8_t* __restrict__ flag, uint32_t count) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const Affine pi = aff_load_ro(&Pi[i]);
    Fr zc = fe_load_ro(&z[i]);
    fe_from_mont(zc, zc);
    Fr yn = fe_load_ro(&y[i]);
    fe_neg(yn, yn);
    fe_from_mont(yn, yn);
    XYZZ acc, p;
    xyzz_from_affine(p, pi);
    xyzz_mul_scalar_w4(acc, p, zc);
    for_w4_digits(yn, [&](int idx, bool neg) {
        Affine t = aff_load_ro(&gtab[idx]);
        if (neg) fe_neg(t.y, t.y);
        xyzz_madd(acc, t);
    });
    xyzz_madd(acc, aff_load_ro(&C[i]));
    Affine a, b = pi;
    xyzz_to_affine(a, acc);
    fe_neg(b.y, pi.y);
    aff_store(&AB[2 * i], a);
    aff_store(&AB[2 * i + 1], b);

    G2XYZZ g;
    g2_xyzz_set_inf(g);
    for_w4_digits(zc, [&](int idx, bool neg) {
        G2Affine t;
        t.x = fq2_load_ro(&tab->g2tab[idx].x);
        t.y = fq2_load_ro(&tab->g2tab[idx].y);
        if (neg) fq2_neg(t.y, t.y);
        g2_xyzz_madd(g, t);
    });
    G2Affine tau;
    tau.x = fq2_load_ro(&tab->tau.x);
    tau.y = fq2_load_ro(&tab->tau.y);
    flag[i] = g2_xyzz_eq_affine(g, tau) ? 2 : 0;
}

// f[i] = f_{6x+2,G2}(A_i) f_{6x+2,[tau]G2}(B_i)
__global__ void __launch_bounds__(64) k_miller(const Affine* __restrict__ AB, const PairingTables* __restrict__ tab,
                                               Fq12* __restrict__ f_out, uint32_t count) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const Affine a = aff_load_ro(&AB[2 * i]), b = aff_load_ro(&AB[2 * i + 1]);
    Fq nxa, nxb;
    fe_neg(nxa, a.x);
    fe_neg(nxb, b.x);
    Fq12 f;
    miller_loop_2(f, nxa, a.y, aff_is_inf(a), nxb, b.y, aff_is_inf(b), [&](int k, int s) {
        Line l;
        l.lam = fq2_load_ro(&tab->lines[k][s].lam);
        l.c = fq2_load_ro(&tab->lines[k][s].c);
        return l;
    });
    f_out[i] = f;
}

// flag[i] = 1 if f[i]^(m (p^12 - 1) / r) == 1, else 0; entries flagged 2 by k_pairing_prep keep their flag
__global__ void __launch_bounds__(64) k_final_exp(const Fq12* __restrict__ f, uint8_t* __restrict__ flag, uint32_t count) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count || flag[i] == 2) return;
    Fq12 r;
    fq12_final_exp(r, f[i]);
    flag[i] = fq12_is_one(r) ? 1 : 0;
}

// the parts of PairingTables that do not depend on [tau]G2: the generator's lines and window multiples
const PairingTables* pairing_fixed_tables() {
    static std::unique_ptr<PairingTables> t(new PairingTables());
    static std::once_flag once;
    std::call_once(once, [] {
        G2Affine g;
        const uint32_t w[32] = KZ_G2_GEN;
        fq2_set(g.x, w);
        fq2_set(g.y, w + 16);
        g2_lines(t->lines[0], g);
        G2XYZZ base;
        base.x = g.x; base.y = g.y; fq2_one(base.zz); fq2_one(base.zzz);
        for (int w4 = 0; w4 < 64; w4++) {
            G2Affine b;
            g2_xyzz_to_affine(b, base);
            G2XYZZ m = base;
            for (int d = 0; d < 8; d++) {
                if (d) g2_xyzz_madd(m, b);
                g2_xyzz_to_affine(t->g2tab[8 * w4 + d], m);
            }
            for (int s = 0; s < 4; s++) g2_xyzz_dbl(base, base);
        }
    });
    return t.get();
}

// the 4 little-endian words at w hold a value below p
bool fq_words_reduced(const uint64_t* w) {
    uint32_t p[8];
    FeConst<FQ>::mod(p);
    for (int k = 7; k >= 0; k--) {
        const uint32_t x = (uint32_t)(w[k / 2] >> (32 * (k & 1)));
        if (x != p[k]) return x < p[k];
    }
    return false;
}

}  // namespace

G2Affine default_g2_tau() {
    G2Affine q;
    const uint32_t w[32] = KZ_G2_TAU;
    fq2_set(q.x, w);
    fq2_set(q.y, w + 16);
    return q;
}

int ensure_pairing_tables(kzgb_ctx* c) {
    if (c->pair_tab && !c->pair_stale) return KZGB_OK;
    std::unique_ptr<PairingTables> h(new PairingTables(*pairing_fixed_tables()));
    h->tau = c->g2_tau;
    g2_lines(h->lines[1], c->g2_tau);
    if (!c->pair_tab) CK(c, dev_alloc(c->pair_tab, sizeof(PairingTables)));
    CK(c, cudaMemcpy(c->pair_tab.get(), h.get(), sizeof(PairingTables), cudaMemcpyHostToDevice));
    c->pair_stale = false;
    return KZGB_OK;
}

size_t pairing_workspace_bytes(uint32_t count) {
    return (size_t)count * (2 * sizeof(Affine) + sizeof(Fq12) + 1);
}

uint8_t* pairing_check_launch(const Affine* C, const Affine* Pi, const Fr* z_mont, const Fr* y_mont, const Affine* gen_table,
                              const PairingTables* tab, void* ws, uint32_t count, cudaStream_t st) {
    Fq12* f = (Fq12*)ws;
    Affine* AB = (Affine*)(f + count);
    uint8_t* flag = (uint8_t*)(AB + 2 * count);
    if (!count) return flag;
    const uint32_t blocks = (count + 63) / 64;
    k_pairing_prep<<<blocks, 64, 0, st>>>(C, Pi, z_mont, y_mont, gen_table, tab, AB, flag, count);
    k_miller<<<blocks, 64, 0, st>>>(AB, tab, f, count);
    k_final_exp<<<blocks, 64, 0, st>>>(f, flag, count);
    g_launch_count += 3;
    return flag;
}

// flags of pairing_check_launch -> ok[], or the error of the lowest opening whose z is tau (ok untouched)
int pairing_finish(kzgb_ctx* c, const std::vector<uint8_t>& flags, uint8_t* ok) {
    for (size_t i = 0; i < flags.size(); i++)
        if (flags[i] == 2) return fail(c, KZGB_ERR_GENERIC, "Evaluation point equals trusted setup secret");
    memcpy(ok, flags.data(), flags.size());
    return KZGB_OK;
}

}  // namespace kzgb

using namespace kzgb;

extern "C" {

int kzgb_set_g2_tau(kzgb_ctx* c, const uint64_t xy[16]) {
    Guard g(c);
    G2Affine q = default_g2_tau();
    if (xy) {
        bool ok = true;
        for (int k = 0; k < 4; k++) ok = ok && fq_words_reduced(xy + 4 * k);
        if (ok) {
            memcpy(&q, xy, sizeof(q));
            ok = g2_on_curve(q);  // the identity (all zero) is not on the twist
        }
        if (ok) {  // order r: [r] q == O
            uint32_t r[8];
            FeConst<FR>::mod(r);
            G2XYZZ acc;
            g2_xyzz_set_inf(acc);
            for (int b = 253; b >= 0; b--) {
                g2_xyzz_dbl(acc, acc);
                if ((r[b / 32] >> (b % 32)) & 1) g2_xyzz_madd(acc, q);
            }
            ok = g2_xyzz_is_inf(acc);
        }
        if (!ok) return fail(c, KZGB_ERR_NOT_ON_CURVE, "Invalid trusted setup: G2_TAU not on curve");
    }
    c->g2_tau = q;
    c->pair_stale = true;
    return KZGB_OK;
}

}  // extern "C"
