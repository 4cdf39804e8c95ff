// BN254 G1 (y^2 = x^3 + 3 over Fq; reference primitives/src/helpers.rs:202) in
// affine and extended-Jacobian "XYZZ" coordinates (x = X/ZZ, y = Y/ZZZ, ZZ^3 = ZZZ^2).
// XYZZ is what the bucket accumulators use: a mixed addition is 8M + 2S with no
// inversion, and the exceptional cases (identity, P + P, P + (-P)) are handled exactly,
// because results must be bit-identical to the reference's arkworks path, not
// probabilistically right.
//
// Conventions: affine identity = (0, 0) (not on the curve, so it is a safe sentinel);
// XYZZ identity = ZZ == 0.
#pragma once
#include "field.cuh"

namespace kzgb {

struct alignas(16) Affine {
    Fq x, y;
};
struct alignas(16) XYZZ {
    Fq x, y, zz, zzz;
};

KZ_HD bool aff_is_inf(const Affine& p) { return fe_is_zero(p.x) && fe_is_zero(p.y); }
KZ_HD void aff_set_inf(Affine& p) { fe_zero(p.x); fe_zero(p.y); }
KZ_HD bool xyzz_is_inf(const XYZZ& p) { return fe_is_zero(p.zz); }
KZ_HD void xyzz_set_inf(XYZZ& p) { fe_zero(p.x); fe_zero(p.y); fe_zero(p.zz); fe_zero(p.zzz); }
KZ_HD void xyzz_from_affine(XYZZ& r, const Affine& p) {
    if (aff_is_inf(p)) { xyzz_set_inf(r); return; }
    r.x = p.x; r.y = p.y; fe_one(r.zz); fe_one(r.zzz);
}
KZ_HD void xyzz_neg(XYZZ& r, const XYZZ& p) { r = p; fe_neg(r.y, p.y); }

// r = 2 * (affine p)          (EFD mdbl-2008-s-1, a = 0)
KZ_HD void xyzz_dbl_affine(XYZZ& r, const Affine& p) {
    if (aff_is_inf(p) || fe_is_zero(p.y)) { xyzz_set_inf(r); return; }
    Fq U, V, W, S, M, t;
    fe_dbl(U, p.y);
    fe_sqr(V, U);
    fe_mul(W, U, V);
    fe_mul(S, p.x, V);
    fe_sqr(t, p.x);
    fe_dbl(M, t); fe_add(M, M, t);  // 3 x^2
    fe_sqr(r.x, M);
    fe_sub(r.x, r.x, S); fe_sub(r.x, r.x, S);
    fe_sub(t, S, r.x);
    fe_mul2sub(r.y, M, t, W, p.y);  // M (S - X3) - W y, one reduction
    r.zz = V;
    r.zzz = W;
}

// r = 2 * p                   (EFD dbl-2008-s-1, a = 0)
KZ_HD void xyzz_dbl(XYZZ& r, const XYZZ& p) {
    if (xyzz_is_inf(p) || fe_is_zero(p.y)) { xyzz_set_inf(r); return; }
    Fq U, V, W, S, M, t, X3;
    fe_dbl(U, p.y);
    fe_sqr(V, U);
    fe_mul(W, U, V);
    fe_mul(S, p.x, V);
    fe_sqr(t, p.x);
    fe_dbl(M, t); fe_add(M, M, t);
    fe_sqr(X3, M);
    fe_sub(X3, X3, S); fe_sub(X3, X3, S);
    fe_sub(t, S, X3);
    {
        Fq y1 = p.y;  // r may alias p
        fe_mul2sub(r.y, M, t, W, y1);  // M (S - X3) - W Y1, one reduction
    }
    r.x = X3;
    fe_mul(r.zz, V, p.zz);
    fe_mul(r.zzz, W, p.zzz);
}

// acc += affine q             (EFD madd-2008-s: 8M + 2S), exact on all inputs; every product reduced on its
// own (10 Montgomery reductions) -- kept for the kernel variant sweep, xyzz_madd below is the one in use
KZ_HD void xyzz_madd_classic(XYZZ& acc, const Affine& q) {
    if (aff_is_inf(q)) return;
    if (xyzz_is_inf(acc)) { acc.x = q.x; acc.y = q.y; fe_one(acc.zz); fe_one(acc.zzz); return; }
    Fq U2, S2, Pp, Rr, PP, PPP, Q, t;
    fe_mul(U2, q.x, acc.zz);
    fe_mul(S2, q.y, acc.zzz);
    fe_sub(Pp, U2, acc.x);
    fe_sub(Rr, S2, acc.y);
    if (fe_is_zero(Pp)) {
        if (fe_is_zero(Rr)) xyzz_dbl_affine(acc, q);
        else xyzz_set_inf(acc);
        return;
    }
    fe_sqr(PP, Pp);
    fe_mul(PPP, Pp, PP);
    fe_mul(Q, acc.x, PP);
    fe_sqr(t, Rr);
    fe_sub(t, t, PPP); fe_sub(t, t, Q); fe_sub(t, t, Q);  // X3
    fe_sub(Q, Q, t);
    fe_mul(Q, Rr, Q);
    fe_mul(S2, acc.y, PPP);
    fe_sub(acc.y, Q, S2);
    acc.x = t;
    fe_mul(acc.zz, acc.zz, PP);
    fe_mul(acc.zzz, acc.zzz, PPP);
}

// The same addition with the difference of products  Y3 = R*(Q - X3) - Y1*PPP  reduced ONCE
// (fe_mul2sub): 9 Montgomery reductions instead of 10, bit-identical results
// (1.245 -> 1.195 ms for the 2^19 accumulation, profiles/r01_sweep_slice.txt).
KZ_HD void xyzz_madd(XYZZ& acc, const Affine& q) {
    if (aff_is_inf(q)) return;
    if (xyzz_is_inf(acc)) { acc.x = q.x; acc.y = q.y; fe_one(acc.zz); fe_one(acc.zzz); return; }
    Fq U2, S2, Pp, Rr, PP, PPP, Q, t;
    fe_mul(U2, q.x, acc.zz);
    fe_mul(S2, q.y, acc.zzz);
    fe_sub(Pp, U2, acc.x);
    fe_sub(Rr, S2, acc.y);
    if (fe_is_zero(Pp)) {
        if (fe_is_zero(Rr)) xyzz_dbl_affine(acc, q);
        else xyzz_set_inf(acc);
        return;
    }
    fe_sqr(PP, Pp);
    fe_mul(PPP, Pp, PP);
    fe_mul(Q, acc.x, PP);
    fe_mul(acc.zz, acc.zz, PP);
    fe_mul(acc.zzz, acc.zzz, PPP);
    fe_sqr(t, Rr);
    fe_sub(t, t, PPP); fe_sub(t, t, Q); fe_sub(t, t, Q);  // X3
    fe_sub(Q, Q, t);
    fe_mul2sub(acc.y, Rr, Q, acc.y, PPP);
    acc.x = t;
}

#ifdef __CUDACC__
// ---- the same addition on RELAXED coordinates: every coordinate of acc lives in [0, 2p) instead of
// [0, p).  4p < 2^256, so a Montgomery product of operands below 2p is again below 2p without its final
// conditional subtraction (gen_field.py "mulnr"/"mul2subnr", ranges asserted by the emulator), and
// a - b + 2p (if negative) stays in [0, 2p) ("sub2p").  Nine conditional subtractions less per
// addition; the caller normalises with xyzz_relaxed_normalise before the accumulator leaves the loop.
// q is canonical.  Zero tests are "congruent to 0": the value 0 or p.
KZ_D bool fq_is_zero_mod(const Fq& a) {
    const uint32_t pm[8] = FQ_MOD_LIMBS;
    uint32_t z = 0, e = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) { z |= a.l[i]; e |= a.l[i] ^ pm[i]; }
    return z == 0 || e == 0;
}
KZ_D void xyzz_madd_relaxed(XYZZ& acc, const Affine& q) {
    if (aff_is_inf(q)) return;
    if (xyzz_is_inf(acc)) { acc.x = q.x; acc.y = q.y; fe_one(acc.zz); fe_one(acc.zzz); return; }
    Fq U2, S2, Pp, Rr, PP, PPP, Q, t;
    fq_mulnr_ptx(U2.l, q.x.l, acc.zz.l);
    fq_mulnr_ptx(S2.l, q.y.l, acc.zzz.l);
    fq_sub2p_ptx(Pp.l, U2.l, acc.x.l);
    fq_sub2p_ptx(Rr.l, S2.l, acc.y.l);
    if (fq_is_zero_mod(Pp)) {
        if (fq_is_zero_mod(Rr)) xyzz_dbl_affine(acc, q);  // canonical result from the canonical q
        else xyzz_set_inf(acc);
        return;
    }
    fq_mulnr_ptx(PP.l, Pp.l, Pp.l);
    fq_mulnr_ptx(PPP.l, Pp.l, PP.l);
    fq_mulnr_ptx(Q.l, acc.x.l, PP.l);
    fq_mulnr_ptx(acc.zz.l, acc.zz.l, PP.l);
    fq_mulnr_ptx(acc.zzz.l, acc.zzz.l, PPP.l);
    fq_mulnr_ptx(t.l, Rr.l, Rr.l);
    fq_sub2p_ptx(t.l, t.l, PPP.l); fq_sub2p_ptx(t.l, t.l, Q.l); fq_sub2p_ptx(t.l, t.l, Q.l);  // X3
    fq_sub2p_ptx(Q.l, Q.l, t.l);
    fq_mul2subnr_ptx(acc.y.l, Rr.l, Q.l, acc.y.l, PPP.l);
    acc.x = t;
}
// back to canonical coordinates (identity stays all-zero: zz == 0 exactly)
KZ_D void xyzz_relaxed_normalise(XYZZ& acc) {
    fq_reduce_once_ptx(acc.x.l, acc.x.l);
    fq_reduce_once_ptx(acc.y.l, acc.y.l);
    fq_reduce_once_ptx(acc.zz.l, acc.zz.l);
    fq_reduce_once_ptx(acc.zzz.l, acc.zzz.l);
}
#endif

// acc += q                    (EFD add-2008-s: 12M + 2S), exact on all inputs
KZ_HD void xyzz_add(XYZZ& acc, const XYZZ& q) {
    if (xyzz_is_inf(q)) return;
    if (xyzz_is_inf(acc)) { acc = q; return; }
    Fq U1, U2, S1, S2, Pp, Rr, PP, PPP, Q, t;
    fe_mul(U1, acc.x, q.zz);
    fe_mul(U2, q.x, acc.zz);
    fe_mul(S1, acc.y, q.zzz);
    fe_mul(S2, q.y, acc.zzz);
    fe_sub(Pp, U2, U1);
    fe_sub(Rr, S2, S1);
    if (fe_is_zero(Pp)) {
        if (fe_is_zero(Rr)) xyzz_dbl(acc, q);
        else xyzz_set_inf(acc);
        return;
    }
    fe_sqr(PP, Pp);
    fe_mul(PPP, Pp, PP);
    fe_mul(Q, U1, PP);
    fe_sqr(t, Rr);
    fe_sub(t, t, PPP); fe_sub(t, t, Q); fe_sub(t, t, Q);  // X3
    fe_sub(Q, Q, t);
    fe_mul2sub(acc.y, Rr, Q, S1, PPP);  // R (Q - X3) - S1 PPP, one reduction
    acc.x = t;
    fe_mul(acc.zz, acc.zz, q.zz);
    fe_mul(acc.zz, acc.zz, PP);
    fe_mul(acc.zzz, acc.zzz, q.zzz);
    fe_mul(acc.zzz, acc.zzz, PPP);
}

// r = k * p for a small unsigned scalar (left-to-right binary)
KZ_HD void xyzz_mul_small(XYZZ& r, const XYZZ& p, uint32_t k) {
    XYZZ acc; xyzz_set_inf(acc);
    for (int b = 31; b >= 0; b--) {
        xyzz_dbl(acc, acc);
        if ((k >> b) & 1) xyzz_add(acc, p);
    }
    r = acc;
}

// r = k * p for a canonical (non-Montgomery) scalar k < 2^254, signed 4-bit windows: K = k + 0x88..8 (64 nibbles of 8)
// has base-16 digits e_i with k = sum (e_i - 8) 16^i, so each digit lies in [-8, 7] with no carry pass.  A table of
// 1p .. 8p (one doubling, six additions; local memory, indexed by the digit), then 252 doublings and at most 64
// additions -- against ~127 additions for plain double-and-add.  Exact for every input (k = 0, p = identity).
KZ_HD void xyzz_mul_scalar_w4(XYZZ& r, const XYZZ& p, const Fr& k) {
    XYZZ tab[8];
    tab[0] = p;
    xyzz_dbl(tab[1], p);
    for (int j = 2; j < 8; j++) { tab[j] = tab[j - 1]; xyzz_add(tab[j], p); }
    uint32_t K[8];
    uint64_t carry = 0;
    for (int w = 0; w < 8; w++) {
        carry += (uint64_t)k.l[w] + 0x88888888u;
        K[w] = (uint32_t)carry;
        carry >>= 32;
    }
    XYZZ acc; xyzz_set_inf(acc);
    for (int w = 7; w >= 0; w--) {
        for (int q = 7; q >= 0; q--) {
            for (int d = 0; d < 4; d++) xyzz_dbl(acc, acc);  // returns at once while acc is the identity
            const int v = (int)((K[w] >> (4 * q)) & 15u) - 8;
            if (v > 0) {
                xyzz_add(acc, tab[v - 1]);
            } else if (v < 0) {
                XYZZ t;
                xyzz_neg(t, tab[-v - 1]);
                xyzz_add(acc, t);
            }
        }
    }
    r = acc;
}

// Affine from XYZZ given inv = 1/ZZZ:  1/Z = inv*ZZ, x = X/Z^2, y = Y*inv
KZ_HD void xyzz_to_affine_with_inv(Affine& r, const XYZZ& p, const Fq& inv_zzz) {
    Fq zi, zi2;
    fe_mul(zi, inv_zzz, p.zz);
    fe_sqr(zi2, zi);
    fe_mul(r.x, p.x, zi2);
    fe_mul(r.y, p.y, inv_zzz);
}
KZ_HD void xyzz_to_affine(Affine& r, const XYZZ& p) {
    if (xyzz_is_inf(p)) { aff_set_inf(r); return; }
    Fq inv; fe_inv_fast(inv, p.zzz);
    xyzz_to_affine_with_inv(r, p, inv);
}
KZ_HD bool aff_on_curve(const Affine& p) {
    if (aff_is_inf(p)) return true;
    Fq y2, x3, b, three;
    fe_sqr(y2, p.y);
    fe_sqr(x3, p.x); fe_mul(x3, x3, p.x);
    fe_one(b); fe_dbl(three, b); fe_add(three, three, b);
    fe_add(x3, x3, three);
    return fe_eq(y2, x3);
}

#ifdef __CUDACC__
KZ_D Affine aff_load_ro(const Affine* p) {
    Affine r;
    r.x = fe_load_ro(&p->x);
    r.y = fe_load_ro(&p->y);
    return r;
}
// Random 64-byte gather from a table far larger than L2: ask L2 to fetch only the 64 B that are used
// (the default promotes a miss to the whole 128 B line, doubling DRAM traffic of the MSM gather).
KZ_D Affine aff_gather_ro(const Affine* p) {
    Affine r;
    const uint4* q = reinterpret_cast<const uint4*>(p);
    uint4 v[4];
#pragma unroll
    for (int k = 0; k < 4; k++)
        asm volatile("ld.global.nc.L2::64B.v4.u32 {%0,%1,%2,%3}, [%4];"
                     : "=r"(v[k].x), "=r"(v[k].y), "=r"(v[k].z), "=r"(v[k].w) : "l"(q + k));
    r.x.l[0] = v[0].x; r.x.l[1] = v[0].y; r.x.l[2] = v[0].z; r.x.l[3] = v[0].w;
    r.x.l[4] = v[1].x; r.x.l[5] = v[1].y; r.x.l[6] = v[1].z; r.x.l[7] = v[1].w;
    r.y.l[0] = v[2].x; r.y.l[1] = v[2].y; r.y.l[2] = v[2].z; r.y.l[3] = v[2].w;
    r.y.l[4] = v[3].x; r.y.l[5] = v[3].y; r.y.l[6] = v[3].z; r.y.l[7] = v[3].w;
    return r;
}
KZ_D void aff_store(Affine* p, const Affine& v) { fe_store(&p->x, v.x); fe_store(&p->y, v.y); }
KZ_D XYZZ xyzz_load(const XYZZ* p) {
    XYZZ r;
    r.x = fe_load(&p->x); r.y = fe_load(&p->y); r.zz = fe_load(&p->zz); r.zzz = fe_load(&p->zzz);
    return r;
}
KZ_D void xyzz_store(XYZZ* p, const XYZZ& v) {
    fe_store(&p->x, v.x); fe_store(&p->y, v.y); fe_store(&p->zz, v.zz); fe_store(&p->zzz, v.zzz);
}
#endif

}  // namespace kzgb
