// Test-only shim: the HOST build of csrc/pairing.cuh (the source the pairing kernels use), for tests/test_pairing_host.py.
#include "../../rust-kzg-bn254_b200/csrc/pairing.cuh"
using namespace kzgb;
extern "C" {
// out (96 words) = the reduced pairing e(p, q)^m of pairing.cuh, over q's own line table.  q: x.c0, x.c1, y.c0, y.c1;
// p: x, y; Montgomery words; p all zero = the identity.
void t_pairing(uint32_t* out, const uint32_t* q, const uint32_t* p) {
    static Line lines[PAIRING_LINES];
    g2_lines(lines, *(const G2Affine*)q);
    const Affine& P = *(const Affine*)p;
    Fq nx;
    fe_neg(nx, P.x);
    Fq12 f;
    miller_loop_2(f, nx, P.y, aff_is_inf(P), nx, P.y, true, [&](int, int i) { return lines[i]; });
    fq12_final_exp(*(Fq12*)out, f);
}
// the default [tau]G2 of the library (x.c0, x.c1, y.c0, y.c1, Montgomery)
void t_default_g2_tau(uint32_t* out) {
    const uint32_t t[32] = KZ_G2_TAU;
    for (int i = 0; i < 32; i++) out[i] = t[i];
}
// a * a through the cyclotomic squaring and through the generic one, after the easy part of the final exponentiation
void t_cyclotomic_sqr(uint32_t* out_cyc, uint32_t* out_gen, const uint32_t* a) {
    const Fq12& f = *(const Fq12*)a;
    Fq12 r, t;
    fq12_inv(t, f);
    fq12_conj(r, f);
    fq12_mul(r, r, t);
    fq12_frobenius(t, r, 2);
    fq12_mul(r, t, r);
    fq12_cyclotomic_sqr(*(Fq12*)out_cyc, r);
    fq12_sqr(*(Fq12*)out_gen, r);
}
}
