// The BN254 optimal ate pairing for the per-opening checks of kzgb_verify_proofs / kzgb_verify_blob_proofs
// (verifier/src/verify.rs:10-115): the tower Fq2 -> Fq6 -> Fq12, the sparse line multiplication, the Miller loop over
// precomputed lines and the final exponentiation.  Written KZ_HD on Fe<FQ> as ec.cuh is, so the same source builds the
// host line tables (pairing.cu) and the device kernels, and is checked on the CPU (tests/test_pairing_host.py).
//
// Tower (the layout of arkworks' Fq12 over Fq6 over Fq2):
//   Fq2  = Fq[u] / (u^2 + 1)          c0 + c1 u
//   Fq6  = Fq2[v] / (v^3 - xi)        c0 + c1 v + c2 v^2,  xi = 9 + u
//   Fq12 = Fq6[w] / (w^2 - v)         c0 + c1 w            (w^6 = xi)
// G2 lives on the D-type sextic twist y^2 = x^3 + 3 / xi over Fq2; psi(x, y) = (x w^2, y w^3) maps it into E(Fq12).
//
// The line through R and S of the twist (slope lambda in Fq2), untwisted and evaluated at a G1 point P = (xP, yP), is
//   l(P) = yP - lambda xP w + (lambda xR - yR) w^3
// -- up to the factor -1, which the final exponentiation removes.  Only lambda and c = lambda xR - yR depend on the G2
// point, so the host precomputes them once per G2 point (g2_lines) and the device evaluates each line with two Fq
// multiplications and multiplies it into f sparsely (fq12_mul_by_line).
//
// The final exponentiation raises to m (p^12 - 1) / r with m = 2x (6x^2 + 3x + 1), x = 4965661367192848881 (the hard
// part is the chain of Fuentes-Castaneda, Knapp and Rodriguez-Henriquez, "Faster hashing to G2", as arkworks computes
// it).  gcd(m, r) = 1, so f^(m (p^12 - 1) / r) == 1 exactly when the reduced pairing is 1.
#pragma once
#include "ec.cuh"

// The Fq6 / Fq12 / G2 operations are out-of-line calls on the device: inlined, one final exponentiation is tens of
// thousands of instructions and a kernel takes ptxas minutes to compile.
#ifdef __CUDACC__
#define KZ_HD_CALL inline __host__ __device__ __noinline__
#else
#define KZ_HD_CALL inline
#endif

namespace kzgb {

struct Fq2 { Fq c0, c1; };
struct Fq6 { Fq2 c0, c1, c2; };
struct Fq12 { Fq6 c0, c1; };
struct G2Affine { Fq2 x, y; };           // identity: all zero (not on the twist)
struct G2XYZZ { Fq2 x, y, zz, zzz; };    // ec.cuh's XYZZ over Fq2; identity: zz == 0
struct Line { Fq2 lam, c; };             // one Miller-loop line of a fixed G2 point

// x of BN254 and the Miller loop's 6x + 2 = 2^64 + KZ_ATE_LOW (65 bits)
constexpr uint64_t KZ_BN_X = 4965661367192848881ull;
constexpr uint64_t KZ_ATE_LOW = 0x9d797039be763ba8ull;
// lines of one G2 point: 64 doublings, one addition per set bit of KZ_ATE_LOW (36), the two Frobenius steps
constexpr int PAIRING_LINES = 64 + 36 + 2;

// Montgomery words of the constants (c0 then c1, 8 x u32 each), from the exact integers:
//   KZ_FROBk_V1 = xi^((p^k - 1) / 3), V2 = xi^(2 (p^k - 1) / 3), W0 = xi^((p^k - 1) / 6), W1 = V1 W0, W2 = V2 W0:
//   the factors by which the p^k-power Frobenius map multiplies the coefficients of v, v^2, w, v w and v^2 w
// KZ_TWIST_B = 3 / xi; KZ_G2_GEN = the G2 generator (x.c0, x.c1, y.c0, y.c1); KZ_G2_TAU = the reference's G2_TAU
// (primitives/src/consts.rs:55-64)
#define KZ_FROB1_V1 {0x4563ab30u, 0xb5773b10u, 0xa9aa6454u, 0x347f91c8u, 0x242e0991u, 0x7a007127u, 0x118214ecu, 0x1956bcd8u, \
    0xa0aa4757u, 0x6e849f1eu, 0x89f89141u, 0xaa1c7b6du, 0xfae0ca3au, 0xb6e713cdu, 0x4e82ebc3u, 0x26694fbbu}
#define KZ_FROB1_V2 {0x843abe92u, 0x7361d77fu, 0x273411fbu, 0xa5bb2bd3u, 0x4b3e2399u, 0x9c941f31u, 0xbb9fd3ecu, 0x15df9cddu, \
    0x4bd8c949u, 0x5dddfd15u, 0xa4445b60u, 0x62cb29a5u, 0x0c7dd2b9u, 0x37bc870au, 0x3171f0fdu, 0x24830a9du}
#define KZ_FROB1_W0 {0x33144907u, 0xaf9ba696u, 0x87afb78au, 0xca6b1d73u, 0xf08a2087u, 0x11bded5eu, 0x1a1f3a7cu, 0x02f34d75u, \
    0x4c492d72u, 0xa222ae23u, 0x565de15bu, 0xd00f02a4u, 0x53dfc926u, 0xdc2ff3a2u, 0xb3899551u, 0x10a75716u}
#define KZ_FROB1_W1 {0x2936b629u, 0xe4bbdd0cu, 0xe133bacbu, 0xbb30f162u, 0xf9645366u, 0x31a9d1b6u, 0xa500f8ddu, 0x253570beu, \
    0x5ffe77c7u, 0xa1d77ce4u, 0x7826d1dbu, 0x07affd11u, 0xbb7edc6bu, 0x6d16bd27u, 0x85defeccu, 0x2c872002u}
#define KZ_FROB1_W2 {0x41690fe7u, 0xc970692fu, 0x27694b0bu, 0xe2403421u, 0x83c459e8u, 0x32bee66bu, 0x0ab08841u, 0x12aabcedu, \
    0x40aebfa9u, 0x0d485d23u, 0xab2fcc57u, 0x05193418u, 0x8a4910f5u, 0xd3b0a40bu, 0x35d2925au, 0x2f21ebb5u}
#define KZ_FROB2_V1 {0x13e80b9cu, 0x3350c88eu, 0xdb5e56b9u, 0x7dce557cu, 0xb615564au, 0x6001b4b8u, 0x020217e0u, 0x2682e617u, \
    0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u}
#define KZ_FROB2_V2 {0xd782e155u, 0x71930c11u, 0xffbe3323u, 0xa6bb947cu, 0xd4741444u, 0xaa303344u, 0x26594943u, 0x2c3b3f0du, \
    0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u}
#define KZ_FROB2_W0 {0x00fa1bf2u, 0xca8d8005u, 0x68b39769u, 0xf0c5d614u, 0xad0d4418u, 0x0e201271u, 0xbad856e6u, 0x04290f65u, \
    0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u}
#define KZ_FROB2_W1 {0x12edefaau, 0x68c34889u, 0x72aabf4fu, 0x8d087f68u, 0x09081231u, 0x51e1a247u, 0x4729c0fau, 0x2259d6b1u, \
    0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u}
#define KZ_FROB2_W2 {0xc494f1abu, 0x08cfc388u, 0x8d1373d4u, 0x19b31514u, 0xcb6c0213u, 0x584e90fdu, 0xdf2f8849u, 0x09e1685bu, \
    0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u, 0x00000000u}
#define KZ_FROB3_V1 {0x16ad6badu, 0xc9af22f7u, 0x4aa662b2u, 0xb311782au, 0xe248c7f4u, 0x19eeaf64u, 0xe3439f82u, 0x20273e77u, \
    0xf7ce93acu, 0xacc02860u, 0x7ba76b4cu, 0x3933d581u, 0x446c8467u, 0x69e6188bu, 0x4417cc55u, 0x0a46036du}
#define KZ_FROB3_V2 {0x7b6762dfu, 0x448a93a5u, 0x28fdeadfu, 0xbfd62df5u, 0x0e9bd47au, 0xd858f5d0u, 0x3476ec58u, 0x06b03d4du, \
    0xbcc936d1u, 0x2b19daf4u, 0x56f4299fu, 0xa1a54e7au, 0x5adeaef1u, 0xb533eee0u, 0x84dda0b2u, 0x170c812bu}
#define KZ_FROB3_W0 {0x4e46d97du, 0x36531618u, 0xd4c96d9fu, 0x0af7129eu, 0xca1009b5u, 0x659da72fu, 0x83a20d23u, 0x08116d89u, \
    0xc39c1939u, 0xb1df4af7u, 0x8a73bf7fu, 0x3d9f0287u, 0x8caf0ae0u, 0x9b222092u, 0xeff054a6u, 0x26684515u}
#define KZ_FROB3_W1 {0xaf46471eu, 0x5764af0au, 0x873e0fc1u, 0xdc50792eu, 0x881d04f6u, 0x86a673ffu, 0x3c30a74cu, 0x0b2eddb4u, \
    0x787e8580u, 0x9a490f32u, 0xf04af8b1u, 0x8fd16d7fu, 0xc6027bf2u, 0x4b39888eu, 0x5b52a15du, 0x03dd2e70u}
#define KZ_FROB3_W2 {0x75cf559fu, 0xe0bc4b22u, 0xc154e60fu, 0xc238b945u, 0x929a7d5eu, 0x803982a5u, 0xf7e4a37eu, 0x15ce052du, \
    0xbf3799a7u, 0x2d28efbdu, 0x1ad60773u, 0x9b097e3cu, 0xaf4a535bu, 0x982d4113u, 0xe3056063u, 0x24e18991u}
#define KZ_TWIST_B {0x77b802a8u, 0x3bf938e3u, 0x3633535du, 0x020b1b27u, 0x49755260u, 0x26b7edf0u, 0x4384a86du, 0x2514c632u, \
    0xd1dcff67u, 0x38e7ecccu, 0x93ce0d3eu, 0x65f0b37du, 0x22ac00aau, 0xd749d0ddu, 0x4a688d4du, 0x0141b9ceu}
#define KZ_G2_GEN {0x02bc2026u, 0x8e83b5d1u, 0x497b0172u, 0xdceb1935u, 0x97811adfu, 0xfbb82647u, 0xaf96503bu, 0x19573841u, \
    0xa84c6140u, 0xafb4737du, 0x5802d8c4u, 0x6043dd5au, 0x52a02f86u, 0x09e950fcu, 0x3aea7b6bu, 0x14fef083u, \
    0x886be9f6u, 0x619dfa9du, 0xf59e9b78u, 0xfe7fd297u, 0x231b7dfeu, 0xff9e1a62u, 0xae9e4206u, 0x28fd7eebu, \
    0xc71856eeu, 0x64095b56u, 0x327d3cbbu, 0xdc57f922u, 0x33351076u, 0x55f935beu, 0x93fd6482u, 0x0da4a0e6u}
#define KZ_G2_TAU {0xae0114e9u, 0x51893240u, 0x48b7a1deu, 0x4821cf25u, 0x86d6cfcdu, 0x952ef47au, 0x95f191a5u, 0x05a42d3du, \
    0x8f9c504cu, 0x423e5741u, 0x6f0d3351u, 0xffc8d9f3u, 0x6a8748aau, 0xc4fbe8c8u, 0x29f4b1b6u, 0x0f79abd3u, \
    0xe17998ceu, 0xa604320du, 0x7d87edfcu, 0x149b3e2du, 0x1754b4fbu, 0x7bbc7df7u, 0x448e8657u, 0x291a0781u, \
    0xc784f0d6u, 0xdad98146u, 0x2f38352au, 0xd7cbbd12u, 0x5e03976cu, 0x8a73f3b8u, 0xd965c75fu, 0x188e3d35u}

KZ_HD void fq2_set(Fq2& r, const uint32_t* t) {
    for (int i = 0; i < 8; i++) { r.c0.l[i] = t[i]; r.c1.l[i] = t[8 + i]; }
}
KZ_HD void fq2_zero(Fq2& r) { fe_zero(r.c0); fe_zero(r.c1); }
KZ_HD void fq2_one(Fq2& r) { fe_one(r.c0); fe_zero(r.c1); }
KZ_HD bool fq2_is_zero(const Fq2& a) { return fe_is_zero(a.c0) && fe_is_zero(a.c1); }
KZ_HD bool fq2_eq(const Fq2& a, const Fq2& b) { return fe_eq(a.c0, b.c0) && fe_eq(a.c1, b.c1); }
KZ_HD void fq2_add(Fq2& r, const Fq2& a, const Fq2& b) { fe_add(r.c0, a.c0, b.c0); fe_add(r.c1, a.c1, b.c1); }
KZ_HD void fq2_sub(Fq2& r, const Fq2& a, const Fq2& b) { fe_sub(r.c0, a.c0, b.c0); fe_sub(r.c1, a.c1, b.c1); }
KZ_HD void fq2_dbl(Fq2& r, const Fq2& a) { fe_dbl(r.c0, a.c0); fe_dbl(r.c1, a.c1); }
KZ_HD void fq2_neg(Fq2& r, const Fq2& a) { fe_neg(r.c0, a.c0); fe_neg(r.c1, a.c1); }
KZ_HD void fq2_conj(Fq2& r, const Fq2& a) { r.c0 = a.c0; fe_neg(r.c1, a.c1); }
// (a0 b0 - a1 b1) + (a0 b1 + a1 b0) u, each a difference of products with one reduction
KZ_HD void fq2_mul(Fq2& r, const Fq2& a, const Fq2& b) {
    Fq na1, c0;
    fe_neg(na1, a.c1);
    fe_mul2sub(c0, a.c0, b.c0, a.c1, b.c1);
    fe_mul2sub(r.c1, a.c0, b.c1, na1, b.c0);
    r.c0 = c0;
}
KZ_HD void fq2_sqr(Fq2& r, const Fq2& a) {  // (a0 + a1)(a0 - a1) + 2 a0 a1 u
    Fq s, d, t;
    fe_add(s, a.c0, a.c1);
    fe_sub(d, a.c0, a.c1);
    fe_mul(t, a.c0, a.c1);
    fe_mul(r.c0, s, d);
    fe_dbl(r.c1, t);
}
KZ_HD void fq2_mul_fq(Fq2& r, const Fq2& a, const Fq& s) { fe_mul(r.c0, a.c0, s); fe_mul(r.c1, a.c1, s); }
KZ_HD void fq2_mul_xi(Fq2& r, const Fq2& a) {  // (9 + u)(a0 + a1 u) = (9 a0 - a1) + (9 a1 + a0) u
    Fq t0, t1;
    fe_dbl(t0, a.c0); fe_dbl(t0, t0); fe_dbl(t0, t0); fe_add(t0, t0, a.c0);
    fe_dbl(t1, a.c1); fe_dbl(t1, t1); fe_dbl(t1, t1); fe_add(t1, t1, a.c1);
    fe_sub(t0, t0, a.c1);
    fe_add(r.c1, t1, a.c0);
    r.c0 = t0;
}
KZ_HD void fq2_inv(Fq2& r, const Fq2& a) {  // conj(a) / (a0^2 + a1^2); 0 -> 0
    Fq n, t;
    fe_sqr(n, a.c0);
    fe_sqr(t, a.c1);
    fe_add(n, n, t);
    fe_inv_fast(n, n);
    fe_mul(r.c0, a.c0, n);
    fe_mul(t, a.c1, n);
    fe_neg(r.c1, t);
}

// ---- Fq6
KZ_HD void fq6_add(Fq6& r, const Fq6& a, const Fq6& b) { fq2_add(r.c0, a.c0, b.c0); fq2_add(r.c1, a.c1, b.c1); fq2_add(r.c2, a.c2, b.c2); }
KZ_HD void fq6_sub(Fq6& r, const Fq6& a, const Fq6& b) { fq2_sub(r.c0, a.c0, b.c0); fq2_sub(r.c1, a.c1, b.c1); fq2_sub(r.c2, a.c2, b.c2); }
KZ_HD void fq6_neg(Fq6& r, const Fq6& a) { fq2_neg(r.c0, a.c0); fq2_neg(r.c1, a.c1); fq2_neg(r.c2, a.c2); }
KZ_HD void fq6_mul_v(Fq6& r, const Fq6& a) {  // a v = xi a2 + a0 v + a1 v^2
    Fq2 t;
    fq2_mul_xi(t, a.c2);
    r.c2 = a.c1;
    r.c1 = a.c0;
    r.c0 = t;
}
// Karatsuba over the three coefficients: 6 Fq2 multiplications
KZ_HD_CALL void fq6_mul(Fq6& r, const Fq6& a, const Fq6& b) {
    Fq2 t0, t1, t2, s, u, c0, c1, c2;
    fq2_mul(t0, a.c0, b.c0);
    fq2_mul(t1, a.c1, b.c1);
    fq2_mul(t2, a.c2, b.c2);
    fq2_add(s, a.c1, a.c2); fq2_add(u, b.c1, b.c2); fq2_mul(c0, s, u);
    fq2_sub(c0, c0, t1); fq2_sub(c0, c0, t2); fq2_mul_xi(c0, c0); fq2_add(c0, c0, t0);
    fq2_add(s, a.c0, a.c1); fq2_add(u, b.c0, b.c1); fq2_mul(c1, s, u);
    fq2_sub(c1, c1, t0); fq2_sub(c1, c1, t1); fq2_mul_xi(s, t2); fq2_add(c1, c1, s);
    fq2_add(s, a.c0, a.c2); fq2_add(u, b.c0, b.c2); fq2_mul(c2, s, u);
    fq2_sub(c2, c2, t0); fq2_sub(c2, c2, t2); fq2_add(c2, c2, t1);
    r.c0 = c0; r.c1 = c1; r.c2 = c2;
}
// a (b0 + b1 v): 5 Fq2 multiplications
KZ_HD_CALL void fq6_mul_by_01(Fq6& r, const Fq6& a, const Fq2& b0, const Fq2& b1) {
    Fq2 t0, t1, s, u, c0, c1, c2;
    fq2_mul(t0, a.c0, b0);
    fq2_mul(t1, a.c1, b1);
    fq2_mul(c0, a.c2, b1); fq2_mul_xi(c0, c0); fq2_add(c0, c0, t0);
    fq2_add(s, a.c0, a.c1); fq2_add(u, b0, b1); fq2_mul(c1, s, u); fq2_sub(c1, c1, t0); fq2_sub(c1, c1, t1);
    fq2_mul(c2, a.c2, b0); fq2_add(c2, c2, t1);
    r.c0 = c0; r.c1 = c1; r.c2 = c2;
}
KZ_HD void fq6_mul_fq(Fq6& r, const Fq6& a, const Fq& s) { fq2_mul_fq(r.c0, a.c0, s); fq2_mul_fq(r.c1, a.c1, s); fq2_mul_fq(r.c2, a.c2, s); }
KZ_HD_CALL void fq6_inv(Fq6& r, const Fq6& a) {
    Fq2 t0, t1, t2, s, d;
    fq2_sqr(t0, a.c0); fq2_mul(s, a.c1, a.c2); fq2_mul_xi(s, s); fq2_sub(t0, t0, s);  // a0^2 - xi a1 a2
    fq2_sqr(t1, a.c2); fq2_mul_xi(t1, t1); fq2_mul(s, a.c0, a.c1); fq2_sub(t1, t1, s);  // xi a2^2 - a0 a1
    fq2_sqr(t2, a.c1); fq2_mul(s, a.c0, a.c2); fq2_sub(t2, t2, s);                      // a1^2 - a0 a2
    fq2_mul(d, a.c2, t1); fq2_mul(s, a.c1, t2); fq2_add(d, d, s); fq2_mul_xi(d, d);
    fq2_mul(s, a.c0, t0); fq2_add(d, d, s);
    fq2_inv(d, d);
    fq2_mul(r.c0, t0, d); fq2_mul(r.c1, t1, d); fq2_mul(r.c2, t2, d);
}

// ---- Fq12
KZ_HD void fq12_one(Fq12& r) {
    fq2_one(r.c0.c0); fq2_zero(r.c0.c1); fq2_zero(r.c0.c2);
    fq2_zero(r.c1.c0); fq2_zero(r.c1.c1); fq2_zero(r.c1.c2);
}
KZ_HD bool fq12_is_one(const Fq12& a) {
    Fq2 one; fq2_one(one);
    return fq2_eq(a.c0.c0, one) && fq2_is_zero(a.c0.c1) && fq2_is_zero(a.c0.c2) && fq2_is_zero(a.c1.c0) &&
           fq2_is_zero(a.c1.c1) && fq2_is_zero(a.c1.c2);
}
KZ_HD void fq12_conj(Fq12& r, const Fq12& a) { r.c0 = a.c0; fq6_neg(r.c1, a.c1); }  // a^(p^6); the inverse in the cyclotomic subgroup
KZ_HD_CALL void fq12_mul(Fq12& r, const Fq12& a, const Fq12& b) {  // 3 Fq6 multiplications
    Fq6 t0, t1, s, u;
    fq6_mul(t0, a.c0, b.c0);
    fq6_mul(t1, a.c1, b.c1);
    fq6_add(s, a.c0, a.c1); fq6_add(u, b.c0, b.c1); fq6_mul(s, s, u);
    fq6_sub(s, s, t0); fq6_sub(r.c1, s, t1);
    fq6_mul_v(t1, t1); fq6_add(r.c0, t0, t1);
}
KZ_HD_CALL void fq12_sqr(Fq12& r, const Fq12& a) {  // complex squaring: 2 Fq6 multiplications
    Fq6 t, s, u;
    fq6_mul(t, a.c0, a.c1);
    fq6_add(s, a.c0, a.c1);
    fq6_mul_v(u, a.c1); fq6_add(u, u, a.c0);
    fq6_mul(s, s, u);
    fq6_sub(s, s, t);
    fq6_mul_v(u, t); fq6_sub(r.c0, s, u);
    fq6_add(r.c1, t, t);
}
KZ_HD_CALL void fq12_inv(Fq12& r, const Fq12& a) {  // conj(a) / (a0^2 - v a1^2)
    Fq6 t, s;
    fq6_mul(t, a.c0, a.c0);
    fq6_mul(s, a.c1, a.c1); fq6_mul_v(s, s);
    fq6_sub(t, t, s);
    fq6_inv(t, t);
    fq6_mul(r.c0, a.c0, t);
    fq6_mul(s, a.c1, t); fq6_neg(r.c1, s);
}
// f * l with l = a0 + (b0 + b1 v) w, a0 in Fq: the shape of every line (see the top of this file)
KZ_HD_CALL void fq12_mul_by_line(Fq12& f, const Fq& a0, const Fq2& b0, const Fq2& b1) {
    Fq6 t0, t1, t2;
    fq6_mul_fq(t0, f.c0, a0);
    fq6_mul_by_01(t1, f.c1, b0, b1);
    fq6_mul_by_01(t2, f.c0, b0, b1);
    fq6_mul_fq(f.c1, f.c1, a0);
    fq6_add(f.c1, f.c1, t2);
    fq6_mul_v(t1, t1);
    fq6_add(f.c0, t0, t1);
}
// a^(p^k), k = 1, 2, 3
KZ_HD_CALL void fq12_frobenius(Fq12& r, const Fq12& a, int k) {
    Fq2 g[5];
    if (k == 1) {
        const uint32_t t[5][16] = {KZ_FROB1_V1, KZ_FROB1_V2, KZ_FROB1_W0, KZ_FROB1_W1, KZ_FROB1_W2};
        for (int i = 0; i < 5; i++) fq2_set(g[i], t[i]);
    } else if (k == 2) {
        const uint32_t t[5][16] = {KZ_FROB2_V1, KZ_FROB2_V2, KZ_FROB2_W0, KZ_FROB2_W1, KZ_FROB2_W2};
        for (int i = 0; i < 5; i++) fq2_set(g[i], t[i]);
    } else {
        const uint32_t t[5][16] = {KZ_FROB3_V1, KZ_FROB3_V2, KZ_FROB3_W0, KZ_FROB3_W1, KZ_FROB3_W2};
        for (int i = 0; i < 5; i++) fq2_set(g[i], t[i]);
    }
    Fq2 c[6] = {a.c0.c0, a.c0.c1, a.c0.c2, a.c1.c0, a.c1.c1, a.c1.c2};
    if (k & 1)
        for (int i = 0; i < 6; i++) fq2_conj(c[i], c[i]);  // the p-power map on Fq2
    r.c0.c0 = c[0];
    fq2_mul(r.c0.c1, c[1], g[0]);
    fq2_mul(r.c0.c2, c[2], g[1]);
    fq2_mul(r.c1.c0, c[3], g[2]);
    fq2_mul(r.c1.c1, c[4], g[3]);
    fq2_mul(r.c1.c2, c[5], g[4]);
}
// a^2 for a in the cyclotomic subgroup (Granger and Scott, "Faster squaring in the cyclotomic subgroup of sixth degree
// extensions"): three Fq4 squarings
KZ_HD void fq2_sqr_fq4(Fq2& t0, Fq2& t1, const Fq2& a, const Fq2& b) {  // (a + b y)^2 = t0 + t1 y over y^2 = xi
    Fq2 ab, s, u;
    fq2_mul(ab, a, b);
    fq2_add(s, a, b);
    fq2_mul_xi(u, b); fq2_add(u, u, a);
    fq2_mul(s, s, u);
    fq2_sub(s, s, ab);
    fq2_mul_xi(u, ab);
    fq2_sub(t0, s, u);
    fq2_dbl(t1, ab);
}
KZ_HD_CALL void fq12_cyclotomic_sqr(Fq12& r, const Fq12& a) {
    Fq2 t0, t1, t2, t3, t4, t5, s;
    fq2_sqr_fq4(t0, t1, a.c0.c0, a.c1.c1);
    fq2_sqr_fq4(t2, t3, a.c1.c0, a.c0.c2);
    fq2_sqr_fq4(t4, t5, a.c0.c1, a.c1.c2);
    // z0 = 3 t0 - 2 z0, z1 = 3 t1 + 2 z1
    fq2_sub(s, t0, a.c0.c0); fq2_dbl(s, s); fq2_add(r.c0.c0, s, t0);
    fq2_add(s, t1, a.c1.c1); fq2_dbl(s, s); fq2_add(r.c1.c1, s, t1);
    // z2 = 3 xi t5 + 2 z2, z3 = 3 t4 - 2 z3
    Fq2 x5; fq2_mul_xi(x5, t5);
    fq2_add(s, x5, a.c1.c0); fq2_dbl(s, s); fq2_add(r.c1.c0, s, x5);
    fq2_sub(s, t4, a.c0.c2); fq2_dbl(s, s); fq2_add(r.c0.c2, s, t4);
    // z4 = 3 t2 - 2 z4, z5 = 3 t3 + 2 z5
    fq2_sub(s, t2, a.c0.c1); fq2_dbl(s, s); fq2_add(r.c0.c1, s, t2);
    fq2_add(s, t3, a.c1.c2); fq2_dbl(s, s); fq2_add(r.c1.c2, s, t3);
}
// a^x in the cyclotomic subgroup (x = KZ_BN_X, 63 bits)
KZ_HD_CALL void fq12_cyclotomic_exp_x(Fq12& r, const Fq12& a) {
    Fq12 acc = a;
    for (int b = 61; b >= 0; b--) {
        fq12_cyclotomic_sqr(acc, acc);
        if ((KZ_BN_X >> b) & 1) fq12_mul(acc, acc, a);
    }
    r = acc;
}
KZ_HD void fq12_exp_by_neg_x(Fq12& r, const Fq12& a) {
    fq12_cyclotomic_exp_x(r, a);
    fq12_conj(r, r);
}
// f^(m (p^12 - 1) / r), m = 2x (6x^2 + 3x + 1).  The easy part (p^6 - 1)(p^2 + 1) lands in the cyclotomic subgroup; the
// hard part is arkworks' chain for BN curves.
KZ_HD_CALL void fq12_final_exp(Fq12& out, const Fq12& f) {
    Fq12 r, t, y0, y1, y3, y4, y6, y8, y9;
    fq12_inv(t, f);
    fq12_conj(r, f);
    fq12_mul(r, r, t);         // f^(p^6 - 1)
    fq12_frobenius(t, r, 2);
    fq12_mul(r, t, r);         // f^((p^6 - 1)(p^2 + 1))
    fq12_exp_by_neg_x(y0, r);
    fq12_cyclotomic_sqr(y1, y0);
    fq12_cyclotomic_sqr(t, y1);
    fq12_mul(y3, t, y1);
    fq12_exp_by_neg_x(y4, y3);
    fq12_cyclotomic_sqr(t, y4);
    fq12_exp_by_neg_x(y6, t);
    fq12_conj(y3, y3);
    fq12_conj(y6, y6);
    fq12_mul(t, y6, y4);       // y7
    fq12_mul(y8, t, y3);
    fq12_mul(y9, y8, y1);
    fq12_mul(t, y8, y4);       // y10
    fq12_mul(t, t, r);         // y11
    fq12_frobenius(y0, y9, 1); // y12
    fq12_mul(t, y0, t);        // y13
    fq12_frobenius(y8, y8, 2);
    fq12_mul(t, y8, t);        // y14
    fq12_conj(r, r);
    fq12_mul(y0, r, y9);
    fq12_frobenius(y0, y0, 3); // y15
    fq12_mul(out, y0, t);
}

// ---- G2 on the twist (the formulas of ec.cuh over Fq2; a = 0 in both)
KZ_HD bool g2_is_inf(const G2Affine& p) { return fq2_is_zero(p.x) && fq2_is_zero(p.y); }
KZ_HD void g2_xyzz_set_inf(G2XYZZ& p) { fq2_zero(p.x); fq2_zero(p.y); fq2_zero(p.zz); fq2_zero(p.zzz); }
KZ_HD bool g2_xyzz_is_inf(const G2XYZZ& p) { return fq2_is_zero(p.zz); }
KZ_HD bool g2_on_curve(const G2Affine& p) {  // identity excluded
    Fq2 y2, x3, b;
    const uint32_t tb[16] = KZ_TWIST_B;
    fq2_set(b, tb);
    fq2_sqr(y2, p.y);
    fq2_sqr(x3, p.x); fq2_mul(x3, x3, p.x); fq2_add(x3, x3, b);
    return !g2_is_inf(p) && fq2_eq(y2, x3);
}
// r = 2 p                     (EFD dbl-2008-s-1)
KZ_HD_CALL void g2_xyzz_dbl(G2XYZZ& r, const G2XYZZ& p) {
    if (g2_xyzz_is_inf(p) || fq2_is_zero(p.y)) { g2_xyzz_set_inf(r); return; }
    Fq2 U, V, W, S, M, t, X3;
    fq2_dbl(U, p.y);
    fq2_sqr(V, U);
    fq2_mul(W, U, V);
    fq2_mul(S, p.x, V);
    fq2_sqr(t, p.x);
    fq2_dbl(M, t); fq2_add(M, M, t);
    fq2_sqr(X3, M);
    fq2_sub(X3, X3, S); fq2_sub(X3, X3, S);
    fq2_sub(t, S, X3);
    fq2_mul(t, M, t);
    fq2_mul(S, W, p.y);
    fq2_sub(r.y, t, S);
    r.x = X3;
    fq2_mul(r.zz, V, p.zz);
    fq2_mul(r.zzz, W, p.zzz);
}
// acc += affine q             (EFD madd-2008-s), exact on all inputs
KZ_HD_CALL void g2_xyzz_madd(G2XYZZ& acc, const G2Affine& q) {
    if (g2_is_inf(q)) return;
    if (g2_xyzz_is_inf(acc)) { acc.x = q.x; acc.y = q.y; fq2_one(acc.zz); fq2_one(acc.zzz); return; }
    Fq2 U2, S2, Pp, Rr, PP, PPP, Q, t;
    fq2_mul(U2, q.x, acc.zz);
    fq2_mul(S2, q.y, acc.zzz);
    fq2_sub(Pp, U2, acc.x);
    fq2_sub(Rr, S2, acc.y);
    if (fq2_is_zero(Pp)) {
        if (fq2_is_zero(Rr)) {
            G2XYZZ d; d.x = q.x; d.y = q.y; fq2_one(d.zz); fq2_one(d.zzz);
            g2_xyzz_dbl(acc, d);
        } else {
            g2_xyzz_set_inf(acc);
        }
        return;
    }
    fq2_sqr(PP, Pp);
    fq2_mul(PPP, Pp, PP);
    fq2_mul(Q, acc.x, PP);
    fq2_mul(acc.zz, acc.zz, PP);
    fq2_mul(acc.zzz, acc.zzz, PPP);
    fq2_sqr(t, Rr);
    fq2_sub(t, t, PPP); fq2_sub(t, t, Q); fq2_sub(t, t, Q);  // X3
    fq2_sub(Q, Q, t);
    fq2_mul(Q, Rr, Q);
    fq2_mul(S2, acc.y, PPP);
    fq2_sub(acc.y, Q, S2);
    acc.x = t;
}
KZ_HD_CALL void g2_xyzz_to_affine(G2Affine& r, const G2XYZZ& p) {
    if (g2_xyzz_is_inf(p)) { fq2_zero(r.x); fq2_zero(r.y); return; }
    Fq2 inv, zi;
    fq2_inv(inv, p.zzz);
    fq2_mul(zi, inv, p.zz);   // 1/Z
    fq2_sqr(zi, zi);
    fq2_mul(r.x, p.x, zi);
    fq2_mul(r.y, p.y, inv);
}
// acc == q (affine, not the identity), with no inversion
KZ_HD bool g2_xyzz_eq_affine(const G2XYZZ& acc, const G2Affine& q) {
    if (g2_xyzz_is_inf(acc)) return false;
    Fq2 t;
    fq2_mul(t, q.x, acc.zz);
    if (!fq2_eq(t, acc.x)) return false;
    fq2_mul(t, q.y, acc.zzz);
    return fq2_eq(t, acc.y);
}
// the p-power Frobenius endomorphism of the twist: (conj(x) xi^((p-1)/3), conj(y) xi^((p-1)/2))
KZ_HD void g2_frobenius(G2Affine& r, const G2Affine& q) {
    Fq2 g;
    const uint32_t tv[16] = KZ_FROB1_V1, tw[16] = KZ_FROB1_W1;
    Fq2 x, y;
    fq2_conj(x, q.x);
    fq2_conj(y, q.y);
    fq2_set(g, tv); fq2_mul(r.x, x, g);
    fq2_set(g, tw); fq2_mul(r.y, y, g);
}

// ---- the Miller loop's lines of a fixed G2 point q (on the twist, not the identity), in the order the loop uses
// them: for each bit of 6x + 2 below the top one, the tangent at R (R = 2R), then, where the bit is set, the line
// through R and q (R = R + q); last the lines through R and pi(q) and through R + pi(q) and -pi^2(q).  Affine, with
// one Fq2 inversion per line: this runs on the host, once per G2 point.  None of the steps meets an exceptional case
// for q of order r: R = kq with 1 < k < r at every step.
KZ_HD_CALL void g2_line_step(Line& l, G2Affine& R, const G2Affine* s) {  // s == nullptr: tangent
    Fq2 num, den, t;
    if (s) {
        fq2_sub(num, s->y, R.y);
        fq2_sub(den, s->x, R.x);
    } else {
        fq2_sqr(t, R.x); fq2_dbl(num, t); fq2_add(num, num, t);
        fq2_dbl(den, R.y);
    }
    fq2_inv(den, den);
    fq2_mul(l.lam, num, den);
    fq2_mul(t, l.lam, R.x);
    fq2_sub(l.c, t, R.y);
    // R + s (or 2R): x3 = lam^2 - xR - xs, y3 = lam (xR - x3) - yR
    Fq2 x3, y3;
    fq2_sqr(x3, l.lam);
    fq2_sub(x3, x3, R.x);
    fq2_sub(x3, x3, s ? s->x : R.x);
    fq2_sub(t, R.x, x3);
    fq2_mul(y3, l.lam, t);
    fq2_sub(y3, y3, R.y);
    R.x = x3;
    R.y = y3;
}
KZ_HD_CALL void g2_lines(Line* out, const G2Affine& q) {
    G2Affine R = q, q1, q2;
    int n = 0;
    for (int b = 63; b >= 0; b--) {
        g2_line_step(out[n++], R, nullptr);
        if ((KZ_ATE_LOW >> b) & 1) g2_line_step(out[n++], R, &q);
    }
    g2_frobenius(q1, q);
    g2_frobenius(q2, q1);
    fq2_neg(q2.y, q2.y);
    g2_line_step(out[n++], R, &q1);
    g2_line_step(out[n++], R, &q2);
}

// ---- the two-pair Miller loop f = f_{6x+2,Q0}(P0) f_{6x+2,Q1}(P1) with the line tables of Q0 and Q1; an identity
// P_k contributes 1 (its lines are skipped).  nx_k = -x(P_k).
template <class LoadLine>
KZ_HD void miller_loop_2(Fq12& f, const Fq& nx0, const Fq& y0, bool inf0, const Fq& nx1, const Fq& y1, bool inf1,
                         LoadLine load) {
    fq12_one(f);
    int n = 0;
    auto both = [&](int i) {
        Line l;
        Fq2 b0;
        if (!inf0) { l = load(0, i); fq2_mul_fq(b0, l.lam, nx0); fq12_mul_by_line(f, y0, b0, l.c); }
        if (!inf1) { l = load(1, i); fq2_mul_fq(b0, l.lam, nx1); fq12_mul_by_line(f, y1, b0, l.c); }
    };
    for (int b = 63; b >= 0; b--) {
        if (b != 63) fq12_sqr(f, f);  // f = 1 before the first line
        both(n++);
        if ((KZ_ATE_LOW >> b) & 1) both(n++);
    }
    both(n++);
    both(n++);
}

}  // namespace kzgb
