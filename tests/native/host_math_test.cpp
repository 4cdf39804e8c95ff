// Test-only shim: exposes the HOST path of csrc/field.cuh + csrc/ec.cuh + sha256 + the transcript to Python so the
// exact formulas the kernels use (same source, compiled for the host) can be checked on CPU.
#include "../../rust-kzg-bn254_b200/csrc/ec.cuh"
#include "../../rust-kzg-bn254_b200/csrc/sha256.hpp"
#include "../../rust-kzg-bn254_b200/csrc/transcript.hpp"
using namespace kzgb;
extern "C" {
void t_fq_mul(uint32_t* r, const uint32_t* a, const uint32_t* b) { fe_mul(*(Fq*)r, *(const Fq*)a, *(const Fq*)b); }
void t_fr_mul(uint32_t* r, const uint32_t* a, const uint32_t* b) { fe_mul(*(Fr*)r, *(const Fr*)a, *(const Fr*)b); }
void t_fq_add(uint32_t* r, const uint32_t* a, const uint32_t* b) { fe_add(*(Fq*)r, *(const Fq*)a, *(const Fq*)b); }
void t_fq_sub(uint32_t* r, const uint32_t* a, const uint32_t* b) { fe_sub(*(Fq*)r, *(const Fq*)a, *(const Fq*)b); }
void t_fr_add(uint32_t* r, const uint32_t* a, const uint32_t* b) { fe_add(*(Fr*)r, *(const Fr*)a, *(const Fr*)b); }
void t_fr_sub(uint32_t* r, const uint32_t* a, const uint32_t* b) { fe_sub(*(Fr*)r, *(const Fr*)a, *(const Fr*)b); }
void t_fq_inv(uint32_t* r, const uint32_t* a) { fe_inv(*(Fq*)r, *(const Fq*)a); }
void t_fr_inv(uint32_t* r, const uint32_t* a) { fe_inv(*(Fr*)r, *(const Fr*)a); }
void t_fq_inv_fast(uint32_t* r, const uint32_t* a) { fe_inv_fast(*(Fq*)r, *(const Fq*)a); }
void t_fr_inv_fast(uint32_t* r, const uint32_t* a) { fe_inv_fast(*(Fr*)r, *(const Fr*)a); }
void t_fq_to_mont(uint32_t* r, const uint32_t* a) { fe_to_mont(*(Fq*)r, *(const Fq*)a); }
void t_fr_to_mont(uint32_t* r, const uint32_t* a) { fe_to_mont(*(Fr*)r, *(const Fr*)a); }
void t_fq_from_mont(uint32_t* r, const uint32_t* a) { fe_from_mont(*(Fq*)r, *(const Fq*)a); }
int t_fq_lex_largest(const uint32_t* a) { return fe_lexicographically_largest(*(const Fq*)a) ? 1 : 0; }
// XYZZ ops on (x,y,zz,zzz) Montgomery; affine (x,y) Montgomery, (0,0) = identity
void t_madd(uint32_t* acc, const uint32_t* q) { xyzz_madd(*(XYZZ*)acc, *(const Affine*)q); }
void t_add(uint32_t* acc, const uint32_t* q) { xyzz_add(*(XYZZ*)acc, *(const XYZZ*)q); }
void t_dbl(uint32_t* r, const uint32_t* p) { XYZZ t; xyzz_dbl(t, *(const XYZZ*)p); *(XYZZ*)r = t; }
void t_to_affine(uint32_t* r, const uint32_t* p) { xyzz_to_affine(*(Affine*)r, *(const XYZZ*)p); }
void t_mul_small(uint32_t* r, const uint32_t* p, uint32_t k) { xyzz_mul_small(*(XYZZ*)r, *(const XYZZ*)p, k); }
int t_on_curve(const uint32_t* p) { return aff_on_curve(*(const Affine*)p) ? 1 : 0; }
void t_sha256(const uint8_t* d, size_t n, uint8_t* out) { sha256(d, n, out); }
void t_sha256_chunked(const uint8_t* d, size_t n, size_t step, uint8_t* out) {
    Sha256 s;
    for (size_t i = 0; i < n; i += step) s.update(d + i, (n - i) < step ? (n - i) : step);
    s.finish(out);
}
int t_has_shani() { return sha256_has_shani() ? 1 : 0; }
int t_has_mb16() { return sha256_has_mb16() ? 1 : 0; }
// 16 messages of nblk 64-byte blocks each, msgs = 16 x (64 nblk) bytes back to back; out = 16 x 8 state words after the blocks
// (no padding: the raw compression chain).  flip != 0 installs a fix-up that xors 0xff into byte 1 of flagged chunks.
static void flip_fix(uint8_t b[64]) { if (b[0] >= 0x30) b[1] ^= 0xff; if (b[32] >= 0x30) b[33] ^= 0xff; }
void t_sha256_mb16(const uint8_t* msgs, size_t nblk, int flip, uint32_t* out) {
    static const uint32_t iv[8] = {0x6a09e667, 0xbb67ae85, 0x3c6ef372, 0xa54ff53a, 0x510e527f, 0x9b05688c, 0x1f83d9ab, 0x5be0cd19};
    uint32_t st[16][8];
    const uint8_t* p[16];
    for (int m = 0; m < 16; m++) { for (int j = 0; j < 8; j++) st[m][j] = iv[j]; p[m] = msgs + (size_t)m * 64 * nblk; }
    sha256_mb16_blocks(st, p, nblk, flip ? flip_fix : nullptr);
    for (int m = 0; m < 16; m++) for (int j = 0; j < 8; j++) out[8 * m + j] = st[m][j];
}
// the same chain through the single-stream implementation (update() without finish): state after nblk blocks
void t_sha256_state(const uint8_t* msg, size_t nblk, uint32_t* out) {
    Sha256 s;
    s.update(msg, 64 * nblk);
    for (int j = 0; j < 8; j++) out[j] = s.h[j];
}
// Fiat-Shamir transcript midstates, each finished by SHA-256 padding alone (out: 32-byte digests).
void t_challenge_midstate(const uint8_t* blob, size_t len, size_t n, uint8_t* out) {
    Sha256 s;
    challenge_midstate(s, blob, len, n);
    s.finish(out);
}
// `members` blobs of 32 n bytes back to back, hashed in lockstep, each midstate finished by challenge_midstate_resume
void t_challenge_midstates_mb16(const uint8_t* blobs, size_t members, size_t n, uint8_t* out) {
    const uint8_t* p[16];
    for (size_t m = 0; m < members; m++) p[m] = blobs + 32 * n * m;
    uint32_t st[16][8];
    challenge_midstates_mb16(p, members, n, st);
    for (size_t m = 0; m < members; m++) challenge_midstate_resume(st[m], p[m], n).finish(out + 32 * m);
}
// the single-stream state after chunks 0 .. n-2 (what the device hands over), finished by challenge_midstate_resume:
// for even n those chunks end on a block boundary, so the one zero chunk of padding stays in the buffer, out of h
void t_challenge_midstate_resumed(const uint8_t* blob, size_t n, uint8_t* out) {
    Sha256 s;
    challenge_midstate(s, blob, 32 * (n - 1), n);
    challenge_midstate_resume(s.h, blob, n).finish(out);
}
}
