// Host Fiat-Shamir transcript (transcript.hpp).
#include "transcript.hpp"

#include <string.h>

namespace kzgb {

namespace {
const uint8_t FR_MOD_BE[32] = {0x30, 0x64, 0x4e, 0x72, 0xe1, 0x31, 0xa0, 0x29, 0xb8, 0x50, 0x45, 0xb6, 0x81, 0x81, 0x58, 0x5d,
                               0x28, 0x33, 0xe8, 0x48, 0x79, 0xb9, 0x70, 0x91, 0x43, 0xe1, 0xf5, 0x93, 0xf0, 0x00, 0x00, 0x01};
const char TAG[] = "EIGENDA_FSBLOBVERIFY_V1_";

void put_u64_be(uint8_t out[8], uint64_t v) {
    for (int i = 0; i < 8; i++) out[i] = (uint8_t)(v >> (56 - 8 * i));
}
}  // namespace

Fr fr_from_be_bytes(const uint8_t* b) {
    Fr a;
    for (int k = 0; k < 8; k++)
        a.l[7 - k] = ((uint32_t)b[4 * k] << 24) | ((uint32_t)b[4 * k + 1] << 16) | ((uint32_t)b[4 * k + 2] << 8) | b[4 * k + 3];
    fe_to_mont(a, a);
    return a;
}

void serialize_compressed(const Affine& a, uint8_t out[32]) {
    memset(out, 0, 32);
    if (aff_is_inf(a)) { out[31] = 0x40; return; }
    Fq xc; fe_from_mont(xc, a.x);
    memcpy(out, xc.l, 32);
    if (fe_lexicographically_largest(a.y)) out[31] |= 0x80;  // y > -y  <=>  y > (p-1)/2
}

const uint8_t* fr_reduce_chunk(const uint8_t in[32], uint8_t out[32]) {
    if (in[0] < 0x30 || memcmp(in, FR_MOD_BE, 32) < 0) return in;
    fe_to_be_bytes(fr_from_be_bytes(in), out);
    return out;
}

void challenge_midstate(Sha256& sh, const uint8_t* blob, size_t len, size_t n) {
    sh.reset();
    sh.update(TAG, 24);
    uint8_t nb[8];
    put_u64_be(nb, n);
    sh.update(nb, 8);
    size_t full = len / 32;
    size_t run_start = 0;
    uint8_t red[32];
    for (size_t i = 0; i < full; i++) {
        if (fr_reduce_chunk(blob + 32 * i, red) != red) continue;  // canonical: hash in place
        if (i > run_start) sh.update(blob + 32 * run_start, 32 * (i - run_start));
        sh.update(red, 32);
        run_start = i + 1;
    }
    if (full > run_start) sh.update(blob + 32 * run_start, 32 * (full - run_start));
    size_t done = full;
    if (len % 32) {  // trailing partial chunk, right-padded with zeros (helpers.rs:47-51)
        uint8_t last[32];
        memset(last, 0, 32);
        memcpy(last, blob + 32 * full, len % 32);
        sh.update(fr_reduce_chunk(last, last), 32);
        done++;
    }
    static const uint8_t zeros[4096] = {0};
    size_t pad = (n - done) * 32;
    while (pad) { size_t t = pad < sizeof(zeros) ? pad : sizeof(zeros); sh.update(zeros, t); pad -= t; }
}

Fr challenge_finish(Sha256 sh, const Affine& commitment) {
    uint8_t cb[32], dg[32];
    serialize_compressed(commitment, cb);
    sh.update(cb, 32);
    sh.finish(dg);
    return fr_from_be_bytes(dg);  // hash_to_field_element (helpers.rs:382-390)
}

bool hash_mb_eligible(size_t len) { const size_t n = len / 32; return len % 32 == 0 && n >= 1024 && (n & (n - 1)) == 0; }

// the fix-up hook of sha256_mb16_blocks: both chunks of a transcript block reduced mod r
static void hash_fix_block(uint8_t block[64]) {
    for (int h = 0; h < 64; h += 32) fr_reduce_chunk(block + h, block + h);
}

void challenge_midstates_mb16(const uint8_t* const* blobs, size_t members, size_t n, uint32_t out[16][8]) {
    static const uint32_t iv[8] = {0x6a09e667, 0xbb67ae85, 0x3c6ef372, 0xa54ff53a, 0x510e527f, 0x9b05688c, 0x1f83d9ab, 0x5be0cd19};
    alignas(64) uint8_t first[16][64];
    const uint8_t* p[16];
    for (size_t m = 0; m < 16; m++) {
        const uint8_t* blob = blobs[m < members ? m : 0];
        memcpy(first[m], TAG, 24);
        put_u64_be(first[m] + 24, n);
        memcpy(first[m] + 32, blob, 32);
        fr_reduce_chunk(first[m] + 32, first[m] + 32);
        memcpy(out[m], iv, 32);
        p[m] = first[m];
    }
    sha256_mb16_blocks(out, p, 1, nullptr);
    for (size_t m = 0; m < 16; m++) p[m] = blobs[m < members ? m : 0] + 32;  // block b >= 1 holds chunks 2b - 1, 2b
    sha256_mb16_blocks(out, p, n / 2 - 1, hash_fix_block);
}

Sha256 challenge_midstate_resume(const uint32_t state[8], const uint8_t* blob, size_t n) {
    Sha256 sh;
    memcpy(sh.h, state, 32);
    sh.total = 32 * (uint64_t)n;  // tag (24) + u64 (8) + chunks 0 .. n-2
    uint8_t red[32];
    sh.update(fr_reduce_chunk(blob + 32 * (n - 1), red), 32);
    return sh;
}

}  // namespace kzgb
