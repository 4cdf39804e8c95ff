#include "sha256.hpp"

#include <string.h>
#if defined(__x86_64__)
#include <immintrin.h>
#endif

namespace kzgb {

static const uint32_t K256[64] = {
    0x428a2f98, 0x71374491, 0xb5c0fbcf, 0xe9b5dba5, 0x3956c25b, 0x59f111f1, 0x923f82a4, 0xab1c5ed5, 0xd807aa98, 0x12835b01,
    0x243185be, 0x550c7dc3, 0x72be5d74, 0x80deb1fe, 0x9bdc06a7, 0xc19bf174, 0xe49b69c1, 0xefbe4786, 0x0fc19dc6, 0x240ca1cc,
    0x2de92c6f, 0x4a7484aa, 0x5cb0a9dc, 0x76f988da, 0x983e5152, 0xa831c66d, 0xb00327c8, 0xbf597fc7, 0xc6e00bf3, 0xd5a79147,
    0x06ca6351, 0x14292967, 0x27b70a85, 0x2e1b2138, 0x4d2c6dfc, 0x53380d13, 0x650a7354, 0x766a0abb, 0x81c2c92e, 0x92722c85,
    0xa2bfe8a1, 0xa81a664b, 0xc24b8b70, 0xc76c51a3, 0xd192e819, 0xd6990624, 0xf40e3585, 0x106aa070, 0x19a4c116, 0x1e376c08,
    0x2748774c, 0x34b0bcb5, 0x391c0cb3, 0x4ed8aa4a, 0x5b9cca4f, 0x682e6ff3, 0x748f82ee, 0x78a5636f, 0x84c87814, 0x8cc70208,
    0x90befffa, 0xa4506ceb, 0xbef9a3f7, 0xc67178f2};

static inline uint32_t rotr(uint32_t x, int n) { return (x >> n) | (x << (32 - n)); }

static void blocks_portable(uint32_t st[8], const uint8_t* p, size_t nblk) {
    while (nblk--) {
        uint32_t w[64];
        for (int i = 0; i < 16; i++)
            w[i] = ((uint32_t)p[4 * i] << 24) | ((uint32_t)p[4 * i + 1] << 16) | ((uint32_t)p[4 * i + 2] << 8) | p[4 * i + 3];
        for (int i = 16; i < 64; i++) {
            uint32_t s0 = rotr(w[i - 15], 7) ^ rotr(w[i - 15], 18) ^ (w[i - 15] >> 3);
            uint32_t s1 = rotr(w[i - 2], 17) ^ rotr(w[i - 2], 19) ^ (w[i - 2] >> 10);
            w[i] = w[i - 16] + s0 + w[i - 7] + s1;
        }
        uint32_t a = st[0], b = st[1], c = st[2], d = st[3], e = st[4], f = st[5], g = st[6], h = st[7];
        for (int i = 0; i < 64; i++) {
            uint32_t S1 = rotr(e, 6) ^ rotr(e, 11) ^ rotr(e, 25);
            uint32_t ch = (e & f) ^ (~e & g);
            uint32_t t1 = h + S1 + ch + K256[i] + w[i];
            uint32_t S0 = rotr(a, 2) ^ rotr(a, 13) ^ rotr(a, 22);
            uint32_t mj = (a & b) ^ (a & c) ^ (b & c);
            uint32_t t2 = S0 + mj;
            h = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
        }
        st[0] += a; st[1] += b; st[2] += c; st[3] += d; st[4] += e; st[5] += f; st[6] += g; st[7] += h;
        p += 64;
    }
}

#if defined(__x86_64__)
__attribute__((target("sha,sse4.1,ssse3"))) static void blocks_shani(uint32_t st[8], const uint8_t* p, size_t nblk) {
    const __m128i MASK = _mm_set_epi64x(0x0c0d0e0f08090a0bULL, 0x0405060700010203ULL);
    __m128i tmp = _mm_loadu_si128((const __m128i*)&st[0]);
    __m128i s1 = _mm_loadu_si128((const __m128i*)&st[4]);
    tmp = _mm_shuffle_epi32(tmp, 0xB1);
    s1 = _mm_shuffle_epi32(s1, 0x1B);
    __m128i s0 = _mm_alignr_epi8(tmp, s1, 8);
    s1 = _mm_blend_epi16(s1, tmp, 0xF0);
    while (nblk--) {
        const __m128i save0 = s0, save1 = s1;
        __m128i m[4];
#pragma GCC unroll 16
        for (int i = 0; i < 16; i++) {
            if (i < 4) {
                m[i] = _mm_shuffle_epi8(_mm_loadu_si128((const __m128i*)(p + 16 * i)), MASK);
            } else {
                __m128i x0 = m[i & 3], x1 = m[(i + 1) & 3], x2 = m[(i + 2) & 3], x3 = m[(i + 3) & 3];
                __m128i t = _mm_add_epi32(_mm_sha256msg1_epu32(x0, x1), _mm_alignr_epi8(x3, x2, 4));
                m[i & 3] = _mm_sha256msg2_epu32(t, x3);
            }
            __m128i msg = _mm_add_epi32(m[i & 3], _mm_loadu_si128((const __m128i*)&K256[4 * i]));
            s1 = _mm_sha256rnds2_epu32(s1, s0, msg);
            msg = _mm_shuffle_epi32(msg, 0x0E);
            s0 = _mm_sha256rnds2_epu32(s0, s1, msg);
        }
        s0 = _mm_add_epi32(s0, save0);
        s1 = _mm_add_epi32(s1, save1);
        p += 64;
    }
    tmp = _mm_shuffle_epi32(s0, 0x1B);
    s1 = _mm_shuffle_epi32(s1, 0xB1);
    s0 = _mm_blend_epi16(tmp, s1, 0xF0);
    s1 = _mm_alignr_epi8(s1, tmp, 8);
    _mm_storeu_si128((__m128i*)&st[0], s0);
    _mm_storeu_si128((__m128i*)&st[4], s1);
}
#endif

bool sha256_has_shani() {
#if defined(__x86_64__)
    static const bool has = __builtin_cpu_supports("sha") && __builtin_cpu_supports("sse4.1") && __builtin_cpu_supports("ssse3");
    return has;
#else
    return false;
#endif
}

#if defined(__x86_64__)
// ---------------------------------------------------------------------------------------------------------------
// Sixteen messages in lockstep, one per 32-bit lane of the AVX-512 registers ("multi-buffer" SHA-256).  A single SHA-NI
// stream is bound by the latency chain of its 32 sha256rnds2 per block (1.8 GB/s on one core of this box, 2.4 GB/s per
// core with both hardware threads hashing); here a round is 6 rotates + 4 ternary logic ops + 7 additions for SIXTEEN
// blocks, so one core sustains about twice that -- at the price of latency: the sixteen digests arrive together.  Used by
// the blob-batch pipeline when a deep batch meets a host whose SHA-NI pool cannot keep up with the GPU (batch.cu HashStage).
// ---------------------------------------------------------------------------------------------------------------
#define KZ_MB_TARGET __attribute__((target("avx512f,avx512bw,avx512vl")))

KZ_MB_TARGET static inline void transpose16(__m512i r[16]) {
    __m512i t[16];
    for (int i = 0; i < 16; i += 2) { t[i] = _mm512_unpacklo_epi32(r[i], r[i + 1]); t[i + 1] = _mm512_unpackhi_epi32(r[i], r[i + 1]); }
    for (int i = 0; i < 16; i += 4) {
        r[i] = _mm512_unpacklo_epi64(t[i], t[i + 2]); r[i + 1] = _mm512_unpackhi_epi64(t[i], t[i + 2]);
        r[i + 2] = _mm512_unpacklo_epi64(t[i + 1], t[i + 3]); r[i + 3] = _mm512_unpackhi_epi64(t[i + 1], t[i + 3]);
    }
    // r[4q + j] now holds, in 128-bit lane L, words 4L + j of rows 4q .. 4q + 3
    for (int j = 0; j < 4; j++) {
        t[j] = _mm512_shuffle_i32x4(r[j], r[4 + j], 0x88);          // lanes 0, 2 of rows 0-3 | 4-7
        t[4 + j] = _mm512_shuffle_i32x4(r[j], r[4 + j], 0xdd);      // lanes 1, 3
        t[8 + j] = _mm512_shuffle_i32x4(r[8 + j], r[12 + j], 0x88);
        t[12 + j] = _mm512_shuffle_i32x4(r[8 + j], r[12 + j], 0xdd);
    }
    for (int j = 0; j < 4; j++) {
        r[j] = _mm512_shuffle_i32x4(t[j], t[8 + j], 0x88);          // word j       of rows 0 .. 15
        r[8 + j] = _mm512_shuffle_i32x4(t[j], t[8 + j], 0xdd);      // word 8 + j
        r[4 + j] = _mm512_shuffle_i32x4(t[4 + j], t[12 + j], 0x88); // word 4 + j
        r[12 + j] = _mm512_shuffle_i32x4(t[4 + j], t[12 + j], 0xdd);// word 12 + j
    }
}

KZ_MB_TARGET void sha256_mb16_blocks(uint32_t st[16][8], const uint8_t* const p[16], size_t nblk, void (*fix)(uint8_t block[64])) {
    const __m512i BSWAP = _mm512_broadcast_i32x4(_mm_set_epi64x(0x0c0d0e0f08090a0bULL, 0x0405060700010203ULL));
    const __m512i THIRTY = _mm512_set1_epi8(0x30);
    __m512i s[16];
    for (int m = 0; m < 16; m++) s[m] = _mm512_zextsi256_si512(_mm256_loadu_si256((const __m256i*)st[m]));
    transpose16(s);  // s[j] = state word j of the 16 messages (j < 8)
    __m512i a = s[0], b = s[1], c = s[2], d = s[3], e = s[4], f = s[5], g = s[6], h = s[7];
    for (size_t k = 0; k < nblk; k++) {
        __m512i w[16];
        for (int m = 0; m < 16; m++) {
            w[m] = _mm512_loadu_si512((const void*)(p[m] + 64 * k));
            // a 32-byte chunk whose first byte is >= 0x30 may need the caller's fix-up (value >= r): rare, out of line
            if (fix && _mm512_mask_cmpge_epu8_mask(0x0000000100000001ULL, w[m], THIRTY)) {
                alignas(64) uint8_t tmp[64];
                _mm512_store_si512((void*)tmp, w[m]);
                fix(tmp);
                w[m] = _mm512_load_si512((const void*)tmp);
            }
            if (k + 4 < nblk) _mm_prefetch((const char*)(p[m] + 64 * (k + 4)), _MM_HINT_T0);
        }
        transpose16(w);
        for (int t = 0; t < 16; t++) w[t] = _mm512_shuffle_epi8(w[t], BSWAP);
        const __m512i a0 = a, b0 = b, c0 = c, d0 = d, e0 = e, f0 = f, g0 = g, h0 = h;
#define KZ_ROUND(A, B, C, D, E, F, G, H, T)                                                                                     \
    do {                                                                                                                        \
        __m512i S1 = _mm512_ternarylogic_epi32(_mm512_ror_epi32(E, 6), _mm512_ror_epi32(E, 11), _mm512_ror_epi32(E, 25), 0x96); \
        __m512i t1 = _mm512_add_epi32(_mm512_add_epi32(H, S1), _mm512_add_epi32(_mm512_ternarylogic_epi32(E, F, G, 0xca),       \
                                                                                 _mm512_add_epi32(w[(T) & 15], _mm512_set1_epi32((int)K256[T])))); \
        __m512i S0 = _mm512_ternarylogic_epi32(_mm512_ror_epi32(A, 2), _mm512_ror_epi32(A, 13), _mm512_ror_epi32(A, 22), 0x96); \
        D = _mm512_add_epi32(D, t1);                                                                                            \
        H = _mm512_add_epi32(t1, _mm512_add_epi32(S0, _mm512_ternarylogic_epi32(A, B, C, 0xe8)));                               \
    } while (0)
#define KZ_SCHED(T)                                                                                                             \
    do {                                                                                                                        \
        const __m512i w15 = w[((T) + 1) & 15], w2 = w[((T) + 14) & 15];                                                         \
        __m512i s0 = _mm512_ternarylogic_epi32(_mm512_ror_epi32(w15, 7), _mm512_ror_epi32(w15, 18), _mm512_srli_epi32(w15, 3), 0x96);   \
        __m512i s1 = _mm512_ternarylogic_epi32(_mm512_ror_epi32(w2, 17), _mm512_ror_epi32(w2, 19), _mm512_srli_epi32(w2, 10), 0x96);    \
        w[(T) & 15] = _mm512_add_epi32(_mm512_add_epi32(w[(T) & 15], s0), _mm512_add_epi32(w[((T) + 9) & 15], s1));             \
    } while (0)
#define KZ_ROUND8(T, SCHED)                                  \
    do {                                                     \
        if (SCHED) KZ_SCHED((T) + 0); KZ_ROUND(a, b, c, d, e, f, g, h, (T) + 0); \
        if (SCHED) KZ_SCHED((T) + 1); KZ_ROUND(h, a, b, c, d, e, f, g, (T) + 1); \
        if (SCHED) KZ_SCHED((T) + 2); KZ_ROUND(g, h, a, b, c, d, e, f, (T) + 2); \
        if (SCHED) KZ_SCHED((T) + 3); KZ_ROUND(f, g, h, a, b, c, d, e, (T) + 3); \
        if (SCHED) KZ_SCHED((T) + 4); KZ_ROUND(e, f, g, h, a, b, c, d, (T) + 4); \
        if (SCHED) KZ_SCHED((T) + 5); KZ_ROUND(d, e, f, g, h, a, b, c, (T) + 5); \
        if (SCHED) KZ_SCHED((T) + 6); KZ_ROUND(c, d, e, f, g, h, a, b, (T) + 6); \
        if (SCHED) KZ_SCHED((T) + 7); KZ_ROUND(b, c, d, e, f, g, h, a, (T) + 7); \
    } while (0)
        KZ_ROUND8(0, 0); KZ_ROUND8(8, 0);
        KZ_ROUND8(16, 1); KZ_ROUND8(24, 1); KZ_ROUND8(32, 1); KZ_ROUND8(40, 1); KZ_ROUND8(48, 1); KZ_ROUND8(56, 1);
#undef KZ_ROUND8
#undef KZ_SCHED
#undef KZ_ROUND
        a = _mm512_add_epi32(a, a0); b = _mm512_add_epi32(b, b0); c = _mm512_add_epi32(c, c0); d = _mm512_add_epi32(d, d0);
        e = _mm512_add_epi32(e, e0); f = _mm512_add_epi32(f, f0); g = _mm512_add_epi32(g, g0); h = _mm512_add_epi32(h, h0);
    }
    s[0] = a; s[1] = b; s[2] = c; s[3] = d; s[4] = e; s[5] = f; s[6] = g; s[7] = h;
    for (int j = 8; j < 16; j++) s[j] = _mm512_setzero_si512();
    transpose16(s);  // s[m] = the 8 state words of message m (low half)
    for (int m = 0; m < 16; m++) _mm256_storeu_si256((__m256i*)st[m], _mm512_castsi512_si256(s[m]));
}
#endif

bool sha256_has_mb16() {
#if defined(__x86_64__)
    static const bool has = __builtin_cpu_supports("avx512f") && __builtin_cpu_supports("avx512bw") && __builtin_cpu_supports("avx512vl");
    return has;
#else
    return false;
#endif
}
#if !defined(__x86_64__)
void sha256_mb16_blocks(uint32_t[16][8], const uint8_t* const[16], size_t, void (*)(uint8_t[64])) {}
#endif

static inline void blocks(uint32_t st[8], const uint8_t* p, size_t nblk) {
#if defined(__x86_64__)
    if (sha256_has_shani()) { blocks_shani(st, p, nblk); return; }
#endif
    blocks_portable(st, p, nblk);
}

void Sha256::reset() {
    static const uint32_t iv[8] = {0x6a09e667, 0xbb67ae85, 0x3c6ef372, 0xa54ff53a, 0x510e527f, 0x9b05688c, 0x1f83d9ab, 0x5be0cd19};
    memcpy(h, iv, sizeof(iv));
    total = 0;
    fill = 0;
}

void Sha256::update(const void* data, size_t len) {
    const uint8_t* p = (const uint8_t*)data;
    total += len;
    if (fill) {
        size_t take = 64 - fill < len ? 64 - fill : len;
        memcpy(buf + fill, p, take);
        fill += take; p += take; len -= take;
        if (fill == 64) { blocks(h, buf, 1); fill = 0; }
    }
    if (len >= 64) {
        size_t nb = len / 64;
        blocks(h, p, nb);
        p += nb * 64; len -= nb * 64;
    }
    if (len) { memcpy(buf, p, len); fill = len; }
}

void Sha256::finish(uint8_t out[32]) {
    uint64_t bits = total * 8;
    uint8_t pad[72];
    size_t padlen = (fill < 56) ? (56 - fill) : (120 - fill);
    memset(pad, 0, sizeof(pad));
    pad[0] = 0x80;
    for (int i = 0; i < 8; i++) pad[padlen + i] = (uint8_t)(bits >> (56 - 8 * i));
    uint64_t keep = total;
    update(pad, padlen + 8);
    total = keep;
    for (int i = 0; i < 8; i++) {
        out[4 * i] = (uint8_t)(h[i] >> 24); out[4 * i + 1] = (uint8_t)(h[i] >> 16);
        out[4 * i + 2] = (uint8_t)(h[i] >> 8); out[4 * i + 3] = (uint8_t)h[i];
    }
}

void sha256(const void* data, size_t len, uint8_t out[32]) {
    Sha256 s;
    s.update(data, len);
    s.finish(out);
}

}  // namespace kzgb
