// Host side of the Fiat-Shamir transcript of compute_challenge (reference primitives/src/helpers.rs:411-472) and the
// host encodings it needs.  Plain C++ (transcript.cpp is compiled by the host compiler like sha256.cpp): nothing here
// touches the GPU, so every form of the midstate -- single stream, 16-way multi-buffer, finished from a device state --
// can be checked against each other on any host.
#pragma once
#include <stddef.h>
#include <stdint.h>
#include "ec.cuh"
#include "sha256.hpp"

namespace kzgb {

// 32 big-endian bytes (any value) -> Fr Montgomery, reduced mod r
Fr fr_from_be_bytes(const uint8_t* b);
template <int F>
void fe_to_be_bytes(const Fe<F>& mont, uint8_t* out) {
    Fe<F> c; fe_from_mont(c, mont);
    for (int k = 0; k < 8; k++) {
        uint32_t w = c.l[7 - k];
        out[4 * k] = (uint8_t)(w >> 24); out[4 * k + 1] = (uint8_t)(w >> 16);
        out[4 * k + 2] = (uint8_t)(w >> 8); out[4 * k + 3] = (uint8_t)w;
    }
}
// arkworks serialize_compressed (reference primitives/src/helpers.rs:458-460)
void serialize_compressed(const Affine& a, uint8_t out[32]);

// The transcript hashes every 32-byte chunk as a field element, so a big-endian value >= r is replaced by its residue
// (to_fr_array, helpers.rs:32-34).  Returns `in` when it is below r, else `out` holding in mod r (out may equal in).
const uint8_t* fr_reduce_chunk(const uint8_t in[32], uint8_t out[32]);

// Absorb tag || u64_be(n) || n canonical 32-byte evaluations (zero padded) -- everything of the
// compute_challenge transcript (helpers.rs:424-456) except the trailing commitment.
void challenge_midstate(Sha256& sh, const uint8_t* blob, size_t len, size_t n);
// Absorb the commitment and hash to the field (hash_to_field_element, helpers.rs:382-390).
Fr challenge_finish(Sha256 sh, const Affine& commitment);

// Blobs the multi-buffer and device hashers take: exactly 32 * 2^j bytes, j >= 10 (whole 64-byte blocks).
bool hash_mb_eligible(size_t len);
// Midstates of up to 16 blobs of exactly 32 n bytes each after tag || u64_be(n) || chunks 0 .. n-2 (all whole blocks),
// hashed in lockstep; out[m] = 8 state words.  Unused slots repeat blob 0.
void challenge_midstates_mb16(const uint8_t* const* blobs, size_t members, size_t n, uint32_t out[16][8]);
// challenge_midstate of a blob of exactly 32 n bytes from the raw state after tag || u64_be(n) || chunks 0 .. n-2
// (challenge_midstates_mb16, or the device's k_fs_midstate_long): appends the reduced last chunk.
Sha256 challenge_midstate_resume(const uint32_t state[8], const uint8_t* blob, size_t n);

}  // namespace kzgb
