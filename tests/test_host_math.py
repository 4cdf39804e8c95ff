"""CPU checks of the library's HOST-side math (same field.cuh/ec.cuh source the kernels use,
compiled for the host), the PTX generator's emulator, SHA-256, and the host-only C-ABI calls."""
import ctypes as C
import hashlib
import os
import random
import subprocess
import sys

import pytest

from oracle import bn254 as o

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
MONT = 1 << 256


@pytest.fixture(scope="module")
def hm():
    src = os.path.join(HERE, "native", "host_math_test.cpp")
    out = os.path.join(HERE, "native", "libhostmath_test.so")
    csrc = os.path.join(ROOT, "rust-kzg-bn254_b200", "csrc")
    sha, transcript = os.path.join(csrc, "sha256.cpp"), os.path.join(csrc, "transcript.cpp")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", out, src, sha, transcript])
    return C.CDLL(out)


def le(x):
    return x.to_bytes(32, "little")


def call2(fn, a, b):
    out = C.create_string_buffer(32)
    fn(out, le(a), le(b))
    return int.from_bytes(out.raw, "little")


def call1(fn, a):
    out = C.create_string_buffer(32)
    fn(out, le(a))
    return int.from_bytes(out.raw, "little")


def test_ptx_generator_emulator():
    sys.path.insert(0, os.path.join(ROOT, "rust-kzg-bn254_b200", "csrc"))
    import gen_field

    gen_field.selftest(iters=60)
    # the committed generated header is what the generator produces now
    cur = open(os.path.join(ROOT, "rust-kzg-bn254_b200", "csrc", "field_gen.cuh")).read()
    assert cur == gen_field.emit_header()


@pytest.mark.parametrize("squaring", [False, True])
def test_relaxed_madd_sequence_on_the_emulator(squaring):
    """squaring: PP and R^2 through the dedicated squaring (gen_field.py sqrnr; k_accumulate uses it for PP).
    The accumulation loop's XYZZ += affine on relaxed [0, 2p) coordinates (ec.cuh xyzz_madd_relaxed), replayed
    instruction by instruction on the PTX emulator: after every addition all coordinates stay below 2p and the
    accumulator equals the oracle's sum -- the carry chains and range invariants checked without a GPU."""
    sys.path.insert(0, os.path.join(ROOT, "rust-kzg-bn254_b200", "csrc"))
    import gen_field as gf
    import golden_data as g

    P = o.P
    mont = lambda v: v * MONT % P
    unmont = lambda v: v * pow(MONT, -1, P) % P
    mulnr = lambda a, b: gf.emulate("fq", "mulnr", a, b)
    sqrnr = (lambda a: gf.emulate("fq", "sqrnr", a)) if squaring else (lambda a: mulnr(a, a))
    sub2p = lambda a, b: gf.emulate("fq", "sub2p", a, b)
    pts = g.srs_points_string()[3:12]
    # a P + (-P) pair and a doubling are handled by the exceptional paths in the kernel; here: distinct points
    x, y = pts[0]
    acc = [mont(x), mont(y), mont(1), mont(1)]  # X, Y, ZZ, ZZZ
    expect = pts[0]
    for q in pts[1:]:
        qx, qy = mont(q[0]), mont(q[1])
        U2 = mulnr(qx, acc[2])
        S2 = mulnr(qy, acc[3])
        Pp = sub2p(U2, acc[0])
        Rr = sub2p(S2, acc[1])
        assert Pp % P != 0
        PP = sqrnr(Pp)
        PPP = mulnr(Pp, PP)
        Q = mulnr(acc[0], PP)
        zz = mulnr(acc[2], PP)
        zzz = mulnr(acc[3], PPP)
        t = sqrnr(Rr)
        t = sub2p(t, PPP)
        t = sub2p(t, Q)
        t = sub2p(t, Q)
        Q = sub2p(Q, t)
        y3 = gf.emulate("fq", "mul2subnr", Rr, Q, acc[1], PPP)
        acc = [t, y3, zz, zzz]
        assert all(v < 2 * P for v in acc)
        expect = o.g1_add(expect, q)
        X, Y, ZZ, ZZZ = (unmont(v % P) for v in acc)
        assert (X * pow(ZZ, -1, P) % P, Y * pow(ZZZ, -1, P) % P) == expect
    # normalisation at the end of the loop
    assert [gf.emulate("fq", "reduce_once", v) for v in acc] == [v % P for v in acc]


def test_host_field_ops(hm):
    rnd = random.Random(7)
    for mod, mul, add, sub, inv in (
        (o.P, hm.t_fq_mul, hm.t_fq_add, hm.t_fq_sub, hm.t_fq_inv),
        (o.R, hm.t_fr_mul, hm.t_fr_add, hm.t_fr_sub, hm.t_fr_inv),
    ):
        rinv = pow(MONT, -1, mod)
        edge = [0, 1, mod - 1, mod - 2, (mod - 1) // 2, MONT % mod]
        cases = [(x, y) for x in edge for y in edge] + [(rnd.randrange(mod), rnd.randrange(mod)) for _ in range(300)]
        for x, y in cases:
            assert call2(mul, x, y) == x * y * rinv % mod
            assert call2(add, x, y) == (x + y) % mod
            assert call2(sub, x, y) == (x - y) % mod
        for _ in range(20):  # word operand may be any 256-bit value
            x, y = rnd.randrange(mod), rnd.randrange(1 << 256)
            assert call2(mul, x, y) == x * y * rinv % mod
        for _ in range(5):
            x = rnd.randrange(1, mod)
            xm = x * MONT % mod
            assert call1(inv, xm) == pow(x, -1, mod) * MONT % mod


def test_montgomery_reduce_kats(hm):
    """The reference's own montgomery_reduce vectors semantics (primitives/src/arith.rs:4-55):
    from_mont(z) == z * 2^-256 mod p."""
    rnd = random.Random(11)
    for _ in range(50):
        z = rnd.randrange(o.P)
        limbs = [(z >> (64 * i)) & ((1 << 64) - 1) for i in range(4)]
        exp = o.montgomery_reduce(*limbs)
        got = call1(hm.t_fq_from_mont, z)
        assert got == sum(v << (64 * i) for i, v in enumerate(exp))


def test_lexicographically_largest(hm):
    for y in (0, 1, (o.P - 1) // 2, (o.P - 1) // 2 + 1, o.P - 1, 12345):
        assert hm.t_fq_lex_largest(le(y * MONT % o.P)) == (1 if o.lexicographically_largest(y) else 0)


def _aff_bytes(pt):
    if pt is None:
        return bytes(64)
    return le(pt[0] * MONT % o.P) + le(pt[1] * MONT % o.P)


def _xyzz_from_aff(pt):
    if pt is None:
        return bytes(128)
    one = le(MONT % o.P)
    return _aff_bytes(pt) + one + one


def _xyzz_to_aff(hm, buf):
    out = C.create_string_buffer(64)
    hm.t_to_affine(out, buf)
    raw = out.raw
    if not any(raw):
        return None
    rinv = pow(MONT, -1, o.P)
    return (int.from_bytes(raw[:32], "little") * rinv % o.P, int.from_bytes(raw[32:], "little") * rinv % o.P)


def test_xyzz_group_law_including_exceptional_cases(hm):
    rnd = random.Random(5)
    G = o.G1_GEN
    pts = [o.g1_mul(G, rnd.randrange(1, o.R)) for _ in range(6)]
    for a in pts[:3]:
        for b in pts[3:] + [a, o.g1_neg(a), None]:
            acc = C.create_string_buffer(_xyzz_from_aff(a), 128)
            hm.t_madd(acc, _aff_bytes(b))
            assert _xyzz_to_aff(hm, acc) == o.g1_add(a, b)
            acc2 = C.create_string_buffer(_xyzz_from_aff(a), 128)
            hm.t_add(acc2, _xyzz_from_aff(b))
            assert _xyzz_to_aff(hm, acc2) == o.g1_add(a, b)
    # identity accumulator
    acc = C.create_string_buffer(bytes(128), 128)
    hm.t_madd(acc, _aff_bytes(pts[0]))
    assert _xyzz_to_aff(hm, acc) == pts[0]
    # non-trivial ZZ: build 5P + Q with projective intermediates, doubling in the middle
    acc = C.create_string_buffer(_xyzz_from_aff(pts[0]), 128)
    hm.t_madd(acc, _aff_bytes(pts[1]))
    d = C.create_string_buffer(128)
    hm.t_dbl(d, acc)
    hm.t_add(d, acc)  # 3(P0+P1)
    assert _xyzz_to_aff(hm, d) == o.g1_mul(o.g1_add(pts[0], pts[1]), 3)
    hm.t_add(d, d)  # aliasing + doubling path of the general add
    assert _xyzz_to_aff(hm, d) == o.g1_mul(o.g1_add(pts[0], pts[1]), 6)
    m = C.create_string_buffer(128)
    hm.t_mul_small(m, acc, 29877)
    assert _xyzz_to_aff(hm, m) == o.g1_mul(o.g1_add(pts[0], pts[1]), 29877)
    assert hm.t_on_curve(_aff_bytes(pts[2])) == 1
    assert hm.t_on_curve(_aff_bytes((pts[2][0], (pts[2][1] + 1) % o.P))) == 0
    assert hm.t_on_curve(bytes(64)) == 1


def test_sha256_matches_hashlib(hm):
    rnd = random.Random(3)
    for n in (0, 1, 55, 56, 63, 64, 65, 119, 120, 1000, 4096 + 17, 70001):
        data = bytes(rnd.getrandbits(8) for _ in range(n))
        out = C.create_string_buffer(32)
        hm.t_sha256(data, n, out)
        assert out.raw == hashlib.sha256(data).digest()
        for step in (1, 7, 64, 100):
            if n and n <= 5000:
                hm.t_sha256_chunked(data, n, step, out)
                assert out.raw == hashlib.sha256(data).digest()


def test_sha256_multibuffer_matches_single_stream(hm):
    """AVX-512 multi-buffer SHA-256 (16 messages in lockstep, sha256.cpp sha256_mb16_blocks): the chaining state after
    nblk blocks of each of the 16 messages equals the single-stream implementation's (itself checked against hashlib
    above), with and without the per-block fix-up hook (which must see exactly the blocks with a flagged chunk)."""
    if not hm.t_has_mb16():
        pytest.skip("no AVX-512 on this host")
    rnd = random.Random(5)
    for nblk in (1, 2, 3, 17, 64):
        msgs = bytearray(rnd.getrandbits(8) for _ in range(16 * 64 * nblk))
        out = (C.c_uint32 * 128)()
        hm.t_sha256_mb16(bytes(msgs), nblk, 0, out)
        for m in range(16):
            one = (C.c_uint32 * 8)()
            hm.t_sha256_state(bytes(msgs[m * 64 * nblk : (m + 1) * 64 * nblk]), nblk, one)
            assert list(out[8 * m : 8 * m + 8]) == list(one), (nblk, m)
        # fix-up hook: reference = apply the same rewrite to the message, then hash it plainly
        hm.t_sha256_mb16(bytes(msgs), nblk, 1, out)
        fixed = bytearray(msgs)
        for off in range(0, len(fixed), 32):
            if fixed[off] >= 0x30:
                fixed[off + 1] ^= 0xFF
        for m in range(16):
            one = (C.c_uint32 * 8)()
            hm.t_sha256_state(bytes(fixed[m * 64 * nblk : (m + 1) * 64 * nblk]), nblk, one)
            assert list(out[8 * m : 8 * m + 8]) == list(one), ("fix", nblk, m)


def test_safegcd_inverse_matches_bigint(hm):
    """fe_inv_fast (Bernstein-Yang division steps, 30-bit batches) against pow(a, -1, p): edge values,
    every bit length, random elements; 0 -> 0 like the Fermat inverse."""
    rnd = random.Random(11)
    for mod, fn in ((o.P, hm.t_fq_inv_fast), (o.R, hm.t_fr_inv_fast)):
        vals = [1, 2, 3, mod - 1, mod - 2, (mod - 1) // 2, (mod + 1) // 2, 1 << 253, (1 << 253) + 1, MONT % mod,
                pow(MONT, -1, mod)]
        vals += [rnd.randrange(1, mod) for _ in range(3000)]
        vals += [rnd.randrange(1 << (k - 1), 1 << k) for k in range(1, 254)]
        for a in vals:
            assert call1(fn, a * MONT % mod) == pow(a, -1, mod) * MONT % mod, hex(a)
        assert call1(fn, 0) == 0


def _transcript_blobs(count, n, seed):
    """count blobs of n random 32-byte chunks, each with values >= r in block 0 (chunk 0), in the middle and in the last
    chunk, plus an all-0xff chunk; the other chunks are random bytes, so about a fifth of them are >= r as well."""
    rnd = random.Random(seed)
    blobs = []
    for k in range(count):
        chunks = [rnd.getrandbits(256).to_bytes(32, "big") for _ in range(n)]
        chunks[0] = (o.R + rnd.randrange(1 << 200)).to_bytes(32, "big")
        chunks[n // 2 + k] = (o.R + k).to_bytes(32, "big")
        chunks[n - 1] = ((1 << 256) - 1 - k).to_bytes(32, "big")
        chunks[1 + k] = b"\xff" * 32
        blobs.append(b"".join(chunks))
    return blobs


def _transcript_digest(blob, n):
    """The compute_challenge transcript without the commitment, every chunk as a field element (helpers.rs:32-34)."""
    chunks = [(int.from_bytes(blob[i : i + 32], "big") % o.R).to_bytes(32, "big") for i in range(0, len(blob), 32)]
    return hashlib.sha256(b"EIGENDA_FSBLOBVERIFY_V1_" + n.to_bytes(8, "big") + b"".join(chunks)).digest()


@pytest.mark.parametrize("members", [16, 9])
def test_multibuffer_transcript_midstates_equal_single_stream(hm, members):
    """The multi-buffer hashing of the blob-batch pipeline (transcript.cpp challenge_midstates_mb16, a full and a partial
    group of equal-size blobs), each finished by challenge_midstate_resume, equals challenge_midstate of the blob and the
    transcript hashed here from the reduced chunks."""
    if not hm.t_has_mb16():
        pytest.skip("no AVX-512 on this host")
    n = 1024
    blobs = _transcript_blobs(members, n, seed=members)
    out = C.create_string_buffer(32 * members)
    hm.t_challenge_midstates_mb16(b"".join(blobs), C.c_size_t(members), C.c_size_t(n), out)
    for m, blob in enumerate(blobs):
        single = C.create_string_buffer(32)
        hm.t_challenge_midstate(blob, C.c_size_t(len(blob)), C.c_size_t(n), single)
        assert single.raw == _transcript_digest(blob, n), m
        assert out.raw[32 * m : 32 * m + 32] == single.raw, m


def test_resumed_transcript_midstate_equals_single_stream(hm):
    """The host half of the device-hashed share: a state taken after chunks 0 .. n-2 and finished by
    challenge_midstate_resume (which appends the last chunk reduced mod r) equals challenge_midstate."""
    n = 1024
    for blob in _transcript_blobs(3, n, seed=3):
        single, resumed = C.create_string_buffer(32), C.create_string_buffer(32)
        hm.t_challenge_midstate(blob, C.c_size_t(len(blob)), C.c_size_t(n), single)
        hm.t_challenge_midstate_resumed(blob, C.c_size_t(n), resumed)
        assert single.raw == _transcript_digest(blob, n)
        assert resumed.raw == single.raw
