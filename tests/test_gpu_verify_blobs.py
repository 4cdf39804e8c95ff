"""kzgb_verify_blob_proofs_g1{,_dev} and kzgb_group_verify_blob_proofs_g1: verify_blob_kzg_proof (verifier/src/verify.rs:77-115)
up to the pairing for a batch of blobs.  Entry i must be what kzgb_verify_blob_proof_g1 returns for (blob i, C_i, proof_i)
alone -- C_i - [y_i] G1, z_i and y_i -- through every hashing route of the shared per-blob stage, and the outputs must satisfy
the pairing relation (G1 form on a synthetic SRS with known tau, the real pairing on the reference's blob)."""
import ctypes as C
import random

import pytest

import golden_data as g
from __graft_entry__ import load_package
from oracle import bn254 as o

pytestmark = pytest.mark.gpu
TAU = o.SYNTH_TAU
FF = b"\xff" * 32
R_BYTES = o.R.to_bytes(32, "big")
OFF_CURVE = (1, 3)


@pytest.fixture(scope="module")
def pkg():
    return load_package()


def _with_large_chunks(rnd, nbytes):
    """Random bytes with chunks >= r: an all-0xff chunk, r itself, r + 1 and an all-0xff partial last chunk."""
    b = bytearray(rnd.randbytes(nbytes))
    for k, chunk in ((0, FF), (1, R_BYTES), (2, (o.R + 1).to_bytes(32, "big"))):
        if 32 * k + 32 <= nbytes:
            b[32 * k : 32 * k + 32] = chunk
    tail = nbytes % 32 or 32
    b[nbytes - tail :] = b"\xff" * tail
    return bytes(b)


def _ragged(rnd, with_2_16=True):
    """Lengths 1, 31, 32, 33, 500, 31*64, 32*2^12, [32*2^16,] then 300 blobs of 2^12 Fr.  Without the 2^16-Fr blob the
    batch is >= 256 blobs of <= 2^13 Fr, which the auto policy of option "fs_device" hashes on the device."""
    lens = [1, 31, 32, 33, 500, 31 * 64, 32 << 12] + ([32 << 16] if with_2_16 else []) + [32 << 12] * 300
    return [_with_large_chunks(rnd, k) for k in lens]


def _blobs(pkg, datas):
    return [pkg.Blob.from_unchecked(d) for d in datas]


def _mixed_inputs(pkg, srs, datas):
    """By i mod 5: an honest (C, proof) pair, the blob's C with the next blob's proof, an unrelated C with the blob's own
    proof, the identity as C and as proof, and the blob's C with the identity as proof."""
    blobs = _blobs(pkg, datas)
    cs = pkg.KZG.commit_blobs(blobs, srs)
    ps = pkg.KZG.compute_blob_proofs(blobs, cs, srs)
    m = len(datas)
    commitments, proofs = [], []
    for i in range(m):
        kind = i % 5
        commitments.append(None if kind == 3 else (o.g1_mul(o.G1_GEN, 7 + i) if kind == 2 else cs[i]))
        proofs.append(None if kind in (3, 4) else (ps[(i + 1) % m] if kind == 1 else ps[i]))
    return commitments, proofs


def _single(pkg, eng, datas, cs, ps):
    return [pkg.verify_blob_kzg_proof_g1(pkg.Blob.from_unchecked(d), c, p, eng) for d, c, p in zip(datas, cs, ps)]


def _host_ptrs(datas):
    keep = [C.create_string_buffer(d, max(1, len(d))) for d in datas]
    return keep, [C.cast(k, C.c_void_p).value for k in keep]


def _raw_verify(pkg, eng, host_ptrs, lens, cs, ps, dev_ptrs=None, out=None):
    """The C call on raw arguments; out = (xy, inf, z, y) buffers to write into (fresh ones by default).  Returns the
    entries as the mirror does, and the raw buffers."""
    count = len(lens)
    cxy, cinf = pkg.g1_to_abi(cs)
    pxy, pinf = pkg.g1_to_abi(ps)
    xy, inf, z, y = out or (C.create_string_buffer(64 * count or 1), C.create_string_buffer(count or 1),
                            C.create_string_buffer(32 * count or 1), C.create_string_buffer(32 * count or 1))
    hp, ln = (C.c_void_p * count)(*host_ptrs), (C.c_size_t * count)(*lens)
    if dev_ptrs is None:
        eng.check(pkg.lib.kzgb_verify_blob_proofs_g1(eng.h, hp, ln, count, cxy, cinf, pxy, pinf, xy, inf, z, y))
    else:
        eng.check(pkg.lib.kzgb_verify_blob_proofs_g1_dev(eng.h, (C.c_void_p * count)(*dev_ptrs), hp, ln, count, cxy, cinf,
                                                         pxy, pinf, xy, inf, z, y))
    outs = pkg.g1_from_abi(xy.raw[: 64 * count], inf.raw[:count])
    got = list(zip(outs, pkg.fr_from_mont_bytes(z.raw[: 32 * count]), pkg.fr_from_mont_bytes(y.raw[: 32 * count])))
    return got, (xy, inf, z, y)


def _set(pkg, name, value):
    assert pkg.lib.kzgb_set_option(name.encode(), value) == 0


@pytest.mark.parametrize("fs_device", [0, 1, -1])
def test_verify_blobs_equal_single_call(pkg, fs_device):
    """Entry i = kzgb_verify_blob_proof_g1(blob i, C_i, proof_i) on a ragged batch holding chunks >= r, with honest pairs,
    wrong proofs, unrelated commitments and identities, for every setting of option "fs_device"; with the auto setting
    the batch without its 2^16-Fr blob is hashed on the device."""
    rnd = random.Random(101 + fs_device)
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(1 << 16, TAU, engine=eng)
    try:
        for with_2_16 in (True, False):
            datas = _ragged(rnd, with_2_16)
            cs, ps = _mixed_inputs(pkg, srs, datas)
            want = _single(pkg, eng, datas, cs, ps)
            _set(pkg, "fs_device", fs_device)
            got = pkg.verify_blob_kzg_proofs_g1(_blobs(pkg, datas), cs, ps, eng)
            _set(pkg, "fs_device", -1)
            assert got == want
            assert len({e[1] for e in got}) == len(datas)  # every blob has a challenge of its own
    finally:
        _set(pkg, "fs_device", -1)
        eng.close()


def _relation_holds(entry, proof):
    """C - [y] G == (tau - z) proof: the G1 form of e(C - [y] G, G2) == e(proof, [tau - z] G2) when [tau] G2 is known."""
    out, z, _ = entry
    return out == o.g1_mul(proof, (TAU - z) % o.R)


def test_verify_blobs_pairing_relation_synthetic_tau(pkg):
    """Honest (C, proof) pairs of kzgb_commit_and_prove_blobs -- 40 blobs of 2^12 Fr and one of 2^19 Fr (16 MiB) -- satisfy
    out_i == (tau - z_i) proof_i on a synthetic SRS; a tampered blob, or a proof swapped in, breaks it at that index only."""
    import numpy as np

    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(1 << 19, TAU, engine=eng)
    rng = np.random.default_rng(8)
    datas = [rng.integers(0, 256, size=32 << 12, dtype=np.uint8).tobytes() for _ in range(40)]
    datas.insert(17, rng.integers(0, 256, size=32 << 19, dtype=np.uint8).tobytes())
    cs32, ps32 = pkg.KZG.commit_and_prove_blobs(_blobs(pkg, datas), srs)
    cs = [o.g1_deserialize_compressed(b) for b in cs32]
    ps = [o.g1_deserialize_compressed(b) for b in ps32]
    got = pkg.verify_blob_kzg_proofs_g1(_blobs(pkg, datas), cs, ps, eng)
    assert all(_relation_holds(e, p) for e, p in zip(got, ps))
    for k in (17, 30):
        tampered = list(datas)
        tampered[k] = bytes([tampered[k][0] ^ 1]) + tampered[k][1:]
        got = pkg.verify_blob_kzg_proofs_g1(_blobs(pkg, tampered), cs, ps, eng)
        assert [i for i, (e, p) in enumerate(zip(got, ps)) if not _relation_holds(e, p)] == [k]
        swapped = list(ps)
        swapped[k] = ps[k - 1]
        got = pkg.verify_blob_kzg_proofs_g1(_blobs(pkg, datas), cs, swapped, eng)
        assert [i for i, (e, p) in enumerate(zip(got, swapped)) if not _relation_holds(e, p)] == [k]
    eng.close()


def test_verify_blobs_reference_fixtures(pkg):
    """The Gettysburg blob on the reference's g1.point SRS: out, z, y = the oracle's C - [y] G, compute_challenge and
    evaluate_polynomial_in_evaluation_form.  The reference's blobs.txt blob (4096 Fr) on a synthetic 2^12 SRS with
    [tau] G2 injected: the real pairing of verify.rs:44-74 accepts the honest proof and rejects another blob's."""
    eng = pkg.Engine(0)
    srs = pkg.SRS.from_gnark_bytes(g.g1_point_bytes()[: 32 * 64], engine=eng)
    raw = g.gettysburg()
    blob = pkg.Blob.from_raw_data(raw)
    kzg = pkg.KZG()
    kzg.calculate_and_store_roots_of_unity(len(blob))
    c = kzg.commit_blob(blob, srs)
    pi = kzg.compute_blob_proof(blob, c, srs)
    bo = o.Blob.from_raw_data(raw)
    z = o.compute_challenge(bo, c)
    y = o.evaluate_polynomial_in_evaluation_form(bo.to_polynomial_eval_form(), z)
    want = (o.g1_add(c, o.g1_neg(o.g1_mul(o.G1_GEN, y))), z, y)
    assert pkg.verify_blob_kzg_proofs_g1([blob, blob], [c, c], [pi, pi], eng) == [want, want]
    eng.close()

    n = 1 << 12
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(n, TAU, engine=eng)
    g2_tau = o.g2_mul(o.G2_GEN, TAU)
    data = g.blobs_txt()
    rnd = random.Random(41)
    other = b"".join(rnd.randrange(o.R).to_bytes(32, "big") for _ in range(n))
    blobs = [pkg.Blob.new(data), pkg.Blob.new(other)]
    cs = pkg.KZG.commit_blobs(blobs, srs)
    ps = pkg.KZG.compute_blob_proofs(blobs, cs, srs)
    (out, z, _), (out_bad, z2, _) = pkg.verify_blob_kzg_proofs_g1([blobs[0], blobs[0]], [cs[0], cs[0]], [ps[0], ps[1]], eng)
    assert z2 == z == o.compute_challenge(o.Blob(data), cs[0])
    x_minus_z = o.g2_add(g2_tau, o.g2_neg(o.g2_mul(o.G2_GEN, z)))
    assert o.pairings_verify(out, o.G2_GEN, ps[0], x_minus_z)
    assert not o.pairings_verify(out_bad, o.G2_GEN, ps[1], x_minus_z)
    eng.close()


def test_verify_blobs_edge_values(pkg):
    """The exceptional branches of C + [-y] G: a constant blob p = v against its own commitment [v] G gives the identity
    (all-zero words, flag set); against [-v] G it gives [-2v] G (the doubling); an all-zero blob gives y = 0 and out = C.
    Each entry = the single call."""
    n = 1 << 12
    eng = pkg.Engine(0)
    rnd = random.Random(12)
    v = rnd.randrange(o.R)
    const = v.to_bytes(32, "big") * n
    zero = bytes(32 * n)
    proof = o.g1_mul(o.G1_GEN, 99)
    datas = [const, const, zero, const[: 32 * 64]]  # the last: p = v on a domain of 64
    cs = [o.g1_mul(o.G1_GEN, v), o.g1_mul(o.G1_GEN, o.R - v), o.g1_mul(o.G1_GEN, 5), o.g1_mul(o.G1_GEN, v)]
    ps = [proof] * 4
    keep, hptrs = _host_ptrs(datas)
    got, (xy, inf, _, _) = _raw_verify(pkg, eng, hptrs, [len(d) for d in datas], cs, ps)
    assert got == _single(pkg, eng, datas, cs, ps)
    assert got[0][0] is None and got[0][2] == v and xy.raw[:64] == bytes(64) and inf.raw[0] == 1
    assert got[3][0] is None and got[3][2] == v
    assert got[1][0] == o.g1_mul(o.G1_GEN, (-2 * v) % o.R) and inf.raw[1] == 0
    assert got[2][2] == 0 and got[2][0] == cs[2]
    eng.close()


def test_verify_blobs_errors(pkg):
    """A bad C at index 3 before a zero-length blob at index 5 is NotOnCurveError, the reverse order the reference's
    GenericError; a bad proof is rejected too, and so is a polynomial over 2^28 elements; each error is the single call's
    and leaves prefilled outputs untouched.  count == 0 writes nothing; lists of different lengths are the mirror's
    GenericError."""
    eng = pkg.Engine(0)
    rnd = random.Random(3)
    datas = [rnd.randbytes(32 * 64) for _ in range(7)]
    keep, hptrs = _host_ptrs(datas)
    good = [o.g1_mul(o.G1_GEN, 3 + i) for i in range(7)]
    huge = (32 << 28) + 1  # never read: the length check fails first
    cases = [  # (lens, commitments, proofs, the (len, C, proof) the single call fails on, variant)
        ([2048] * 5 + [0, 2048], good[:3] + [OFF_CURVE] + good[4:], good, (2048, OFF_CURVE, good[3]), "NotOnCurveError"),
        ([2048] * 3 + [0] + [2048] * 3, good[:5] + [OFF_CURVE, good[6]], good, (0, good[3], good[3]), "GenericError"),
        ([2048] * 7, good, good[:2] + [OFF_CURVE] + good[3:], (2048, good[2], OFF_CURVE), "NotOnCurveError"),
        ([2048] * 4 + [huge, 2048, 2048], good, good, (huge, good[4], good[4]), "GenericError"),
    ]
    for lens, cs, ps, (bad_len, bad_c, bad_p), variant in cases:
        cxy, cinf = pkg.g1_to_abi([bad_c])
        pxy, pinf = pkg.g1_to_abi([bad_p])
        with pytest.raises(pkg.KzgError) as single:
            eng.check(pkg.lib.kzgb_verify_blob_proof_g1(eng.h, hptrs[0], bad_len, cxy, cinf[0], pxy, pinf[0],
                                                        C.create_string_buffer(64), None, None, None))
        sentinel = (C.create_string_buffer(b"\xab" * 448, 448), C.create_string_buffer(b"\xcd" * 7, 7),
                    C.create_string_buffer(b"\xee" * 224, 224), C.create_string_buffer(b"\x11" * 224, 224))
        with pytest.raises(pkg.KzgError) as batch:
            _raw_verify(pkg, eng, hptrs, lens, cs, ps, out=sentinel)
        assert (batch.value.variant, batch.value.msg) == (single.value.variant, single.value.msg)
        assert batch.value.variant == variant
        assert [b.raw for b in sentinel] == [b"\xab" * 448, b"\xcd" * 7, b"\xee" * 224, b"\x11" * 224]
    sentinel = (C.create_string_buffer(b"\xab" * 64, 64), C.create_string_buffer(b"\xcd", 1),
                C.create_string_buffer(b"\xee" * 32, 32), C.create_string_buffer(b"\x11" * 32, 32))
    got, _ = _raw_verify(pkg, eng, [], [], [], [], out=sentinel)
    assert got == [] and [b.raw for b in sentinel] == [b"\xab" * 64, b"\xcd", b"\xee" * 32, b"\x11" * 32]
    assert pkg.lib.kzgb_verify_blob_proofs_g1_dev(eng.h, None, None, None, 0, None, None, None, None, None, None, None, None) == 0
    assert pkg.verify_blob_kzg_proofs_g1([], [], [], eng) == []
    with pytest.raises(pkg.KzgError) as mismatch:
        pkg.verify_blob_kzg_proofs_g1(_blobs(pkg, datas), good, good[:6], eng)
    assert (mismatch.value.variant, mismatch.value.msg) == ("GenericError", "length's of the input are not the same")
    want = _single(pkg, eng, datas, good, good)  # the context stays usable
    assert pkg.verify_blob_kzg_proofs_g1(_blobs(pkg, datas), good, good, eng) == want
    eng.close()


def test_verify_blobs_dev_equals_host(pkg):
    """kzgb_verify_blob_proofs_g1_dev = the host form with the blobs back to back in one device buffer (one conversion per
    run), and scattered over separate, unaligned buffers; on the device-hashed and the host-hashed routes."""
    import torch

    rnd = random.Random(66)
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(1 << 16, TAU, engine=eng)
    try:
        n = 1 << 12
        datas = [_with_large_chunks(rnd, 32 * n) for _ in range(300)]
        cs, ps = _mixed_inputs(pkg, srs, datas)
        keep, hptrs = _host_ptrs(datas)
        lens = [32 * n] * len(datas)
        run = torch.frombuffer(bytearray(b"".join(datas)), dtype=torch.uint8).cuda()
        for fs_device in (1, 0):
            _set(pkg, "fs_device", fs_device)
            want, _ = _raw_verify(pkg, eng, hptrs, lens, cs, ps)
            got, _ = _raw_verify(pkg, eng, hptrs, lens, cs, ps, dev_ptrs=[run.data_ptr() + 32 * n * i for i in range(len(datas))])
            assert got == want
        _set(pkg, "fs_device", -1)
        for with_2_16 in (False, True):
            datas = _ragged(rnd, with_2_16)
            cs, ps = _mixed_inputs(pkg, srs, datas)
            want = pkg.verify_blob_kzg_proofs_g1(_blobs(pkg, datas), cs, ps, eng)
            keep, hptrs = _host_ptrs(datas)
            bufs = [torch.frombuffer(bytearray(b"\x00" * 3 + d + b"\x00" * 5), dtype=torch.uint8).cuda() for d in datas]
            got, _ = _raw_verify(pkg, eng, hptrs, [len(d) for d in datas], cs, ps, dev_ptrs=[b.data_ptr() + 3 for b in bufs])
            assert got == want
    finally:
        _set(pkg, "fs_device", -1)
        eng.close()


def _device_sets():
    import torch

    sets = [[0, 0], [0, 0, 0]]
    n = torch.cuda.device_count()
    if n >= 2:
        sets.append([0, 1])
    if n >= 4:
        sets.append(list(range(n)))
    return sets


@pytest.mark.parametrize("devices", _device_sets() if __import__("torch").cuda.is_available() else [[0, 0]])
def test_group_verify_blobs_equal_single_context(pkg, devices):
    """kzgb_group_verify_blob_proofs_g1 = the one-context call on a ragged batch cut across the members, on fewer blobs
    than members, and on none."""
    rnd = random.Random(len(devices) * 5 + devices[-1])
    datas = [_with_large_chunks(rnd, k) for k in (31 * 64, 31 * 33, 31, 1, 31 * 200, 31 * 128, 500, 32 * 300 + 5)]
    datas += [_with_large_chunks(rnd, 32 << 12) for _ in range(20)]
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(1 << 12, TAU, engine=eng)
    cs, ps = _mixed_inputs(pkg, srs, datas)
    want = pkg.verify_blob_kzg_proofs_g1(_blobs(pkg, datas), cs, ps, eng)
    eng.close()
    grp = pkg.Group(devices)
    assert grp.verify_blob_kzg_proofs_g1(_blobs(pkg, datas), cs, ps) == want
    assert grp.verify_blob_kzg_proofs_g1(_blobs(pkg, datas[:1]), cs[:1], ps[:1]) == want[:1]
    assert grp.verify_blob_kzg_proofs_g1([], [], []) == []
    # out_xy == NULL, as the one-context call allows it: z and y only, every member writing its own share
    _keep, ptrs, lens = pkg._blobs_to_abi(_blobs(pkg, datas))
    cxy, cinf = pkg.g1_to_abi(cs)
    pxy, pinf = pkg.g1_to_abi(ps)
    z, y = C.create_string_buffer(32 * len(datas)), C.create_string_buffer(32 * len(datas))
    grp.check(pkg.lib.kzgb_group_verify_blob_proofs_g1(grp.h, ptrs, lens, len(datas), cxy, cinf, pxy, pinf, None, None, z, y))
    assert pkg.fr_from_mont_bytes(z.raw) == [w[1] for w in want]
    assert pkg.fr_from_mont_bytes(y.raw) == [w[2] for w in want]
    grp.close()
