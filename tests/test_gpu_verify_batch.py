"""The batch verification in its device-resident and multi-GPU forms, and the RLC over evaluated openings:
kzgb_verify_batch_rlc_dev, kzgb_group_verify_batch_rlc and kzgb_verify_kzg_proof_batch_rlc (verifier/src/batch.rs:16-249 up
to the pairing).  Each must give the words of kzgb_verify_batch_rlc -- lhs and rhs are unique group elements, so equal
means bit-identical --, the same errors, and outputs that satisfy the pairing relation rhs == tau * lhs in G1 on a synthetic
SRS of known tau (the G1 form of e(lhs, [tau] G2) == e(rhs, G2))."""
import ctypes as C
import random

import pytest

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


def _ragged(rnd):
    """Lengths 1, 31, 33, 500 and 31 * 64 (partial last chunks), 40 blobs of 2^12 Fr, one of 2^16 Fr, three of 2^12 Fr and
    a 2^16-Fr blob with a partial last chunk."""
    lens = [1, 31, 33, 500, 31 * 64] + [32 << 12] * 40 + [32 << 16] + [32 << 12] * 3 + [(32 << 16) - 17]
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


def _host_ptrs(datas):
    keep = [C.create_string_buffer(d, max(1, len(d))) for d in datas]
    return keep, [C.cast(k, C.c_void_p).value for k in keep]


def _out():
    return (C.create_string_buffer(64), C.c_uint8(0), C.create_string_buffer(64), C.c_uint8(0))


def _sentinel():
    return (C.create_string_buffer(b"\xab" * 64, 64), C.c_uint8(7), C.create_string_buffer(b"\xcd" * 64, 64), C.c_uint8(9))


def _words(out):
    """(lhs words, lhs flag, rhs words, rhs flag) of an output set."""
    return (out[0].raw, out[1].value, out[2].raw, out[3].value)


def _points(pkg, out):
    return pkg.g1_from_abi(out[0].raw, bytes([out[1].value]))[0], pkg.g1_from_abi(out[2].raw, bytes([out[3].value]))[0]


def _rlc_raw(pkg, eng, host_ptrs, lens, cs, ps, dev_ptrs=None, out=None):
    """kzgb_verify_batch_rlc, or kzgb_verify_batch_rlc_dev with dev_ptrs, on raw arguments; returns the output set."""
    count = len(lens)
    cxy, cinf = pkg.g1_to_abi(cs)
    pxy, pinf = pkg.g1_to_abi(ps)
    out = out or _out()
    hp, ln = (C.c_void_p * count)(*host_ptrs), (C.c_size_t * count)(*lens)
    tail = (out[0], C.byref(out[1]), out[2], C.byref(out[3]))
    if dev_ptrs is None:
        eng.check(pkg.lib.kzgb_verify_batch_rlc(eng.h, hp, ln, count, cxy, cinf, pxy, pinf, *tail))
    else:
        eng.check(pkg.lib.kzgb_verify_batch_rlc_dev(eng.h, (C.c_void_p * count)(*dev_ptrs), hp, ln, count, cxy, cinf, pxy,
                                                    pinf, *tail))
    return out


def _group_raw(pkg, grp, host_ptrs, lens, cs, ps, out=None):
    count = len(lens)
    cxy, cinf = pkg.g1_to_abi(cs)
    pxy, pinf = pkg.g1_to_abi(ps)
    out = out or _out()
    grp.check(pkg.lib.kzgb_group_verify_batch_rlc(grp.h, (C.c_void_p * count)(*host_ptrs), (C.c_size_t * count)(*lens), count,
                                                  cxy, cinf, pxy, pinf, out[0], C.byref(out[1]), out[2], C.byref(out[3])))
    return out


def _openings_raw(pkg, eng, cs, ps, z_words, y_words, ns, out=None):
    """kzgb_verify_kzg_proof_batch_rlc on raw Montgomery words of z and y."""
    count = len(cs)
    cxy, cinf = pkg.g1_to_abi(cs)
    pxy, pinf = pkg.g1_to_abi(ps)
    out = out or _out()
    eng.check(pkg.lib.kzgb_verify_kzg_proof_batch_rlc(eng.h, count, cxy, cinf, pxy, pinf, z_words, y_words,
                                                      (C.c_uint64 * max(1, count))(*ns), out[0], C.byref(out[1]), out[2],
                                                      C.byref(out[3])))
    return out


def _zy_words(pkg, eng, datas, cs, ps, with_out=True):
    """The raw z and y words of kzgb_verify_blob_proofs_g1 (out_xy passed, or NULL)."""
    count = len(datas)
    keep, hptrs = _host_ptrs(datas)
    cxy, cinf = pkg.g1_to_abi(cs)
    pxy, pinf = pkg.g1_to_abi(ps)
    z, y = C.create_string_buffer(32 * count), C.create_string_buffer(32 * count)
    xy = C.create_string_buffer(64 * count) if with_out else None
    inf = C.create_string_buffer(count) if with_out else None
    eng.check(pkg.lib.kzgb_verify_blob_proofs_g1(eng.h, (C.c_void_p * count)(*hptrs), (C.c_size_t * count)(*[len(d) for d in datas]),
                                                 count, cxy, cinf, pxy, pinf, xy, inf, z, y))
    return z.raw, y.raw


def _poly_lens(datas):
    return [o.next_power_of_two(-(-len(d) // 32)) for d in datas]


def _set(pkg, name, value):
    assert pkg.lib.kzgb_set_option(name.encode(), value) == 0


def _honest(pkg, srs, datas):
    cs32, ps32 = pkg.KZG.commit_and_prove_blobs(_blobs(pkg, datas), srs)
    return [o.g1_deserialize_compressed(b) for b in cs32], [o.g1_deserialize_compressed(b) for b in ps32]


@pytest.mark.parametrize("fs_device", [0, 1, -1])
def test_dev_equals_host(pkg, fs_device):
    """kzgb_verify_batch_rlc_dev = kzgb_verify_batch_rlc word for word on a ragged batch (2^12, 2^16 and one 2^19 blob,
    partial last chunks, chunks >= r, identities), with the blobs back to back in one device buffer and scattered over
    separate buffers at odd offsets, for every setting of option "fs_device"."""
    import torch

    rnd = random.Random(700 + fs_device)
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(1 << 16, TAU, engine=eng)
    try:
        datas = _ragged(rnd)
        cs, ps = _mixed_inputs(pkg, srs, datas)
        # one 2^19-Fr blob with a partial last chunk, with an unrelated (C, proof): the SRS holds 2^16 points
        datas.insert(46, _with_large_chunks(rnd, (32 << 19) - 5))
        cs.insert(46, o.g1_mul(o.G1_GEN, 1234))
        ps.insert(46, o.g1_mul(o.G1_GEN, 4321))
        lens = [len(d) for d in datas]
        keep, hptrs = _host_ptrs(datas)
        _set(pkg, "fs_device", fs_device)
        want = _words(_rlc_raw(pkg, eng, hptrs, lens, cs, ps))
        offs, pos = [], 0
        for d in datas:
            offs.append(pos)
            pos += len(d)
        run = torch.frombuffer(bytearray(b"".join(datas)), dtype=torch.uint8).cuda()
        got = _words(_rlc_raw(pkg, eng, hptrs, lens, cs, ps, dev_ptrs=[run.data_ptr() + k for k in offs]))
        assert got == want
        bufs = [torch.frombuffer(bytearray(b"\x00" * 3 + d + b"\x00" * 5), dtype=torch.uint8).cuda() for d in datas]
        got = _words(_rlc_raw(pkg, eng, hptrs, lens, cs, ps, dev_ptrs=[b.data_ptr() + 3 for b in bufs]))
        assert got == want
        # full 2^12-Fr blobs back to back: the device form converts each run in one launch
        full = [_with_large_chunks(rnd, 32 << 12) for _ in range(300)]
        fcs, fps = _mixed_inputs(pkg, srs, full)
        keep2, fptrs = _host_ptrs(full)
        want = _words(_rlc_raw(pkg, eng, fptrs, [32 << 12] * 300, fcs, fps))
        frun = torch.frombuffer(bytearray(b"".join(full)), dtype=torch.uint8).cuda()
        got = _words(_rlc_raw(pkg, eng, fptrs, [32 << 12] * 300, fcs, fps,
                              dev_ptrs=[frun.data_ptr() + (32 << 12) * i for i in range(300)]))
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
def test_group_equals_single_context(pkg, devices):
    """kzgb_group_verify_batch_rlc = the one-context call on a ragged batch with identities among commitments and proofs,
    on a batch with one 2^19-Fr blob carrying almost all the bytes (every other member's share empty or tiny), on fewer
    blobs than members, and on none (identities)."""
    rnd = random.Random(len(devices) * 7 + devices[-1])
    datas = [_with_large_chunks(rnd, k) for k in (31 * 64, 31 * 33, 31, 1, 31 * 200, 31 * 128, 500, 32 * 300 + 5)]
    datas += [_with_large_chunks(rnd, 32 << 12) for _ in range(20)]
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(1 << 12, TAU, engine=eng)
    cs, ps = _mixed_inputs(pkg, srs, datas)
    heavy = datas[:3] + [_with_large_chunks(rnd, 32 << 19)] + datas[3:5]
    hcs = cs[:3] + [o.g1_mul(o.G1_GEN, 77)] + cs[3:5]
    hps = ps[:3] + [o.g1_mul(o.G1_GEN, 78)] + ps[3:5]
    cases = [(datas, cs, ps), (heavy, hcs, hps), (datas[:1], cs[:1], ps[:1]), ([], [], [])]
    want = [pkg.verify_blob_kzg_proof_batch_rlc(_blobs(pkg, d), c, p, eng) for d, c, p in cases]
    wwords = []
    for d, c, p in cases:
        keep, hptrs = _host_ptrs(d)
        wwords.append(_words(_rlc_raw(pkg, eng, hptrs, [len(x) for x in d], c, p)))
    eng.close()
    assert want[3] == (None, None) and wwords[3] == (bytes(64), 1, bytes(64), 1)
    grp = pkg.Group(devices)
    for (d, c, p), w, ww in zip(cases, want, wwords):
        assert grp.verify_blob_kzg_proof_batch_rlc(_blobs(pkg, d), c, p) == w
        keep, hptrs = _host_ptrs(d)
        assert _words(_group_raw(pkg, grp, hptrs, [len(x) for x in d], c, p)) == ww
    grp.close()


def test_openings_equal_blob_form_and_oracle(pkg):
    """kzgb_verify_kzg_proof_batch_rlc over the z and y that kzgb_verify_blob_proofs_g1 returns, with n_i of each blob,
    = kzgb_verify_batch_rlc bit for bit; on a small batch both = the oracle's verify_kzg_proof_batch_rlc; changing one n_i
    changes the output (the lengths are hashed); a z or y word >= r is InvalidFieldElement, outputs untouched."""
    rnd = random.Random(5150)
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(1 << 16, TAU, engine=eng)
    datas = [_with_large_chunks(rnd, k) for k in (1, 33, 31 * 64, 32 << 12, 32 << 12, (32 << 16) - 1)]
    datas += [_with_large_chunks(rnd, 32 << 12) for _ in range(294)]
    cs, ps = _mixed_inputs(pkg, srs, datas)
    ns = _poly_lens(datas)
    keep, hptrs = _host_ptrs(datas)
    want = _words(_rlc_raw(pkg, eng, hptrs, [len(d) for d in datas], cs, ps))
    zw, yw = _zy_words(pkg, eng, datas, cs, ps)
    assert _words(_openings_raw(pkg, eng, cs, ps, zw, yw, ns)) == want
    zs, ys = pkg.fr_from_mont_bytes(zw), pkg.fr_from_mont_bytes(yw)
    assert pkg.verify_kzg_proof_batch_rlc(cs, zs, ys, ps, ns, eng) == _points(pkg, _openings_raw(pkg, eng, cs, ps, zw, yw, ns))

    # small m against the oracle, from both entry points
    small = slice(0, 6)
    ref = o.verify_kzg_proof_batch_rlc(cs[small], zs[small], ys[small], ps[small], ns[small])
    assert pkg.verify_kzg_proof_batch_rlc(cs[small], zs[small], ys[small], ps[small], ns[small], eng) == ref
    assert pkg.verify_blob_kzg_proof_batch_rlc(_blobs(pkg, datas[small]), cs[small], ps[small], eng) == ref
    rz, ry = [rnd.randrange(o.R) for _ in range(5)], [rnd.randrange(o.R) for _ in range(5)]
    rc_ = [o.g1_mul(o.G1_GEN, rnd.randrange(1, o.R)) for _ in range(4)] + [None]
    rp = [None] + [o.g1_mul(o.G1_GEN, rnd.randrange(1, o.R)) for _ in range(4)]
    rn = [1, 2, 4096, 65536, 1 << 28]
    assert pkg.verify_kzg_proof_batch_rlc(rc_, rz, ry, rp, rn, eng) == o.verify_kzg_proof_batch_rlc(rc_, rz, ry, rp, rn)

    # the lengths are hashed as given
    for k in (0, 150):
        changed = list(ns)
        changed[k] *= 2
        assert _words(_openings_raw(pkg, eng, cs, ps, zw, yw, changed)) != want

    # words >= r: r itself, r + 1, all ones -- in z or in y, at index 3
    rw = o.R.to_bytes(32, "little")
    for bad in (rw, (o.R + 1).to_bytes(32, "little"), FF):
        for which in ("z", "y"):
            z2, y2 = bytearray(zw), bytearray(yw)
            (z2 if which == "z" else y2)[96:128] = bad
            out = _sentinel()
            with pytest.raises(pkg.KzgError) as err:
                _openings_raw(pkg, eng, cs, ps, bytes(z2), bytes(y2), ns, out=out)
            assert err.value.variant == "InvalidFieldElement"
            assert _words(out) == _words(_sentinel())
    # the largest reduced word, r - 1, is accepted
    y2 = bytearray(yw)
    y2[96:128] = (o.R - 1).to_bytes(32, "little")
    _openings_raw(pkg, eng, cs, ps, zw, bytes(y2), ns)
    eng.close()


def _relation(lhs, rhs):
    return rhs == o.g1_mul(lhs, TAU) if lhs is not None else rhs is None


def test_pairing_relation_every_form(pkg):
    """Honest pairs of kzgb_commit_and_prove_blobs (60 blobs of 2^12 Fr, one of 2^16 Fr) satisfy rhs == tau lhs in the
    host, device, group and openings forms on a synthetic SRS; one tampered proof breaks it in each, and so does one
    tampered y_i in the openings form."""
    import torch

    rnd = random.Random(99)
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(1 << 16, TAU, engine=eng)
    datas = [b"".join(rnd.randrange(o.R).to_bytes(32, "big") for _ in range(1 << 12)) for _ in range(60)]
    datas.insert(25, rnd.randbytes(32 << 16))
    cs, ps = _honest(pkg, srs, datas)
    lens = [len(d) for d in datas]
    keep, hptrs = _host_ptrs(datas)
    bufs = [torch.frombuffer(bytearray(d), dtype=torch.uint8).cuda() for d in datas]
    grp = pkg.Group([0, 0])
    zw, yw = _zy_words(pkg, eng, datas, cs, ps)
    ns = _poly_lens(datas)

    def forms(proofs, y_words=yw):
        return {
            "host": _points(pkg, _rlc_raw(pkg, eng, hptrs, lens, cs, proofs)),
            "dev": _points(pkg, _rlc_raw(pkg, eng, hptrs, lens, cs, proofs, dev_ptrs=[b.data_ptr() for b in bufs])),
            "group": _points(pkg, _group_raw(pkg, grp, hptrs, lens, cs, proofs)),
            "openings": _points(pkg, _openings_raw(pkg, eng, cs, proofs, zw, y_words, ns)),
        }

    got = forms(ps)
    assert all(_relation(*v) for v in got.values()), got
    assert len(set(got.values())) == 1
    for k in (0, 25):
        bad = list(ps)
        bad[k] = o.g1_add(ps[k], o.G1_GEN)
        assert not any(_relation(*v) for v in forms(bad).values())
    y2 = bytearray(yw)
    y2[32 * 7 : 32 * 8] = pkg.fr_to_mont_bytes([(pkg.fr_from_mont_bytes(yw[32 * 7 : 32 * 8])[0] + 1) % o.R])
    assert not _relation(*_points(pkg, _openings_raw(pkg, eng, cs, ps, zw, bytes(y2), ns)))
    grp.close()
    eng.close()


def test_errors_same_in_every_form(pkg):
    """An off-curve commitment or proof at index k, or a zero-length blob, gives the same code and message in the host,
    device and group forms, and leaves the outputs untouched; points are checked before lengths, as in the reference.
    The openings form rejects the same points with the same code and message.  count == 0 gives identities everywhere."""
    import torch

    rnd = random.Random(31)
    eng = pkg.Engine(0)
    grp = pkg.Group([0, 0])
    datas = [rnd.randbytes(32 * 64) for _ in range(7)]
    keep, hptrs = _host_ptrs(datas)
    bufs = [torch.frombuffer(bytearray(d), dtype=torch.uint8).cuda() for d in datas]
    dptrs = [b.data_ptr() for b in bufs]
    good = [o.g1_mul(o.G1_GEN, 3 + i) for i in range(7)]
    cases = [  # (lens, commitments, proofs, variant)
        ([2048] * 5 + [0, 2048], good[:3] + [OFF_CURVE] + good[4:], good, "NotOnCurveError"),
        ([2048] * 7, good, good[:6] + [OFF_CURVE], "NotOnCurveError"),
        ([2048] * 3 + [0] + [2048] * 3, good, good, "GenericError"),
        ([0] + [2048] * 6, good, good, "GenericError"),
    ]
    for lens, cs, ps, variant in cases:
        msgs = set()
        for form in ("host", "dev", "group"):
            out = _sentinel()
            with pytest.raises(pkg.KzgError) as err:
                if form == "group":
                    _group_raw(pkg, grp, hptrs, lens, cs, ps, out=out)
                else:
                    _rlc_raw(pkg, eng, hptrs, lens, cs, ps, dev_ptrs=dptrs if form == "dev" else None, out=out)
            assert err.value.variant == variant
            assert _words(out) == _words(_sentinel())
            msgs.add(err.value.msg)
        assert len(msgs) == 1, msgs
        if variant == "NotOnCurveError":
            out = _sentinel()
            with pytest.raises(pkg.KzgError) as err:
                _openings_raw(pkg, eng, cs, ps, bytes(32 * 7), bytes(32 * 7), [64] * 7, out=out)
            assert (err.value.variant, err.value.msg) == (variant, msgs.pop())
            assert _words(out) == _words(_sentinel())
    ident = (bytes(64), 1, bytes(64), 1)
    assert _words(_rlc_raw(pkg, eng, [], [], [], [], out=_sentinel())) == ident
    assert _words(_rlc_raw(pkg, eng, [], [], [], [], dev_ptrs=[], out=_sentinel())) == ident
    assert _words(_group_raw(pkg, grp, [], [], [], [], out=_sentinel())) == ident
    assert _words(_openings_raw(pkg, eng, [], [], b"", b"", [], out=_sentinel())) == ident
    assert pkg.verify_kzg_proof_batch_rlc([], [], [], [], [], eng) == (None, None)
    with pytest.raises(pkg.KzgError) as mismatch:
        pkg.verify_kzg_proof_batch_rlc(good, [1] * 7, [1] * 7, good, [64] * 6, eng)
    assert (mismatch.value.variant, mismatch.value.msg) == ("GenericError", "length's of the input are not the same")
    with pytest.raises(pkg.KzgError) as mismatch:
        grp.verify_blob_kzg_proof_batch_rlc(_blobs(pkg, datas), good, good[:6])
    assert (mismatch.value.variant, mismatch.value.msg) == ("GenericError", "length's of the input are not the same")
    # both handles stay usable
    want = pkg.verify_blob_kzg_proof_batch_rlc(_blobs(pkg, datas), good, good, eng)
    assert grp.verify_blob_kzg_proof_batch_rlc(_blobs(pkg, datas), good, good) == want
    grp.close()
    eng.close()


@pytest.mark.parametrize("fs_device", [0, 1])
def test_verify_blob_proofs_without_out(pkg, fs_device):
    """kzgb_verify_blob_proofs_g1 with out_xy == NULL returns the z and y it returns with out_xy."""
    rnd = random.Random(17 + fs_device)
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(1 << 16, TAU, engine=eng)
    try:
        datas = [_with_large_chunks(rnd, k) for k in (1, 33, 31 * 64, 32 << 16)] + [_with_large_chunks(rnd, 32 << 12) for _ in range(260)]
        cs, ps = _mixed_inputs(pkg, srs, datas)
        _set(pkg, "fs_device", fs_device)
        assert _zy_words(pkg, eng, datas, cs, ps, with_out=False) == _zy_words(pkg, eng, datas, cs, ps)
    finally:
        _set(pkg, "fs_device", -1)
        eng.close()
