"""kzgb_compute_blob_proofs{,_dev} and kzgb_group_compute_blob_proofs: batched KZG::compute_blob_proof
(prover/src/kzg.rs:288-309) against caller-supplied commitments.  Every proof must be the one kzgb_compute_blob_proof
returns for that (blob, commitment) pair alone, on the grouped small-blob path and the large-blob lanes, and through
every route the hashing plan can take."""
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


@pytest.fixture(scope="module")
def pkg():
    return load_package()


def _poly_len(nbytes):
    return 1 << max(0, (nbytes + 31) // 32 - 1).bit_length()


def _barycentric(evals, z):
    """p(z) for the interpolant of evals on the 2^k domain, O(n) with one batch inversion (z outside the domain)."""
    n = len(evals)
    w = o.PRIMITIVE_ROOTS_OF_UNITY[n.bit_length() - 1]
    roots = [1] * n
    for i in range(1, n):
        roots[i] = roots[i - 1] * w % o.R
    den = [(z - r) % o.R for r in roots]
    pref, acc = [], 1
    for d in den:
        pref.append(acc)
        acc = acc * d % o.R
    inv = pow(acc, -1, o.R)
    total = 0
    for i in range(n - 1, -1, -1):
        di = inv * pref[i] % o.R
        inv = inv * den[i] % o.R
        total = (total + evals[i] * roots[i] % o.R * di) % o.R
    return total * (pow(z, n, o.R) - 1) % o.R * pow(n, -1, o.R) % o.R


def _with_large_chunks(rnd, nbytes):
    """Random bytes with chunks >= r: an all-0xff chunk, r itself, r + 1 and an all-0xff partial last chunk."""
    b = bytearray(rnd.randbytes(nbytes))
    for k, chunk in ((0, FF), (1, R_BYTES), (2, (o.R + 1).to_bytes(32, "big"))):
        if 32 * k + 32 <= nbytes:
            b[32 * k : 32 * k + 32] = chunk
    tail = nbytes % 32 or 32
    b[nbytes - tail :] = b"\xff" * tail
    return bytes(b)


def _ragged(rnd, large=False):
    """Lengths 1, 31, 32, 33, 500, 31*64, 32*2^12, 32*2^16, a run of 70 equal 2^12-Fr blobs (two groups);
    large=True adds one 2^18-Fr blob, which sends the whole batch to the large-blob lanes."""
    lens = [1, 31, 32, 33, 500, 31 * 64, 32 << 12, 32 << 16] + [32 << 12] * 70 + ([32 << 18] if large else [])
    return [_with_large_chunks(rnd, k) for k in lens]


def _blobs(pkg, datas):
    return [pkg.Blob.from_unchecked(d) for d in datas]


def _mixed_commitments(pkg, srs, datas):
    """Blob i's own commitment, an unrelated valid point or the identity, by i mod 3."""
    own = pkg.KZG.commit_blobs(_blobs(pkg, datas), srs)
    return [own[i] if i % 3 == 0 else (o.g1_mul(o.G1_GEN, 7 + i) if i % 3 == 1 else None) for i in range(len(datas))]


def _prove_one(pkg, eng, data, commitment):
    xy, inf = pkg.g1_to_abi([commitment])
    return eng._point_call(lambda h, *a: pkg.lib.kzgb_compute_blob_proof(h, data, len(data), xy, inf[0], *a))


def _raw_proofs(pkg, eng, host_ptrs, lens, commitments, dev_ptrs=None, with_inf=True):
    count = len(lens)
    cxy, cinf = pkg.g1_to_abi(commitments)
    xy = C.create_string_buffer(64 * count if count else 1)
    inf = C.create_string_buffer(count if count else 1)
    hp, ln = (C.c_void_p * count)(*host_ptrs), (C.c_size_t * count)(*lens)
    ci = cinf if with_inf else None
    if dev_ptrs is None:
        eng.check(pkg.lib.kzgb_compute_blob_proofs(eng.h, hp, ln, count, cxy, ci, xy, inf))
    else:
        eng.check(pkg.lib.kzgb_compute_blob_proofs_dev(eng.h, (C.c_void_p * count)(*dev_ptrs), hp, ln, count, cxy, ci, xy, inf))
    return pkg.g1_from_abi(xy.raw[: 64 * count], inf.raw[:count])


def _host_ptrs(datas):
    keep = [C.create_string_buffer(d, max(1, len(d))) for d in datas]
    return keep, [C.cast(k, C.c_void_p).value for k in keep]


def _set(pkg, name, value):
    assert pkg.lib.kzgb_set_option(name.encode(), value) == 0


@pytest.mark.parametrize("lagrange", [1, 0])
@pytest.mark.parametrize("large", [False, True], ids=["groups", "lanes"])
def test_blob_proofs_equal_single_call(pkg, lagrange, large):
    """Proof i = kzgb_compute_blob_proof(blob i, C_i) for a ragged batch holding chunks >= r, with commitments that are
    the blob's own, unrelated points and the identity; with the Lagrange tables of every size resident and with option
    "lagrange" 0 (quotient -> inverse NTT -> monomial table)."""
    rnd = random.Random(21 + 2 * lagrange + large)
    datas = _ragged(rnd, large)
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(1 << (18 if large else 16), TAU, engine=eng)
    try:
        _set(pkg, "lagrange", lagrange)
        if lagrange:
            for n in sorted({_poly_len(len(d)) for d in datas}):
                srs.prepare_lagrange(n)
        cs = _mixed_commitments(pkg, srs, datas)
        got = pkg.KZG.compute_blob_proofs(_blobs(pkg, datas), cs, srs)
        want = [_prove_one(pkg, eng, d, c) for d, c in zip(datas, cs)]
        assert got == want
        assert len(set(got[8:78])) == 70  # the run of equal-size blobs holds 70 different proofs
    finally:
        _set(pkg, "lagrange", 1)
        eng.close()


def test_blob_proofs_equal_commit_and_prove_and_oracle(pkg):
    """With C_i from KZG.commit_blobs, g1_serialize_compressed of every proof = the proof bytes of
    kzgb_commit_and_prove_blobs on the same batch; a few small blobs also = the oracle's compute_blob_proof on the
    reference's g1.point SRS."""
    rnd = random.Random(4)
    raws = [rnd.randbytes(k) for k in (31 * 64, 31 * 33, 31, 1, 31 * 200, 31 * 128, 500, 31 * 64, 31 * 7, 31 * 256)]
    blobs = [pkg.Blob.from_raw_data(r) for r in raws] + [pkg.Blob.from_unchecked(_with_large_chunks(rnd, 32 * 100 + 7))]
    eng = pkg.Engine(0)
    srs = pkg.SRS.from_gnark_bytes(g.g1_point_bytes(), engine=eng)
    cs = pkg.KZG.commit_blobs(blobs, srs)
    proofs = pkg.KZG.compute_blob_proofs(blobs, cs, srs)
    _, ps = pkg.KZG.commit_and_prove_blobs(blobs, srs)
    assert [pkg.g1_serialize_compressed(p) for p in proofs] == ps
    ref = g.srs_points_string()
    for i in (3, 6, 8):
        ob = o.Blob.from_raw_data(raws[i])
        okzg = o.KZG()
        okzg.calculate_and_store_roots_of_unity(len(ob.blob_data))
        assert proofs[i] == okzg.compute_blob_proof(ob, cs[i], ref)
    eng.close()


def test_blob_proofs_closed_form_full_size(pkg):
    """Synthetic SRS: 4 blobs of 2^19 Fr (large-blob lanes) and 256 blobs of 2^12 Fr (groups); each proof against an
    arbitrary valid commitment C is ((p(tau) - y) / (tau - z)) G with z = the oracle's transcript of (blob, C) and
    y = p(z) by barycentric evaluation."""
    import numpy as np

    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(1 << 19, TAU, engine=eng)
    rng = np.random.default_rng(29)
    for logn, count in ((19, 4), (12, 256)):
        a = rng.integers(0, 256, size=(count, 1 << logn, 32), dtype=np.uint8)
        a[:, :: 1 << 9, :] = 0xFF  # chunks >= r all over
        datas = [a[i].tobytes() for i in range(count)]
        cs = [o.g1_mul(o.G1_GEN, 1000 + i) for i in range(count)]
        got = pkg.KZG.compute_blob_proofs(_blobs(pkg, datas), cs, srs)
        for d, c, p in zip(datas, cs, got):
            evals = [int.from_bytes(d[32 * k : 32 * k + 32], "big") % o.R for k in range(1 << logn)]
            z = o.compute_challenge(o.Blob.from_unchecked(d), c)
            y = _barycentric(evals, z)
            q = (_barycentric(evals, TAU) - y) * pow((TAU - z) % o.R, -1, o.R) % o.R
            assert p == o.g1_mul(o.G1_GEN, q)
    eng.close()


def test_blob_proofs_dev_equals_host(pkg):
    """kzgb_compute_blob_proofs_dev = kzgb_compute_blob_proofs with the blobs back to back in one device buffer and
    scattered over separate, unaligned buffers, on groups and on lanes; commitments_inf may be NULL."""
    import torch

    rnd = random.Random(6)
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(1 << 18, TAU, engine=eng)
    for n, count in ((1 << 12, 70), (1 << 18, 3)):
        srs.prepare_lagrange(n)
        datas = [_with_large_chunks(rnd, 32 * n) for _ in range(count)]
        cs = [o.g1_mul(o.G1_GEN, 3 + i) for i in range(count)]  # no identity: the flags can be left out
        want = pkg.KZG.compute_blob_proofs(_blobs(pkg, datas), cs, srs)
        keep, hptrs = _host_ptrs(datas)
        assert _raw_proofs(pkg, eng, hptrs, [32 * n] * count, cs, with_inf=False) == want
        run = torch.frombuffer(bytearray(b"".join(datas)), dtype=torch.uint8).cuda()
        dptrs = [run.data_ptr() + 32 * n * i for i in range(count)]
        assert _raw_proofs(pkg, eng, hptrs, [32 * n] * count, cs, dev_ptrs=dptrs) == want
    for large in (False, True):
        datas = _ragged(rnd, large)
        cs = _mixed_commitments(pkg, srs, datas)
        want = pkg.KZG.compute_blob_proofs(_blobs(pkg, datas), cs, srs)
        keep, hptrs = _host_ptrs(datas)
        bufs = [torch.frombuffer(bytearray(b"\x00" * 3 + d + b"\x00" * 5), dtype=torch.uint8).cuda() for d in datas]
        dptrs = [b.data_ptr() + 3 for b in bufs]  # unaligned sources
        assert _raw_proofs(pkg, eng, hptrs, [len(d) for d in datas], cs, dev_ptrs=dptrs) == want
    eng.close()


ROUTES = {
    "single_stream": {"hash_mb": 0, "device_hash": 0},
    "multi_buffer": {"hash_mb": 1, "device_hash": 0, "hash_threads": 2},  # a single-stream head of 2, then groups of 16
    "device_warp": {"hash_mb": 0, "device_hash": 5, "device_hash_lanes": 0},
    "device_lanes": {"hash_mb": 0, "device_hash": 5, "device_hash_lanes": 1},
    "multi_buffer_and_device": {"hash_mb": 1, "device_hash": 5, "hash_threads": 2},
    "generic_inverses": {"eval_structured": 0},
}
DEFAULTS = {"hash_mb": -1, "device_hash": -1, "device_hash_lanes": -1, "hash_threads": 0, "eval_structured": 1, "group": -1}


@pytest.mark.parametrize("route", list(ROUTES))
def test_blob_proofs_every_hashing_route(pkg, route):
    """Large-blob lanes (option "group" 0) over 40 blobs of exactly 32 * 2^12 bytes between two ragged ones (the
    multi-buffer and device kernels take only the former; the device share is the last blobs): every route the
    hashing plan can choose -- single stream, multi-buffer groups behind a single-stream head, a device share hashed by
    one warp or one lane per transcript (host blobs staged, and device blobs) -- and the generic inverses give the
    proofs of the single call."""
    import torch

    rnd = random.Random(31)
    eligible = [_with_large_chunks(rnd, 32 << 12) for _ in range(40)]
    datas = [_with_large_chunks(rnd, 33)] + eligible[:20] + [_with_large_chunks(rnd, 31 * 64)] + eligible[20:]
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(1 << 12, TAU, engine=eng)
    try:
        cs = _mixed_commitments(pkg, srs, datas)
        want = [_prove_one(pkg, eng, d, c) for d, c in zip(datas, cs)]
        _set(pkg, "group", 0)
        for name, value in ROUTES[route].items():
            _set(pkg, name, value)
        keep, hptrs = _host_ptrs(datas)
        lens = [len(d) for d in datas]
        assert _raw_proofs(pkg, eng, hptrs, lens, cs) == want
        bufs = [torch.frombuffer(bytearray(d), dtype=torch.uint8).cuda() for d in datas]
        assert _raw_proofs(pkg, eng, hptrs, lens, cs, dev_ptrs=[b.data_ptr() for b in bufs]) == want
    finally:
        for name, value in DEFAULTS.items():
            _set(pkg, name, value)
        eng.close()


def test_blob_proofs_errors(pkg):
    """Each error kind behind valid blobs -- a commitment off the curve, a blob of length 0, a blob over the SRS -- fails
    the batch exactly as kzgb_compute_blob_proof fails on that pair, before any work (the outputs stay untouched); the
    lowest-index failing blob wins, and within a blob the commitment is checked first; the context stays usable;
    count == 0 is KZGB_OK; lists of different lengths are the mirror's GenericError."""
    n = 1 << 12
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(n, TAU, engine=eng)
    rnd = random.Random(2)
    good = [rnd.randbytes(32 * n), rnd.randbytes(100)]
    good_cs = [o.g1_mul(o.G1_GEN, 11), None]
    off_curve = (1, 3)
    cases = [  # (lens, commitments, single call that must fail the same way)
        ([32 * n, 100, 100], good_cs + [off_curve], (100, off_curve)),
        ([32 * n, 100, 0], good_cs + [o.G1_GEN], (0, o.G1_GEN)),
        ([32 * n, 100, 32 * n + 1], good_cs + [o.G1_GEN], (32 * n + 1, o.G1_GEN)),
        ([32 * n, 0, 0], [good_cs[0], o.G1_GEN, off_curve], (0, o.G1_GEN)),  # lowest index first
        ([32 * n, 100, 0], good_cs + [off_curve], (0, off_curve)),  # the commitment before the length
    ]
    big = C.create_string_buffer(b"\x01" * (32 * n + 32))
    keep, ptrs = _host_ptrs(good)
    ptrs = ptrs + [C.cast(big, C.c_void_p).value]
    variants = set()
    for lens, cs, (bad_len, bad_c) in cases:
        xy, inf = pkg.g1_to_abi([bad_c])
        with pytest.raises(pkg.KzgError) as single:
            eng.check(pkg.lib.kzgb_compute_blob_proof(eng.h, ptrs[2], bad_len, xy, inf[0], C.create_string_buffer(64), None))
        cxy, cinf = pkg.g1_to_abi(cs)
        out = C.create_string_buffer(b"\xab" * 192, 192)
        out_inf = C.create_string_buffer(b"\xcd" * 3, 3)
        with pytest.raises(pkg.KzgError) as batch:
            eng.check(pkg.lib.kzgb_compute_blob_proofs(eng.h, (C.c_void_p * 3)(*ptrs), (C.c_size_t * 3)(*lens), 3, cxy, cinf,
                                                       out, out_inf))
        assert (batch.value.variant, batch.value.msg) == (single.value.variant, single.value.msg)
        assert out.raw == b"\xab" * 192 and out_inf.raw == b"\xcd" * 3
        variants.add(single.value.variant)
    assert variants == {"NotOnCurveError", "GenericError", "SrsCapacityExceeded"}
    want = [_prove_one(pkg, eng, d, c) for d, c in zip(good, good_cs)]
    assert pkg.KZG.compute_blob_proofs(_blobs(pkg, good), good_cs, srs) == want
    assert pkg.lib.kzgb_compute_blob_proofs(eng.h, None, None, 0, None, None, None, None) == 0
    assert pkg.lib.kzgb_compute_blob_proofs_dev(eng.h, None, None, None, 0, None, None, None, None) == 0
    assert pkg.KZG.compute_blob_proofs([], [], srs) == []
    with pytest.raises(pkg.KzgError) as mismatch:
        pkg.KZG.compute_blob_proofs(_blobs(pkg, good), good_cs[:1], srs)
    assert (mismatch.value.variant, mismatch.value.msg) == ("GenericError", "length's of the input are not the same")
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
def test_group_blob_proofs_equal_single_context(pkg, devices):
    """kzgb_group_compute_blob_proofs = the one-context call on a ragged batch cut across the members, on fewer blobs
    than members, and on none."""
    rnd = random.Random(len(devices) * 7 + devices[-1])
    raws = [rnd.randbytes(k) for k in (31 * 64, 31 * 33, 31, 1, 31 * 200, 31 * 128, 500, 31 * 64, 31 * 7, 31 * 256)]
    blobs = [pkg.Blob.from_raw_data(r) for r in raws] + [pkg.Blob.from_unchecked(_with_large_chunks(rnd, 32 * 300 + 5))]
    eng = pkg.Engine(0)
    srs = pkg.SRS.from_gnark_bytes(g.g1_point_bytes(), engine=eng)
    cs = _mixed_commitments(pkg, srs, [b.blob_data for b in blobs])
    want = pkg.KZG.compute_blob_proofs(blobs, cs, srs)
    eng.close()
    grp = pkg.Group(devices)
    grp.load_srs_gnark_bytes(g.g1_point_bytes())
    assert grp.compute_blob_proofs(blobs, cs) == want
    assert grp.compute_blob_proofs(blobs[:1], cs[:1]) == want[:1]
    assert grp.compute_blob_proofs([], []) == []
    grp.close()
