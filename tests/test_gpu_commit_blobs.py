"""kzgb_commit_blobs{,_dev} and kzgb_group_commit_blobs: batched KZG::commit_blob (prover/src/kzg.rs:182-185) with no
proofs.  Every point must be the one kzgb_commit_blob returns for that blob alone, on the grouped small-blob path, the
large-blob lanes, the byte-fed MSM over the Lagrange tables and the convert-first path without them."""
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


def _barycentric(evals, z):
    """p(z) for the interpolant of evals on the 2^k domain, O(n) with one batch inversion."""
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


def _closed_form(data: bytes):
    """Commitment of blob bytes over SRS_i = tau^i G: p(tau) G, p the interpolant of the (unreduced) 32-byte chunks."""
    n = 1 << max(0, (len(data) + 31) // 32 - 1).bit_length()
    data = data + bytes(32 * n - len(data))
    return o.g1_mul(o.G1_GEN, _barycentric([int.from_bytes(data[32 * k : 32 * k + 32], "big") for k in range(n)], TAU))


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
    """Lengths 0, 1, 31, 32, 33, 500, 31*64, 32*2^12, 32*2^16, a run of 70 equal 2^12-Fr blobs (two groups);
    large=True adds one 2^18-Fr blob, which sends the whole batch to the large-blob lanes."""
    lens = [0, 1, 31, 32, 33, 500, 31 * 64, 32 << 12, 32 << 16] + [32 << 12] * 70 + ([32 << 18] if large else [])
    return [_with_large_chunks(rnd, k) if k else b"" for k in lens]


def _commit_one(pkg, eng, data: bytes):
    return eng._point_call(lambda h, *a: pkg.lib.kzgb_commit_blob(h, data, len(data), *a))


def _raw_commit_blobs(pkg, eng, ptrs, lens, dev=False):
    count = len(lens)
    xy = C.create_string_buffer(64 * count if count else 1)
    inf = C.create_string_buffer(count if count else 1)
    fn = pkg.lib.kzgb_commit_blobs_dev if dev else pkg.lib.kzgb_commit_blobs
    eng.check(fn(eng.h, (C.c_void_p * count)(*ptrs), (C.c_size_t * count)(*lens), count, xy, inf))
    return pkg.g1_from_abi(xy.raw[: 64 * count], inf.raw[:count])


def _set_lagrange(pkg, on):
    assert pkg.lib.kzgb_set_option(b"lagrange", 1 if on else 0) == 0


@pytest.mark.parametrize("lagrange", [1, 0])
@pytest.mark.parametrize("large", [False, True], ids=["groups", "lanes"])
def test_commit_blobs_equal_commit_blob(pkg, lagrange, large):
    """Point i = kzgb_commit_blob on blob i, for a ragged batch holding chunks >= r, with the Lagrange tables of every
    size resident (the byte-fed MSM) and with option "lagrange" 0 (bytes -> Montgomery -> inverse NTT -> monomial
    table)."""
    rnd = random.Random(11 + 2 * lagrange + large)
    datas = _ragged(rnd, large)
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(1 << (18 if large else 16), TAU, engine=eng)
    try:
        _set_lagrange(pkg, lagrange)
        if lagrange:
            for n in sorted({1 << max(0, (len(d) + 31) // 32 - 1).bit_length() for d in datas}):
                srs.prepare_lagrange(n)
        got = pkg.KZG.commit_blobs([pkg.Blob.from_unchecked(d) for d in datas], srs)
        want = [_commit_one(pkg, eng, d) for d in datas]
        assert got == want
        assert got[0] is None  # the zero polynomial
        assert len(set(got[9:79])) == 70  # the run of equal-size blobs holds 70 different blobs
    finally:
        _set_lagrange(pkg, 1)
        eng.close()


def test_commit_blobs_equal_prover_commitments_and_oracle(pkg):
    """g1_serialize_compressed of every point = the commitment bytes kzgb_commit_and_prove_blobs returns for the same
    batch (which rejects length 0, so the empty blob is left out), and = the oracle's commit_blob on the reference's
    g1.point SRS for a few small blobs."""
    rnd = random.Random(3)
    raws = [rnd.randbytes(k) for k in (31 * 64, 31 * 33, 31, 1, 31 * 200, 31 * 128, 500, 31 * 64, 31 * 7, 31 * 256)]
    blobs = [pkg.Blob.from_raw_data(r) for r in raws] + [pkg.Blob.from_unchecked(_with_large_chunks(rnd, 32 * 100 + 7))]
    eng = pkg.Engine(0)
    srs = pkg.SRS.from_gnark_bytes(g.g1_point_bytes(), engine=eng)
    pts = pkg.KZG.commit_blobs(blobs, srs)
    cs, _ = pkg.KZG.commit_and_prove_blobs(blobs, srs)
    assert [pkg.g1_serialize_compressed(p) for p in pts] == cs
    ref = g.srs_points_string()
    okzg = o.KZG()
    for i in (3, 6, 8):
        assert pts[i] == okzg.commit_blob(o.Blob.from_raw_data(raws[i]), ref)
    eng.close()


def test_commit_blobs_closed_form_full_size(pkg):
    """Synthetic SRS: 4 blobs of 2^19 Fr (large-blob lanes) and 256 blobs of 2^12 Fr (groups) each give p(tau) G."""
    import numpy as np

    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(1 << 19, TAU, engine=eng)
    rng = np.random.default_rng(19)
    for logn, count in ((19, 4), (12, 256)):
        a = rng.integers(0, 256, size=(count, 1 << logn, 32), dtype=np.uint8)
        a[:, :: 1 << 9, :] = 0xFF  # chunks >= r all over
        datas = [a[i].tobytes() for i in range(count)]
        got = pkg.KZG.commit_blobs([pkg.Blob.from_unchecked(d) for d in datas], srs)
        assert got == [_closed_form(d) for d in datas]
    eng.close()


def test_commit_blobs_dev_equals_host(pkg):
    """kzgb_commit_blobs_dev = kzgb_commit_blobs with the blobs back to back in one device buffer (one launch reads
    them in place) and scattered over separate buffers (gathered device to device), on groups and on lanes."""
    import torch

    rnd = random.Random(5)
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(1 << 18, TAU, engine=eng)
    for n, count in ((1 << 12, 70), (1 << 18, 3)):
        srs.prepare_lagrange(n)
        datas = [_with_large_chunks(rnd, 32 * n) for _ in range(count)]
        want = pkg.KZG.commit_blobs([pkg.Blob.from_unchecked(d) for d in datas], srs)
        run = torch.frombuffer(bytearray(b"".join(datas)), dtype=torch.uint8).cuda()
        ptrs = [run.data_ptr() + 32 * n * i for i in range(count)]
        assert _raw_commit_blobs(pkg, eng, ptrs, [32 * n] * count, dev=True) == want
    datas = _ragged(rnd)
    want = pkg.KZG.commit_blobs([pkg.Blob.from_unchecked(d) for d in datas], srs)
    bufs = [torch.frombuffer(bytearray(b"\x00" * 3 + d + b"\x00" * 5), dtype=torch.uint8).cuda() for d in datas]
    ptrs = [b.data_ptr() + 3 for b in bufs]  # unaligned sources
    assert _raw_commit_blobs(pkg, eng, ptrs, [len(d) for d in datas], dev=True) == want
    eng.close()


def test_commit_blobs_no_conversion_kernel(pkg):
    """With the Lagrange table prepared the blob bytes feed the MSM directly: k large blobs cost k times the launches
    of one kzgb_commit_eval of that size, which is a bare MSM over the table."""
    n, k = 1 << 19, 3
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(n, TAU, engine=eng)
    srs.prepare_lagrange(n)
    rnd = random.Random(9)
    blobs = [pkg.Blob.from_unchecked(rnd.randbytes(32 * n)) for _ in range(k)]
    pkg.KZG.commit_blobs(blobs, srs)  # lanes, twiddles and tables in place
    evals = pkg.fr_to_mont_bytes([rnd.randrange(o.R) for _ in range(1024)] * (n // 1024))
    out, inf = C.create_string_buffer(64), C.c_uint8(0)
    eng.check(pkg.lib.kzgb_commit_eval(eng.h, evals, n, out, C.byref(inf)))
    c0 = eng.launch_count()
    eng.check(pkg.lib.kzgb_commit_eval(eng.h, evals, n, out, C.byref(inf)))
    one = eng.launch_count() - c0
    c0 = eng.launch_count()
    pkg.KZG.commit_blobs(blobs, srs)
    assert eng.launch_count() - c0 == k * one
    eng.close()


def test_commit_blobs_errors(pkg):
    """A blob over the SRS fails with SrsCapacityExceeded and a blob above 2^28 elements with the GenericError text,
    each exactly as kzgb_commit_blob fails on that blob, before any work (the outputs stay untouched); the context
    stays usable; count == 0 is KZGB_OK."""
    n = 1 << 12
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(n, TAU, engine=eng)
    rnd = random.Random(1)
    good = [rnd.randbytes(32 * n), rnd.randbytes(100)]
    keep = [C.create_string_buffer(d, len(d)) for d in good]
    ptrs = [C.cast(b, C.c_void_p).value for b in keep]
    huge = (32 << 28) + 1  # never read: every blob is checked before any work
    for bad_len, variant in ((32 * n + 1, "SrsCapacityExceeded"), (huge, "GenericError")):
        with pytest.raises(pkg.KzgError) as single:
            eng.check(pkg.lib.kzgb_commit_blob(eng.h, ptrs[0], bad_len, C.create_string_buffer(64), None))
        assert single.value.variant == variant
        lens = [32 * n, 100, bad_len]
        xy = C.create_string_buffer(b"\xab" * 192, 192)
        with pytest.raises(pkg.KzgError) as batch:
            eng.check(pkg.lib.kzgb_commit_blobs(eng.h, (C.c_void_p * 3)(*ptrs, ptrs[0]), (C.c_size_t * 3)(*lens), 3, xy, None))
        assert (batch.value.variant, batch.value.msg) == (single.value.variant, single.value.msg)
        assert xy.raw == b"\xab" * 192
    assert "Input size exceeds maximum polynomial size" in single.value.msg
    want = [_commit_one(pkg, eng, d) for d in good]
    assert pkg.KZG.commit_blobs([pkg.Blob.from_unchecked(d) for d in good], srs) == want
    assert pkg.lib.kzgb_commit_blobs(eng.h, None, None, 0, None, None) == 0
    assert pkg.lib.kzgb_commit_blobs_dev(eng.h, None, None, 0, None, None) == 0
    assert pkg.KZG.commit_blobs([], srs) == []
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
def test_group_commit_blobs_equal_single_context(pkg, devices):
    """kzgb_group_commit_blobs = the one-context call on a ragged batch cut across the members, on fewer blobs than
    members, and on none."""
    rnd = random.Random(len(devices) * 5 + devices[-1])
    raws = [rnd.randbytes(k) for k in (31 * 64, 31 * 33, 0, 31, 1, 31 * 200, 31 * 128, 500, 31 * 64, 31 * 7, 31 * 256)]
    blobs = [pkg.Blob.from_raw_data(r) for r in raws] + [pkg.Blob.from_unchecked(_with_large_chunks(rnd, 32 * 300 + 5))]
    eng = pkg.Engine(0)
    srs = pkg.SRS.from_gnark_bytes(g.g1_point_bytes(), engine=eng)
    want = pkg.KZG.commit_blobs(blobs, srs)
    eng.close()
    grp = pkg.Group(devices)
    grp.load_srs_gnark_bytes(g.g1_point_bytes())
    assert grp.commit_blobs(blobs) == want
    assert grp.commit_blobs(blobs[:1]) == want[:1]
    assert grp.commit_blobs([]) == []
    grp.close()
