"""kzgb_compute_proofs{,_dev}, kzgb_group_compute_proofs and KZG.compute_proofs: KZG::compute_proof (prover/src/kzg.rs:
128-178, 187-234) for many polynomials, each at a point the caller chooses, in one call.  Entry i must be word for word
(proof, identity flag, y) what kzgb_compute_proof returns for polynomial i and z_i alone, for z inside the domain (the
reference's compute_quotient_eval_on_domain branch) and outside it, on every route the batch can take: groups of
equal-size polynomials (one batched launch set each, n <= 2^17), task lanes (larger polynomials), the generic and the
structured inverses, the Lagrange and the monomial tables."""
import ctypes as C
import random

import numpy as np
import pytest

import golden_data as g
from __graft_entry__ import load_package
from oracle import bn254 as o

pytestmark = pytest.mark.gpu
TAU = o.SYNTH_TAU
SRS_N = 1 << 19


@pytest.fixture(scope="module")
def pkg():
    return load_package()


@pytest.fixture(scope="module")
def srs(pkg):
    """The synthetic SRS tau^j G, j < 2^19, on a context of its own."""
    e = pkg.Engine(0)
    yield pkg.SRS.synthetic(SRS_N, TAU, engine=e)
    e.close()


@pytest.fixture(scope="module")
def eng(srs):
    return srs.engine


def _set(pkg, name, value):
    assert pkg.lib.kzgb_set_option(name.encode(), value) == 0


def _rand_words(rng, n):
    """n random reduced Montgomery words (below 2^253 < r), as bytes."""
    a = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    a[:, 31] &= 0x1F
    return a.tobytes()


def _z_mont(pkg, z):
    return pkg.fr_to_mont_bytes([z])


def _root(n, k):
    return pow(o.PRIMITIVE_ROOTS_OF_UNITY[n.bit_length() - 1], k, o.R)


def _points(n, rnd, count):
    """z = 0, w^0, w^(n-1), then roots and non-roots alternating (every group mixes both)."""
    zs = [0, 1, _root(n, n - 1)]
    while len(zs) < count:
        zs.append(_root(n, rnd.randrange(n)) if len(zs) % 2 else rnd.randrange(o.R))
    return zs[:count]


def _single(pkg, eng, evals, z):
    """kzgb_compute_proof: (proof words, identity flag, y words)."""
    xy, y = C.create_string_buffer(64), C.create_string_buffer(32)
    inf = C.c_uint8(7)
    eng.check(pkg.lib.kzgb_compute_proof(eng.h, evals, len(evals) // 32, _z_mont(pkg, z), xy, C.byref(inf), y))
    return xy.raw, inf.value, y.raw


def _batch(pkg, eng, evals, zs, fill=0xAB, with_inf=True, with_y=True):
    """kzgb_compute_proofs on host polynomials: the (proof, flag, y) of each entry; outputs pre-filled with `fill`."""
    count = len(evals)
    keep = [C.create_string_buffer(e, max(32, len(e))) for e in evals]
    ptrs = (C.c_void_p * count)(*[C.cast(k, C.c_void_p).value for k in keep])
    ns = (C.c_size_t * count)(*[len(e) // 32 for e in evals])
    xy = C.create_string_buffer(bytes([fill]) * 64 * count, 64 * count)
    inf = C.create_string_buffer(bytes([fill]) * count, count)
    ys = C.create_string_buffer(bytes([fill]) * 32 * count, 32 * count)
    eng.check(pkg.lib.kzgb_compute_proofs(eng.h, ptrs, ns, count, b"".join(_z_mont(pkg, z) for z in zs), xy,
                                          inf if with_inf else None, ys if with_y else None))
    return _entries(xy.raw, inf.raw, ys.raw, count)


def _entries(xy, inf, ys, count):
    return [(xy[64 * i : 64 * i + 64], inf[i], ys[32 * i : 32 * i + 32]) for i in range(count)]


def _check_equal_single(pkg, eng, evals, zs):
    got = _batch(pkg, eng, evals, zs)
    want = {}
    for i, (e, z) in enumerate(zip(evals, zs)):
        key = (id(e), z)
        if key not in want:
            want[key] = _single(pkg, eng, e, z)
        assert got[i] == want[key], (i, len(e) // 32)
    return got


def test_reference_kat(pkg):
    """kzg.proof.eq.input: the Gettysburg blob's polynomial over the reference's g1.point SRS, 40 times in one call with
    z = w^idx of each row: the 40 proofs of the fixture, and y = evaluation idx of the polynomial."""
    e = pkg.Engine(0)
    try:
        srs = pkg.SRS.from_gnark_bytes(g.g1_point_bytes(), engine=e)
        poly = pkg.Blob.from_raw_data(g.gettysburg()).to_polynomial_eval_form(e)
        n = len(poly)
        rows = g.proof_eq_input()
        assert n == 64 and len(rows) == 40
        proofs, ys = pkg.KZG.compute_proofs([poly] * len(rows), [_root(n, idx) for idx, _, _ in rows], srs)
        assert proofs == [(x, y) for _, x, y in rows]
        assert ys == [poly.evaluations[idx] for idx, _, _ in rows]
    finally:
        e.close()


@pytest.mark.parametrize("logn,count", [(0, 12), (1, 12), (2, 12), (6, 100), (12, 70), (16, 40), (19, 4)])
def test_equal_single_call(pkg, eng, logn, count):
    """Sizes below the structured inverses (1, 2, 4), several groups (2^6, 2^12, 2^16) and task lanes (2^19, above the
    2^17 group limit); z = 0, w^0, w^(n-1), random roots and random points mixed inside every group."""
    n = 1 << logn
    rnd = random.Random(logn)
    rng = np.random.default_rng(logn)
    polys = [_rand_words(rng, n) for _ in range(min(count, 5))]
    evals = [polys[i % len(polys)] for i in range(count)]
    _check_equal_single(pkg, eng, evals, _points(n, rnd, count))


def test_mixed_sizes(pkg, eng):
    """One call whose sizes break the equal-size runs the groups are cut from."""
    rnd = random.Random(5)
    rng = np.random.default_rng(5)
    sizes = [64, 64, 4096, 64, 1, 64, 64, 2, 4096, 4096, 1 << 16, 64, 8, 8, 8, 1 << 10]
    evals = [_rand_words(rng, n) for n in sizes]
    zs = [(_root(n, rnd.randrange(n)) if i % 3 == 0 else rnd.randrange(o.R)) for i, n in enumerate(sizes)]
    _check_equal_single(pkg, eng, evals, zs)


def _barycentric(evals, n, z):
    """p(z) for the interpolant of evals on the domain of size n (z outside it)."""
    w = o.PRIMITIVE_ROOTS_OF_UNITY[n.bit_length() - 1]
    total, r = 0, 1
    for f in evals:
        total = (total + f * r % o.R * pow((z - r) % o.R, -1, o.R)) % o.R
        r = r * w % o.R
    return total * (pow(z, n, o.R) - 1) % o.R * pow(n, -1, o.R) % o.R


@pytest.mark.parametrize("logn", [12, 16])
def test_tau_trick_closed_form(pkg, eng, srs, logn):
    """On the synthetic SRS tau^j G: proof = [(p(tau) - y) / (tau - z)] G and y = the oracle's
    evaluate_polynomial_in_evaluation_form, for roots and random points."""
    n = 1 << logn
    rnd = random.Random(100 + logn)
    evals = [rnd.randrange(o.R) for _ in range(n)]
    zs = [1, _root(n, rnd.randrange(n)), rnd.randrange(o.R), rnd.randrange(o.R)]
    proofs, ys = pkg.KZG.compute_proofs([pkg.PolynomialEvalForm(evals)] * len(zs), zs, srs)
    p_tau = _barycentric(evals, n, TAU)
    po = o.PolynomialEvalForm(evals)
    for z, pi, y in zip(zs, proofs, ys):
        assert y == o.evaluate_polynomial_in_evaluation_form(po, z)
        assert pi == o.g1_mul(o.G1_GEN, (p_tau - y) * pow((TAU - z) % o.R, -1, o.R) % o.R)


def test_round_trip_through_verify_proofs(pkg, eng, srs):
    """Commitments from kzgb_commit_eval, openings from the new call, kzgb_verify_proofs under [tau]G2 of the synthetic
    SRS: all true; with y bumped at {0, 17, last} exactly those are false."""
    n = 1 << 12
    rnd = random.Random(9)
    polys = [pkg.PolynomialEvalForm([rnd.randrange(o.R) for _ in range(n)]) for _ in range(4)]
    kzg = pkg.KZG()
    commits = [kzg.commit_eval_form(p, srs) for p in polys]
    m = 40
    ps = [polys[i % 4] for i in range(m)]
    cs = [commits[i % 4] for i in range(m)]
    zs = _points(n, rnd, m)
    proofs, ys = pkg.KZG.compute_proofs(ps, zs, srs)
    eng.set_g2_tau(o.g2_mul(o.G2_GEN, TAU))
    try:
        assert pkg.verify_proofs(cs, proofs, zs, ys, eng) == [True] * m
        bad = {0, 17, m - 1}
        ys2 = [(y + 1) % o.R if i in bad else y for i, y in enumerate(ys)]
        assert pkg.verify_proofs(cs, proofs, zs, ys2, eng) == [i not in bad for i in range(m)]
    finally:
        eng.set_g2_tau(None)


@pytest.mark.parametrize("option,value,default", [("group", 0, -1), ("lanes", 1, 0), ("lagrange", 0, 1),
                                                  ("eval_structured", 0, 1)])
def test_routes_agree(pkg, eng, option, value, default):
    """One context, one batch (groups of 2^6 and 2^12 with roots and random points mixed, and a lone 2^16), with an
    option that changes the route: the same words as with the defaults."""
    rnd = random.Random(33)
    rng = np.random.default_rng(33)
    sizes = [64] * 70 + [4096] * 9 + [1 << 16]
    polys = {n: [_rand_words(rng, n) for _ in range(3)] for n in set(sizes)}
    evals = [polys[n][i % 3] for i, n in enumerate(sizes)]
    zs = [(_root(n, rnd.randrange(n)) if i % 2 else rnd.randrange(o.R)) for i, n in enumerate(sizes)]
    want = _batch(pkg, eng, evals, zs)
    _set(pkg, option, value)
    try:
        assert _batch(pkg, eng, evals, zs) == want
    finally:
        _set(pkg, option, default)
    assert _batch(pkg, eng, evals, zs) == want


@pytest.mark.parametrize("large", [False, True], ids=["groups", "lanes"])
def test_dev_equals_host(pkg, eng, large):
    """kzgb_compute_proofs_dev with the evaluations back to back in one device buffer and with scattered device
    pointers: the words of the host form."""
    import torch

    rnd = random.Random(44 + large)
    rng = np.random.default_rng(44 + large)
    sizes = [64] * 20 + [4096] * 6 + ([1 << 18, 1 << 18] if large else [])
    evals = [_rand_words(rng, n) for n in sizes]
    zs = [(_root(n, rnd.randrange(n)) if i % 2 else rnd.randrange(o.R)) for i, n in enumerate(sizes)]
    want = _batch(pkg, eng, evals, zs)
    count = len(sizes)
    ns = (C.c_size_t * count)(*sizes)
    zm = b"".join(_z_mont(pkg, z) for z in zs)
    run = torch.frombuffer(bytearray(b"".join(evals)), dtype=torch.uint8).cuda()
    offs = np.cumsum([0] + [32 * n for n in sizes])
    bufs = [torch.frombuffer(bytearray(b"\x00" * 32 + e + b"\x00" * 64), dtype=torch.uint8).cuda() for e in evals]
    for ptrs in ([run.data_ptr() + int(offs[i]) for i in range(count)], [b.data_ptr() + 32 for b in bufs]):
        xy, inf, ys = C.create_string_buffer(64 * count), C.create_string_buffer(count), C.create_string_buffer(32 * count)
        eng.check(pkg.lib.kzgb_compute_proofs_dev(eng.h, (C.c_void_p * count)(*ptrs), ns, count, zm, xy, inf, ys))
        assert _entries(xy.raw, inf.raw, ys.raw, count) == want
    torch.cuda.synchronize()


def test_group_equals_single_context(pkg, eng, srs):
    """Two members (device 0 listed twice): the proofs and y of the one-context call, for a ragged batch."""
    rnd = random.Random(55)
    sizes = [64] * 10 + [4096] * 5 + [1 << 16, 1, 2, 64, 64]
    polys = [pkg.PolynomialEvalForm([rnd.randrange(o.R) for _ in range(n)]) for n in sizes]
    zs = [(_root(n, rnd.randrange(n)) if i % 2 else rnd.randrange(o.R)) for i, n in enumerate(sizes)]
    want = pkg.KZG.compute_proofs(polys, zs, srs)
    grp = pkg.Group([0, 0])
    try:
        grp.load_srs_synthetic(SRS_N, TAU)
        assert grp.compute_proofs(polys, zs) == want
        assert grp.compute_proofs([], []) == ([], [])
    finally:
        grp.close()


def test_errors(pkg, eng, srs):
    """Each error at the lowest failing entry when several entries fail differently, z = r and z = 2^256 - 1 rejected,
    outputs left untouched, count == 0 writes nothing, NULL out_inf and NULL ys_mont accepted."""
    rng = np.random.default_rng(66)
    ok = _rand_words(rng, 64)
    zr = o.R.to_bytes(32, "little")
    zmax = b"\xff" * 32
    zok = _z_mont(pkg, 12345)

    def call(evals, zs_raw, count=None):
        count = len(evals) if count is None else count
        keep = [C.create_string_buffer(e, max(32, len(e))) for e in evals]
        ptrs = (C.c_void_p * max(1, len(evals)))(*[C.cast(k, C.c_void_p).value for k in keep])
        ns = (C.c_size_t * max(1, len(evals)))(*[len(e) // 32 for e in evals])
        xy = C.create_string_buffer(b"\xab" * 64 * max(1, len(evals)))
        inf = C.create_string_buffer(b"\xab" * max(1, len(evals)))
        ys = C.create_string_buffer(b"\xab" * 32 * max(1, len(evals)))
        before = (xy.raw, inf.raw, ys.raw)
        rc = pkg.lib.kzgb_compute_proofs(eng.h, ptrs, ns, count, b"".join(zs_raw) or b"\x00" * 32, xy, inf, ys)
        return rc, (xy.raw, inf.raw, ys.raw) == before

    three = _rand_words(rng, 3)
    big = b"\x00" * (32 * (SRS_N * 2))
    cases = [
        ([ok, ok, three, big], [zok, zr, zok, zok], "InvalidFieldElement"),
        ([ok, three, big, ok], [zok, zok, zok, zmax], "FFTError"),
        ([ok, big, three, ok], [zok, zok, zr, zok], "SrsCapacityExceeded"),
        ([ok, b"", ok], [zok, zok, zok], "FFTError"),
        ([ok, ok], [zok, zmax], "InvalidFieldElement"),
    ]
    for evals, zs_raw, variant in cases:
        rc, untouched = call(evals, zs_raw)
        assert rc != 0 and pkg._capi.STATUS_VARIANT[rc] == variant, (variant, rc)
        assert untouched, variant
        msg = pkg.lib.kzgb_last_error(eng.h).decode()
        if variant == "FFTError":
            assert msg == "length provided is not a power of 2"
        if variant == "InvalidFieldElement":
            assert "1" in msg.split()
    rc, untouched = call([ok], [zok], count=0)
    assert rc == 0 and untouched
    # NULL out_inf and NULL ys_mont
    evals, zs = [ok, ok, _rand_words(rng, 4096)], [5, 1, 7]
    full = _batch(pkg, eng, evals, zs)
    assert [e[0] for e in _batch(pkg, eng, evals, zs, with_inf=False, with_y=False)] == [e[0] for e in full]
    assert [(e[0], e[2]) for e in _batch(pkg, eng, evals, zs, with_inf=False)] == [(e[0], e[2]) for e in full]
    with pytest.raises(pkg.KzgError) as e:
        pkg.KZG.compute_proofs([pkg.PolynomialEvalForm([1, 2])], [1, 2], srs)
    assert e.value.variant == "GenericError" and e.value.msg == "length's of the input are not the same"
    assert pkg.KZG.compute_proofs([], [], srs) == ([], [])
