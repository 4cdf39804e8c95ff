"""kzgb_commit_evals{,_dev}, kzgb_commit_coeffs{,_dev}, their group forms and KZG.commit_eval_forms / commit_coeff_forms:
KZG::commit_eval_form and commit_coeff_form (prover/src/kzg.rs:84-125) for many polynomials in one call.  Entry i must be
word for word (point, identity flag) what kzgb_commit_eval or kzgb_commit_coeff returns for polynomial i alone, on every
route the batch can take: groups cut from the entries sorted by size (one batched launch set each, domain <= 2^17), zero
tails of short coefficient lists, task lanes (larger polynomials, or coefficient lists an SRS cannot pad), the Lagrange and
the monomial tables."""
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
EVALS, COEFFS = "evals", "coeffs"


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


def _single(pkg, eng, form, words):
    """kzgb_commit_eval / kzgb_commit_coeff: (point words, identity flag)."""
    xy, inf = C.create_string_buffer(64), C.c_uint8(7)
    call = pkg.lib.kzgb_commit_eval if form == EVALS else pkg.lib.kzgb_commit_coeff
    eng.check(call(eng.h, words or b"\x00" * 32, len(words) // 32, xy, C.byref(inf)))
    return xy.raw, inf.value


def _entries(xy, inf, count):
    return [(xy[64 * i : 64 * i + 64], inf[i]) for i in range(count)]


def _batch(pkg, eng, form, polys, fill=0xAB, with_inf=True):
    """kzgb_commit_evals / kzgb_commit_coeffs on host polynomials: the (point, flag) of each entry."""
    count = len(polys)
    keep = [C.create_string_buffer(p, max(32, len(p))) for p in polys]
    ptrs = (C.c_void_p * count)(*[C.cast(k, C.c_void_p).value for k in keep])
    ns = (C.c_size_t * count)(*[len(p) // 32 for p in polys])
    xy = C.create_string_buffer(bytes([fill]) * 64 * count, 64 * count)
    inf = C.create_string_buffer(bytes([fill]) * count, count)
    call = pkg.lib.kzgb_commit_evals if form == EVALS else pkg.lib.kzgb_commit_coeffs
    eng.check(call(eng.h, ptrs, ns, count, xy, inf if with_inf else None))
    return _entries(xy.raw, inf.raw, count)


def _check_equal_single(pkg, eng, form, polys):
    got = _batch(pkg, eng, form, polys)
    want = {}
    for i, p in enumerate(polys):
        if id(p) not in want:
            want[id(p)] = _single(pkg, eng, form, p)
        assert got[i] == want[id(p)], (form, i, len(p) // 32)
    return got


def _polys(rng, sizes, distinct=3):
    """A few random polynomials of each size, and the zero polynomial of every size, reused across the batch."""
    pool = {n: [_rand_words(rng, n) for _ in range(distinct)] + [b"\x00" * 32 * n] for n in set(sizes)}
    return [pool[n][i % len(pool[n])] for i, n in enumerate(sizes)]


# interleaved sizes (the sort by size forms the groups), then adjacent runs
EVAL_SIZES = [64, 4096, 1, 64, 2, 4096, 1 << 16, 64, 4, 1 << 10, 4096, 2, 1] + [64] * 7 + [4096] * 4 + [1 << 12]
COEFF_SIZES = [511, 3, 1000, 0, 513, 1, 4097, 511, 1000, 3, 513, 0, 1, 4097, 1000] + [512] * 6 + [1000] * 5


def test_evals_equal_single_call(pkg, eng):
    """Evaluation sizes 1 to 2^16 in groups, interleaved and in runs, zero polynomials included."""
    _check_equal_single(pkg, eng, EVALS, _polys(np.random.default_rng(1), EVAL_SIZES))


def test_coeffs_equal_single_call(pkg, eng):
    """Coefficient lengths 0, 1, 3, 511, 512, 513, 1000 and 4097 in groups with zero tails, zero polynomials included."""
    _check_equal_single(pkg, eng, COEFFS, _polys(np.random.default_rng(2), COEFF_SIZES))


@pytest.mark.parametrize("form", [EVALS, COEFFS])
def test_tasks_equal_single_call(pkg, eng, form):
    """A 2^19 polynomial (above the 2^17 group limit) puts the whole batch on the task lanes, small entries included."""
    sizes = [1 << 19, 64, 1 << 19, 4096, 1] if form == EVALS else [1 << 19, 1000, 0, 4097, 1 << 19, 3]
    _check_equal_single(pkg, eng, form, _polys(np.random.default_rng(3), sizes, distinct=2))


def test_eval_form_equals_coeff_form_of_ifft(pkg, eng, srs):
    """prover/tests/kzg_test.rs:57-89: the commitment of evals in evaluation form is the commitment of IFFT(evals) in
    coefficient form, both sides batched."""
    rnd = random.Random(4)
    polys = [pkg.PolynomialEvalForm([rnd.randrange(o.R) for _ in range(n)]) for n in [4096, 64, 4096, 1 << 16, 64, 2]]
    evals = pkg.KZG.commit_eval_forms(polys, srs)
    coeffs = pkg.KZG.commit_coeff_forms([p.to_coeff_form(eng) for p in polys], srs)
    assert evals == coeffs
    assert evals[0] == pkg.KZG().commit_eval_form(polys[0], srs)


def test_known_answer_gettysburg(pkg):
    """Blob::from_raw_data(gettysburg) over the reference's g1.point SRS, in both forms and three times in one call: the
    oracle's commit_eval_form / commit_coeff_form."""
    e = pkg.Engine(0)
    try:
        srs = pkg.SRS.from_gnark_bytes(g.g1_point_bytes(), engine=e)
        pts = g.srs_points_string()
        blob = pkg.Blob.from_raw_data(g.gettysburg())
        pe = blob.to_polynomial_eval_form(e)
        pc = blob.to_polynomial_coeff_form(e)
        ok = o.KZG()
        want_e = ok.commit_eval_form(o.PolynomialEvalForm(pe.evaluations), pts)
        want_c = ok.commit_coeff_form(o.PolynomialCoeffForm(pc.coeffs), pts)
        assert pkg.KZG.commit_eval_forms([pe] * 3, srs) == [want_e] * 3
        assert pkg.KZG.commit_coeff_forms([pc] * 3, srs) == [want_c] * 3
    finally:
        e.close()


def _barycentric(evals, n, z):
    """p(z) for the interpolant of evals on the domain of size n (z outside it)."""
    w = o.PRIMITIVE_ROOTS_OF_UNITY[n.bit_length() - 1]
    total, r = 0, 1
    for f in evals:
        total = (total + f * r % o.R * pow((z - r) % o.R, -1, o.R)) % o.R
        r = r * w % o.R
    return total * (pow(z, n, o.R) - 1) % o.R * pow(n, -1, o.R) % o.R


def test_tau_closed_form(pkg, eng, srs):
    """On the synthetic SRS tau^j G: [p(tau)] G, evaluation form by the barycentric formula, coefficient form by Horner."""
    rnd = random.Random(6)
    evals = [[rnd.randrange(o.R) for _ in range(n)] for n in (4096, 64, 4096)]
    coeffs = [[rnd.randrange(o.R) for _ in range(n)] for n in (1000, 3, 1000)]
    got_e = pkg.KZG.commit_eval_forms([pkg.PolynomialEvalForm(v) for v in evals], srs)
    assert got_e == [o.g1_mul(o.G1_GEN, _barycentric(v, len(v), TAU)) for v in evals]
    words = [pkg.fr_to_mont_bytes(v) for v in coeffs]  # odd lengths: through the C ABI, unpadded
    got_c = _batch(pkg, eng, COEFFS, words)

    def horner(v):
        acc = 0
        for x in reversed(v):
            acc = (acc * TAU + x) % o.R
        return acc

    want = [o.g1_mul(o.G1_GEN, horner(v)) for v in coeffs]
    assert [pkg.g1_from_abi(xy, bytes([f]))[0] for xy, f in got_c] == want


@pytest.mark.parametrize(
    "option,value,default",
    [("group", 0, -1), ("group", 1, -1), ("lagrange", 0, 1), ("lanes", 1, 0), ("lanes", 6, 0), ("ntt_kernel", 0, -1),
     ("ntt_kernel", 1, -1)],
)
def test_routes_agree(pkg, eng, option, value, default):
    """One context, both forms, with an option that changes the route: the words of the defaults."""
    rng = np.random.default_rng(7)
    ev = _polys(rng, [64] * 40 + [4096] * 9 + [1 << 16])
    co = _polys(rng, [512, 1000, 4096, 511] * 10 + [3, 0])
    want = (_batch(pkg, eng, EVALS, ev), _batch(pkg, eng, COEFFS, co))
    _set(pkg, option, value)
    try:
        assert (_batch(pkg, eng, EVALS, ev), _batch(pkg, eng, COEFFS, co)) == want
    finally:
        _set(pkg, option, default)
    assert (_batch(pkg, eng, EVALS, ev), _batch(pkg, eng, COEFFS, co)) == want


def test_fresh_contexts_and_resident_tables(pkg, eng):
    """The words of the shared context on: a fresh context below lagrange_after (no Lagrange table: the monomial
    routes); a fresh context with a 2^19 monomial window table resident before a batch of 2^12 coefficient lists; a
    fresh context whose 3000-point SRS cannot pad lengths 2049 .. 3000 to 4096 (those run as tasks over ns points)."""
    rng = np.random.default_rng(8)
    co = _polys(rng, [4096] * 20 + [4000, 1000])
    ev = _polys(rng, [4096] * 20 + [64] * 3)
    want = (_batch(pkg, eng, EVALS, ev), _batch(pkg, eng, COEFFS, co))
    short = _polys(rng, [3000, 2049, 17, 3000, 0, 1000])
    want_short = _batch(pkg, eng, COEFFS, short)

    e = pkg.Engine(0)
    try:
        pkg.SRS.synthetic(SRS_N, TAU, engine=e)
        _set(pkg, "lagrange_after", 1 << 20)
        try:
            assert (_batch(pkg, e, EVALS, ev), _batch(pkg, e, COEFFS, co)) == want
        finally:
            _set(pkg, "lagrange_after", 2)
        s = pkg.SRS.synthetic(SRS_N, TAU, engine=e)  # a new SRS: no table of the old one is kept
        s.precompute(SRS_N)
        assert _batch(pkg, e, COEFFS, co) == want[1]
        assert _batch(pkg, e, EVALS, ev) == want[0]
        pkg.SRS.synthetic(3000, TAU, engine=e)
        assert _batch(pkg, e, COEFFS, short) == want_short
        assert _batch(pkg, e, COEFFS, short) == [_single(pkg, e, COEFFS, p) for p in short]
    finally:
        e.close()


@pytest.mark.parametrize("form", [EVALS, COEFFS])
def test_dev_equals_host(pkg, eng, form):
    """The _dev form with the polynomials back to back in one device buffer (read in place where whole) and with
    scattered device pointers; coefficient lists of unequal lengths share a group."""
    import torch

    rng = np.random.default_rng(9)
    sizes = [64] * 12 + [4096] * 6 if form == EVALS else [512] * 8 + [511, 300, 512, 1, 0, 4096, 4000, 4096]
    polys = _polys(rng, sizes)
    want = _batch(pkg, eng, form, polys)
    count = len(sizes)
    ns = (C.c_size_t * count)(*sizes)
    run = torch.frombuffer(bytearray(b"".join(polys) + b"\x00" * 32), dtype=torch.uint8).cuda()
    offs = np.cumsum([0] + [32 * n for n in sizes])
    bufs = [torch.frombuffer(bytearray(b"\x00" * 32 + p + b"\x00" * 64), dtype=torch.uint8).cuda() for p in polys]
    call = pkg.lib.kzgb_commit_evals_dev if form == EVALS else pkg.lib.kzgb_commit_coeffs_dev
    for ptrs in ([run.data_ptr() + int(offs[i]) for i in range(count)], [b.data_ptr() + 32 for b in bufs]):
        before = (run.cpu().numpy().tobytes(), [b.cpu().numpy().tobytes() for b in bufs])
        xy, inf = C.create_string_buffer(64 * count), C.create_string_buffer(count)
        eng.check(call(eng.h, (C.c_void_p * count)(*ptrs), ns, count, xy, inf))
        assert _entries(xy.raw, inf.raw, count) == want
        assert (run.cpu().numpy().tobytes(), [b.cpu().numpy().tobytes() for b in bufs]) == before  # inputs unchanged
    torch.cuda.synchronize()


def test_group_equals_single_context(pkg, eng, srs):
    """Two members (device 0 listed twice): the commitments of the one-context call, both forms, ragged batches."""
    rnd = random.Random(10)
    ev = [pkg.PolynomialEvalForm([rnd.randrange(o.R) for _ in range(n)]) for n in [64] * 6 + [4096] * 5 + [1 << 16, 1, 2]]
    co = [pkg.PolynomialCoeffForm([rnd.randrange(o.R) for _ in range(n)]) for n in [512, 1024, 2048, 512, 1024] * 3 + [1]]
    want = (pkg.KZG.commit_eval_forms(ev, srs), pkg.KZG.commit_coeff_forms(co, srs))
    grp = pkg.Group([0, 0])
    try:
        grp.load_srs_synthetic(SRS_N, TAU)
        assert (grp.commit_eval_forms(ev), grp.commit_coeff_forms(co)) == want
        assert grp.commit_eval_forms([]) == [] and grp.commit_coeff_forms([]) == []
    finally:
        grp.close()


def test_errors(pkg, eng, srs):
    """Each error and its order of checks at the lowest failing entry, outputs left untouched, count == 0 writes nothing,
    NULL out_inf accepted."""
    rng = np.random.default_rng(11)
    ok = _rand_words(rng, 64)
    three = _rand_words(rng, 3)
    big = b"\x00" * (32 * (SRS_N * 2))   # above srs_len, a power of two
    big3 = b"\x00" * (32 * (SRS_N + 3))  # above srs_len, not a power of two

    def call(form, polys, count=None):
        count = len(polys) if count is None else count
        keep = [C.create_string_buffer(p, max(32, len(p))) for p in polys]
        ptrs = (C.c_void_p * max(1, len(polys)))(*[C.cast(k, C.c_void_p).value for k in keep])
        ns = (C.c_size_t * max(1, len(polys)))(*[len(p) // 32 for p in polys])
        xy = C.create_string_buffer(b"\xab" * 64 * max(1, len(polys)))
        inf = C.create_string_buffer(b"\xab" * max(1, len(polys)))
        before = (xy.raw, inf.raw)
        fn = pkg.lib.kzgb_commit_evals if form == EVALS else pkg.lib.kzgb_commit_coeffs
        rc = fn(eng.h, ptrs, ns, count, xy, inf)
        return rc, (xy.raw, inf.raw) == before

    cases = [
        (EVALS, [ok, ok, three, big], "FFTError"),
        (EVALS, [ok, big3, three], "SrsCapacityExceeded"),  # capacity is checked before the power of two
        (EVALS, [ok, big, three], "SrsCapacityExceeded"),
        (EVALS, [ok, b"", big], "FFTError"),
        (COEFFS, [three, b"", ok, big3, big], "SerializationError"),
    ]
    for form, polys, variant in cases:
        rc, untouched = call(form, polys)
        assert rc != 0 and pkg._capi.STATUS_VARIANT[rc] == variant, (form, variant, rc)
        assert untouched, variant
        msg = pkg.lib.kzgb_last_error(eng.h).decode()
        if variant == "FFTError":
            assert msg == "length provided is not a power of 2"
        if variant == "SerializationError":
            assert msg == "polynomial length is not correct"
        if variant == "SrsCapacityExceeded":
            assert f"polynomial_len={len(polys[1]) // 32}" in msg
    for form in (EVALS, COEFFS):
        rc, untouched = call(form, [ok], count=0)
        assert rc == 0 and untouched
        polys = [ok, ok, _rand_words(rng, 4096)]
        assert [e[0] for e in _batch(pkg, eng, form, polys, with_inf=False)] == [e[0] for e in _batch(pkg, eng, form, polys)]
    with pytest.raises(pkg.KzgError) as e:
        pkg.KZG.commit_eval_forms([pkg.PolynomialEvalForm([1] * 64), pkg.PolynomialEvalForm([1] * (2 * SRS_N))], srs)
    assert e.value.variant == "SrsCapacityExceeded"
    assert pkg.KZG.commit_eval_forms([], srs) == [] and pkg.KZG.commit_coeff_forms([], srs) == []


def test_round_trip_through_proofs(pkg, eng, srs):
    """kzgb_commit_evals -> kzgb_compute_proofs -> kzgb_verify_proofs under [tau]G2 of the synthetic SRS: all true; with
    one commitment replaced by another polynomial's, exactly that entry is false."""
    n, m = 1 << 12, 24
    rnd = random.Random(12)
    polys = [pkg.PolynomialEvalForm([rnd.randrange(o.R) for _ in range(n if i % 3 else 64)]) for i in range(m)]
    cs = pkg.KZG.commit_eval_forms(polys, srs)
    zs = [rnd.randrange(o.R) for _ in range(m)]
    proofs, ys = pkg.KZG.compute_proofs(polys, zs, srs)
    eng.set_g2_tau(o.g2_mul(o.G2_GEN, TAU))
    try:
        assert pkg.verify_proofs(cs, proofs, zs, ys, eng) == [True] * m
        bad = 7
        cs2 = list(cs)
        cs2[bad] = cs[bad + 1]
        assert pkg.verify_proofs(cs2, proofs, zs, ys, eng) == [i != bad for i in range(m)]
    finally:
        eng.set_g2_tau(None)
