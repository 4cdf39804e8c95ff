"""kzgb_compute_proofs_all_roots / KZG.compute_proofs_at_all_roots: the proof at every root of the domain in one call
(FK20).  Every proof is a unique group element, so each must be bit-identical to what
KZG::compute_proof_with_known_z_fr_index (prover/src/kzg.rs:187-207) returns for that index alone."""
import ctypes as C
import random

import pytest

import golden_data as g
from __graft_entry__ import load_package
from oracle import bn254 as o

pytestmark = pytest.mark.gpu
TAU = o.SYNTH_TAU


@pytest.fixture(scope="module")
def pkg():
    return load_package()


@pytest.fixture(scope="module")
def eng(pkg):
    e = pkg.Engine(0)
    yield e
    e.close()


@pytest.fixture(scope="module")
def ref_srs(pkg, eng):
    """The reference's prover/tests/test-files/g1.point (3000 points)."""
    return pkg.SRS.from_gnark_bytes(g.g1_point_bytes(), engine=eng)


def _kzg(pkg, n):
    k = pkg.KZG()
    k.calculate_and_store_roots_of_unity(32 * n)
    return k


def _single(pkg, poly, srs, indices):
    k = _kzg(pkg, len(poly))
    return [k.compute_proof_with_known_z_fr_index(poly, i, srs) for i in indices]


def _all(pkg, poly, srs):
    return _kzg(pkg, len(poly)).compute_proofs_at_all_roots(poly, srs)


def _sample(n, rnd, count):
    return sorted({0, 1, n // 2, n - 1} | set(rnd.sample(range(n), min(n, count - 4))))


def _batch_inv(vals):
    pref, acc = [], 1
    for v in vals:
        pref.append(acc)
        acc = acc * v % o.R
    inv = pow(acc, -1, o.R)
    out = [0] * len(vals)
    for i in range(len(vals) - 1, -1, -1):
        out[i] = inv * pref[i] % o.R
        inv = inv * vals[i] % o.R
    return out


def _barycentric(evals, roots, z):
    """p(z) for the interpolant of evals on the domain `roots` (z outside it)."""
    n = len(evals)
    inv = _batch_inv([(z - r) % o.R for r in roots])
    total = sum(e * r % o.R * d for e, r, d in zip(evals, roots, inv)) % o.R
    return total * (pow(z, n, o.R) - 1) % o.R * pow(n, -1, o.R) % o.R


def test_gettysburg_fixture_and_every_index(pkg, ref_srs):
    """kzg.proof.eq.input: all 40 rows; all 64 proofs = the single-index call on the GPU and in the oracle."""
    blob = pkg.Blob.from_raw_data(g.gettysburg())
    poly = blob.to_polynomial_eval_form(ref_srs.engine)
    assert len(poly) == 64
    got = _all(pkg, poly, ref_srs)
    for idx, x, y in g.proof_eq_input():
        assert got[idx] == (x, y), idx
    assert got == _single(pkg, poly, ref_srs, range(64))
    ko = o.KZG()
    ko.calculate_and_store_roots_of_unity(len(blob))
    po = o.Blob.from_raw_data(g.gettysburg()).to_polynomial_eval_form()
    ref = g.srs_points_string()
    assert got == [ko.compute_proof_with_known_z_fr_index(po, i, ref) for i in range(64)]


def test_every_size_equals_single_index(pkg, ref_srs):
    """n = 1 .. 2048 on g1.point, random evaluations: every index up to n = 256, 32 indices (0, 1, n/2, n-1 among them)
    above; every index against the oracle up to n = 16; n = 1 gives the identity."""
    rnd = random.Random(7)
    ref = g.srs_points_string()
    for logn in range(12):
        n = 1 << logn
        evals = [rnd.randrange(o.R) for _ in range(n)]
        poly = pkg.PolynomialEvalForm(evals)
        got = _all(pkg, poly, ref_srs)
        assert len(got) == n
        idx = list(range(n)) if n <= 256 else _sample(n, rnd, 32)
        assert [got[i] for i in idx] == _single(pkg, poly, ref_srs, idx), n
        if n <= 16:
            ko = o.KZG()
            ko.calculate_and_store_roots_of_unity(32 * n)
            po = o.PolynomialEvalForm(evals)
            assert got == [ko.compute_proof_with_known_z_fr_index(po, i, ref) for i in range(n)], n
    assert _all(pkg, pkg.PolynomialEvalForm([rnd.randrange(o.R)]), ref_srs) == [None]


@pytest.mark.parametrize("logn", [12, 16, 19])
def test_closed_form_full_size(pkg, logn):
    """Synthetic SRS tau^j G: sum_k rho^k pi_k = [sum_k rho^k q_k(tau)] G with q_k(tau) = (p(tau) - f_k) / (tau - w^k),
    one random linear combination (an MSM on the GPU) that checks all n proofs; 16 indices against the single-index
    call."""
    n = 1 << logn
    rnd = random.Random(logn)
    eng = pkg.Engine(0)
    try:
        srs = pkg.SRS.synthetic(n, TAU, engine=eng)
        evals = [rnd.randrange(o.R) for _ in range(n)]
        poly = pkg.PolynomialEvalForm(evals)
        got = _all(pkg, poly, srs)
        w = o.PRIMITIVE_ROOTS_OF_UNITY[logn]
        roots = [1] * n
        for i in range(1, n):
            roots[i] = roots[i - 1] * w % o.R
        p_tau = _barycentric(evals, roots, TAU)
        inv = _batch_inv([(TAU - r) % o.R for r in roots])
        rho = rnd.randrange(1, o.R)
        rho_k = [1] * n
        for i in range(1, n):
            rho_k[i] = rho_k[i - 1] * rho % o.R
        want = sum(rk * ((p_tau - f) * d % o.R) for rk, f, d in zip(rho_k, evals, inv)) % o.R
        assert pkg.g1_lincomb(got, rho_k, eng) == o.g1_mul(o.G1_GEN, want)
        idx = _sample(n, rnd, 16)
        assert [got[i] for i in idx] == _single(pkg, poly, srs, idx)
    finally:
        eng.close()


def test_adversarial_polynomials(pkg, ref_srs):
    """n = 2^10: zero and constant polynomials (every proof the identity, also for the constant r - 1), one non-zero
    evaluation, degree 1 (every proof the same point b * SRS_0), and sparse coefficients that zero a quarter of
    DFT_2n(c || 0)."""
    n = 1 << 10
    rnd = random.Random(10)
    ref = g.srs_points_string()
    one_hot = [0] * n
    one_hot[rnd.randrange(n)] = rnd.randrange(1, o.R)
    a, b = rnd.randrange(o.R), rnd.randrange(1, o.R)
    sparse = [0] * n
    sparse[3], sparse[n // 2 + 3] = o.R - 5, 5  # 5 X^3 (X^(n/2) - 1): zero at every 4th root of unity of order 2n
    cases = {
        "zero": [0] * n,
        "constant": [rnd.randrange(o.R)] * n,
        "all r-1": [o.R - 1] * n,
        "one non-zero": one_hot,
        "degree 1": o.fft([a, b] + [0] * (n - 2)),
        "sparse coefficients": o.fft(sparse),
    }
    for name, evals in cases.items():
        poly = pkg.PolynomialEvalForm(evals)
        got = _all(pkg, poly, ref_srs)
        assert got == _single(pkg, poly, ref_srs, range(n)), name
        if name in ("zero", "constant", "all r-1"):
            assert got == [None] * n, name
        if name == "degree 1":
            assert got == [o.g1_mul(ref[0], b)] * n


def test_table_cache(pkg):
    """Two calls and prepare-then-call give the same points; after the SRS is reloaded (another tau, then g1.point) the
    proofs follow the new SRS; kzgb_g1_ifft(64) still gives lagrangeG1SRS.txt after an all-roots call."""
    n = 64
    rnd = random.Random(3)
    poly = pkg.PolynomialEvalForm([rnd.randrange(o.R) for _ in range(n)])
    eng = pkg.Engine(0)
    try:
        srs = pkg.SRS.synthetic(1024, TAU, engine=eng)
        first = _all(pkg, poly, srs)
        assert _all(pkg, poly, srs) == first
        eng2 = pkg.Engine(0)
        srs2 = pkg.SRS.synthetic(1024, TAU, engine=eng2)
        srs2.prepare_all_roots(n)
        assert _all(pkg, poly, srs2) == first
        eng2.close()
        other = pkg.SRS.synthetic(1024, TAU + 1, engine=eng)
        got = _all(pkg, poly, other)
        assert got != first
        assert got == _single(pkg, poly, other, range(n))
        ref_srs = pkg.SRS.from_gnark_bytes(g.g1_point_bytes(), engine=eng)
        blob = pkg.Blob.from_raw_data(g.gettysburg())
        got = _all(pkg, blob.to_polynomial_eval_form(eng), ref_srs)
        for idx, x, y in g.proof_eq_input():
            assert got[idx] == (x, y), idx
        assert pkg.KZG().g1_ifft(64, ref_srs) == g.lagrange_srs_64()
    finally:
        eng.close()


def test_errors(pkg, eng, ref_srs):
    """n = 3: FFTError; n = 4096 over the 3000-point SRS: SrsCapacityExceeded (both also from the prepare call); a
    roots-of-unity table of another length: the mirror's GenericError with the reference's text; the context stays
    usable."""
    evals = pkg.fr_to_mont_bytes(list(range(4096)))
    out, inf = C.create_string_buffer(64 * 4096), C.create_string_buffer(4096)
    for n, variant in ((3, "FFTError"), (0, "FFTError"), (4096, "SrsCapacityExceeded")):
        with pytest.raises(pkg.KzgError) as e:
            eng.check(pkg.lib.kzgb_compute_proofs_all_roots(eng.h, evals, n, out, inf))
        assert e.value.variant == variant
        if variant == "FFTError":
            assert e.value.msg == "length provided is not a power of 2"
        with pytest.raises(pkg.KzgError) as e:
            ref_srs.prepare_all_roots(n)
        assert e.value.variant == variant
    k = pkg.KZG()
    k.calculate_and_store_roots_of_unity(32 * 32)
    with pytest.raises(pkg.KzgError) as e:
        k.compute_proofs_at_all_roots(pkg.PolynomialEvalForm([1] * 64), ref_srs)
    assert e.value.variant == "GenericError" and e.value.msg == "inconsistent length between blob and root of unities"
    poly = pkg.PolynomialEvalForm([5, 6, 7, 8])
    assert _all(pkg, poly, ref_srs) == _single(pkg, poly, ref_srs, range(4))

