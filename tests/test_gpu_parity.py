"""GPU parity tests: every result of the CUDA path is compared bit-for-bit with the CPU oracle
and with the reference's own fixtures.  All calls go through the C ABI (via the Python mirror)."""
import random

import pytest

import golden_data as g
from __graft_entry__ import load_package
from oracle import bn254 as o

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    return load_package()


@pytest.fixture(scope="module")
def eng(pkg):
    return pkg.Engine(0)


@pytest.fixture(scope="module")
def ref_srs(pkg, eng):
    """The reference's prover/tests/test-files/g1.point loaded through the GPU decompressor."""
    return pkg.SRS.from_gnark_bytes(g.g1_point_bytes(), engine=eng)


@pytest.fixture(scope="module")
def ref_srs_points():
    return g.srs_points_string()


def test_integer_pipe_microbench(pkg, eng):
    import ctypes as C

    for kind in range(4):
        v = C.c_double(0)
        eng.check(pkg.lib.kzgb_microbench(eng.h, kind, C.byref(v)))
        assert v.value > 1e9
        print(f"microbench kind {kind}: {v.value:.4e} ops/s")


def test_srs_decompression_kat(ref_srs, ref_srs_points):
    """read_g1_point_from_bytes_be (helpers.rs:175-226) vs srs.g1.points.string: 3000/3000."""
    assert len(ref_srs) == 3000
    assert ref_srs.points() == ref_srs_points


def test_srs_load_errors(pkg, eng):
    bad = bytearray(g.g1_point_bytes()[: 32 * 8])
    # x = 4 with flag 0b10: 4^3 + 3 = 67 is a non-residue?  find one deterministically
    x = 2
    while o.fq_sqrt((x**3 + 3) % o.P) is not None:
        x += 1
    bad[32 * 5 : 32 * 6] = bytes([0x80]) + x.to_bytes(31, "big")
    with pytest.raises(pkg.KzgError) as e:
        pkg.SRS.from_gnark_bytes(bytes(bad), engine=pkg.Engine(0))
    assert e.value.variant == "NotOnCurveError" and "point 5" in e.value.msg
    inf_bad = bytes([0x40]) + bytes(30) + b"\x01"
    with pytest.raises(pkg.KzgError) as e:
        pkg.SRS.from_gnark_bytes(inf_bad, engine=pkg.Engine(0))
    assert e.value.variant == "DeserializationError"
    s = pkg.SRS.from_gnark_bytes(bytes([0x40]) + bytes(31) + g.g1_point_bytes()[:32], engine=pkg.Engine(0))
    assert s.points() == [None, (1, 2)]


def test_srs_new_order_error(pkg, tmp_path):
    # prover/tests/kzg_test.rs:19-28
    p = tmp_path / "g1.point"
    p.write_bytes(g.g1_point_bytes())
    with pytest.raises(pkg.KzgError) as e:
        pkg.SRS(str(p), 3000, 3001)
    assert e.value.msg == "Number of points to load exceeds SRS order."
    s = pkg.SRS(str(p), 3000, 100)
    assert s.points() == g.srs_points_string()[:100]


def test_streamed_ingest_and_point_cache(pkg, ref_srs_points, tmp_path):
    """SRS::new through the chunked loader (chunks of 257 points: 12 chunks for the 3000-point fixture), a bad
    point in a late chunk, and the decompressed-point cache round trip incl. a damaged cache."""
    lib = pkg.lib
    raw = g.g1_point_bytes()
    path = tmp_path / "g1.point"
    path.write_bytes(raw)
    try:
        assert lib.kzgb_set_option(b"srs_chunk_points", 257) == 0
        srs = pkg.SRS(str(path), 3000, 3000, engine=pkg.Engine(0))
        assert srs.points() == ref_srs_points
        assert pkg.SRS(str(path), 3000, 1000, engine=pkg.Engine(0)).points() == ref_srs_points[:1000]
        with pytest.raises(pkg.KzgError) as e:
            pkg.SRS(str(path), 3001, 3001, engine=pkg.Engine(0))  # file shorter than points_to_load
        assert "Failed to read G1 points" in e.value.msg
        x = 2
        while o.fq_sqrt((x**3 + 3) % o.P) is not None:
            x += 1
        bad = bytearray(raw)
        bad[32 * 2345 : 32 * 2346] = bytes([0x80]) + x.to_bytes(31, "big")
        with pytest.raises(pkg.KzgError) as e:
            pkg.SRS.from_gnark_bytes(bytes(bad), engine=pkg.Engine(0))
        assert e.value.variant == "NotOnCurveError" and "point 2345" in e.value.msg
        bad[32 * 700 : 32 * 701] = bytes([0x40, 1]) + bytes(30)  # infinity flag with stray bits, in an earlier chunk
        with pytest.raises(pkg.KzgError) as e:
            pkg.SRS.from_gnark_bytes(bytes(bad), engine=pkg.Engine(0))
        assert e.value.variant == "DeserializationError" and "point 700" in e.value.msg
        cache = tmp_path / "g1.cache"
        srs.save_cache(str(cache))
        assert cache.stat().st_size == 64 + 64 * 3000
        assert pkg.SRS.from_cache(str(cache), engine=pkg.Engine(0)).points() == ref_srs_points
        part = pkg.SRS.from_cache(str(cache), 1500, engine=pkg.Engine(0))
        assert len(part) == 1500 and part.points() == ref_srs_points[:1500]
        with pytest.raises(pkg.KzgError) as e:
            pkg.SRS.from_cache(str(cache), 3001, engine=pkg.Engine(0))
        assert e.value.msg == "Number of points to load exceeds SRS order."
        blob = bytearray(cache.read_bytes())
        blob[64 + 64 * 2000 + 5] ^= 0x10  # one flipped bit in point 2000
        dmg = tmp_path / "damaged.cache"
        dmg.write_bytes(bytes(blob))
        with pytest.raises(pkg.KzgError) as e:
            pkg.SRS.from_cache(str(dmg), engine=pkg.Engine(0))
        assert e.value.variant == "NotOnCurveError" and "2000" in e.value.msg
        dmg.write_bytes(bytes(blob[: 64 + 64 * 100]))  # truncated
        with pytest.raises(pkg.KzgError):
            pkg.SRS.from_cache(str(dmg), 3000, engine=pkg.Engine(0))
        dmg.write_bytes(raw)
        with pytest.raises(pkg.KzgError) as e:
            pkg.SRS.from_cache(str(dmg), engine=pkg.Engine(0))
        assert e.value.variant == "DeserializationError"
    finally:
        lib.kzgb_set_option(b"srs_chunk_points", 0)


def test_roots_of_unity_match_the_reference_table(pkg, eng):
    """helpers::calculate_roots_of_unity (helpers.rs:553-610) on the GPU vs the oracle and the literal
    table of primitives/tests/helpers_test.rs:587-628 (first/last entries); error texts of :554-566."""
    for nbytes in (1, 32, 33, 1536, 32 * 4096, 32 * 5000):
        got = pkg.calculate_roots_of_unity(nbytes, eng)
        assert got == o.calculate_roots_of_unity(nbytes)
    n = 1 << 19
    big = pkg.calculate_roots_of_unity(32 * n, eng)
    w = o.PRIMITIVE_ROOTS_OF_UNITY[19]
    assert len(big) == n and big[0] == 1 and big[1] == w and big[n // 2] == o.R - 1
    assert big[n - 1] == pow(w, n - 1, o.R) and big[12345] == pow(w, 12345, o.R)
    with pytest.raises(pkg.KzgError) as e:
        pkg.calculate_roots_of_unity(0, eng)
    assert e.value.msg == "Length of data after padding is 0"
    with pytest.raises(pkg.KzgError) as e:
        pkg.calculate_roots_of_unity(32 * ((1 << 28) + 1), eng)
    assert e.value.msg == "the length of data after padding is not valid with respect to the SRS"


def test_to_fr_array_kat(pkg, eng):
    assert pkg.to_fr_array(g.blobs_txt(), eng) == g.blobs_from_fr()
    for raw in (b"", b"\x01", bytes(range(33)), b"\xff" * 95, g.gettysburg()):
        assert pkg.to_fr_array(raw, eng) == o.to_fr_array(raw)
    frs = g.blobs_from_fr()[:77] + [0, 1, o.R - 1]
    assert pkg.to_byte_array(frs, 32 * len(frs), eng) == o.to_byte_array(frs, 32 * len(frs))
    assert pkg.to_byte_array(frs, 100, eng) == o.to_byte_array(frs, 100)


@pytest.fixture(params=[0, 1], ids=["smem-tiles", "warp-resident"])
def ntt_kernel(pkg, request):
    """Both Fr NTT implementations (ntt.cu: shared-memory tile passes, and the register / warp-shuffle / bulk-copy passes)."""
    pkg.lib.kzgb_set_option(b"ntt_kernel", request.param)
    yield request.param
    pkg.lib.kzgb_set_option(b"ntt_kernel", -1)


@pytest.mark.parametrize("logn", [0, 1, 2, 3, 4, 5, 7, 8, 9, 10, 11, 12, 13])
def test_ntt_matches_oracle(pkg, eng, logn, ntt_kernel):
    rnd = random.Random(100 + logn)
    n = 1 << logn
    v = [rnd.randrange(o.R) for _ in range(n)]
    assert pkg._ntt(v, False, eng) == o.fft(v)
    assert pkg._ntt(v, True, eng) == o.ifft(v)


@pytest.mark.parametrize("logn", [16, 17, 19, 21])
def test_ntt_roundtrip_large(pkg, eng, logn, ntt_kernel):
    """FFT o IFFT identity (primitives/tests/polynomial_test.rs:47-64) at bench sizes, plus a
    delta-function known answer: fft(e_1)[i] = w^i."""
    import ctypes as C

    n = 1 << logn
    rnd = random.Random(logn)
    seed = [rnd.randrange(o.R) for _ in range(256)]
    vals = (seed * (n // 256))[:n]
    buf = C.create_string_buffer(pkg.fr_to_mont_bytes(seed) * (n // 256), 32 * n)
    orig = buf.raw
    eng.check(pkg.lib.kzgb_ntt_fr(eng.h, buf, n, 0))
    assert buf.raw != orig
    eng.check(pkg.lib.kzgb_ntt_fr(eng.h, buf, n, 1))
    assert buf.raw == orig
    delta = C.create_string_buffer(bytes(32) + pkg.fr_to_mont_bytes([1]) + bytes(32 * (n - 2)), 32 * n)
    eng.check(pkg.lib.kzgb_ntt_fr(eng.h, delta, n, 0))
    w = o.PRIMITIVE_ROOTS_OF_UNITY[logn]
    for i in (0, 1, 2, 3, n // 2, n - 1, 12345 % n):
        assert pkg.fr_from_mont_bytes(delta.raw[32 * i : 32 * i + 32])[0] == pow(w, i, o.R)
    del vals


def test_msm_var_matches_oracle(pkg, eng, ref_srs_points):
    rnd = random.Random(1)
    for m in (1, 2, 33, 300):
        pts = ref_srs_points[:m]
        sc = [rnd.randrange(o.R) for _ in range(m)]
        assert pkg.g1_lincomb(pts, sc, eng) == o.msm(pts, sc)
    # edge cases: zero scalars, identity bases, duplicate bases with equal scalars (forces P + P in a
    # bucket), P and -P with equal scalars (forces P + (-P)), scalars 1 and r - 1
    P1, P2 = ref_srs_points[1], ref_srs_points[2]
    pts = [P1, P1, P2, o.g1_neg(P2), None, P1, P2, P2]
    sc = [5, 5, 77, 77, 123456, 0, o.R - 1, 1]
    assert pkg.g1_lincomb(pts, sc, eng) == o.msm(pts, sc)
    assert pkg.g1_lincomb([P1, P2], [0, 0], eng) is None
    assert pkg.g1_lincomb([], [], eng) is None
    big = [rnd.randrange(o.R) for _ in range(64)]
    same = [ref_srs_points[7]] * 64
    assert pkg.g1_lincomb(same, big, eng) == o.g1_mul(ref_srs_points[7], sum(big) % o.R)
    with pytest.raises(pkg.KzgError) as e:
        pkg.g1_lincomb([P1], [1, 2], eng)
    assert e.value.variant == "MsmError"


def test_msm_fixed_base_matches_oracle(pkg, ref_srs, ref_srs_points):
    rnd = random.Random(2)
    kzg = pkg.KZG()
    for n in (1, 2, 64, 1024):
        sc = [rnd.randrange(o.R) for _ in range(n)]
        got = kzg.commit_coeff_form(pkg.PolynomialCoeffForm(sc), ref_srs)
        assert got == o.msm(ref_srs_points[:n], sc)
    # all-equal coefficients: every point of a window lands in one bucket (chunk-spanning buckets)
    sc = [0x1234567890ABCDEF1234567890ABCDEF] * 2048
    assert kzg.commit_coeff_form(pkg.PolynomialCoeffForm(sc), ref_srs) == o.msm(ref_srs_points[:2048], sc)
    zero = kzg.commit_coeff_form(pkg.PolynomialCoeffForm([0] * 64), ref_srs)
    assert zero is None  # zero polynomial -> identity (verifier/tests/tests.rs:239-269)
    with pytest.raises(pkg.KzgError) as e:
        kzg.commit_coeff_form(pkg.PolynomialCoeffForm([1] * 4096), ref_srs)
    assert e.value.variant == "SerializationError" and e.value.msg == "polynomial length is not correct"


def test_gettysburg_commit_and_proof_kats(pkg, ref_srs, ref_srs_points):
    """kzg.proof.eq.input: 40 proofs at roots of unity (z in the domain -> kzg.rs:237-260)."""
    blob = pkg.Blob.from_raw_data(g.gettysburg())
    kzg = pkg.KZG()
    kzg.calculate_and_store_roots_of_unity(len(blob))
    c = kzg.commit_blob(blob, ref_srs)
    assert pkg.g1_to_gnark_be(c).hex() == "868bf472ebc0e26c297f8a9257c3f42a38af1e4612b60f6ac64d57dc272d50b1"
    poly = blob.to_polynomial_eval_form(ref_srs.engine)
    assert len(poly) == 64
    assert kzg.commit_eval_form(poly, ref_srs) == c
    assert kzg.commit_coeff_form(poly.to_coeff_form(ref_srs.engine), ref_srs) == c  # kzg_test.rs:57-89
    for idx, x, y in g.proof_eq_input():
        assert kzg.compute_proof_with_known_z_fr_index(poly, idx, ref_srs) == (x, y)


def test_g1_ifft_kat(pkg, ref_srs):
    kzg = pkg.KZG()
    assert kzg.g1_ifft(64, ref_srs) == g.lagrange_srs_64()
    with pytest.raises(pkg.KzgError) as e:
        kzg.g1_ifft(15, ref_srs)
    assert e.value.variant == "FFTError" and "length provided is not a power of 2" in e.value.msg


def test_evaluate_polynomial(pkg, eng):
    rnd = random.Random(3)
    for raw in (g.gettysburg(), b"short", bytes(rnd.getrandbits(8) for _ in range(31 * 300))):
        bo = o.Blob.from_raw_data(raw)
        po = bo.to_polynomial_eval_form()
        pg = pkg.PolynomialEvalForm(po.evaluations[: len(bo) // 32])
        roots = o.calculate_roots_of_unity(len(bo))
        for z in (rnd.randrange(o.R), 0, 1, roots[-1], roots[len(roots) // 3]):
            assert pkg.evaluate_polynomial_in_evaluation_form(pg, z, eng) == o.evaluate_polynomial_in_evaluation_form(po, z)


@pytest.mark.parametrize("logn", [6, 7, 9, 12, 16])
def test_structured_and_generic_denominators_agree(pkg, logn):
    """1/(z - w_i) from the factorisation of z^n - 1 (z outside the domain) vs the generic prefix/suffix
    products: same evaluation y and same proof, also for z = 0, z = 1 + r - 1 (= 0), z = 2 and a root (generic path)."""
    n = 1 << logn
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(n, o.SYNTH_TAU, engine=eng)
    rnd = random.Random(300 + logn)
    ev = [rnd.randrange(o.R) for _ in range(n)]
    poly = pkg.PolynomialEvalForm(ev)
    kzg = pkg.KZG()
    kzg.calculate_and_store_roots_of_unity(32 * n)
    w = o.PRIMITIVE_ROOTS_OF_UNITY[logn]
    zs = [rnd.randrange(o.R), 0, 2, o.R - 1 if logn == 0 else pow(w, 3, o.R), rnd.randrange(o.R)]
    got = {}
    try:
        for mode in (1, 0):
            assert pkg.lib.kzgb_set_option(b"eval_structured", mode) == 0
            got[mode] = [(pkg.evaluate_polynomial_in_evaluation_form(poly, z, eng), kzg.compute_proof(poly, z, srs)) for z in zs]
    finally:
        pkg.lib.kzgb_set_option(b"eval_structured", 1)
    assert got[0] == got[1]
    if logn <= 9:
        po = o.PolynomialEvalForm(ev)
        for z, (y, _) in zip(zs, got[1]):
            assert y == o.evaluate_polynomial_in_evaluation_form(po, z)


def test_blob_proof_matches_oracle(pkg, ref_srs, ref_srs_points):
    rnd = random.Random(4)
    for raw in (g.gettysburg(), b"a", bytes(rnd.getrandbits(8) for _ in range(31 * 100 + 5))):
        blob = pkg.Blob.from_raw_data(raw)
        bo = o.Blob.from_raw_data(raw)
        kzg, ko = pkg.KZG(), o.KZG()
        kzg.calculate_and_store_roots_of_unity(len(blob))
        ko.calculate_and_store_roots_of_unity(len(bo))
        c = kzg.commit_blob(blob, ref_srs)
        assert c == ko.commit_blob(bo, ref_srs_points)
        assert kzg.compute_blob_proof(blob, c, ref_srs) == ko.compute_blob_proof(bo, c, ref_srs_points)
    # full-range canonical blob (blobs.txt prefix), ragged non-canonical blob
    full = g.blobs_txt()[: 32 * 200]
    blob, bo = pkg.Blob.new(full), o.Blob(full)
    kzg, ko = pkg.KZG(), o.KZG()
    kzg.calculate_and_store_roots_of_unity(len(blob))
    ko.calculate_and_store_roots_of_unity(len(bo))
    c = kzg.commit_blob(blob, ref_srs)
    assert c == ko.commit_blob(bo, ref_srs_points)
    assert kzg.compute_blob_proof(blob, c, ref_srs) == ko.compute_blob_proof(bo, c, ref_srs_points)
    ragged = b"\xff" * 45 + bytes(range(50))
    blob, bo = pkg.Blob.from_unchecked(ragged), o.Blob.from_unchecked(ragged)
    kzg.calculate_and_store_roots_of_unity(len(blob))
    ko.calculate_and_store_roots_of_unity(len(bo))
    c = kzg.commit_blob(blob, ref_srs)
    assert c == ko.commit_blob(bo, ref_srs_points)
    assert kzg.compute_blob_proof(blob, c, ref_srs) == ko.compute_blob_proof(bo, c, ref_srs_points)
    # invalid commitment rejected (prover/tests/kzg_test.rs:163-196)
    with pytest.raises(pkg.KzgError) as e:
        kzg.compute_blob_proof(blob, (1, 3), ref_srs)
    assert e.value.variant == "NotOnCurveError"
    # roots not stored for this length -> GenericError (kzg.rs:135-139)
    with pytest.raises(pkg.KzgError) as e:
        pkg.KZG().compute_blob_proof(blob, c, ref_srs)
    assert e.value.msg == "inconsistent length between blob and root of unities"


def test_srs_capacity_error(pkg, eng):
    srs = pkg.SRS.from_gnark_bytes(g.g1_point_bytes()[: 32 * 16], engine=pkg.Engine(0))
    with pytest.raises(pkg.KzgError) as e:
        pkg.KZG().commit_blob(pkg.Blob.from_raw_data(g.gettysburg()), srs)
    assert e.value.variant == "SrsCapacityExceeded"


def test_synthetic_srs_and_tau_trick(pkg):
    """SRS_i = tau^i G generated on the GPU; MSM == (sum s_i tau^i) G (SURVEY.md 0.9), n = 2^12 (config 1)."""
    n = 1 << 12
    srs = pkg.SRS.synthetic(n, o.SYNTH_TAU)
    ref = o.synthetic_srs(64)
    assert srs.points(0, 64) == ref
    assert srs.points(n - 1, 1) == [o.g1_mul(o.G1_GEN, pow(o.SYNTH_TAU, n - 1, o.R))]
    blob = pkg.Blob.new(g.blobs_txt())  # exactly 4096 full-range canonical Fr (config 1 blob)
    kzg = pkg.KZG()
    kzg.calculate_and_store_roots_of_unity(len(blob))
    c = kzg.commit_blob(blob, srs)
    evals = g.blobs_from_fr()
    coeffs = o.ifft(evals)
    assert c == o.tau_trick_msm(coeffs)
    bo = o.Blob(g.blobs_txt())
    z = o.compute_challenge(bo, c)
    assert pkg.compute_challenge(blob, c) == z
    y = o.evaluate_polynomial_in_evaluation_form(bo.to_polynomial_eval_form(), z)
    ptau = 0
    for cf in reversed(coeffs):
        ptau = (ptau * o.SYNTH_TAU + cf) % o.R
    expect = o.g1_mul(o.G1_GEN, (ptau - y) * o.fr_inv((o.SYNTH_TAU - z) % o.R) % o.R)
    assert kzg.compute_blob_proof(blob, c, srs) == expect


def test_batch_commit_and_prove(pkg, ref_srs, ref_srs_points):
    rnd = random.Random(6)
    raws = [g.gettysburg(), b"b", bytes(rnd.getrandbits(8) for _ in range(31 * 64)), bytes(31 * 17), g.gettysburg()[:500],
            bytes(rnd.getrandbits(8) for _ in range(31 * 256 - 3)), b"zz" * 40]
    blobs = [pkg.Blob.from_raw_data(r) for r in raws]
    cs, ps = pkg.KZG.commit_and_prove_blobs(blobs, ref_srs)
    for r, cb, pb in zip(raws, cs, ps):
        bo = o.Blob.from_raw_data(r)
        ko = o.KZG()
        ko.calculate_and_store_roots_of_unity(len(bo))
        c = ko.commit_blob(bo, ref_srs_points)
        assert cb == o.g1_serialize_compressed(c)
        assert pb == o.g1_serialize_compressed(ko.compute_blob_proof(bo, c, ref_srs_points))


def test_batch_groups_of_equal_size_blobs(pkg, ref_srs, ref_srs_points):
    """Small blobs go through the grouped path (one batched MSM / evaluation launch set per group): same
    bytes as one blob at a time, with and without the Lagrange-basis table, and as the oracle."""
    rnd = random.Random(16)
    raws = [bytes(rnd.getrandbits(8) for _ in range(31 * 64 - k)) for k in (0, 1, 40, 0, 7)]          # n = 64, ragged lengths
    raws += [bytes(rnd.getrandbits(8) for _ in range(31 * 256 - 3 * k)) for k in range(4)]            # n = 256
    raws += [bytes(31 * 64), raws[0], raws[0]]                                                        # zero blob, duplicates
    raws += [b"q"]                                                                                    # n = 1
    blobs = [pkg.Blob.from_raw_data(r) for r in raws]
    lib = pkg.lib
    outs = {}
    try:
        for lag in (1, 0):
            for group in (-1, 0, 3):
                lib.kzgb_set_option(b"lagrange", lag)
                lib.kzgb_set_option(b"group", group)
                srs = pkg.SRS.from_gnark_bytes(g.g1_point_bytes(), engine=pkg.Engine(0))
                outs[(lag, group)] = pkg.KZG.commit_and_prove_blobs(blobs, srs)
    finally:
        lib.kzgb_set_option(b"lagrange", 1)
        lib.kzgb_set_option(b"group", -1)
    first = outs[(1, -1)]
    for k, v in outs.items():
        assert v == first, k
    for i in (1, 5, 9, 12):
        bo = o.Blob.from_raw_data(raws[i])
        ko = o.KZG()
        ko.calculate_and_store_roots_of_unity(len(bo))
        c = ko.commit_blob(bo, ref_srs_points)
        assert first[0][i] == o.g1_serialize_compressed(c)
        assert first[1][i] == o.g1_serialize_compressed(ko.compute_blob_proof(bo, c, ref_srs_points))


def test_device_hashed_transcripts_equal_host_hashed(pkg):
    """Long-transcript hashing on the device (fs.cu k_fs_midstate_long, one warp per blob, from the resident blob bytes)
    forced on for the tail of a batch: same commitments and proofs as the host SHA-256 pool and as the oracle's
    compute_challenge.  Covers chunks >= r inside a blob and in its last chunk (reduced in place, helpers.rs:32-34),
    blobs that do not qualify (ragged length -> host), host-buffer and device-resident entry points, every split."""
    import ctypes as C

    import torch

    rnd = random.Random(77)
    n = 1 << 11
    TAU = o.SYNTH_TAU
    datas = []
    for k in range(6):
        chunks = [rnd.randrange(o.R).to_bytes(32, "big") for _ in range(n)]
        if k == 1:
            chunks[5] = (o.R + 12345).to_bytes(32, "big")          # >= r in the middle
            chunks[2 * 700] = b"\xff" * 32                          # the largest 256-bit value
        if k == 2:
            chunks[n - 1] = (2 * o.R + 7).to_bytes(32, "big")      # >= r in the chunk the host appends
            chunks[0] = (o.R).to_bytes(32, "big")                  # exactly r in block 0
        datas.append(b"".join(chunks))
    datas.insert(0, datas[0][: 32 * n - 40])                        # ragged: ends the eligible tail, stays on the host pool
    blobs = [pkg.Blob.from_unchecked(d) for d in datas]
    lib = pkg.lib
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(n, TAU, engine=eng)
    outs = {}
    try:
        lib.kzgb_set_option(b"group", 0)  # small blobs through the large-blob pipeline (where device hashing lives)
        for k in (0, 1, 4, 7):
            lib.kzgb_set_option(b"device_hash", k)
            outs[k] = pkg.KZG.commit_and_prove_blobs(blobs, srs)
        for lanes in (0, 1):  # one warp per transcript / one lane per transcript
            lib.kzgb_set_option(b"device_hash_lanes", lanes)
            lib.kzgb_set_option(b"device_hash", 5)
            outs["lanes%d" % lanes] = pkg.KZG.commit_and_prove_blobs(blobs, srs)
        lib.kzgb_set_option(b"device_hash_lanes", -1)
        # device-resident entry point
        dev = [torch.frombuffer(bytearray(d), dtype=torch.uint8).cuda() for d in datas]
        cnt = len(datas)
        keep = [C.create_string_buffer(d, len(d)) for d in datas]
        hp = (C.c_void_p * cnt)(*[C.cast(kb, C.c_void_p).value for kb in keep])
        dp = (C.c_void_p * cnt)(*[t.data_ptr() for t in dev])
        lens = (C.c_size_t * cnt)(*[len(d) for d in datas])
        cm, pf = C.create_string_buffer(32 * cnt), C.create_string_buffer(32 * cnt)
        lib.kzgb_set_option(b"device_hash", 4)
        eng.check(lib.kzgb_commit_and_prove_blobs_dev(eng.h, dp, hp, lens, cnt, cm, pf))
        outs["dev"] = ([cm.raw[32 * i : 32 * i + 32] for i in range(cnt)], [pf.raw[32 * i : 32 * i + 32] for i in range(cnt)])
    finally:
        lib.kzgb_set_option(b"group", -1)
        lib.kzgb_set_option(b"device_hash", -1)
        lib.kzgb_set_option(b"device_hash_lanes", -1)
    for k, v in outs.items():
        assert v == outs[0], k
    # z of the device-hashed blobs against the oracle's transcript: proof = ((p(tau) - y)/(tau - z)) G needs the right z
    for i in (2, 3):  # the blobs with chunks >= r
        bo = o.Blob.from_unchecked(datas[i])
        c = o.g1_deserialize_compressed(outs[0][0][i])
        z = o.compute_challenge(bo, c)
        poly = bo.to_polynomial_eval_form()
        y = o.evaluate_polynomial_in_evaluation_form(poly, z)
        ptau = o.evaluate_polynomial_in_evaluation_form(poly, TAU)
        assert c == o.g1_mul(o.G1_GEN, ptau)
        q = (ptau - y) * pow(TAU - z, -1, o.R) % o.R
        assert outs[7][1][i] == o.g1_serialize_compressed(o.g1_mul(o.G1_GEN, q))


def test_multibuffer_hashed_transcripts_equal_single_stream(pkg):
    """Host transcripts hashed 16 at a time on AVX-512 (sha256.cpp sha256_mb16_blocks via transcript.cpp challenge_midstates_mb16),
    forced on: same commitments and proofs as the single-stream pool and as the oracle's compute_challenge.  37 blobs =
    two full groups + a group of 5 that falls back to single streams; values >= r in block 0, in the middle, in the last
    chunk (which the host appends after the lockstep part) and a ragged blob that splits a run."""
    if not pkg.lib.kzgb_set_option(b"hash_mb", 1) == 0:
        pytest.fail("option hash_mb missing")
    rnd = random.Random(79)
    n = 1 << 10
    TAU = o.SYNTH_TAU
    datas = []
    for k in range(37):
        chunks = [rnd.randrange(o.R).to_bytes(32, "big") for _ in range(n)]
        if k == 3:
            chunks[0] = (o.R + 5).to_bytes(32, "big")
            chunks[77] = b"\xff" * 32
            chunks[78] = (o.R).to_bytes(32, "big")
        if k == 17:
            chunks[n - 1] = (3 * o.R + 11).to_bytes(32, "big")
            chunks[n - 2] = (o.R + 1).to_bytes(32, "big")
        datas.append(b"".join(chunks))
    datas[20] = datas[20][: 32 * n - 7]  # ragged: single stream, and it ends the run of equal sizes
    blobs = [pkg.Blob.from_unchecked(d) for d in datas]
    lib = pkg.lib
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(n, TAU, engine=eng)
    try:
        lib.kzgb_set_option(b"group", 0)
        lib.kzgb_set_option(b"device_hash", 0)
        lib.kzgb_set_option(b"hash_mb", 0)
        single = pkg.KZG.commit_and_prove_blobs(blobs, srs)
        lib.kzgb_set_option(b"hash_mb", 1)
        multi = pkg.KZG.commit_and_prove_blobs(blobs, srs)
        lib.kzgb_set_option(b"device_hash", 6)  # multi-buffer groups in front, the device's share behind
        mixed = pkg.KZG.commit_and_prove_blobs(blobs, srs)
    finally:
        lib.kzgb_set_option(b"group", -1)
        lib.kzgb_set_option(b"device_hash", -1)
        lib.kzgb_set_option(b"hash_mb", -1)
    assert multi == single and mixed == single
    for i in (3, 17):
        bo = o.Blob.from_unchecked(datas[i])
        c = o.g1_deserialize_compressed(single[0][i])
        z = o.compute_challenge(bo, c)
        poly = bo.to_polynomial_eval_form()
        y = o.evaluate_polynomial_in_evaluation_form(poly, z)
        ptau = o.evaluate_polynomial_in_evaluation_form(poly, TAU)
        q = (ptau - y) * pow(TAU - z, -1, o.R) % o.R
        assert multi[1][i] == o.g1_serialize_compressed(o.g1_mul(o.G1_GEN, q))


def test_verify_batch_rlc(pkg, ref_srs, ref_srs_points):
    """verifier/src/batch.rs:16-249 up to the pairing: both G1 outputs equal the oracle's."""
    rnd = random.Random(8)
    raws = [g.gettysburg(), b"hello", bytes(rnd.getrandbits(8) for _ in range(31 * 30)), g.gettysburg()]
    blobs_o = [o.Blob.from_raw_data(r) for r in raws]
    cs, ps = [], []
    for bo in blobs_o:
        ko = o.KZG()
        ko.calculate_and_store_roots_of_unity(len(bo))
        c = ko.commit_blob(bo, ref_srs_points)
        cs.append(c)
        ps.append(ko.compute_blob_proof(bo, c, ref_srs_points))
    lhs_o, rhs_o = o.verify_blob_kzg_proof_batch_rlc(blobs_o, cs, ps)
    blobs = [pkg.Blob.from_raw_data(r) for r in raws]
    lhs, rhs = pkg.verify_blob_kzg_proof_batch_rlc(blobs, cs, ps, ref_srs.engine)
    assert (lhs, rhs) == (lhs_o, rhs_o)
    with pytest.raises(pkg.KzgError) as e:
        pkg.verify_blob_kzg_proof_batch_rlc(blobs, [(1, 3)] + cs[1:], ps, ref_srs.engine)
    assert e.value.variant == "NotOnCurveError"
    with pytest.raises(pkg.KzgError):
        pkg.verify_blob_kzg_proof_batch_rlc(blobs, cs[:2], ps, ref_srs.engine)


@pytest.mark.parametrize("waves", [1, 4, 32])
def test_msm_exceptional_pairs_exact(pkg, eng, ref_srs, ref_srs_points, waves):
    """Bucket accumulation, chunk stitching and the quad-cooperative 2-D bucket reduction at small sizes, for
    several chunkings of the sorted list: results must equal the oracle for random inputs and for every
    exceptional pair -- identity bases (pass-through), duplicate bases with equal digits (P + P ->
    tangent), P and -P (-> identity), all-equal scalars (one hot bucket), zeros."""
    rnd = random.Random(100 + waves)
    try:
        pkg.lib.kzgb_set_option(b"acc_waves", waves)
        P1, P2, P3 = ref_srs_points[1], ref_srs_points[2], ref_srs_points[3]
        # variable-base: duplicates / negations / identity with equal scalars land in the same buckets
        pts = [P1, P1, P2, o.g1_neg(P2), None, P1, P2, P2, P3, P3, P3, P3, None, o.g1_neg(P1), P1, P1]
        sc = [5, 5, 77, 77, 123456, 0, o.R - 1, 1, 9, 9, 9, 9, 3, 5, 5, 5]
        assert pkg.g1_lincomb(pts, sc, eng) == o.msm(pts, sc)
        same = [ref_srs_points[7]] * 100
        big = [rnd.randrange(o.R) for _ in range(100)]
        assert pkg.g1_lincomb(same, big, eng) == o.g1_mul(ref_srs_points[7], sum(big) % o.R)
        assert pkg.g1_lincomb(same, [12345] * 100, eng) == o.g1_mul(ref_srs_points[7], 1234500)
        assert pkg.g1_lincomb([P1, o.g1_neg(P1)] * 8, [7] * 16, eng) is None
        for m in (1, 2, 3, 33, 300):
            pts = ref_srs_points[:m]
            sc = [rnd.randrange(o.R) for _ in range(m)]
            assert pkg.g1_lincomb(pts, sc, eng) == o.msm(pts, sc)
        # fixed-base table path
        kzg = pkg.KZG()
        for n in (1, 2, 64, 1024):
            sc = [rnd.randrange(o.R) for _ in range(n)]
            assert kzg.commit_coeff_form(pkg.PolynomialCoeffForm(sc), ref_srs) == o.msm(ref_srs_points[:n], sc)
        sc = [0x1234567890ABCDEF1234567890ABCDEF] * 2048
        assert kzg.commit_coeff_form(pkg.PolynomialCoeffForm(sc), ref_srs) == o.msm(ref_srs_points[:2048], sc)
        assert kzg.commit_coeff_form(pkg.PolynomialCoeffForm([0] * 64), ref_srs) is None
        # many points, few distinct digits: hot buckets that span dozens of chunks of either tier
        sc = [rnd.choice([3, 1 << 40, o.R - 2]) for _ in range(2048)]
        assert kzg.commit_coeff_form(pkg.PolynomialCoeffForm(sc), ref_srs) == o.msm(ref_srs_points[:2048], sc)
        sc = [rnd.randrange(o.R) for _ in range(2048)]
        assert kzg.commit_coeff_form(pkg.PolynomialCoeffForm(sc), ref_srs) == o.msm(ref_srs_points[:2048], sc)
    finally:
        pkg.lib.kzgb_set_option(b"acc_waves", 4)


def test_lagrange_table_and_monomial_paths_agree(pkg, ref_srs_points):
    """Evaluation-form commits/proofs through the resident Lagrange-basis table (one MSM on the evaluations,
    the cached form of kzg.rs:98) and through Fr-IFFT + monomial table give the oracle's group element."""
    rnd = random.Random(21)
    lib = pkg.lib
    try:
        results = {}
        for mode in (0, 1):
            assert lib.kzgb_set_option(b"lagrange", mode) == 0
            srs = pkg.SRS.from_gnark_bytes(g.g1_point_bytes(), engine=pkg.Engine(0))  # fresh context: no tables yet
            kzg = pkg.KZG()
            out = []
            for n in (2, 8, 64, 512, 2048):
                rr = random.Random(100 + n)
                ev = [rr.randrange(o.R) for _ in range(n)]
                if n == 8:
                    ev = [0] * n  # zero polynomial -> identity
                if n == 512:
                    ev = [ev[0]] * n  # constant polynomial: every evaluation in the same buckets
                poly = pkg.PolynomialEvalForm(ev)
                kzg.calculate_and_store_roots_of_unity(32 * n)
                out.append(kzg.commit_eval_form(poly, srs))
                out.append(kzg.compute_proof(poly, rr.randrange(o.R), srs))
                out.append(kzg.compute_proof_with_known_z_fr_index(poly, n // 3, srs))
            results[mode] = out
        assert results[0] == results[1]
        # oracle check of the Lagrange path at the sizes the big-int oracle finishes quickly
        lib.kzgb_set_option(b"lagrange", 1)
        srs = pkg.SRS.from_gnark_bytes(g.g1_point_bytes(), engine=pkg.Engine(0))
        srs.prepare_lagrange(64)
        ev = [rnd.randrange(o.R) for _ in range(64)]
        ko = o.KZG()
        ko.calculate_and_store_roots_of_unity(32 * 64)
        po = o.PolynomialEvalForm(ev)
        kzg = pkg.KZG()
        kzg.calculate_and_store_roots_of_unity(32 * 64)
        z = rnd.randrange(o.R)
        assert kzg.commit_eval_form(pkg.PolynomialEvalForm(ev), srs) == ko.commit_eval_form(po, ref_srs_points)
        assert kzg.compute_proof(pkg.PolynomialEvalForm(ev), z, srs) == ko.compute_proof(po, z, ref_srs_points)
        with pytest.raises(pkg.KzgError) as e:
            srs.prepare_lagrange(48)
        assert e.value.variant == "FFTError"
        with pytest.raises(pkg.KzgError) as e:
            srs.prepare_lagrange(4096)  # 3000-point SRS
        assert e.value.variant == "SrsCapacityExceeded"
    finally:
        lib.kzgb_set_option(b"lagrange", 1)


def test_lagrange_table_tau_trick_large(pkg):
    """n = 2^16 on the synthetic SRS: commitment through the Lagrange table == p(tau) G, proof == ((p(tau)-y)/(tau-z)) G."""
    n = 1 << 16
    srs = pkg.SRS.synthetic(n, o.SYNTH_TAU)
    srs.prepare_lagrange(n)
    rnd = random.Random(22)
    ev = [rnd.randrange(o.R) for _ in range(n)]
    kzg = pkg.KZG()
    kzg.calculate_and_store_roots_of_unity(32 * n)
    poly = pkg.PolynomialEvalForm(ev)
    c = kzg.commit_eval_form(poly, srs)
    coeffs = poly.to_coeff_form(srs.engine).coeffs
    ptau = 0
    for cf in reversed(coeffs):
        ptau = (ptau * o.SYNTH_TAU + cf) % o.R
    assert c == o.g1_mul(o.G1_GEN, ptau)
    z = rnd.randrange(o.R)
    y = pkg.evaluate_polynomial_in_evaluation_form(poly, z, srs.engine)
    expect = o.g1_mul(o.G1_GEN, (ptau - y) * o.fr_inv((o.SYNTH_TAU - z) % o.R) % o.R)
    assert kzg.compute_proof(poly, z, srs) == expect
    pkg.lib.kzgb_set_option(b"lagrange", 0)
    try:
        assert kzg.commit_eval_form(poly, srs) == c
    finally:
        pkg.lib.kzgb_set_option(b"lagrange", 1)


def test_g1_ifft_kernel_sizes_and_identities(pkg, eng, ref_srs, ref_srs_points):
    """The G1 inverse-NTT kernels (kzg.rs:263-285) beyond the 64-point fixture: tiny sizes against the
    big-int oracle, the defining identity commit_eval_form(f) == MSM(g1_ifft(n), f) (prover/src/lib.rs:36-49)
    at n = 1024, an SRS containing the identity and repeated points, and the error paths."""
    kzg = pkg.KZG()
    rnd = random.Random(21)
    for n in (1, 2, 4, 16):
        assert kzg.g1_ifft(n, ref_srs) == o.g1_ifft(n, ref_srs_points[:n])
    n = 1024
    lag = kzg.g1_ifft(n, ref_srs)
    evals = [rnd.randrange(o.R) for _ in range(n)]
    assert pkg.g1_lincomb(lag, evals, eng) == kzg.commit_eval_form(pkg.PolynomialEvalForm(evals), ref_srs)
    # sum of the Lagrange basis = commitment to the constant polynomial 1 = SRS[0]
    assert pkg.g1_lincomb(lag, [1] * n, eng) == ref_srs_points[0]
    odd = [ref_srs_points[1], None, ref_srs_points[1], o.g1_neg(ref_srs_points[1]), ref_srs_points[2], None, None, ref_srs_points[2]]
    srs2 = pkg.SRS.from_points(odd, engine=pkg.Engine(0))
    assert kzg.g1_ifft(8, srs2) == o.g1_ifft(8, odd)
    with pytest.raises(pkg.KzgError) as e:
        kzg.g1_ifft(4096, ref_srs)  # only 3000 points loaded
    assert e.value.variant == "SrsCapacityExceeded"


def test_g1_ifft_closed_form_large(pkg):
    """n = 2^14 on the synthetic SRS tau^j G: L_i = l_i(tau) G with l_i(tau) = (tau^n - 1) / (n (tau w^-i - 1))."""
    n = 1 << 14
    srs = pkg.SRS.synthetic(n, o.SYNTH_TAU)
    lag = pkg.KZG().g1_ifft(n, srs)
    w = o.PRIMITIVE_ROOTS_OF_UNITY[14]
    tn = (pow(o.SYNTH_TAU, n, o.R) - 1) % o.R
    for i in (0, 1, 2, 77, n // 2, n - 1):
        den = n * ((o.SYNTH_TAU * pow(w, -i, o.R) - 1) % o.R) % o.R
        assert lag[i] == o.g1_mul(o.G1_GEN, tn * o.fr_inv(den) % o.R), i


def test_device_fiat_shamir_matches_host_and_oracle(pkg, ref_srs, ref_srs_points):
    """The per-blob challenges of verify_blob_kzg_proof_batch hashed on the GPU (fs.cu, one thread per
    transcript) against the host SHA-256 pool and the oracle: polynomial lengths 1, 2, 4, 16, 32, 64, 256, 1024
    (odd / even block structure of the transcript), ragged and non-canonical blobs, identity commitment."""
    rnd = random.Random(33)
    eng = ref_srs.engine
    raws = [b"x", b"y" * 31, b"ab" * 20, b"cd" * 40, g.gettysburg(), g.gettysburg()[:700], bytes(31 * 200), b"z",
            bytes(rnd.getrandbits(8) for _ in range(31 * 256 - 7)), bytes(rnd.getrandbits(8) for _ in range(31 * 250)),
            bytes(rnd.getrandbits(8) for _ in range(31 * 10)), bytes(rnd.getrandbits(8) for _ in range(31 * 13)),
            bytes(rnd.getrandbits(8) for _ in range(31 * 1000))]  # n = 16 (quad kernel, 7 middle blocks), 16, 1024
    blobs = [pkg.Blob.from_raw_data(r) for r in raws]
    blobs.append(pkg.Blob.from_unchecked(b"\xff" * 45 + bytes(range(50))))  # non-canonical, ragged
    blobs.sort(key=lambda b: len(b))  # equal lengths adjacent -> batched chunks
    cs, ps = pkg.KZG.commit_and_prove_blobs(blobs, ref_srs)
    cpts = [o.g1_deserialize_compressed(c) for c in cs]
    ppts = [o.g1_deserialize_compressed(p) for p in ps]
    try:
        pkg.lib.kzgb_set_option(b"fs_device", 1)
        dev = pkg.verify_blob_kzg_proof_batch_rlc(blobs, cpts, ppts, eng)
        pkg.lib.kzgb_set_option(b"fs_force_generic", 1)  # device-side choice: generic inverses for every polynomial
        dev_generic = pkg.verify_blob_kzg_proof_batch_rlc(blobs, cpts, ppts, eng)
        pkg.lib.kzgb_set_option(b"fs_force_generic", 0)
        pkg.lib.kzgb_set_option(b"fs_device", 0)
        host = pkg.verify_blob_kzg_proof_batch_rlc(blobs, cpts, ppts, eng)
    finally:
        pkg.lib.kzgb_set_option(b"fs_device", -1)
        pkg.lib.kzgb_set_option(b"fs_force_generic", 0)
    assert dev == host == dev_generic
    bo = [o.Blob.from_unchecked(b.data()) for b in blobs]
    assert dev == o.verify_blob_kzg_proof_batch_rlc(bo, cpts, ppts)
    assert pkg.lib.kzgb_set_option(b"no_such_option", 1) != 0
