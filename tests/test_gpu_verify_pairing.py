"""kzgb_verify_proofs, kzgb_verify_blob_proofs{,_dev}, kzgb_group_verify_blob_proofs and kzgb_{group_,}set_g2_tau:
verify_proof / verify_blob_kzg_proof (verifier/src/verify.rs:10-115) through the pairing on the GPU, one bool per
opening.  With [tau]G2 = [t]G2 for the synthetic t, an opening C = [c]G1, pi = [b]G1 verifies exactly when
c - y = b (t - z) mod r, so thousands of bools are checked with no oracle pairing; a few cases are checked against the
oracle's own pairing."""
import ctypes as C
import random

import pytest

import golden_data as g
from __graft_entry__ import load_package
from oracle import bn254 as o

pytestmark = pytest.mark.gpu
T = o.SYNTH_TAU
R = o.R


@pytest.fixture(scope="module")
def pkg():
    return load_package()


@pytest.fixture(scope="module")
def g2_t():
    return o.g2_mul(o.G2_GEN, T)


def _set(pkg, name, value):
    assert pkg.lib.kzgb_set_option(name.encode(), value) == 0


def _g1_many(pkg, eng, scalars):
    """[k]G1 for every k, as the GPU's variable-base MSM of one term (the oracle's g1_mul is slow for thousands)."""
    return [o.g1_mul(o.G1_GEN, k) if k < 1000 else pkg.g1_lincomb([o.G1_GEN], [k], eng) for k in scalars]


def _closed_form_openings(rnd, count):
    """(c, b, z, y, expected): half honest (c - y = b (t - z)), half off by one in a random coordinate, and the identity
    cases pi = O with C = [y]G1, C = O, y = 0 among them."""
    out = []
    for i in range(count):
        b, z, y = rnd.randrange(R), rnd.randrange(R), rnd.randrange(R)
        kind = i % 8
        if kind == 5:
            b = 0  # pi = O, C = [y]G1
        if kind == 7:
            y = 0
        if kind == 6:  # C = O: y = -b (t - z)
            y = -b * (T - z) % R
        c = (y + b * (T - z)) % R
        honest = i % 2 == 0 or kind in (5, 6, 7)
        if not honest:
            j = rnd.randrange(4)
            if j == 0:
                c = (c + 1) % R
            elif j == 1:
                b = (b + 1) % R
            elif j == 2:
                z = (z + 1) % R
            else:
                y = (y + 1) % R
        out.append((c, b, z, y, honest))
    return out


def test_closed_form_thousands(pkg, g2_t):
    rnd = random.Random(1)
    eng = pkg.Engine(0)
    ops = _closed_form_openings(rnd, 2048)
    cs = _g1_many(pkg, eng, [c for c, *_ in ops])
    ps = _g1_many(pkg, eng, [b for _, b, *_ in ops])
    assert any(c is None for c in cs) and any(p is None for p in ps)
    zs, ys = [op[2] for op in ops], [op[3] for op in ops]
    eng.set_g2_tau(g2_t)
    assert pkg.verify_proofs(cs, ps, zs, ys, eng) == [op[4] for op in ops]
    # the default (mainnet) [tau]G2: honest openings fail, except those that hold for every tau (pi = O, C = [y]G1)
    eng.set_g2_tau(None)
    got = pkg.verify_proofs(cs, ps, zs, ys, eng)
    assert got == [op[1] == 0 and op[0] == op[3] for op in ops]
    eng.close()


def test_agrees_with_oracle_bools(pkg, g2_t):
    rnd = random.Random(2)
    eng = pkg.Engine(0)
    ops = []
    for k in range(3):
        z, y, b = rnd.randrange(R), rnd.randrange(R), rnd.randrange(R)
        c = (y + b * (T - z) + (k == 2)) % R
        ops.append((o.g1_mul(o.G1_GEN, c), o.g1_mul(o.G1_GEN, b), z, y))
    for tau in (g2_t, o.G2_TAU):
        eng.set_g2_tau(tau)
        got = pkg.verify_proofs([a[0] for a in ops], [a[1] for a in ops], [a[2] for a in ops], [a[3] for a in ops], eng)
        assert got == [o.verify_proof(cc, pp, y, z, tau) for cc, pp, z, y in ops]
    # config 1: the reference's blobs.txt blob on a synthetic 2^12 SRS with [tau]G2 injected
    srs = pkg.SRS.synthetic(1 << 12, T, engine=eng)
    data = g.blobs_txt()
    other = b"".join(rnd.randrange(R).to_bytes(32, "big") for _ in range(1 << 12))
    blobs = [pkg.Blob.new(data), pkg.Blob.new(other)]
    cs = pkg.KZG.commit_blobs(blobs, srs)
    ps = pkg.KZG.compute_blob_proofs(blobs, cs, srs)
    eng.set_g2_tau(g2_t)
    got = pkg.verify_blob_kzg_proofs([blobs[0], blobs[0]], [cs[0], cs[0]], [ps[0], ps[1]], eng)
    ob = o.Blob.from_unchecked(data)
    assert got == [o.verify_blob_kzg_proof(ob, cs[0], ps[0], g2_t), o.verify_blob_kzg_proof(ob, cs[0], ps[1], g2_t)]
    assert got == [True, False]
    eng.close()


def _random_blob(rnd, n):
    """n random bytes, every 32-byte chunk below r"""
    b = bytearray(rnd.randbytes(n))
    b[0::32] = bytes(x & 0x1F for x in b[0::32])
    return bytes(b)


def _ragged_honest(pkg, srs, rnd):
    """Honest (C, proof) pairs of 300 blobs of 2^12 Fr, one of 2^16, one of 2^19 and two short ones."""
    lens = [32 << 12] * 150 + [32 << 16, 31 * 5] + [32 << 12] * 150 + [32 << 19, 100]
    datas = [_random_blob(rnd, n) for n in lens]
    blobs = [pkg.Blob.from_unchecked(d) for d in datas]
    cs32, ps32 = pkg.KZG.commit_and_prove_blobs(blobs, srs)
    return datas, [o.g1_deserialize_compressed(b) for b in cs32], [o.g1_deserialize_compressed(b) for b in ps32]


def _tamper(rnd, datas, cs, ps):
    """Scattered indices with a wrong proof, a wrong commitment or a changed blob byte."""
    datas, cs, ps = list(datas), list(cs), list(ps)
    bad = sorted(rnd.sample(range(len(datas)), 12))
    for k, i in enumerate(bad):
        if k % 3 == 0:
            ps[i] = ps[(i + 1) % len(ps)] if ps[(i + 1) % len(ps)] != ps[i] else o.g1_mul(o.G1_GEN, 3)
        elif k % 3 == 1:
            cs[i] = o.g1_add(cs[i], o.G1_GEN)
        else:
            d = bytearray(datas[i])
            d[-1] ^= 1
            datas[i] = bytes(d)
    return datas, cs, ps, bad


def _raw_ok(pkg, eng, datas, cs, ps, dev_ptrs=None):
    count = len(datas)
    keep = [C.create_string_buffer(d, max(1, len(d))) for d in datas]
    hp = (C.c_void_p * count)(*[C.cast(k, C.c_void_p).value for k in keep])
    ln = (C.c_size_t * count)(*[len(d) for d in datas])
    cxy, cinf = pkg.g1_to_abi(cs)
    pxy, pinf = pkg.g1_to_abi(ps)
    ok = C.create_string_buffer(count or 1)
    if dev_ptrs is None:
        eng.check(pkg.lib.kzgb_verify_blob_proofs(eng.h, hp, ln, count, cxy, cinf, pxy, pinf, ok))
    else:
        eng.check(pkg.lib.kzgb_verify_blob_proofs_dev(eng.h, (C.c_void_p * count)(*dev_ptrs), hp, ln, count, cxy, cinf,
                                                      pxy, pinf, ok))
    return [bool(b) for b in ok.raw[:count]]


@pytest.mark.parametrize("fs_device", [0, 1, -1])
def test_blob_forms(pkg, g2_t, fs_device):
    import torch

    rnd = random.Random(10 + fs_device)
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(1 << 19, T, engine=eng)
    eng.set_g2_tau(g2_t)
    datas, cs, ps = _ragged_honest(pkg, srs, rnd)
    _set(pkg, "fs_device", fs_device)
    try:
        assert all(_raw_ok(pkg, eng, datas, cs, ps))
        tdatas, tcs, tps, bad = _tamper(rnd, datas, cs, ps)
        want = [i not in bad for i in range(len(datas))]
        assert _raw_ok(pkg, eng, tdatas, tcs, tps) == want
        offs, pos = [], 0
        for d in tdatas:
            offs.append(pos)
            pos += len(d)
        run = torch.frombuffer(bytearray(b"".join(tdatas)), dtype=torch.uint8).cuda()
        assert _raw_ok(pkg, eng, tdatas, tcs, tps, dev_ptrs=[run.data_ptr() + k for k in offs]) == want
        bufs = [torch.frombuffer(bytearray(b"\x00" * 3 + d + b"\x00" * 5), dtype=torch.uint8).cuda() for d in tdatas]
        assert _raw_ok(pkg, eng, tdatas, tcs, tps, dev_ptrs=[b.data_ptr() + 3 for b in bufs]) == want
        if fs_device == -1:
            # ok[i] agrees with the _g1 call followed by the oracle's pairing on a small sample
            sample = [0, bad[0], bad[1], bad[2], 151]
            sb = [pkg.Blob.from_unchecked(tdatas[i]) for i in sample]
            g1 = pkg.verify_blob_kzg_proofs_g1(sb, [tcs[i] for i in sample], [tps[i] for i in sample], eng)
            for (out, z, _), i in zip(g1, sample):
                x_minus_z = o.g2_add(g2_t, o.g2_neg(o.g2_mul(o.G2_GEN, z)))
                assert o.pairings_verify(out, o.G2_GEN, tps[i], x_minus_z) == want[i]
    finally:
        _set(pkg, "fs_device", -1)
        eng.close()


def test_group_equals_single_context(pkg, g2_t):
    rnd = random.Random(20)
    eng = pkg.Engine(0)
    srs = pkg.SRS.synthetic(1 << 12, T, engine=eng)
    lens = [32 << 12] * 40 + [31 * 7, 64]
    datas = [_random_blob(rnd, n) for n in lens]
    blobs = [pkg.Blob.from_unchecked(d) for d in datas]
    cs = pkg.KZG.commit_blobs(blobs, srs)
    ps = pkg.KZG.compute_blob_proofs(blobs, cs, srs)
    tdatas, tcs, tps, bad = _tamper(rnd, datas, cs, ps)
    tblobs = [pkg.Blob.from_unchecked(d) for d in tdatas]
    eng.set_g2_tau(g2_t)
    cases = [(tblobs, tcs, tps), (tblobs[:1], tcs[:1], tps[:1]), ([], [], [])]
    want = [pkg.verify_blob_kzg_proofs(b, c, p, eng) for b, c, p in cases]
    assert want[0] == [i not in bad for i in range(len(tdatas))]
    eng.close()
    grp = pkg.Group([0, 0])
    grp.set_g2_tau(g2_t)
    for (b, c, p), w in zip(cases, want):
        assert grp.verify_blob_kzg_proofs(b, c, p) == w
    grp.set_g2_tau(None)
    assert grp.verify_blob_kzg_proofs(*cases[0]) == [False] * len(tdatas)
    grp.close()


def _ok_raw_openings(pkg, eng, cs, ps, zw, yw, ok):
    cxy, cinf = pkg.g1_to_abi(cs)
    pxy, pinf = pkg.g1_to_abi(ps)
    return pkg.lib.kzgb_verify_proofs(eng.h, len(cs), cxy, cinf, pxy, pinf, zw, yw, ok)


def _words(vals):
    return b"".join(v.to_bytes(32, "little") for v in vals)


def test_errors(pkg, g2_t):
    rnd = random.Random(30)
    eng = pkg.Engine(0)
    eng.set_g2_tau(g2_t)
    mont = lambda v: v * (1 << 256) % R
    ops = _closed_form_openings(rnd, 8)
    cs = [o.g1_mul(o.G1_GEN, c) for c, *_ in ops]
    ps = [o.g1_mul(o.G1_GEN, b) for _, b, *_ in ops]
    zs, ys = [op[2] for op in ops], [op[3] for op in ops]
    # z = t at indices 3 and 5: the error of index 3, ok untouched
    zt = list(zs)
    zt[3] = zt[5] = T
    ok = C.create_string_buffer(b"\x07" * 8, 8)
    rc = _ok_raw_openings(pkg, eng, cs, ps, _words(map(mont, zt)), _words(map(mont, ys)), ok)
    assert rc == -1 and pkg.lib.kzgb_last_error(eng.h).decode() == "Evaluation point equals trusted setup secret"
    assert ok.raw == b"\x07" * 8
    with pytest.raises(pkg.KzgError) as e:
        pkg.verify_proofs(cs, ps, zt, ys, eng)
    assert e.value.variant == "GenericError"
    # words >= r, off-curve points: the RLC openings form's codes, ok untouched
    for zw, yw in ((_words([R] + [mont(z) for z in zs[1:]]), _words(map(mont, ys))),
                   (_words(map(mont, zs)), _words([mont(y) for y in ys[:7]] + [(1 << 256) - 1]))):
        rc = _ok_raw_openings(pkg, eng, cs, ps, zw, yw, ok)
        assert rc == -9 and ok.raw == b"\x07" * 8
    rc = _ok_raw_openings(pkg, eng, cs[:2] + [(1, 3)] + cs[3:], ps, _words(map(mont, zs)), _words(map(mont, ys)), ok)
    assert rc == -5 and ok.raw == b"\x07" * 8
    with pytest.raises(pkg.KzgError) as e:
        pkg.verify_proofs(cs, ps, zs, ys[:7], eng)
    assert e.value.msg == "length's of the input are not the same"
    # blob forms: the _g1 calls' codes and messages
    blob = pkg.Blob.from_unchecked(bytes(64))
    for bad_c, msg_variant in (((1, 3), "NotOnCurveError"),):
        with pytest.raises(pkg.KzgError) as e:
            pkg.verify_blob_kzg_proofs([blob, blob], [None, bad_c], [None, None], eng)
        assert e.value.variant == msg_variant
    with pytest.raises(pkg.KzgError) as e:
        pkg.verify_blob_kzg_proofs([blob, pkg.Blob.from_unchecked(b"")], [None, None], [None, None], eng)
    assert e.value.msg == "Length of data after padding is 0"
    # a length above 2^28 elements, lengths only: rejected before any byte is read
    ok2 = C.create_string_buffer(b"\x07" * 2, 2)
    hp = (C.c_void_p * 2)(C.cast(C.create_string_buffer(64), C.c_void_p).value, 1)
    ln = (C.c_size_t * 2)(64, (32 << 28) + 1)
    cxy, cinf = pkg.g1_to_abi([None, None])
    rc = pkg.lib.kzgb_verify_blob_proofs(eng.h, hp, ln, 2, cxy, cinf, cxy, cinf, ok2)
    assert rc == -1 and pkg.lib.kzgb_last_error(eng.h).decode() == "Input size exceeds maximum polynomial size"
    assert ok2.raw == b"\x07" * 2
    # count == 0 writes nothing
    assert _ok_raw_openings(pkg, eng, [], [], b"", b"", ok) == 0 and ok.raw == b"\x07" * 8
    assert pkg.lib.kzgb_verify_blob_proofs(eng.h, None, None, 0, None, None, None, None, ok) == 0 and ok.raw == b"\x07" * 8
    assert pkg.verify_blob_kzg_proofs([], [], [], eng) == []
    eng.close()


def _fq2_sqrt(a):
    """A square root in Fq2 = Fq[u]/(u^2 + 1), or None (p = 3 mod 4)."""
    p = o.P
    a0, a1 = a
    n = (a0 * a0 + a1 * a1) % p
    s = pow(n, (p + 1) // 4, p)
    if s * s % p != n:
        return None
    for t in (s, -s % p):
        h = (a0 + t) * pow(2, -1, p) % p
        x0 = pow(h, (p + 1) // 4, p)
        if x0 * x0 % p != h or x0 == 0:
            continue
        x1 = a1 * pow(2 * x0, -1, p) % p
        if o.fq2_mul((x0, x1), (x0, x1)) == (a0 % p, a1 % p):
            return (x0, x1)
    return None


def test_set_g2_tau_rejects(pkg, g2_t):
    eng = pkg.Engine(0)
    eng.set_g2_tau(g2_t)
    # a twist point outside the r-torsion: x = k, y = sqrt(x^3 + b')
    q = None
    for k in range(1, 100):
        x = (k, 1)
        y = _fq2_sqrt(o.fq2_add(o.fq2_mul(o.fq2_mul(x, x), x), o._TWIST_B))
        if y is not None:
            q = (x, y)
            break
    assert q is not None and o.g2_is_on_curve(q) and o.g2_mul(q, R - 1) != o.g2_neg(q)
    off = (o.G2_GEN[0], (o.G2_GEN[1][0], (o.G2_GEN[1][1] + 1) % o.P))
    for bad in (off, ((0, 0), (0, 0)), q):
        with pytest.raises(pkg.KzgError) as e:
            eng.set_g2_tau(bad)
        assert e.value.variant == "NotOnCurveError" and e.value.msg == "Invalid trusted setup: G2_TAU not on curve"
    # the previous setting is still in force
    c, b, z, y = 5, 7, 11, 0
    y = (c - b * (T - z)) % R
    assert pkg.verify_proofs([o.g1_mul(o.G1_GEN, c)], [o.g1_mul(o.G1_GEN, b)], [z], [y], eng) == [True]
    grp = pkg.Group([0, 0])
    with pytest.raises(pkg.KzgError):
        grp.set_g2_tau(off)
    eng.close()
    grp.close()
