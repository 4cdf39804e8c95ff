"""CPU checks of csrc/pairing.cuh, compiled for the host: the tower, the line tables and the final exponentiation that
the pairing kernels run give the oracle's pairing raised to the fixed m of the final exponentiation (DESIGN.md section 4),
the reduced pairing is bilinear, and the library's default [tau]G2 is the reference's G2_TAU."""
import ctypes as C
import os
import random
import subprocess

import pytest

from oracle import bn254 as o

HERE = os.path.dirname(os.path.abspath(__file__))
MONT = 1 << 256
X = 4965661367192848881
M_EXP = 2 * X * (6 * X * X + 3 * X + 1)  # the final exponentiation computes f^(M_EXP (p^12 - 1) / r)


@pytest.fixture(scope="module")
def ph(tmp_path_factory):
    src = os.path.join(HERE, "native", "pairing_host_test.cpp")
    out = str(tmp_path_factory.mktemp("pairing") / "libpairing_host_test.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", out, src])
    return C.CDLL(out)


def _w(v):
    return (v % o.P * MONT % o.P).to_bytes(32, "little")


def _g2(q):
    return _w(q[0][0]) + _w(q[0][1]) + _w(q[1][0]) + _w(q[1][1])


def _g1(p):
    return bytes(64) if p is None else _w(p[0]) + _w(p[1])


def _f12(raw):
    """Fq12 words of the tower (c0 + c1 w over Fq6 = Fq2[v], v = w^2, Fq2 = Fq[u], u = w^6 - 9) -> the oracle's
    coefficients of w^0 .. w^11."""
    rinv = pow(MONT, -1, o.P)
    c = [int.from_bytes(raw[32 * i : 32 * i + 32], "little") * rinv % o.P for i in range(12)]
    out = [0] * 12
    for half in range(2):
        for j in range(3):
            x, y = c[6 * half + 2 * j], c[6 * half + 2 * j + 1]
            k = 2 * j + half
            out[k] = (out[k] + x - 9 * y) % o.P
            out[k + 6] = (out[k + 6] + y) % o.P
    return out


def _pair(ph, q, p):
    out = C.create_string_buffer(384)
    ph.t_pairing(out, _g2(q), _g1(p))
    return _f12(out.raw)


def test_pairing_equals_oracle_to_the_m(ph):
    rnd = random.Random(5)
    a, b = rnd.randrange(1, o.R), rnd.randrange(1, o.R)
    cases = [(o.G2_GEN, o.G1_GEN), (o.G2_TAU, o.G1_GEN), (o.g2_mul(o.G2_GEN, b), o.g1_mul(o.G1_GEN, a))]
    for q, p in cases:
        assert _pair(ph, q, p) == o._f12_pow(o.pairing(q, p), M_EXP)
    assert _pair(ph, o.G2_TAU, None) == o._F12_ONE  # the identity in G1


def test_bilinear(ph):
    rnd = random.Random(6)
    a, b = rnd.randrange(1, o.R), rnd.randrange(1, o.R)
    e = _pair(ph, o.G2_GEN, o.G1_GEN)
    assert e != o._F12_ONE
    assert _pair(ph, o.g2_mul(o.G2_GEN, b), o.g1_mul(o.G1_GEN, a)) == o._f12_pow(e, a * b % o.R)
    assert o._f12_pow(e, o.R) == o._F12_ONE


def test_cyclotomic_squaring(ph):
    rnd = random.Random(7)
    for _ in range(3):
        a = b"".join(_w(rnd.randrange(o.P)) for _ in range(12))
        cyc, gen = C.create_string_buffer(384), C.create_string_buffer(384)
        ph.t_cyclotomic_sqr(cyc, gen, a)
        assert cyc.raw == gen.raw


def test_default_g2_tau_is_the_reference_constant(ph):
    out = C.create_string_buffer(128)
    ph.t_default_g2_tau(out)
    assert out.raw == _g2(o.G2_TAU)
