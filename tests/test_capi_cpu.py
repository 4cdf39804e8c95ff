"""No-GPU checks of the C-ABI library: it loads, exports every symbol include/kzg_bn254_b200.h
(and the measurement header kzg_bn254_b200_bench.h) declares, the host-only entry points agree with the oracle, and a context cannot be created
without a GPU (no silent CPU fallback)."""
import ctypes as C
import os
import re

import pytest

import golden_data as g
from __graft_entry__ import ROOT, load_package
from oracle import bn254 as o


@pytest.fixture(scope="module")
def pkg():
    return load_package()


def test_header_symbols_exported(pkg):
    hdr = open(os.path.join(ROOT, "include", "kzg_bn254_b200.h")).read()
    hdr += open(os.path.join(ROOT, "include", "kzg_bn254_b200_bench.h")).read()  # measurement hooks, same library
    declared = set(re.findall(r"\b(kzgb_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 35
    lib = pkg._capi.lib
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert declared == set(pkg._capi.SIGNATURES), declared ^ set(pkg._capi.SIGNATURES)


def test_point_codecs_match_oracle(pkg):
    pts = g.srs_points_string()[:40] + [None]
    raw = g.g1_point_bytes()
    for i, p in enumerate(pts):
        assert pkg.g1_serialize_compressed(p) == o.g1_serialize_compressed(p)
        assert pkg.g1_to_gnark_be(p) == o.g1_to_gnark_be(p)
        if p is not None:
            assert pkg.g1_to_gnark_be(p) == raw[32 * i : 32 * i + 32]
            assert o.g1_deserialize_compressed(pkg.g1_serialize_compressed(p)) == p


def test_host_g1_add(pkg):
    pts = g.srs_points_string()
    assert pkg.g1_add(pts[1], pts[2]) == o.g1_add(pts[1], pts[2])
    assert pkg.g1_add(pts[3], pts[3]) == o.g1_add(pts[3], pts[3])
    assert pkg.g1_add(pts[3], o.g1_neg(pts[3])) is None
    assert pkg.g1_add(None, pts[4]) == pts[4]


def test_fiat_shamir_challenge_matches_oracle(pkg):
    """helpers.rs:411-472 runs on the host inside the library (SHA-256, mod-r reduction)."""
    c = g.srs_points_string()[5]
    for raw in (g.gettysburg(), b"x", bytes(100), g.gettysburg()[:31 * 7]):
        blob_o = o.Blob.from_raw_data(raw)
        assert pkg.compute_challenge(pkg.Blob.from_raw_data(raw), c) == o.compute_challenge(blob_o, c)
    # non-canonical / ragged blob (From<Vec<u8>>): chunks >= r are reduced, the tail is right-padded
    ragged = b"\xff" * 45 + bytes(range(50))
    assert pkg.compute_challenge(pkg.Blob.from_unchecked(ragged), c) == o.compute_challenge(o.Blob.from_unchecked(ragged), c)
    full = g.blobs_txt()[: 32 * 100]
    assert pkg.compute_challenge(pkg.Blob.new(full), None) == o.compute_challenge(o.Blob(full), None)
    with pytest.raises(pkg.KzgError) as e:
        pkg.compute_challenge(pkg.Blob.from_raw_data(b"abc"), (1, 3))
    assert e.value.variant == "NotOnCurveError"


def test_verify_proof_g1_side_matches_oracle(pkg):
    """verifier/src/verify.rs:18-42 on the host side of the library (no GPU needed): C - [y] G1, and the validation errors."""
    import ctypes as C

    pts = g.srs_points_string()
    for y in (0, 1, 5, o.R - 1, 0x1234567890ABCDEF1234567890ABCDEF1234567890ABCDEF):
        cxy, cinf = pkg.g1_to_abi([pts[7]])
        pxy, pinf = pkg.g1_to_abi([pts[9]])
        out, inf = C.create_string_buffer(64), C.c_uint8(0)
        assert pkg.lib.kzgb_verify_proof_g1(None, cxy, cinf[0], pxy, pinf[0], pkg.fr_to_mont_bytes([y]), out, C.byref(inf)) == 0
        want = o.g1_add(pts[7], o.g1_neg(o.g1_mul(o.G1_GEN, y)))
        assert pkg.g1_from_abi(out.raw, bytes([inf.value]))[0] == want
    # C = [y] G -> the identity; a point off the curve -> NotOnCurveError
    cxy, cinf = pkg.g1_to_abi([o.g1_mul(o.G1_GEN, 77)])
    out, inf = C.create_string_buffer(64), C.c_uint8(0)
    assert pkg.lib.kzgb_verify_proof_g1(None, cxy, cinf[0], pxy, pinf[0], pkg.fr_to_mont_bytes([77]), out, C.byref(inf)) == 0 and inf.value == 1
    bad, binf = pkg.g1_to_abi([(1, 3)])
    assert pkg.lib.kzgb_verify_proof_g1(None, bad, binf[0], pxy, pinf[0], pkg.fr_to_mont_bytes([1]), out, C.byref(inf)) == -5
    assert pkg.lib.kzgb_verify_proof_g1(None, cxy, cinf[0], bad, binf[0], pkg.fr_to_mont_bytes([1]), out, C.byref(inf)) == -5


def test_host_side_containers(pkg):
    assert pkg.pad_payload(b"hi") == o.pad_payload(b"hi")
    b = pkg.Blob.from_raw_data(g.gettysburg())
    assert b.data() == o.pad_payload(g.gettysburg()) and len(b) == 1536
    assert b.to_raw_data()[: len(g.gettysburg())] == g.gettysburg()
    with pytest.raises(pkg.KzgError):
        pkg.Blob.new(bytes(62))
    with pytest.raises(pkg.KzgError):
        pkg.Blob.new(b"\xff" * 32)
    assert pkg.calculate_roots_of_unity(1536) == o.calculate_roots_of_unity(1536)
    with pytest.raises(pkg.KzgError):
        pkg.calculate_roots_of_unity(0)
    assert [pkg.get_primitive_root_of_unity(k) for k in range(29)] == o.PRIMITIVE_ROOTS_OF_UNITY


def test_no_cpu_fallback_without_gpu(pkg):
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(pkg.KzgError):
        pkg.Engine(0)


def test_bench_clock_sampler_addresses_visible_devices(monkeypatch):
    """bench.py samples clocks through NVML / nvidia-smi, which enumerate every GPU of the box whatever CUDA_VISIBLE_DEVICES
    says: CUDA ordinal i of the job must map to the i-th entry of the mask (index or UUID), and to i itself without a mask."""
    import bench

    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "3, 5,GPU-1234")
    s = bench.ClockSampler(range(3))
    assert s.targets == ["3", "5", "GPU-1234"]
    assert bench.ClockSampler(1).targets == ["5"]
    monkeypatch.delenv("CUDA_VISIBLE_DEVICES")
    assert bench.ClockSampler(range(2)).targets == ["0", "1"]
    empty = bench.ClockSampler([]).summary()
    assert empty["samples"] == 0 and empty["reasons"] == [] and empty["sm_mhz"] is None


def test_bench_payload_blob_distribution():
    """D1 'payload' blobs: byte 0 of every 32-byte element is 0 (what Blob::from_raw_data yields), seeded."""
    import bench

    a, b = bench.make_blob(64, 7), bench.make_blob(64, 7)
    assert a.shape == (64 * 32,) and (a == b).all() and (a.reshape(64, 32)[:, 0] == 0).all()
    assert (bench.make_blob(64, 8) != a).any()


def test_bench_dump_outputs_round_trip(tmp_path):
    """--dump-outputs: every 32-byte point becomes one float32 row of its bytes, read back exactly."""
    import numpy as np

    import bench

    raw = bytes(range(256)) * 3
    bench.dump_outputs(str(tmp_path / "out"), {"commitments": raw, "proofs": raw[:32]})
    got = np.load(tmp_path / "out" / "commitments.npy")
    assert got.dtype == np.float32 and got.shape == (24, 32)
    assert got.astype(np.uint8).tobytes() == raw
    assert np.load(tmp_path / "out" / "proofs.npy").shape == (1, 32)


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--dump-outputs", "d", "--config", "c3"], ["--dump-outputs", "d", "--impl", "reference"]])
def test_bench_rejects_arguments_it_cannot_honour(argv, tmp_path):
    import subprocess
    import sys

    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 2 and "error" in r.stderr
    assert not (tmp_path / "d").exists()
