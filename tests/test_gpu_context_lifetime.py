"""kzgb_ctx_destroy frees every resource a context built, the lazily created ones included, and never destroys a stream
the caller handed to kzgb_ctx_create."""
import ctypes as C

import numpy as np
import pytest

from __graft_entry__ import load_package
from oracle import bn254 as o

pytestmark = pytest.mark.gpu
T = o.SYNTH_TAU
SRS_N = 1 << 22
BLOB_N = 1 << 18
ALL_ROOTS_N = 1 << 12


@pytest.fixture(scope="module")
def pkg():
    return load_package()


@pytest.fixture(scope="module")
def torch():
    import torch

    return torch


@pytest.fixture(scope="module")
def inputs(pkg):
    """Host MSM scalars over the whole SRS, four blobs of BLOB_N field elements, one polynomial of ALL_ROOTS_N and [T]G2."""
    rng = np.random.default_rng(5)
    scalars = rng.integers(0, 1 << 64, size=(SRS_N, 4), dtype=np.uint64)
    scalars[:, 3] &= (1 << 60) - 1  # below r: valid Montgomery words
    blobs = []
    for _ in range(4):
        data = rng.integers(0, 256, size=(BLOB_N, 32), dtype=np.uint8)
        data[:, 0] &= 0x1F  # big-endian elements below r
        blobs.append(pkg.Blob.from_unchecked(data.tobytes()))
    evals = pkg.fr_to_mont_bytes([int(v) for v in rng.integers(0, 1 << 62, size=ALL_ROOTS_N)])
    return scalars, blobs, evals, o.g2_mul(o.G2_GEN, T)


def _cycle(pkg, inputs):
    """One context that builds every lazily created resource: SRS and monomial window table, the pipelined upload's copy
    stream, a Lagrange table, the lanes and the hashing stream of a device-hashed batch, an all-roots table, the
    generator and pairing tables, the trace events and the timer.  Returns what it computed; destroys the context."""
    lib = pkg.lib
    scalars, blobs, evals, g2_t = inputs
    eng = pkg.Engine(0)
    try:
        srs = pkg.SRS.synthetic(SRS_N, T, engine=eng)
        srs.precompute(SRS_N)
        xy, inf = C.create_string_buffer(64), C.c_uint8(0)
        eng.check(lib.kzgb_msm_srs_range(eng.h, scalars.ctypes.data, 0, SRS_N, xy, C.byref(inf)))
        msm = pkg.g1_from_abi(xy.raw, bytes([inf.value]))[0]
        srs.prepare_lagrange(BLOB_N)
        eng.check(lib.kzgb_trace_begin(eng.h))
        eng.check(lib.kzgb_timer_begin(eng.h))
        cs, ps = pkg.KZG.commit_and_prove_blobs(blobs, srs)
        ms, nrec = C.c_double(0), C.c_size_t(0)
        eng.check(lib.kzgb_timer_end(eng.h, C.byref(ms)))
        eng.check(lib.kzgb_trace_end(eng.h, None, 0, C.byref(nrec)))
        assert ms.value > 0 and nrec.value > 0
        rxy, rinf = C.create_string_buffer(64 * ALL_ROOTS_N), C.create_string_buffer(ALL_ROOTS_N)
        eng.check(lib.kzgb_compute_proofs_all_roots(eng.h, evals, ALL_ROOTS_N, rxy, rinf))
        eng.set_g2_tau(g2_t)
        ok = pkg.verify_blob_kzg_proofs(
            blobs, [o.g1_deserialize_compressed(c) for c in cs], [o.g1_deserialize_compressed(p) for p in ps], eng
        )
        assert ok == [True] * len(blobs)
        return msm, cs, ps, rxy.raw, rinf.raw, ok
    finally:
        eng.close()


def test_teardown_returns_what_the_context_built(pkg, torch, inputs):
    """Three create / use / destroy cycles give the same results, and the device's free memory after each destroy stays
    within 1 GiB of the first (one cycle holds more than 3 GiB, the window table alone 3 GiB)."""
    lib = pkg.lib
    outs, free_after = [], []
    try:
        assert lib.kzgb_set_option(b"device_hash", 2) == 0  # the last two blobs hash on the device: the hashing stream
        for _ in range(3):
            outs.append(_cycle(pkg, inputs))
            free_after.append(torch.cuda.mem_get_info(0)[0])
    finally:
        lib.kzgb_set_option(b"device_hash", -1)
    for out in outs[1:]:
        assert out == outs[0]
    for free in free_after[1:]:
        assert abs(free - free_after[0]) <= 1 << 30, free_after


def test_caller_stream_survives_the_context(pkg, torch):
    s = torch.cuda.Stream(device=0)
    eng = pkg.Engine(0, stream=s.cuda_stream)
    try:
        srs = pkg.SRS.synthetic(1 << 12, T, engine=eng)
        blob = pkg.Blob.from_raw_data(b"context on a caller's stream")
        assert pkg.KZG().commit_blob(blob, srs) is not None
    finally:
        eng.close()
    with torch.cuda.stream(s):
        x = torch.arange(1 << 20, device="cuda", dtype=torch.float64) * 2
        total = x.sum()
    s.synchronize()
    assert total.item() == float((1 << 20) * ((1 << 20) - 1))
