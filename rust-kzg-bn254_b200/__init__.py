"""Host-side mirror of the rust-kzg-bn254 API over the B200 engine (libkzgbn254_b200.so).

Same names, argument meaning and error behaviour as the reference's Rust API
(``prover::kzg::KZG``, ``prover::srs::SRS``, ``primitives::blob::Blob``,
``primitives::polynomial::Polynomial{Eval,Coeff}Form``, ``primitives::helpers``,
``verifier::batch``), so the parity tests read like the reference's own tests.  The Rust
toolchain is not available in this image, so this Python layer plays the role of the Rust
shim described in INTEGRATION.md: it only marshals, performs the reference's cheap
pre-condition checks, and calls the C ABI.  All arithmetic runs in the CUDA library; there is
no CPU fallback.

Field elements are Python ints (canonical); G1 points are ``(x, y)`` int tuples, ``None`` is
the identity.  Across the ABI they travel as arkworks-layout Montgomery limbs.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

from . import _capi
from ._capi import lib

P = 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47
R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
_MONT = 1 << 256
_RINV_R = pow(_MONT, -1, R)
_RINV_P = pow(_MONT, -1, P)
BYTES_PER_FIELD_ELEMENT = 32  # primitives/src/consts.rs:4
MAINNET_SRS_G1_SIZE = 268435456  # consts.rs:66

Affine = Optional[Tuple[int, int]]


class KzgError(Exception):
    """primitives/src/errors.rs:32-86: ``variant`` is the enum variant name, ``msg`` its payload."""

    def __init__(self, variant: str, msg: str = ""):
        super().__init__(f"{variant}: {msg}" if msg else variant)
        self.variant = variant
        self.msg = msg


# ---------------------------------------------------------------- marshalling
def fr_to_mont_bytes(vals: Sequence[int]) -> bytes:
    return b"".join(((v % R) * _MONT % R).to_bytes(32, "little") for v in vals)


def fr_from_mont_bytes(buf: bytes) -> List[int]:
    return [int.from_bytes(buf[i : i + 32], "little") * _RINV_R % R for i in range(0, len(buf), 32)]


def g1_to_abi(pts: Sequence[Affine]) -> Tuple[bytes, bytes]:
    xy = bytearray()
    inf = bytearray()
    for p in pts:
        if p is None:
            xy += bytes(64)
            inf.append(1)
        else:
            xy += (p[0] % P * _MONT % P).to_bytes(32, "little") + (p[1] % P * _MONT % P).to_bytes(32, "little")
            inf.append(0)
    return bytes(xy), bytes(inf)


def g1_from_abi(xy: bytes, inf: Optional[bytes] = None) -> List[Affine]:
    out: List[Affine] = []
    for i in range(len(xy) // 64):
        if (inf is not None and inf[i]) or not any(xy[64 * i : 64 * i + 64]):
            out.append(None)
        else:
            x = int.from_bytes(xy[64 * i : 64 * i + 32], "little") * _RINV_P % P
            y = int.from_bytes(xy[64 * i + 32 : 64 * i + 64], "little") * _RINV_P % P
            out.append((x, y))
    return out


def _blobs_to_abi(blobs: Sequence["Blob"]):
    """The (blob pointers, lengths) arguments of the blob-batch calls, and the buffers the pointers point into: the
    caller keeps those alive for the length of the call."""
    keep = [C.create_string_buffer(b.blob_data, max(1, len(b.blob_data))) for b in blobs]
    ptrs = (C.c_void_p * len(blobs))(*[C.cast(k, C.c_void_p).value for k in keep])
    lens = (C.c_size_t * len(blobs))(*[len(b.blob_data) for b in blobs])
    return keep, ptrs, lens


def _next_pow2(n: int) -> int:
    return 1 if n <= 1 else 1 << (n - 1).bit_length()


# ---------------------------------------------------------------- engine context
class Engine:
    """One GPU context (``kzgb_ctx``): HBM-resident SRS, twiddles, streams and workspaces."""

    def __init__(self, device: int = 0, stream: Optional[int] = None):
        h = C.c_void_p()
        rc = lib.kzgb_ctx_create(C.byref(h), device, stream)
        if rc != 0:
            raise KzgError("GenericError", f"kzgb_ctx_create failed ({rc}): no usable CUDA device {device}")
        self.h = h
        self.device = device
        self._owned = True

    def close(self):
        if getattr(self, "h", None):
            if getattr(self, "_owned", True):
                lib.kzgb_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc: int):
        if rc != 0:
            msg = lib.kzgb_last_error(self.h)
            raise KzgError(_capi.STATUS_VARIANT.get(rc, "GenericError"), msg.decode() if msg else "")

    # -- raw helpers returning affine points -------------------------------------------
    def _point_call(self, fn, *args) -> Affine:
        out = C.create_string_buffer(64)
        inf = C.c_uint8(0)
        self.check(fn(self.h, *args, out, C.byref(inf)))
        return g1_from_abi(out.raw, bytes([inf.value]))[0]

    def launch_count(self) -> int:
        return int(lib.kzgb_launch_count(self.h))


class Group:
    """Several GPUs of one box behind one handle (``kzgb_group``): batches of blobs are cut by blob, one large
    MSM by point range; the SRS is decompressed once and replicated device to device.  ``devices=None`` takes
    every visible GPU; a device may be listed twice (independent contexts on one GPU)."""

    def __init__(self, devices: Optional[Sequence[int]] = None):
        h = C.c_void_p()
        if devices is None:
            rc = lib.kzgb_group_create(C.byref(h), None, 0)
        else:
            arr = (C.c_int * len(devices))(*devices)
            rc = lib.kzgb_group_create(C.byref(h), arr, len(devices))
        if rc != 0:
            raise KzgError("GenericError", f"kzgb_group_create failed ({rc})")
        self.h = h

    def close(self):
        if getattr(self, "h", None):
            lib.kzgb_group_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self):
        return int(lib.kzgb_group_size(self.h))

    def check(self, rc: int):
        if rc != 0:
            msg = lib.kzgb_group_last_error(self.h)
            raise KzgError(_capi.STATUS_VARIANT.get(rc, "GenericError"), msg.decode() if msg else "")

    def member(self, i: int) -> "Engine":
        """Borrowed view of member i's context (owned by the group)."""
        e = Engine.__new__(Engine)
        e.h = C.c_void_p(lib.kzgb_group_ctx(self.h, i))
        e._owned = False
        e.device = -1
        return e

    # -- SRS ----------------------------------------------------------------------------
    def load_srs_file(self, path: str, order: int, points_to_load: int) -> None:
        self.check(lib.kzgb_group_srs_load_file(self.h, path.encode(), order, points_to_load))

    def load_srs_gnark_bytes(self, data: bytes) -> None:
        self.check(lib.kzgb_group_srs_load_gnark_be(self.h, data, len(data) // 32))

    def load_srs_points(self, pts: Sequence[Affine]) -> None:
        xy, inf = g1_to_abi(pts)
        self.check(lib.kzgb_group_srs_load_affine_mont(self.h, xy, inf, len(pts)))

    def load_srs_synthetic(self, n: int, tau: int) -> None:
        self.check(lib.kzgb_group_srs_load_synthetic(self.h, fr_to_mont_bytes([tau]), n))

    def prepare_lagrange(self, n: int) -> None:
        self.check(lib.kzgb_group_srs_prepare_lagrange(self.h, n))

    def precompute_ranges(self, n: int, window_bits: int = 0) -> None:
        self.check(lib.kzgb_group_srs_precompute_ranges(self.h, n, window_bits))

    # -- the sharded calls --------------------------------------------------------------
    def commit_and_prove_blobs(self, blobs: Sequence["Blob"]) -> Tuple[List[bytes], List[bytes]]:
        count = len(blobs)
        keep, ptrs, lens = _blobs_to_abi(blobs)  # keep: the buffers ptrs points into
        cs = C.create_string_buffer(32 * count if count else 1)
        ps = C.create_string_buffer(32 * count if count else 1)
        self.check(lib.kzgb_group_commit_and_prove_blobs(self.h, ptrs, lens, count, cs, ps))
        return ([cs.raw[32 * i : 32 * i + 32] for i in range(count)], [ps.raw[32 * i : 32 * i + 32] for i in range(count)])

    def commit_coeff_form(self, polynomial: "PolynomialCoeffForm") -> Affine:
        """KZG::commit_coeff_form with the points cut into one range per GPU (prover/src/kzg.rs:107-125)."""
        out = C.create_string_buffer(64)
        inf = C.c_uint8(0)
        self.check(lib.kzgb_group_msm_srs(self.h, fr_to_mont_bytes(polynomial.coeffs), len(polynomial), out, C.byref(inf)))
        return g1_from_abi(out.raw, bytes([inf.value]))[0]


_default_engine: Optional[Engine] = None


def default_engine() -> Engine:
    global _default_engine
    if _default_engine is None:
        _default_engine = Engine(0)
    return _default_engine


# ---------------------------------------------------------------- primitives::helpers (host-cheap parts)
def pad_payload(data: bytes) -> bytes:
    """primitives/src/helpers.rs:823-840."""
    out = bytearray()
    for i in range(0, len(data), 31):
        ch = data[i : i + 31]
        out += b"\x00" + ch + bytes(31 - len(ch))
    return bytes(out)


def remove_internal_padding(padded: bytes) -> bytes:
    """primitives/src/helpers.rs:856-874."""
    if len(padded) % 32 != 0:
        raise KzgError("InvalidInputLength")
    return b"".join(padded[i + 1 : i + 32] for i in range(0, len(padded), 32))


def validate_blob_data_as_canonical_field_elements(data: bytes) -> None:
    """primitives/src/helpers.rs:784-811."""
    if len(data) % 32 != 0:
        raise KzgError("InvalidInputLength")
    for i in range(0, len(data), 32):
        if int.from_bytes(data[i : i + 32], "big") >= R:
            raise KzgError("InvalidFieldElement", f"Field element at position {i // 32} is not canonical or invalid")


def to_fr_array(data: bytes, engine: Optional[Engine] = None) -> List[int]:
    """primitives/src/helpers.rs:40-57 on the GPU (k_bytes_to_fr)."""
    e = engine or default_engine()
    n = (len(data) + 31) // 32
    out = C.create_string_buffer(32 * n if n else 1)
    e.check(lib.kzgb_to_fr_array(e.h, data, len(data), out))
    return fr_from_mont_bytes(out.raw[: 32 * n])


def to_byte_array(frs: Sequence[int], max_output_size: int, engine: Optional[Engine] = None) -> bytes:
    """primitives/src/helpers.rs:80-119 (conversion on the GPU, truncation on the host)."""
    e = engine or default_engine()
    n = len(frs)
    out = C.create_string_buffer(32 * n if n else 1)
    e.check(lib.kzgb_to_byte_array(e.h, fr_to_mont_bytes(frs), n, out))
    return out.raw[: min(32 * n, max_output_size)]


def g1_serialize_compressed(pt: Affine) -> bytes:
    """arkworks ``serialize_compressed`` (call sites helpers.rs:458-460, batch.rs:128,149-151)."""
    xy, inf = g1_to_abi([pt])
    out = C.create_string_buffer(32)
    lib.kzgb_g1_serialize_compressed(xy, inf[0], out)
    return out.raw


def g1_to_gnark_be(pt: Affine) -> bytes:
    xy, inf = g1_to_abi([pt])
    out = C.create_string_buffer(32)
    lib.kzgb_g1_to_gnark_be(xy, inf[0], out)
    return out.raw


def g1_add(a: Affine, b: Affine) -> Affine:
    axy, ainf = g1_to_abi([a])
    bxy, binf = g1_to_abi([b])
    out = C.create_string_buffer(64)
    oinf = C.c_uint8(0)
    lib.kzgb_g1_add(axy, ainf[0], bxy, binf[0], out, C.byref(oinf))
    return g1_from_abi(out.raw, bytes([oinf.value]))[0]


def validate_g1_point(pt: Affine, engine: Optional[Engine] = None) -> None:
    """primitives/src/helpers.rs:694-708."""
    e = engine or default_engine()
    xy, inf = g1_to_abi([pt])
    e.check(lib.kzgb_validate_g1_points(e.h, xy, inf, 1))


def g1_lincomb(points: Sequence[Affine], scalars: Sequence[int], engine: Optional[Engine] = None) -> Affine:
    """primitives/src/helpers.rs:328-337 (variable-base MSM on the GPU)."""
    if len(points) != len(scalars):
        raise KzgError("MsmError", str(min(len(points), len(scalars))))
    e = engine or default_engine()
    xy, inf = g1_to_abi(points)
    return e._point_call(lambda h, *a: lib.kzgb_msm_var(h, xy, inf, fr_to_mont_bytes(scalars), len(points), *a))


def calculate_roots_of_unity(length_of_data_after_padding: int, engine: Optional["Engine"] = None) -> List[int]:
    """primitives/src/helpers.rs:553-610.  With an engine: kzgb_roots_of_unity (one kernel on the GPU); without: the
    host loop below (the no-GPU tests use it)."""
    if engine is not None:
        n = C.c_size_t(0)
        engine.check(lib.kzgb_roots_of_unity(engine.h, length_of_data_after_padding, None, 0, C.byref(n)))
        out = C.create_string_buffer(32 * n.value)
        engine.check(lib.kzgb_roots_of_unity(engine.h, length_of_data_after_padding, out, n.value, C.byref(n)))
        return fr_from_mont_bytes(out.raw)
    if length_of_data_after_padding == 0:
        raise KzgError("GenericError", "Length of data after padding is 0")
    nelem = -(-length_of_data_after_padding // 32)
    if nelem > MAINNET_SRS_G1_SIZE:
        raise KzgError("GenericError", "the length of data after padding is not valid with respect to the SRS")
    n = _next_pow2(nelem)
    w = get_primitive_root_of_unity(n.bit_length() - 1)
    roots = [1] * n
    for i in range(1, n):
        roots[i] = roots[i - 1] * w % R
    return roots


_TWO_ADIC_ROOT = 19103219067921713944291392827692070036145651957329286315305642004821462161904


def get_primitive_root_of_unity(power: int) -> int:
    """primitives/src/helpers.rs:365-370 / consts.rs:22-52."""
    if power > 28 or power < 0:
        raise KzgError("GenericError", "power must be <= 28")
    return pow(_TWO_ADIC_ROOT, 1 << (28 - power), R)


# ---------------------------------------------------------------- containers
class PolynomialEvalForm:
    """primitives/src/polynomial.rs:13-140."""

    def __init__(self, evals: Sequence[int], len_underlying_blob_bytes: Optional[int] = None):
        if len(evals) > MAINNET_SRS_G1_SIZE:
            raise KzgError("GenericError", "Input size exceeds maximum polynomial size")
        self.len_underlying_blob_bytes = len(evals) * 32 if len_underlying_blob_bytes is None else len_underlying_blob_bytes
        n = _next_pow2(len(evals))
        self.evaluations = [e % R for e in evals] + [0] * (n - len(evals))

    def __len__(self):
        return len(self.evaluations)

    def len_underlying_blob_field_elements(self) -> int:
        return self.len_underlying_blob_bytes // 32

    def get_evalualtion(self, i: int) -> Optional[int]:
        return self.evaluations[i] if 0 <= i < len(self.evaluations) else None

    def to_bytes_be(self) -> bytes:
        return to_byte_array(self.evaluations, self.len_underlying_blob_bytes)

    def to_coeff_form(self, engine: Optional[Engine] = None) -> "PolynomialCoeffForm":
        """polynomial.rs:130-140 -- Fr IFFT on the GPU."""
        return PolynomialCoeffForm(_ntt(self.evaluations, True, engine), self.len_underlying_blob_bytes)


class PolynomialCoeffForm:
    """primitives/src/polynomial.rs:143-251."""

    def __init__(self, coeffs: Sequence[int], len_underlying_blob_bytes: Optional[int] = None):
        if len(coeffs) > MAINNET_SRS_G1_SIZE:
            raise KzgError("GenericError", "Input size exceeds maximum polynomial size")
        self.len_underlying_blob_bytes = len(coeffs) * 32 if len_underlying_blob_bytes is None else len_underlying_blob_bytes
        n = _next_pow2(len(coeffs))
        self.coeffs = [c % R for c in coeffs] + [0] * (n - len(coeffs))

    def __len__(self):
        return len(self.coeffs)

    def to_bytes_be(self) -> bytes:
        return to_byte_array(self.coeffs, self.len_underlying_blob_bytes)

    def to_eval_form(self, engine: Optional[Engine] = None) -> PolynomialEvalForm:
        """polynomial.rs:241-251 -- Fr FFT on the GPU."""
        return PolynomialEvalForm(_ntt(self.coeffs, False, engine), self.len_underlying_blob_bytes)


def _ntt(vals: Sequence[int], inverse: bool, engine: Optional[Engine]) -> List[int]:
    e = engine or default_engine()
    buf = C.create_string_buffer(fr_to_mont_bytes(vals), 32 * len(vals))
    e.check(lib.kzgb_ntt_fr(e.h, buf, len(vals), 1 if inverse else 0))
    return fr_from_mont_bytes(buf.raw)


class Blob:
    """primitives/src/blob.rs:15-97."""

    def __init__(self, blob_data: bytes, _validate: bool = True):
        if _validate:
            validate_blob_data_as_canonical_field_elements(blob_data)
        self.blob_data = bytes(blob_data)

    @classmethod
    def new(cls, blob_data: bytes) -> "Blob":
        return cls(blob_data)

    @classmethod
    def from_raw_data(cls, raw: bytes) -> "Blob":
        return cls(pad_payload(raw), _validate=False)

    @classmethod
    def from_unchecked(cls, data: bytes) -> "Blob":
        """``impl From<Vec<u8>> for Blob`` (blob.rs:90-97)."""
        return cls(data, _validate=False)

    def to_raw_data(self) -> bytes:
        return remove_internal_padding(self.blob_data)

    def data(self) -> bytes:
        return self.blob_data

    def __len__(self):
        return len(self.blob_data)

    def is_empty(self) -> bool:
        return len(self.blob_data) == 0

    def __eq__(self, other):
        return isinstance(other, Blob) and self.blob_data == other.blob_data

    def to_polynomial_eval_form(self, engine: Optional[Engine] = None) -> PolynomialEvalForm:
        return PolynomialEvalForm(to_fr_array(self.blob_data, engine))

    def to_polynomial_coeff_form(self, engine: Optional[Engine] = None) -> PolynomialCoeffForm:
        return PolynomialCoeffForm(to_fr_array(self.blob_data, engine))


class SRS:
    """prover/src/srs.rs:11-49.  The points live in HBM inside an :class:`Engine`;
    ``g1`` reads them back (the reference's ``pub g1`` field)."""

    def __init__(self, path_to_g1_points: str, order: int, points_to_load: int, engine: Optional[Engine] = None):
        self.engine = engine or Engine(0)
        self.order = order
        self.engine.check(lib.kzgb_srs_load_file(self.engine.h, path_to_g1_points.encode(), order, points_to_load))

    @classmethod
    def _blank(cls, engine: Optional[Engine], order: int) -> "SRS":
        s = cls.__new__(cls)
        s.engine = engine or Engine(0)
        s.order = order
        return s

    @classmethod
    def from_gnark_bytes(cls, data: bytes, engine: Optional[Engine] = None) -> "SRS":
        s = cls._blank(engine, len(data) // 32)
        s.engine.check(lib.kzgb_srs_load_gnark_be(s.engine.h, data, len(data) // 32))
        return s

    @classmethod
    def from_cache(cls, path: str, points_to_load: int = 0, engine: Optional[Engine] = None) -> "SRS":
        """Decompressed-point cache written by :meth:`save_cache` (no square roots; on-curve check on the GPU)."""
        s = cls._blank(engine, points_to_load)
        s.engine.check(lib.kzgb_srs_load_cache(s.engine.h, path.encode(), points_to_load))
        s.order = len(s)
        return s

    def save_cache(self, path: str) -> None:
        self.engine.check(lib.kzgb_srs_save_cache(self.engine.h, path.encode()))

    @classmethod
    def from_points(cls, pts: Sequence[Affine], engine: Optional[Engine] = None) -> "SRS":
        s = cls._blank(engine, len(pts))
        xy, inf = g1_to_abi(pts)
        s.engine.check(lib.kzgb_srs_load_affine_mont(s.engine.h, xy, inf, len(pts)))
        return s

    @classmethod
    def synthetic(cls, n: int, tau: int, engine: Optional[Engine] = None, first: int = 0) -> "SRS":
        """SRS_i = tau^(first+i) * G generated on the GPU (SURVEY.md 8d synthetic inputs); `first` selects a
        point range of the same SRS for point-range sharding."""
        s = cls._blank(engine, n)
        s.engine.check(lib.kzgb_srs_load_synthetic_range(s.engine.h, fr_to_mont_bytes([tau]), first, n))
        return s

    def __len__(self):
        return int(lib.kzgb_srs_len(self.engine.h))

    def points(self, start: int = 0, count: Optional[int] = None) -> List[Affine]:
        count = len(self) - start if count is None else count
        xy = C.create_string_buffer(64 * count if count else 1)
        inf = C.create_string_buffer(count if count else 1)
        self.engine.check(lib.kzgb_srs_get_affine_mont(self.engine.h, start, count, xy, inf))
        return g1_from_abi(xy.raw[: 64 * count], inf.raw[:count])

    @property
    def g1(self) -> List[Affine]:
        return self.points()

    def precompute(self, max_n: int = 0, window_bits: int = 0) -> None:
        self.engine.check(lib.kzgb_srs_precompute(self.engine.h, max_n, window_bits))

    def prepare_lagrange(self, n: int) -> None:
        """Resident Lagrange-basis window table for evaluation-form polynomials of n elements: the cached
        equivalent of the g1_ifft that KZG::commit_eval_form runs on every call (prover/src/kzg.rs:98)."""
        self.engine.check(lib.kzgb_srs_prepare_lagrange(self.engine.h, n))


class KZG:
    """prover/src/kzg.rs:25-309."""

    def __init__(self):
        self.expanded_roots_of_unity: List[int] = []

    @classmethod
    def new(cls) -> "KZG":
        return cls()

    def calculate_and_store_roots_of_unity(self, length_of_data_after_padding: int) -> None:
        self.expanded_roots_of_unity = calculate_roots_of_unity(length_of_data_after_padding)

    def get_roots_of_unities(self) -> List[int]:
        return list(self.expanded_roots_of_unity)

    def get_nth_root_of_unity(self, i: int) -> Optional[int]:
        return self.expanded_roots_of_unity[i] if 0 <= i < len(self.expanded_roots_of_unity) else None

    def commit_eval_form(self, polynomial: PolynomialEvalForm, srs: SRS) -> Affine:
        """kzg.rs:84-104."""
        e = srs.engine
        m = fr_to_mont_bytes(polynomial.evaluations)
        return e._point_call(lambda h, *a: lib.kzgb_commit_eval(h, m, len(polynomial), *a))

    def commit_coeff_form(self, polynomial: PolynomialCoeffForm, srs: SRS) -> Affine:
        """kzg.rs:107-125."""
        e = srs.engine
        m = fr_to_mont_bytes(polynomial.coeffs)
        return e._point_call(lambda h, *a: lib.kzgb_commit_coeff(h, m, len(polynomial), *a))

    def commit_blob(self, blob: Blob, srs: SRS) -> Affine:
        """kzg.rs:182-185."""
        e = srs.engine
        return e._point_call(lambda h, *a: lib.kzgb_commit_blob(h, blob.blob_data, len(blob.blob_data), *a))

    def compute_proof(self, polynomial: PolynomialEvalForm, z_fr: int, srs: SRS) -> Affine:
        """kzg.rs:215-234 (+ compute_proof_impl :128-178)."""
        if len(polynomial) != len(self.expanded_roots_of_unity):
            raise KzgError("GenericError", "inconsistent length between blob and root of unities")
        e = srs.engine
        m = fr_to_mont_bytes(polynomial.evaluations)
        z = fr_to_mont_bytes([z_fr])
        return e._point_call(lambda h, out, inf: lib.kzgb_compute_proof(h, m, len(polynomial), z, out, inf, None))

    def compute_proof_with_known_z_fr_index(self, polynomial: PolynomialEvalForm, index: int, srs: SRS) -> Affine:
        """kzg.rs:187-207."""
        z = self.get_nth_root_of_unity(index)
        if z is None:
            raise KzgError("GenericError", "Root of unity not found")
        return self.compute_proof(polynomial, z, srs)

    def g1_ifft(self, length: int, srs: SRS) -> List[Affine]:
        """kzg.rs:263-285."""
        e = srs.engine
        if length <= 0 or length & (length - 1):
            raise KzgError("FFTError", "length provided is not a power of 2")
        xy = C.create_string_buffer(64 * length)
        inf = C.create_string_buffer(length)
        e.check(lib.kzgb_g1_ifft(e.h, length, xy, inf))
        return g1_from_abi(xy.raw, inf.raw)

    def compute_blob_proof(self, blob: Blob, commitment: Affine, srs: SRS) -> Affine:
        """kzg.rs:288-309."""
        e = srs.engine
        xy, inf = g1_to_abi([commitment])
        n = _next_pow2((len(blob.blob_data) + 31) // 32)
        if n != len(self.expanded_roots_of_unity):  # compute_proof_impl's check (kzg.rs:135-139)
            validate_g1_point(commitment, e)  # keeps the reference's order of checks (kzg.rs:295)
            raise KzgError("GenericError", "inconsistent length between blob and root of unities")
        return e._point_call(
            lambda h, *a: lib.kzgb_compute_blob_proof(h, blob.blob_data, len(blob.blob_data), xy, inf[0], *a)
        )

    # -- fused hot path: commit + proof for a batch of blobs (sharded by blob across GPUs) ---
    @staticmethod
    def commit_and_prove_blobs(blobs: Sequence[Blob], srs: SRS) -> Tuple[List[bytes], List[bytes]]:
        """commit_blob + compute_blob_proof per blob, pipelined inside the library.  Returns the
        arkworks-compressed commitment and proof bytes."""
        e = srs.engine
        count = len(blobs)
        keep, ptrs, lens = _blobs_to_abi(blobs)  # keep: the buffers ptrs points into
        cs = C.create_string_buffer(32 * count if count else 1)
        ps = C.create_string_buffer(32 * count if count else 1)
        e.check(lib.kzgb_commit_and_prove_blobs(e.h, ptrs, lens, count, cs, ps))
        return ([cs.raw[32 * i : 32 * i + 32] for i in range(count)], [ps.raw[32 * i : 32 * i + 32] for i in range(count)])


def compute_challenge(blob: Blob, commitment: Affine, engine: Optional[Engine] = None) -> int:
    """primitives/src/helpers.rs:411-472 (host SHA-256 inside the library)."""
    xy, inf = g1_to_abi([commitment])
    out = C.create_string_buffer(32)
    h = engine.h if engine else None
    rc = lib.kzgb_compute_challenge(h, blob.blob_data, len(blob.blob_data), xy, inf[0], out)
    if rc != 0:
        raise KzgError(_capi.STATUS_VARIANT.get(rc, "GenericError"), "G1 point not on curve")
    return fr_from_mont_bytes(out.raw)[0]


def evaluate_polynomial_in_evaluation_form(polynomial: PolynomialEvalForm, z: int, engine: Optional[Engine] = None) -> int:
    """primitives/src/helpers.rs:475-535 (GPU barycentric evaluation with batched inversion)."""
    if polynomial.len_underlying_blob_bytes == 0:
        raise KzgError("GenericError", "Length of data after padding is 0")
    if len(polynomial) != _next_pow2(-(-polynomial.len_underlying_blob_bytes // 32)):
        raise KzgError("InvalidInputLength")
    e = engine or default_engine()
    out = C.create_string_buffer(32)
    e.check(lib.kzgb_evaluate_polynomial(e.h, fr_to_mont_bytes(polynomial.evaluations), len(polynomial), fr_to_mont_bytes([z]), out))
    return fr_from_mont_bytes(out.raw)[0]


def verify_proof_g1(commitment: Affine, proof: Affine, value_fr: int, engine: Optional[Engine] = None) -> Affine:
    """verifier/src/verify.rs:10-42: validates both points and returns ``commitment - [value] G1``, the first argument of the
    final ``pairings_verify`` (which, with ``[tau - z] G2``, stays in the reference's code)."""
    e = engine or default_engine()
    cxy, cinf = g1_to_abi([commitment])
    pxy, pinf = g1_to_abi([proof])
    out = C.create_string_buffer(64)
    inf = C.c_uint8(0)
    e.check(lib.kzgb_verify_proof_g1(e.h, cxy, cinf[0], pxy, pinf[0], fr_to_mont_bytes([value_fr]), out, C.byref(inf)))
    return g1_from_abi(out.raw, bytes([inf.value]))[0]


def verify_blob_kzg_proof_g1(blob: "Blob", commitment: Affine, proof: Affine, engine: Optional[Engine] = None) -> Tuple[Affine, int, int]:
    """verifier/src/verify.rs:77-115 up to the pairing: returns ``(commitment - [y] G1, z, y)``."""
    e = engine or default_engine()
    cxy, cinf = g1_to_abi([commitment])
    pxy, pinf = g1_to_abi([proof])
    out = C.create_string_buffer(64)
    inf = C.c_uint8(0)
    z, y = C.create_string_buffer(32), C.create_string_buffer(32)
    e.check(lib.kzgb_verify_blob_proof_g1(e.h, blob.blob_data, len(blob.blob_data), cxy, cinf[0], pxy, pinf[0], out, C.byref(inf), z, y))
    return g1_from_abi(out.raw, bytes([inf.value]))[0], fr_from_mont_bytes(z.raw)[0], fr_from_mont_bytes(y.raw)[0]


def verify_blob_kzg_proof_batch_rlc(
    blobs: Sequence[Blob], commitments: Sequence[Affine], proofs: Sequence[Affine], engine: Optional[Engine] = None
) -> Tuple[Affine, Affine]:
    """verifier/src/batch.rs:16-249 up to (not including) the pairing: returns the two G1 inputs
    ``(proof_lincomb, rhs_g1)`` of ``pairings_verify`` (batch.rs:253-254), which stays in the
    reference's code."""
    if not (len(commitments) == len(blobs) and len(proofs) == len(blobs)):
        raise KzgError("GenericError", "length's of the input are not the same")
    e = engine or default_engine()
    count = len(blobs)
    keep, ptrs, lens = _blobs_to_abi(blobs)  # keep: the buffers ptrs points into
    cxy, cinf = g1_to_abi(commitments)
    pxy, pinf = g1_to_abi(proofs)
    lhs = C.create_string_buffer(64)
    rhs = C.create_string_buffer(64)
    li = C.c_uint8(0)
    ri = C.c_uint8(0)
    e.check(lib.kzgb_verify_batch_rlc(e.h, ptrs, lens, count, cxy, cinf, pxy, pinf, lhs, C.byref(li), rhs, C.byref(ri)))
    return g1_from_abi(lhs.raw, bytes([li.value]))[0], g1_from_abi(rhs.raw, bytes([ri.value]))[0]
