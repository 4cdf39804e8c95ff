"""ctypes binding of libkzgbn254_b200.so (the C ABI in include/kzg_bn254_b200.h).

The library is the product; this file only declares its entry points.  There is no
fallback of any kind: if the shared library is missing the import fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libkzgbn254_b200.so")

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} not found: build the CUDA library first "
        "(python -c 'import __graft_entry__ as g; g.build()' or make -C rust-kzg-bn254_b200/csrc)"
    )

lib = C.CDLL(LIB_PATH)

u8p = C.POINTER(C.c_uint8)
u64p = C.POINTER(C.c_uint64)
ctx_p = C.c_void_p
grp_p = C.c_void_p
buf = C.c_void_p  # any host/device buffer: bytes, ctypes arrays or integer addresses

# name -> (restype, argtypes); mirrors include/kzg_bn254_b200.h one to one
SIGNATURES = {
    "kzgb_ctx_create": (C.c_int, [C.POINTER(ctx_p), C.c_int, C.c_void_p]),
    "kzgb_ctx_destroy": (None, [ctx_p]),
    "kzgb_last_error": (C.c_char_p, [ctx_p]),
    "kzgb_sync": (C.c_int, [ctx_p]),
    "kzgb_srs_load_file": (C.c_int, [ctx_p, C.c_char_p, C.c_uint32, C.c_uint32]),
    "kzgb_srs_save_cache": (C.c_int, [ctx_p, C.c_char_p]),
    "kzgb_srs_load_cache": (C.c_int, [ctx_p, C.c_char_p, C.c_uint32]),
    "kzgb_srs_load_gnark_be": (C.c_int, [ctx_p, buf, C.c_size_t]),
    "kzgb_srs_load_affine_mont": (C.c_int, [ctx_p, buf, buf, C.c_size_t]),
    "kzgb_srs_load_synthetic": (C.c_int, [ctx_p, buf, C.c_size_t]),
    "kzgb_srs_load_synthetic_range": (C.c_int, [ctx_p, buf, C.c_size_t, C.c_size_t]),
    "kzgb_srs_len": (C.c_size_t, [ctx_p]),
    "kzgb_srs_get_affine_mont": (C.c_int, [ctx_p, C.c_size_t, C.c_size_t, buf, buf]),
    "kzgb_srs_precompute": (C.c_int, [ctx_p, C.c_size_t, C.c_int]),
    "kzgb_srs_prepare_lagrange": (C.c_int, [ctx_p, C.c_size_t]),
    "kzgb_msm_srs": (C.c_int, [ctx_p, buf, C.c_size_t, buf, u8p]),
    "kzgb_msm_srs_range": (C.c_int, [ctx_p, buf, C.c_size_t, C.c_size_t, buf, u8p]),
    "kzgb_msm_srs_range_dev": (C.c_int, [ctx_p, buf, C.c_size_t, C.c_size_t, buf, u8p]),
    "kzgb_fr_powers_dev": (C.c_int, [ctx_p, buf, C.c_size_t, C.c_size_t, buf]),
    "kzgb_msm_var": (C.c_int, [ctx_p, buf, buf, buf, C.c_size_t, buf, u8p]),
    "kzgb_g1_add": (C.c_int, [buf, C.c_uint8, buf, C.c_uint8, buf, u8p]),
    "kzgb_roots_of_unity": (C.c_int, [ctx_p, C.c_uint64, buf, C.c_size_t, C.POINTER(C.c_size_t)]),
    "kzgb_ntt_fr": (C.c_int, [ctx_p, buf, C.c_size_t, C.c_int]),
    "kzgb_to_fr_array": (C.c_int, [ctx_p, buf, C.c_size_t, buf]),
    "kzgb_to_byte_array": (C.c_int, [ctx_p, buf, C.c_size_t, buf]),
    "kzgb_commit_eval": (C.c_int, [ctx_p, buf, C.c_size_t, buf, u8p]),
    "kzgb_commit_coeff": (C.c_int, [ctx_p, buf, C.c_size_t, buf, u8p]),
    "kzgb_commit_blob": (C.c_int, [ctx_p, buf, C.c_size_t, buf, u8p]),
    "kzgb_g1_ifft": (C.c_int, [ctx_p, C.c_size_t, buf, buf]),
    "kzgb_compute_proof": (C.c_int, [ctx_p, buf, C.c_size_t, buf, buf, u8p, buf]),
    "kzgb_evaluate_polynomial": (C.c_int, [ctx_p, buf, C.c_size_t, buf, buf]),
    "kzgb_compute_challenge": (C.c_int, [ctx_p, buf, C.c_size_t, buf, C.c_uint8, buf]),
    "kzgb_compute_blob_proof": (C.c_int, [ctx_p, buf, C.c_size_t, buf, C.c_uint8, buf, u8p]),
    "kzgb_commit_and_prove_blobs": (
        C.c_int,
        [ctx_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_size_t, buf, buf],
    ),
    "kzgb_commit_and_prove_blobs_dev": (
        C.c_int,
        [ctx_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_size_t, buf, buf],
    ),
    "kzgb_commit_blobs": (C.c_int, [ctx_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_size_t, buf, buf]),
    "kzgb_commit_blobs_dev": (C.c_int, [ctx_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_size_t, buf, buf]),
    "kzgb_verify_batch_rlc": (
        C.c_int,
        [ctx_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_size_t, buf, buf, buf,
         buf, buf, u8p, buf, u8p],
    ),
    "kzgb_g1_serialize_compressed": (C.c_int, [buf, C.c_uint8, buf]),
    "kzgb_g1_to_gnark_be": (C.c_int, [buf, C.c_uint8, buf]),
    "kzgb_validate_g1_points": (C.c_int, [ctx_p, buf, buf, C.c_size_t]),
    "kzgb_microbench": (C.c_int, [ctx_p, C.c_int, C.POINTER(C.c_double)]),
    "kzgb_bench_msm": (C.c_int, [ctx_p, C.c_size_t, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "kzgb_bench_ntt": (C.c_int, [ctx_p, C.c_int, C.c_size_t, C.c_int, C.POINTER(C.c_double)]),
    "kzgb_launch_count": (C.c_uint64, [ctx_p]),
    "kzgb_timer_begin": (C.c_int, [ctx_p]),
    "kzgb_timer_end": (C.c_int, [ctx_p, C.POINTER(C.c_double)]),
    "kzgb_stats": (C.c_int, [ctx_p, C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.c_int]),
    "kzgb_set_option": (C.c_int, [C.c_char_p, C.c_long]),
    "kzgb_msm_config": (C.c_int, [ctx_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_size_t)]),
    "kzgb_verify_proof_g1": (C.c_int, [ctx_p, buf, C.c_uint8, buf, C.c_uint8, buf, buf, u8p]),
    "kzgb_verify_blob_proof_g1": (C.c_int, [ctx_p, buf, C.c_size_t, buf, C.c_uint8, buf, C.c_uint8, buf, u8p, buf, buf]),
    "kzgb_trace_begin": (C.c_int, [ctx_p]),
    "kzgb_trace_end": (C.c_int, [ctx_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "kzgb_srs_precompute_range": (C.c_int, [ctx_p, C.c_size_t, C.c_size_t, C.c_int]),
    "kzgb_srs_clone": (C.c_int, [ctx_p, ctx_p]),
    # multi-GPU group
    "kzgb_group_create": (C.c_int, [C.POINTER(grp_p), C.POINTER(C.c_int), C.c_int]),
    "kzgb_group_destroy": (None, [grp_p]),
    "kzgb_group_size": (C.c_int, [grp_p]),
    "kzgb_group_ctx": (ctx_p, [grp_p, C.c_int]),
    "kzgb_group_last_error": (C.c_char_p, [grp_p]),
    "kzgb_group_sync": (C.c_int, [grp_p]),
    "kzgb_group_srs_load_file": (C.c_int, [grp_p, C.c_char_p, C.c_uint32, C.c_uint32]),
    "kzgb_group_srs_load_cache": (C.c_int, [grp_p, C.c_char_p, C.c_uint32]),
    "kzgb_group_srs_load_gnark_be": (C.c_int, [grp_p, buf, C.c_size_t]),
    "kzgb_group_srs_load_affine_mont": (C.c_int, [grp_p, buf, buf, C.c_size_t]),
    "kzgb_group_srs_load_synthetic": (C.c_int, [grp_p, buf, C.c_size_t]),
    "kzgb_group_srs_prepare_lagrange": (C.c_int, [grp_p, C.c_size_t]),
    "kzgb_group_srs_precompute_ranges": (C.c_int, [grp_p, C.c_size_t, C.c_int]),
    "kzgb_group_commit_and_prove_blobs": (C.c_int, [grp_p, C.c_void_p, C.c_void_p, C.c_size_t, buf, buf]),
    "kzgb_group_commit_blobs": (C.c_int, [grp_p, C.c_void_p, C.c_void_p, C.c_size_t, buf, buf]),
    "kzgb_group_msm_srs": (C.c_int, [grp_p, buf, C.c_size_t, buf, C.POINTER(C.c_uint8)]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)  # AttributeError here = the library does not export what the header declares
    _fn.restype = _res
    _fn.argtypes = _args

STATUS_VARIANT = {
    -1: "GenericError",
    -2: "SrsCapacityExceeded",
    -3: "SerializationError",
    -4: "FFTError",
    -5: "NotOnCurveError",
    -6: "MsmError",
    -7: "InvalidInputLength",
    -8: "DeserializationError",
    -9: "InvalidFieldElement",
    -100: "GenericError",  # CUDA failure surfaces as GenericError(<cuda string>)
}
