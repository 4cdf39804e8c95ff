"""Proofs at every root of the domain (kzgb_compute_proofs_all_roots, FK20) against the loop a caller of
KZG::compute_proof_with_known_z_fr_index would run, on a synthetic SRS (tau^j G, 2^19 points) at n = 2^12, 2^16, 2^19.

Per size it records: the one-off kzgb_srs_prepare_all_roots time; the best of --reps all-roots calls (host clock around a
call that returns host results, so it ends in a device synchronise) after one warm-up call; the time of --single
kzgb_compute_proof calls at w^0 .. w^(single-1) (Lagrange table prepared, one warm-up call), scaled by n / single and
labelled extrapolated; the rate in Fq multiplications per second under the cost model below, as a fraction of the
integer-pipe roof measured live (IMAD/s / 136, as bench.py).  Every run also checks its output: the single proofs must
equal the all-roots proofs at those indices bit for bit, and sum_k rho^k pi_k must equal [sum_k rho^k q_k(tau)] G with
q_k(tau) = (p(tau) - f_k) / (tau - w^k) (one random linear combination, an MSM on the GPU, covers all n proofs).

Cost model: a G1 scalar multiplication is ~4000 Fq-mul; a call does 2n (Hadamard) + n log2(2n) (inverse 2n-point G1
NTT) + (n/2) log2(n) (forward n-point G1 NTT) of them, the table n log2(2n) (forward 2n-point G1 NTT).  The loop costs
~10 W n Fq-mul per proof (one n-point MSM).

    python scripts/all_roots_bench.py [--sizes 12,16,19] [--reps 3] [--single 64] [--out-dir DIR]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import random
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

FQMUL_PER_SCALAR_MUL = 4000
IMAD_PER_FQMUL = 136


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def scalar_muls_per_call(logn):
    n = 1 << logn
    return 2 * n + n * (logn + 1) + (n // 2) * logn


def closed_form_ok(pkg, o, eng, proofs, evals, logn, rnd):
    n = 1 << logn
    w = o.PRIMITIVE_ROOTS_OF_UNITY[logn]
    roots = [1] * n
    for i in range(1, n):
        roots[i] = roots[i - 1] * w % o.R
    den = [(o.SYNTH_TAU - r) % o.R for r in roots]
    pref, acc = [], 1
    for d in den:
        pref.append(acc)
        acc = acc * d % o.R
    inv, dinv = pow(acc, -1, o.R), [0] * n
    for i in range(n - 1, -1, -1):
        dinv[i] = inv * pref[i] % o.R
        inv = inv * den[i] % o.R
    p_tau = sum(f * r % o.R * d for f, r, d in zip(evals, roots, dinv)) % o.R
    p_tau = p_tau * (pow(o.SYNTH_TAU, n, o.R) - 1) % o.R * pow(n, -1, o.R) % o.R
    rho = rnd.randrange(1, o.R)
    rho_k = [1] * n
    for i in range(1, n):
        rho_k[i] = rho_k[i - 1] * rho % o.R
    want = sum(rk * ((p_tau - f) * d % o.R) for rk, f, d in zip(rho_k, evals, dinv)) % o.R
    return pkg.g1_lincomb(proofs, rho_k, eng) == o.g1_mul(o.G1_GEN, want)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="12,16,19")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--single", type=int, default=64, help="kzgb_compute_proof calls timed for the loop estimate")
    ap.add_argument("--out-dir", default=None)
    args = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU")
    from __graft_entry__ import load_package
    from oracle import bn254 as o

    pkg = load_package()
    lib = pkg.lib
    name = card()
    eng = pkg.Engine(0)
    sizes = [int(s) for s in args.sizes.split(",")]
    pkg.SRS.synthetic(1 << max(sizes), o.SYNTH_TAU, engine=eng)
    imad = C.c_double(0)
    eng.check(lib.kzgb_microbench(eng.h, 0, C.byref(imad)))
    roof = imad.value / IMAD_PER_FQMUL
    results = []
    for logn in sizes:
        n = 1 << logn
        rnd = random.Random(logn)
        evals = [rnd.randrange(o.R) for _ in range(n)]
        m = pkg.fr_to_mont_bytes(evals)
        xy, inf = C.create_string_buffer(64 * n), C.create_string_buffer(n)

        t0 = time.perf_counter()
        eng.check(lib.kzgb_srs_prepare_all_roots(eng.h, n))
        prepare_s = time.perf_counter() - t0

        def call():
            t = time.perf_counter()
            eng.check(lib.kzgb_compute_proofs_all_roots(eng.h, m, n, xy, inf))
            return time.perf_counter() - t

        call()
        call_s = min(call() for _ in range(args.reps))
        proofs = pkg.g1_from_abi(xy.raw, inf.raw)

        eng.check(lib.kzgb_srs_prepare_lagrange(eng.h, n))
        w = o.PRIMITIVE_ROOTS_OF_UNITY[logn]
        k = min(args.single, n)
        zs = [pkg.fr_to_mont_bytes([pow(w, i, o.R)]) for i in range(k)]
        sxy, sinf = C.create_string_buffer(64 * k), C.create_string_buffer(k)

        def single(i):
            eng.check(lib.kzgb_compute_proof(eng.h, m, n, zs[i], C.cast(C.addressof(sxy) + 64 * i, C.c_void_p),
                                             C.cast(C.addressof(sinf) + i, C.POINTER(C.c_uint8)), None))

        single(0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(k):
            single(i)
        single_s = (time.perf_counter() - t0) / k
        single_equal = pkg.g1_from_abi(sxy.raw, sinf.raw) == proofs[:k]
        closed = closed_form_ok(pkg, o, eng, proofs, evals, logn, rnd)

        work = scalar_muls_per_call(logn) * FQMUL_PER_SCALAR_MUL
        rec = {"n": n, "card": name, "reps": args.reps,
               "prepare_s": round(prepare_s, 4),
               "prepare_fqmul_per_s": n * (logn + 1) * FQMUL_PER_SCALAR_MUL / prepare_s,
               "all_roots_call_s": round(call_s, 4),
               "call_fqmul_per_s": work / call_s, "call_fraction_of_roof": round(work / call_s / roof, 3),
               "single_proof_ms": round(single_s * 1e3, 3), "single_proofs_timed": k,
               "loop_all_proofs_s_extrapolated": round(single_s * n, 2),
               "speedup_vs_loop_extrapolated": round(single_s * n / call_s, 1),
               "roof_fqmul_per_s": roof, "roof_source": "kzgb_microbench IMAD/s / 136, measured in this run",
               "single_equal_all_roots": single_equal, "closed_form_ok": closed}
        print(json.dumps(rec), flush=True)
        results.append(rec)
    eng.close()
    if args.out_dir:
        os.makedirs(args.out_dir, exist_ok=True)
        with open(os.path.join(args.out_dir, "all_roots_bench.jsonl"), "w") as f:
            for rec in results:
                f.write(json.dumps(rec) + "\n")
    if not all(r["single_equal_all_roots"] and r["closed_form_ok"] for r in results):
        raise SystemExit("all-roots proofs differ from the single-index proofs or the closed form")


if __name__ == "__main__":
    main()
