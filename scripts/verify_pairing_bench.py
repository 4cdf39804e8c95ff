"""Blobs per second of per-blob verification through the pairing (kzgb_verify_blob_proofs{,_dev},
kzgb_group_verify_blob_proofs), each next to the G1-only call of the same shape (kzgb_verify_blob_proofs_g1{,_dev},
kzgb_group_verify_blob_proofs_g1), and openings per second of kzgb_verify_proofs, on the shapes a verifier sees:

  4096 x 2^12 Fr and 64 x 2^19 Fr (blobs); 4096 and 65 536 openings.

Inputs are seeded random blobs (canonical elements) with their own commitments and proofs on a synthetic SRS of known
tau, and [tau]G2 set to match (untimed); the proofs of two blobs are swapped.  Before any timing counts, every leg's output
is checked: 1 at every honest blob, 0 at the two swapped ones.  The openings are the (C_i, pi_i, z_i, y_i) of the blob
batch, repeated to the wanted count.  Every leg is warmed up once and timed over --reps calls (host clock; the calls end
in a device synchronise).  The group legs run over one member on GPU 0.  The pairing kernels' time per opening comes from
torch.profiler (CUDA activities) around one more openings call; their Fq-mul count per opening is computed below from the
structure of pairing.cuh, and set against the integer-pipe roof measured in the same run (kzgb_microbench IMAD/s / 136,
as all_roots_bench.py).  Prints the card and its power limit, then one JSON line per shape, and writes them to --out.

    python scripts/verify_pairing_bench.py [--reps 3] [--out file.jsonl]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

SHAPES = {"4096x2^12": (12, 4096), "64x2^19": (19, 64)}
OPENINGS = (4096, 65536)
IMAD_PER_FQMUL = 136
KERNELS = ("k_pairing_prep", "k_miller", "k_final_exp")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def fq_mul_per_opening():
    """Montgomery products per opening in pairing.cu, counted from pairing.cuh / ec.cuh (a difference of two products
    with one reduction counts as two).  The inversions (safegcd) are not products and are left out."""
    fq2_mul, fq2_sqr, fq2_mul_fq = 4, 2, 2
    fq6_mul, fq6_mul01, fq6_mul_fq = 6 * fq2_mul, 5 * fq2_mul, 3 * fq2_mul_fq
    fq12_mul, fq12_sqr = 3 * fq6_mul, 2 * fq6_mul
    line = 2 * fq6_mul_fq + 2 * fq6_mul01 + fq2_mul_fq
    cyc = 3 * 2 * fq2_mul
    x = 4965661367192848881
    lines = 64 + bin(6 * x + 2 - (1 << 64)).count("1") + 2
    miller = 63 * fq12_sqr + 2 * lines * line
    exp_x = (x.bit_length() - 1) * cyc + (bin(x).count("1") - 1) * fq12_mul
    fq6_inv = 9 * fq2_mul + 3 * fq2_sqr + 3
    final = (4 * fq6_mul + fq6_inv) + 2 * fq12_mul + 5 * fq2_mul + 3 * exp_x + 3 * cyc + 10 * fq12_mul + 15 * fq2_mul
    g1_dbl, g1_add, g1_madd = 9, 14, 10  # xyzz_dbl, xyzz_add, xyzz_madd
    prep_g1 = 252 * g1_dbl + 64 * g1_add + 7 * g1_add + 65 * g1_madd + 6
    prep_g2 = 64 * (8 * fq2_mul + 2 * fq2_sqr) + 2 * fq2_mul
    return {"miller": miller, "final_exp": final, "prep_g1": prep_g1, "prep_g2": prep_g2,
            "total": miller + final + prep_g1 + prep_g2}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU")
    from __graft_entry__ import load_package
    from oracle import bn254 as o

    pkg = load_package()
    lib = pkg.lib
    h = C.c_void_p()
    assert lib.kzgb_ctx_create(C.byref(h), 0, None) == 0

    def check(rc, err=lambda: lib.kzgb_last_error(h)):
        if rc:
            raise RuntimeError(f"{rc}: {err().decode()}")

    tau2 = pkg.g2_to_abi(o.g2_mul(o.G2_GEN, o.SYNTH_TAU))
    check(lib.kzgb_srs_load_synthetic(h, pkg.fr_to_mont_bytes([o.SYNTH_TAU]), 1 << 19))
    check(lib.kzgb_set_g2_tau(h, tau2))
    grp = C.c_void_p()
    assert lib.kzgb_group_create(C.byref(grp), (C.c_int * 1)(0), 1) == 0
    check(lib.kzgb_group_set_g2_tau(grp, tau2), lambda: lib.kzgb_group_last_error(grp))
    imad = C.c_double(0)
    check(lib.kzgb_microbench(h, 0, C.byref(imad)))
    roof = imad.value / IMAD_PER_FQMUL
    model = fq_mul_per_opening()
    name = card()
    print(json.dumps({"card": name, "cpu_count": os.cpu_count(), "roof_fqmul_per_s": roof,
                      "fq_mul_per_opening": model}), flush=True)
    results = []
    for shape in args.shapes.split(","):
        logn, count = SHAPES[shape]
        n = 1 << logn
        check(lib.kzgb_srs_prepare_lagrange(h, n))
        rng = np.random.default_rng(logn * 1000 + count)
        host = torch.empty((count, 32 * n), dtype=torch.uint8).pin_memory()
        step = max(1, (1 << 27) // (32 * n))
        for i in range(0, count, step):
            a = rng.integers(0, 256, size=(min(step, count - i), n, 32), dtype=np.uint8)
            a[:, :, 0] &= 0x1F
            host[i : i + len(a)] = torch.from_numpy(a.reshape(len(a), -1))
        dbuf = host.cuda()
        lens = (C.c_size_t * count)(*[32 * n] * count)
        hptrs = (C.c_void_p * count)(*[host[i].data_ptr() for i in range(count)])
        dptrs = (C.c_void_p * count)(*[dbuf[i].data_ptr() for i in range(count)])
        cxy, cinf = C.create_string_buffer(64 * count), C.create_string_buffer(count)
        pxy, pinf = C.create_string_buffer(64 * count), C.create_string_buffer(count)
        check(lib.kzgb_commit_blobs(h, hptrs, lens, count, cxy, cinf))
        check(lib.kzgb_compute_blob_proofs(h, hptrs, lens, count, cxy, cinf, pxy, pinf))
        swapped = (1, count // 2)
        p = bytearray(pxy.raw)
        p[64 * swapped[0] : 64 * swapped[0] + 64], p[64 * swapped[1] : 64 * swapped[1] + 64] = (
            p[64 * swapped[1] : 64 * swapped[1] + 64], p[64 * swapped[0] : 64 * swapped[0] + 64])
        pxy = C.create_string_buffer(bytes(p), len(p))
        want = bytes(0 if i in swapped else 1 for i in range(count))
        ok = {leg: C.create_string_buffer(count) for leg in ("host", "dev", "group")}
        g1 = tuple(C.create_string_buffer(k * count) for k in (64, 1, 32, 32))

        def bools(leg):
            if leg == "dev":
                check(lib.kzgb_verify_blob_proofs_dev(h, dptrs, hptrs, lens, count, cxy, cinf, pxy, pinf, ok[leg]))
            elif leg == "group":
                check(lib.kzgb_group_verify_blob_proofs(grp, hptrs, lens, count, cxy, cinf, pxy, pinf, ok[leg]),
                      lambda: lib.kzgb_group_last_error(grp))
            else:
                check(lib.kzgb_verify_blob_proofs(h, hptrs, lens, count, cxy, cinf, pxy, pinf, ok[leg]))

        def g1_only(leg):
            if leg == "dev":
                check(lib.kzgb_verify_blob_proofs_g1_dev(h, dptrs, hptrs, lens, count, cxy, cinf, pxy, pinf, *g1))
            elif leg == "group":
                check(lib.kzgb_group_verify_blob_proofs_g1(grp, hptrs, lens, count, cxy, cinf, pxy, pinf, *g1),
                      lambda: lib.kzgb_group_last_error(grp))
            else:
                check(lib.kzgb_verify_blob_proofs_g1(h, hptrs, lens, count, cxy, cinf, pxy, pinf, *g1))

        for leg in ok:
            bools(leg)
            if ok[leg].raw != want:
                raise SystemExit(f"{shape}: {leg} bools wrong at {[i for i in range(count) if ok[leg].raw[i] != want[i]][:8]}")

        def timed(fn, items, *a):
            fn(*a)
            rates = []
            for _ in range(args.reps):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn(*a)
                torch.cuda.synchronize()
                rates.append(items / (time.perf_counter() - t0))
            return rates

        rec = {"shape": shape, "card": name, "reps": args.reps, "group_gpus": 1}
        for leg in ("host", "dev", "group"):
            rec[f"bool_{leg}_blobs_per_s"] = [round(r, 1) for r in timed(bools, count, leg)]
            rec[f"g1_{leg}_blobs_per_s"] = [round(r, 1) for r in timed(g1_only, count, leg)]
        print(json.dumps(rec), flush=True)
        results.append(rec)
        if logn == 12:  # the openings of this batch, repeated
            g1_only("host")
            zw, yw = g1[2].raw, g1[3].raw
            for m in OPENINGS:
                k = m // count
                oc, oci, op, opi = cxy.raw * k, cinf.raw * k, pxy.raw * k, pinf.raw * k
                oz, oy = zw * k, yw * k
                oo = C.create_string_buffer(m)

                def openings():
                    check(lib.kzgb_verify_proofs(h, m, oc, oci, op, opi, oz, oy, oo))

                openings()
                if oo.raw != want * k:
                    raise SystemExit(f"openings {m}: bools wrong")
                rates = timed(openings, m)
                with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                    openings()
                    torch.cuda.synchronize()
                per_kernel = {}
                for e in prof.key_averages():
                    for kname in KERNELS:
                        if kname in e.key:
                            per_kernel[kname] = per_kernel.get(kname, 0) + (
                                getattr(e, "device_time_total", 0) or getattr(e, "cuda_time_total", 0))
                k_us = sum(per_kernel.values())
                orec = {"openings": m, "card": name, "verify_proofs_per_s": [round(r, 1) for r in rates],
                        "kernel_us": {k: round(v, 1) for k, v in per_kernel.items()},
                        "kernel_ns_per_opening": round(1000 * k_us / m, 1),
                        "fq_mul_per_opening": model["total"],
                        "fq_mul_per_s": round(model["total"] * m / (k_us * 1e-6)) if k_us else None,
                        "share_of_roof": round(model["total"] * m / (k_us * 1e-6) / roof, 3) if k_us else None}
                print(json.dumps(orec), flush=True)
                results.append(orec)
        del dbuf, host
        torch.cuda.empty_cache()
    lib.kzgb_group_destroy(grp)
    lib.kzgb_ctx_destroy(h)
    if args.out:
        with open(args.out, "a") as f:
            for rec in results:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
