"""Blobs per second of the per-blob verification batch (kzgb_verify_blob_proofs_g1{,_dev}, kzgb_group_verify_blob_proofs_g1)
against a loop of kzgb_verify_blob_proof_g1 on the same inputs, on the shapes a verifier sees:

  4096 x 2^12 Fr (BASELINE config 5's shape) and 64 x 2^19 Fr (16 MiB blobs).

Inputs are seeded random blobs (canonical elements, 0.5-2 GiB per shape, larger than the 126 MB L2) with their own
commitments and proofs on a synthetic SRS of known tau (kzgb_commit_blobs + kzgb_compute_blob_proofs, untimed); the proofs
of two blobs are swapped, so the batch holds both outcomes.  Before any timing counts, the output of the batch call is
checked against the pairing relation in G1, out_i == (tau - z_i) proof_i: it must hold for every honest blob (every one at
64 blobs, every 8th at 4096) and fail at the two swapped ones.  Every leg is warmed up once and timed over --reps calls,
each ending in a device synchronise (the calls return host results), and every leg must return the same outputs.  The
loop is timed over --loop-blobs blobs (a rate per blob).  The group leg runs over every visible GPU.  The time of
k_commit_minus_value alone comes from torch.profiler (CUDA activities) around one more batch call, after the timed ones.
--lib loads another build of the library (same ABI).  Prints the card and its power limit and the host's CPU count, then
one JSON line per shape, and writes them to --out when given.

    python scripts/verify_blobs_bench.py [--lib path/to/libkzgbn254_b200.so] [--reps 3] [--out file.jsonl]
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


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--loop-blobs", type=int, default=64, help="blobs timed in the kzgb_verify_blob_proof_g1 loop")
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
    if args.lib:
        lib = C.CDLL(os.path.abspath(args.lib))
        for name, (res, argt) in pkg._capi.SIGNATURES.items():
            getattr(lib, name).restype, getattr(lib, name).argtypes = res, argt
    h = C.c_void_p()
    assert lib.kzgb_ctx_create(C.byref(h), 0, None) == 0

    def check(rc, err=lambda: lib.kzgb_last_error(h)):
        if rc:
            raise RuntimeError(f"{rc}: {err().decode()}")

    check(lib.kzgb_srs_load_synthetic(h, pkg.fr_to_mont_bytes([o.SYNTH_TAU]), 1 << 19))
    grp = C.c_void_p()
    assert lib.kzgb_group_create(C.byref(grp), None, 0) == 0
    members = lib.kzgb_group_size(grp)
    name = card()
    print(json.dumps({"card": name, "lib": args.lib or "package", "gpus_in_group": members, "cpu_count": os.cpu_count(),
                      "cpus_usable": len(os.sched_getaffinity(0))}), flush=True)
    results = []
    for shape in args.shapes.split(","):
        logn, count = SHAPES[shape]
        n = 1 << logn
        check(lib.kzgb_srs_prepare_lagrange(h, n))
        rng = np.random.default_rng(logn * 1000 + count)
        host = torch.empty((count, 32 * n), dtype=torch.uint8).pin_memory()
        step = max(1, (1 << 27) // (32 * n))  # generate in ~128 MiB slices
        for i in range(0, count, step):
            a = rng.integers(0, 256, size=(min(step, count - i), n, 32), dtype=np.uint8)
            a[:, :, 0] &= 0x1F  # canonical: < 2^253 < r
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
        outs = {leg: tuple(C.create_string_buffer(k * count) for k in (64, 1, 32, 32)) for leg in ("host", "dev", "group")}

        def batch(leg="host"):
            xy, inf, z, y = outs[leg]
            if leg == "dev":
                check(lib.kzgb_verify_blob_proofs_g1_dev(h, dptrs, hptrs, lens, count, cxy, cinf, pxy, pinf, xy, inf, z, y))
            elif leg == "group":
                check(lib.kzgb_group_verify_blob_proofs_g1(grp, hptrs, lens, count, cxy, cinf, pxy, pinf, xy, inf, z, y),
                      lambda: lib.kzgb_group_last_error(grp))
            else:
                check(lib.kzgb_verify_blob_proofs_g1(h, hptrs, lens, count, cxy, cinf, pxy, pinf, xy, inf, z, y))

        loop_n = min(count, args.loop_blobs)
        loop_out = tuple(C.create_string_buffer(k * loop_n) for k in (64, 1, 32, 32))

        def at(buf, off, typ=C.c_void_p):
            return C.cast(C.addressof(buf) + off, typ)

        def loop():
            lxy, linf, lz, ly = loop_out
            for i in range(loop_n):
                check(lib.kzgb_verify_blob_proof_g1(h, hptrs[i], 32 * n, at(cxy, 64 * i), cinf.raw[i], at(pxy, 64 * i),
                                                    pinf.raw[i], at(lxy, 64 * i), at(linf, i, C.POINTER(C.c_uint8)),
                                                    at(lz, 32 * i), at(ly, 32 * i)))

        # relation 2 before any timing: out_i == (tau - z_i) proof_i exactly where the proof is the blob's own
        batch()
        xy, inf, z, _ = outs["host"]
        got = pkg.g1_from_abi(xy.raw, inf.raw)
        zs = pkg.fr_from_mont_bytes(z.raw)
        proofs = pkg.g1_from_abi(pxy.raw, pinf.raw)
        checked = sorted(set(range(0, count, 1 if count <= 64 else 8)) | set(swapped))
        for i in checked:
            holds = got[i] == o.g1_mul(proofs[i], (o.SYNTH_TAU - zs[i]) % o.R)
            if holds == (i in swapped):
                raise SystemExit(f"{shape}: the pairing relation {'holds' if holds else 'fails'} at blob {i}")

        def timed(fn, blobs, *a):
            fn(*a)  # warm-up: lanes, workspaces, twiddles
            rates = []
            for _ in range(args.reps):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn(*a)
                torch.cuda.synchronize()
                rates.append(blobs / (time.perf_counter() - t0))
            return rates

        r_batch = timed(batch, count, "host")
        r_dev = timed(batch, count, "dev")
        r_group = timed(batch, count, "group")
        r_loop = timed(loop, loop_n)
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            batch()
            torch.cuda.synchronize()
        kern = [e for e in prof.key_averages() if "k_commit_minus_value" in e.key]
        k_us = sum(getattr(e, "device_time_total", 0) or getattr(e, "cuda_time_total", 0) for e in kern)
        k_launches = sum(e.count for e in kern)
        ref = [b.raw for b in outs["host"]]
        same = all([b.raw for b in outs[leg]] == ref for leg in ("dev", "group"))
        same = same and all(loop_out[k].raw == ref[k][: len(loop_out[k].raw)] for k in range(4))
        rec = {"shape": shape, "card": name, "lib": args.lib or "package", "reps": args.reps,
               "verify_blob_proofs_per_s": [round(r, 1) for r in r_batch],
               "verify_blob_proofs_dev_per_s": [round(r, 1) for r in r_dev],
               "group_verify_blob_proofs_per_s": [round(r, 1) for r in r_group], "group_gpus": members,
               "verify_blob_proof_loop_per_s": [round(r, 1) for r in r_loop], "loop_blobs": loop_n,
               "k_commit_minus_value_us": round(k_us, 1), "k_commit_minus_value_launches": k_launches,
               "relation_checked_blobs": len(checked),
               "outputs_equal": same}
        print(json.dumps(rec), flush=True)
        results.append(rec)
        del dbuf, host
        torch.cuda.empty_cache()
    lib.kzgb_group_destroy(grp)
    lib.kzgb_ctx_destroy(h)
    if args.out:
        with open(args.out, "a") as f:
            for rec in results:
                f.write(json.dumps(rec) + "\n")
    if not all(r["outputs_equal"] for r in results):
        raise SystemExit("outputs differ between the legs")


if __name__ == "__main__":
    main()
