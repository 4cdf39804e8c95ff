"""Blobs per second of the batch verification up to the pairing in each of its forms, on the shapes a verifier sees:

  4096 x 2^12 Fr (BASELINE config 5's shape) and 64 x 2^19 Fr (16 MiB blobs).

Legs: kzgb_verify_batch_rlc (host blobs), kzgb_verify_batch_rlc_dev (blobs in HBM), kzgb_group_verify_batch_rlc on a group
of one GPU and on a group of every visible GPU, and kzgb_verify_kzg_proof_batch_rlc alone over the z and y of the same
batch (no blob hashed or read).  Inputs are seeded random blobs of canonical elements (0.5-1 GiB per shape, larger than
the 126 MB L2) with their own commitments and proofs on a synthetic SRS of known tau (kzgb_commit_blobs +
kzgb_compute_blob_proofs, untimed).  Before any timing counts, the host form's output is checked against the pairing
relation in G1, rhs == tau lhs, and every leg must return the host form's words.  Every leg is warmed up once and timed
over --reps calls, each ending in a device synchronise (the calls return host results).  Prints the card, its power
limit and the host's thread count, then one JSON line per shape, and writes them to --out when given.

    python scripts/verify_batch_bench.py [--reps 3] [--shapes 4096x2^12,64x2^19] [--out file.jsonl]
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

    check(lib.kzgb_srs_load_synthetic(h, pkg.fr_to_mont_bytes([o.SYNTH_TAU]), 1 << 19))
    groups = {}
    g1 = C.c_void_p()
    assert lib.kzgb_group_create(C.byref(g1), (C.c_int * 1)(0), 1) == 0
    groups["group_1gpu"] = g1
    n_gpus = torch.cuda.device_count()
    if n_gpus > 1:
        ga = C.c_void_p()
        assert lib.kzgb_group_create(C.byref(ga), None, 0) == 0
        groups[f"group_{n_gpus}gpu"] = ga
    name = card()
    print(json.dumps({"card": name, "visible_gpus": n_gpus, "cpu_count": os.cpu_count(),
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
        zs, ys = C.create_string_buffer(32 * count), C.create_string_buffer(32 * count)
        check(lib.kzgb_verify_blob_proofs_g1(h, hptrs, lens, count, cxy, cinf, pxy, pinf, None, None, zs, ys))
        ns = (C.c_uint64 * count)(*[n] * count)
        legs = ["host", "dev", *groups, "openings"]
        outs = {leg: (C.create_string_buffer(64), C.c_uint8(0), C.create_string_buffer(64), C.c_uint8(0)) for leg in legs}

        def call(leg):
            lx, li, rx, ri = outs[leg]
            tail = (lx, C.byref(li), rx, C.byref(ri))
            if leg == "host":
                check(lib.kzgb_verify_batch_rlc(h, hptrs, lens, count, cxy, cinf, pxy, pinf, *tail))
            elif leg == "dev":
                check(lib.kzgb_verify_batch_rlc_dev(h, dptrs, hptrs, lens, count, cxy, cinf, pxy, pinf, *tail))
            elif leg == "openings":
                check(lib.kzgb_verify_kzg_proof_batch_rlc(h, count, cxy, cinf, pxy, pinf, zs, ys, ns, *tail))
            else:
                g = groups[leg]
                check(lib.kzgb_group_verify_batch_rlc(g, hptrs, lens, count, cxy, cinf, pxy, pinf, *tail),
                      lambda: lib.kzgb_group_last_error(g))

        # the pairing relation before any timing: rhs == tau lhs for honest inputs
        call("host")
        lx, li, rx, ri = outs["host"]
        lhs = pkg.g1_from_abi(lx.raw, bytes([li.value]))[0]
        rhs = pkg.g1_from_abi(rx.raw, bytes([ri.value]))[0]
        if lhs is None or rhs != o.g1_mul(lhs, o.SYNTH_TAU):
            raise SystemExit(f"{shape}: rhs != tau lhs for honest inputs")

        def timed(leg):
            call(leg)  # warm-up: lanes, workspaces, twiddles
            rates = []
            for _ in range(args.reps):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                call(leg)
                torch.cuda.synchronize()
                rates.append(count / (time.perf_counter() - t0))
            return rates

        rates = {leg: timed(leg) for leg in legs}

        def words(leg):
            lx, li, rx, ri = outs[leg]
            return lx.raw, li.value, rx.raw, ri.value

        same = all(words(leg) == words("host") for leg in legs)
        rec = {"shape": shape, "card": name, "reps": args.reps, "relation_holds": True, "outputs_equal": same}
        for leg in legs:
            rec[f"{leg}_blobs_per_s"] = [round(r, 1) for r in rates[leg]]
        print(json.dumps(rec), flush=True)
        results.append(rec)
        del dbuf, host
        torch.cuda.empty_cache()
    for g in groups.values():
        lib.kzgb_group_destroy(g)
    lib.kzgb_ctx_destroy(h)
    if args.out:
        with open(args.out, "a") as f:
            for rec in results:
                f.write(json.dumps(rec) + "\n")
    if not all(r["outputs_equal"] for r in results):
        raise SystemExit("outputs differ between the legs")


if __name__ == "__main__":
    main()
