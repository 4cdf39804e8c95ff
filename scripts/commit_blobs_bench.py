"""Blobs per second of the commit-only batch (kzgb_commit_blobs{,_dev}) against kzgb_commit_and_prove_blobs and a loop
of kzgb_commit_blob on the same inputs, on the workloads a caller looping KZG::commit_blob sees:

  64 x 2^19 Fr in pinned host memory, the same 64 blobs resident in HBM (_dev), 1024 x 2^16 and 4096 x 2^12.

Inputs are seeded random blobs (canonical elements) of 0.5-2 GiB per workload, larger than the 126 MB L2.  Every leg
is warmed up once and timed over --reps calls, each ending in a device synchronise (the calls return host results).
All three legs must return the same commitments.  --lib loads another build of the library (same ABI) in place of
the package's, so two builds can be compared in one GPU session.  Prints one JSON line per workload and writes them
to --out when given.

    python scripts/commit_blobs_bench.py [--lib path/to/libkzgbn254_b200.so] [--reps 3] [--out file.jsonl]
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

WORKLOADS = {"64x2^19": (19, 64, False), "64x2^19_dev": (19, 64, True), "1024x2^16": (16, 1024, False), "4096x2^12": (12, 4096, False)}


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
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--loop-blobs", type=int, default=64, help="blobs timed in the kzgb_commit_blob loop (rate per blob)")
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

    def check(rc):
        if rc:
            raise RuntimeError(f"{rc}: {lib.kzgb_last_error(h).decode()}")

    check(lib.kzgb_srs_load_synthetic(h, pkg.fr_to_mont_bytes([o.SYNTH_TAU]), 1 << 19))
    name = card()
    results = []
    for wl in args.workloads.split(","):
        logn, count, dev = WORKLOADS[wl]
        n = 1 << logn
        check(lib.kzgb_srs_prepare_lagrange(h, n))
        rng = np.random.default_rng(logn * 1000 + count)
        host = torch.empty((count, 32 * n), dtype=torch.uint8).pin_memory()
        step = max(1, (1 << 27) // (32 * n))  # generate in ~128 MiB slices
        for i in range(0, count, step):
            a = rng.integers(0, 256, size=(min(step, count - i), n, 32), dtype=np.uint8)
            a[:, :, 0] &= 0x1F  # canonical: < 2^253 < r
            host[i : i + len(a)] = torch.from_numpy(a.reshape(len(a), -1))
        dbuf = host.cuda() if dev else None
        lens = (C.c_size_t * count)(*[32 * n] * count)
        hptrs = (C.c_void_p * count)(*[host[i].data_ptr() for i in range(count)])
        dptrs = (C.c_void_p * count)(*[dbuf[i].data_ptr() for i in range(count)]) if dev else None
        xy, inf = C.create_string_buffer(64 * count), C.create_string_buffer(count)
        cm, pf = C.create_string_buffer(32 * count), C.create_string_buffer(32 * count)

        def commit_blobs():
            if dev:
                check(lib.kzgb_commit_blobs_dev(h, dptrs, lens, count, xy, inf))
            else:
                check(lib.kzgb_commit_blobs(h, hptrs, lens, count, xy, inf))

        def prove():
            if dev:
                check(lib.kzgb_commit_and_prove_blobs_dev(h, dptrs, hptrs, lens, count, cm, pf))
            else:
                check(lib.kzgb_commit_and_prove_blobs(h, hptrs, lens, count, cm, pf))

        loop_n = min(count, args.loop_blobs)
        lxy, linf = C.create_string_buffer(64 * loop_n), C.create_string_buffer(loop_n)

        def loop():
            for i in range(loop_n):
                check(lib.kzgb_commit_blob(h, hptrs[i], 32 * n, C.cast(C.addressof(lxy) + 64 * i, C.c_void_p),
                                           C.cast(C.addressof(linf) + i, C.POINTER(C.c_uint8))))

        def timed(fn, blobs):
            fn()  # warm-up: lanes, workspaces, tables
            rates = []
            for _ in range(args.reps):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn()
                torch.cuda.synchronize()
                rates.append(blobs / (time.perf_counter() - t0))
            return rates

        r_commit = timed(commit_blobs, count)
        r_prove = timed(prove, count)
        r_loop = timed(loop, loop_n)
        pts = pkg.g1_from_abi(xy.raw, inf.raw)
        same = [pkg.g1_serialize_compressed(p) for p in pts] == [cm.raw[32 * i : 32 * i + 32] for i in range(count)]
        same = same and pkg.g1_from_abi(lxy.raw, linf.raw) == pts[:loop_n]
        rec = {"workload": wl, "card": name, "lib": args.lib or "package", "reps": args.reps,
               "commit_blobs_per_s": [round(r, 1) for r in r_commit],
               "commit_and_prove_per_s": [round(r, 1) for r in r_prove],
               "commit_blob_loop_per_s": [round(r, 1) for r in r_loop], "loop_blobs": loop_n,
               "commitments_equal": same}
        print(json.dumps(rec), flush=True)
        results.append(rec)
        del dbuf, host
        torch.cuda.empty_cache()
    lib.kzgb_ctx_destroy(h)
    if args.out:
        with open(args.out, "a") as f:
            for rec in results:
                f.write(json.dumps(rec) + "\n")
    if not all(r["commitments_equal"] for r in results):
        raise SystemExit("commitments differ between the legs")


if __name__ == "__main__":
    main()
