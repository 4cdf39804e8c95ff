"""Proofs per second of kzgb_compute_proofs{,_dev} (KZG::compute_proof for many polynomials, each at a point the caller
chooses) against a loop of kzgb_compute_proof and against kzgb_compute_blob_proofs on the same polynomials given as blob
bytes (the same GPU work plus the SHA-256 transcripts), on the workloads

  64 x 2^19 Fr in pinned host memory, the same 64 polynomials resident in HBM (_dev), 1024 x 2^16 and 4096 x 2^12,

each with three sets of points: random z outside the domain ("outside"), roots w^k only ("roots"), and the two
alternating, so that every group holds both ("mixed").  Inputs are seeded canonical evaluations of 0.5-2 GiB per
workload, larger than the 126 MB L2; the kzgb_compute_blob_proofs leg gets the same evaluations as big-endian bytes and
their own commitments (kzgb_commit_blobs, untimed).  Every leg is warmed up once and timed over --reps calls, each ending
in a device synchronise (the calls return host results).  All legs that take the caller's points must return the same
proofs, checked before anything is timed.  --lib loads another build of the library (same ABI) in place of the
package's; --group-devices d0,d1,.. adds kzgb_group_compute_proofs over those devices.  Prints the card and its power
limit and the host's CPU count, then one JSON line per workload and point set, and writes them to --out when given.

    python scripts/compute_proofs_bench.py [--lib path/to/libkzgbn254_b200.so] [--reps 3] [--profile DIR] [--out file.jsonl]
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
POINT_SETS = ("outside", "roots", "mixed")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def profile_call(fn, trace_path):
    """fn() once under torch.profiler: the device time of the 12 largest kernels and copies it ran (ms, by name), and
    the trace at trace_path."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    os.makedirs(os.path.dirname(trace_path), exist_ok=True)
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    prof.export_chrome_trace(trace_path)
    totals = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = getattr(ev, "cuda_time_total", 0)
        if t:
            totals[ev.key] = totals.get(ev.key, 0.0) + t / 1e3
    return {k: round(v, 3) for k, v in sorted(totals.items(), key=lambda kv: -kv[1])[:12]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--points", default=",".join(POINT_SETS))
    ap.add_argument("--loop-polys", type=int, default=64, help="polynomials timed in the kzgb_compute_proof loop (rate per proof)")
    ap.add_argument("--group-devices", default=None, help="also time kzgb_group_compute_proofs over these devices")
    ap.add_argument("--profile", default=None, metavar="DIR",
                    help="after timing, one kzgb_compute_proofs call per point set under torch.profiler: its kernel totals "
                         "are printed and its trace written to DIR")
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

    tau = pkg.fr_to_mont_bytes([o.SYNTH_TAU])
    check(lib.kzgb_srs_load_synthetic(h, tau, 1 << 19))
    grp = None
    if args.group_devices:
        devs = [int(d) for d in args.group_devices.split(",")]
        grp = C.c_void_p()
        assert lib.kzgb_group_create(C.byref(grp), (C.c_int * len(devs))(*devs), len(devs)) == 0
        check(lib.kzgb_group_srs_load_synthetic(grp, tau, 1 << 19), lambda: lib.kzgb_group_last_error(grp))
    name = card()
    print(json.dumps({"card": name, "lib": args.lib or "package", "cpu_count": os.cpu_count(),
                      "cpus_usable": len(os.sched_getaffinity(0))}), flush=True)
    results = []
    for wl in args.workloads.split(","):
        logn, count, dev = WORKLOADS[wl]
        n = 1 << logn
        check(lib.kzgb_srs_prepare_lagrange(h, n))
        if grp:
            check(lib.kzgb_group_srs_prepare_lagrange(grp, n), lambda: lib.kzgb_group_last_error(grp))
        rng = np.random.default_rng(logn * 1000 + count)
        # canonical evaluations as big-endian blob bytes (the blob-proof leg) and as Montgomery words (the other legs)
        blobs = torch.empty((count, 32 * n), dtype=torch.uint8).pin_memory()
        mont = torch.empty((count, 32 * n), dtype=torch.uint8).pin_memory()
        step = max(1, (1 << 27) // (32 * n))  # generate in ~128 MiB slices
        for i in range(0, count, step):
            k = min(step, count - i)
            a = rng.integers(0, 256, size=(k, n, 32), dtype=np.uint8)
            a[:, :, 0] &= 0x1F  # canonical: < 2^253 < r
            blobs[i : i + k] = torch.from_numpy(a.reshape(k, -1))
            d = torch.from_numpy(np.ascontiguousarray(a.reshape(k, -1)))
            check(lib.kzgb_to_fr_array(h, d.data_ptr(), k * 32 * n, mont[i : i + k].data_ptr()))
        dmont = mont.cuda() if dev else None
        lens = (C.c_size_t * count)(*[32 * n] * count)
        ns = (C.c_size_t * count)(*[n] * count)
        bptrs = (C.c_void_p * count)(*[blobs[i].data_ptr() for i in range(count)])
        mptrs = (C.c_void_p * count)(*[mont[i].data_ptr() for i in range(count)])
        dptrs = (C.c_void_p * count)(*[dmont[i].data_ptr() for i in range(count)]) if dev else None
        cxy, cinf = C.create_string_buffer(64 * count), C.create_string_buffer(count)
        check(lib.kzgb_commit_blobs(h, bptrs, lens, count, cxy, cinf))
        bxy, binf = C.create_string_buffer(64 * count), C.create_string_buffer(count)

        def blob_proofs():
            check(lib.kzgb_compute_blob_proofs(h, bptrs, lens, count, cxy, cinf, bxy, binf))

        r_blob = None
        w = o.PRIMITIVE_ROOTS_OF_UNITY[logn]
        prng = np.random.default_rng(logn)
        for ps in args.points.split(","):
            zs = []
            for i in range(count):
                root = ps == "roots" or (ps == "mixed" and i % 2)
                zs.append(pow(w, int(prng.integers(0, n)), o.R) if root else int.from_bytes(prng.bytes(32), "little") % o.R)
            zm = pkg.fr_to_mont_bytes(zs)
            xy, inf, ys = C.create_string_buffer(64 * count), C.create_string_buffer(count), C.create_string_buffer(32 * count)
            gxy, ginf = C.create_string_buffer(64 * count), C.create_string_buffer(count)

            def proofs():
                if dev:
                    check(lib.kzgb_compute_proofs_dev(h, dptrs, ns, count, zm, xy, inf, ys))
                else:
                    check(lib.kzgb_compute_proofs(h, mptrs, ns, count, zm, xy, inf, ys))

            def group_proofs():
                check(lib.kzgb_group_compute_proofs(grp, mptrs, ns, count, zm, gxy, ginf, None), lambda: lib.kzgb_group_last_error(grp))

            loop_n = min(count, args.loop_polys)
            lxy, linf = C.create_string_buffer(64 * loop_n), C.create_string_buffer(loop_n)

            def loop():
                for i in range(loop_n):
                    check(lib.kzgb_compute_proof(h, mptrs[i], n, zm[32 * i : 32 * i + 32], C.cast(C.addressof(lxy) + 64 * i, C.c_void_p),
                                                 C.cast(C.addressof(linf) + i, C.POINTER(C.c_uint8)), None))

            # the legs agree before anything is timed
            proofs()
            loop()
            if grp:
                group_proofs()
            same = lxy.raw == xy.raw[: 64 * loop_n] and linf.raw == inf.raw[:loop_n]
            same = same and (not grp or (gxy.raw == xy.raw and ginf.raw == inf.raw))
            if not same:
                raise SystemExit(f"{wl} {ps}: proofs differ between the legs")

            def timed(fn, items):
                fn()  # warm-up: lanes, workspaces, tables
                rates = []
                for _ in range(args.reps):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    fn()
                    torch.cuda.synchronize()
                    rates.append(items / (time.perf_counter() - t0))
                return rates

            r_proofs = timed(proofs, count)
            r_loop = timed(loop, loop_n)
            r_group = timed(group_proofs, count) if grp else None
            if r_blob is None:
                r_blob = timed(blob_proofs, count)
            rec = {"workload": wl, "points": ps, "card": name, "lib": args.lib or "package", "reps": args.reps,
                   "compute_proofs_per_s": [round(r, 1) for r in r_proofs],
                   "compute_proof_loop_per_s": [round(r, 1) for r in r_loop], "loop_polys": loop_n,
                   "compute_blob_proofs_per_s": [round(r, 1) for r in r_blob], "proofs_equal": same}
            if grp:
                rec["group_devices"] = args.group_devices
                rec["group_compute_proofs_per_s"] = [round(r, 1) for r in r_group]
            if args.profile:
                rec["profile_kernels_ms"] = profile_call(proofs, os.path.join(args.profile, f"compute_proofs_{wl}_{ps}.pt.trace.json"))
            print(json.dumps(rec), flush=True)
            results.append(rec)
        del dmont, mont, blobs
        torch.cuda.empty_cache()
    if grp:
        lib.kzgb_group_destroy(grp)
    lib.kzgb_ctx_destroy(h)
    if args.out:
        with open(args.out, "a") as f:
            for rec in results:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
