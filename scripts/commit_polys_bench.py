"""Commitments per second of kzgb_commit_evals{,_dev} and kzgb_commit_coeffs{,_dev} (KZG::commit_eval_form /
commit_coeff_form for many polynomials in one call) against a loop of the single call (kzgb_commit_eval /
kzgb_commit_coeff), against kzgb_commit_blobs on the same values given as blob bytes (evaluation form: the blob job reads
the same 32 bytes per element, so it is that form's reference rate), and the kzgb_group_commit_* call over every visible
GPU, on the workloads

  evals_/coeffs_  64x2^19, 1024x2^16, 4096x2^12   values in pinned host memory, and the same resident in HBM (_dev)
  ref_mixed / ref_sorted                          the reference's commit benchmark (bench_kzg_commit_{10000,30000,50000}):
                                                  Blob::from_raw_data of random printable payloads of 10000, 30000 and
                                                  50000 bytes in coefficient form (512, 1024 and 2048 coefficients after
                                                  padding), --ref-count of each, in random order and sorted by size
  coeffs_8x2^22                                   coefficient form, host values, on an SRS of 2^22 points

Inputs are seeded canonical values (the large workloads 0.5-2 GiB, larger than the 126 MB L2).  Every leg is warmed up
once and timed over --reps calls, each ending in a device synchronise (the calls return host results).  Before anything
is timed, --loop-polys entries sampled across the batch must equal the single call, and the group's points the batch's.
--routes instead times coefficient-form groups of 512 .. 4096 coefficients on a fresh context and with a 2^19 monomial
window table resident: the route the library selects (option lagrange = 1) against one batched MSM over the monomial
window table (lagrange = 0, no Lagrange table).  Prints the card and its power limit, then one JSON
line per workload, and appends them to --out when given.

    python scripts/commit_polys_bench.py [--reps 3] [--workloads a,b] [--routes] [--profile DIR] [--out file.jsonl]
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

# name: (form, log2 n, count, device-resident)
WORKLOADS = {}
for _form in ("evals", "coeffs"):
    for _logn, _count in ((19, 64), (16, 1024), (12, 4096)):
        for _dev in (False, True):
            WORKLOADS[f"{_form}_{_count}x2^{_logn}{'_dev' if _dev else ''}"] = (_form, _logn, _count, _dev)
WORKLOADS["ref_mixed"] = ("coeffs", None, None, False)
WORKLOADS["ref_sorted"] = ("coeffs", None, None, False)
WORKLOADS["coeffs_8x2^22"] = ("coeffs", 22, 8, False)
REF_PAYLOADS = (10000, 30000, 50000)


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


def timed(fn, items, reps):
    import torch

    fn()  # warm-up: lanes, workspaces, tables
    rates = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        rates.append(round(items / (time.perf_counter() - t0), 1))
    return rates


class Lib:
    """The package's library with one context (and optionally one group) over a synthetic SRS of srs_n points."""

    def __init__(self, pkg, srs_n, group_devices=None):
        from oracle import bn254 as o

        self.lib = pkg.lib
        self.h = C.c_void_p()
        assert self.lib.kzgb_ctx_create(C.byref(self.h), 0, None) == 0
        self.tau = pkg.fr_to_mont_bytes([o.SYNTH_TAU])
        self.check(self.lib.kzgb_srs_load_synthetic(self.h, self.tau, srs_n))
        self.grp = None
        if group_devices:
            self.grp = C.c_void_p()
            assert self.lib.kzgb_group_create(C.byref(self.grp), (C.c_int * len(group_devices))(*group_devices), len(group_devices)) == 0
            self.gcheck(self.lib.kzgb_group_srs_load_synthetic(self.grp, self.tau, srs_n))

    def check(self, rc):
        if rc:
            raise RuntimeError(f"{rc}: {self.lib.kzgb_last_error(self.h).decode()}")

    def gcheck(self, rc):
        if rc:
            raise RuntimeError(f"{rc}: {self.lib.kzgb_group_last_error(self.grp).decode()}")

    def close(self):
        if self.grp:
            self.lib.kzgb_group_destroy(self.grp)
        self.lib.kzgb_ctx_destroy(self.h)


def make_values(L, rng, sizes, pad_to=None):
    """Seeded canonical values: blob bytes (big-endian, pinned) and their Montgomery words (pinned), one row per entry of
    max(sizes) slots; entry i fills sizes[i] of them (the rest zero)."""
    import numpy as np
    import torch

    width = max(sizes)
    count = len(sizes)
    blobs = torch.zeros((count, 32 * width), dtype=torch.uint8).pin_memory()
    mont = torch.zeros((count, 32 * width), dtype=torch.uint8).pin_memory()
    step = max(1, (1 << 27) // (32 * width))  # ~128 MiB slices
    for i in range(0, count, step):
        k = min(step, count - i)
        a = rng.integers(0, 256, size=(k, width, 32), dtype=np.uint8)
        a[:, :, 0] &= 0x1F  # canonical: < 2^253 < r
        for j in range(k):
            a[j, sizes[i + j]:] = 0
        d = torch.from_numpy(np.ascontiguousarray(a.reshape(k, -1)))
        blobs[i : i + k] = d
        L.check(L.lib.kzgb_to_fr_array(L.h, d.data_ptr(), k * 32 * width, mont[i : i + k].data_ptr()))
    return blobs, mont


def ref_values(L, rng, count_each, sort):
    """The reference's commit benchmark: pad_payload of random printable payloads of 10000, 30000 and 50000 bytes,
    count_each of each, as coefficient-form Montgomery words (ns = the next power of two of the padded elements, as
    Blob::to_polynomial_coeff_form pads them), in random order or sorted by size."""
    import torch
    from oracle import bn254 as o

    sizes_b = [s for s in REF_PAYLOADS for _ in range(count_each)]
    if not sort:
        rng.shuffle(sizes_b)
    padded = [o.pad_payload(bytes(rng.integers(32, 127, size=s, dtype="uint8"))) for s in sizes_b]
    ns = [1 << max(0, (len(p) // 32 - 1).bit_length()) for p in padded]
    width = max(ns)
    mont = torch.zeros((len(ns), 32 * width), dtype=torch.uint8).pin_memory()
    for i, p in enumerate(padded):
        L.check(L.lib.kzgb_to_fr_array(L.h, p, len(p), mont[i].data_ptr()))
    return ns, mont


def run_workload(pkg, L, wl, args, name):
    import numpy as np
    import torch

    lib = L.lib
    form, logn, count, dev = WORKLOADS[wl]
    rng = np.random.default_rng(sum(map(ord, wl)))
    blobs = None
    if wl.startswith("ref_"):
        ns, mont = ref_values(L, rng, args.ref_count, wl == "ref_sorted")
        count = len(ns)
    else:
        ns = [1 << logn] * count
        blobs, mont = make_values(L, rng, ns)
    dmont = mont.cuda() if dev else None
    c_ns = (C.c_size_t * count)(*ns)
    ptrs = (C.c_void_p * count)(*[(dmont if dev else mont)[i].data_ptr() for i in range(count)])
    hptrs = (C.c_void_p * count)(*[mont[i].data_ptr() for i in range(count)])
    xy, inf = C.create_string_buffer(64 * count), C.create_string_buffer(count)
    gxy, ginf = C.create_string_buffer(64 * count), C.create_string_buffer(count)
    batch_fn = {("evals", False): lib.kzgb_commit_evals, ("evals", True): lib.kzgb_commit_evals_dev,
                ("coeffs", False): lib.kzgb_commit_coeffs, ("coeffs", True): lib.kzgb_commit_coeffs_dev}[(form, dev)]
    single_fn = lib.kzgb_commit_eval if form == "evals" else lib.kzgb_commit_coeff
    group_fn = lib.kzgb_group_commit_evals if form == "evals" else lib.kzgb_group_commit_coeffs

    def batch():
        L.check(batch_fn(L.h, ptrs, c_ns, count, xy, inf))

    def group():
        L.gcheck(group_fn(L.grp, hptrs, c_ns, count, gxy, ginf))

    loop_n = min(count, args.loop_polys)
    sample = sorted(rng.choice(count, size=loop_n, replace=False).tolist())
    lxy, linf = C.create_string_buffer(64 * loop_n), C.create_string_buffer(loop_n)

    def loop():
        for k, i in enumerate(sample):
            L.check(single_fn(L.h, hptrs[i], ns[i], C.cast(C.addressof(lxy) + 64 * k, C.c_void_p),
                              C.cast(C.addressof(linf) + k, C.POINTER(C.c_uint8))))

    batch()
    loop()
    same = all(lxy.raw[64 * k : 64 * k + 64] == xy.raw[64 * i : 64 * i + 64] and linf.raw[k] == inf.raw[i]
               for k, i in enumerate(sample))
    if L.grp:
        group()
        same = same and gxy.raw == xy.raw and ginf.raw == inf.raw
    if not same:
        raise SystemExit(f"{wl}: commitments differ between the legs")
    rec = {"workload": wl, "card": name, "reps": args.reps, "count": count,
           "batch_per_s": timed(batch, count, args.reps),
           "loop_per_s": timed(loop, loop_n, args.reps), "loop_polys": loop_n, "sampled_equal": same}
    if form == "evals" and blobs is not None:
        lens = (C.c_size_t * count)(*[32 * n for n in ns])
        bptrs = (C.c_void_p * count)(*[blobs[i].data_ptr() for i in range(count)])
        bxy, binf = C.create_string_buffer(64 * count), C.create_string_buffer(count)
        if dev:
            dblobs = blobs.cuda()
            dbptrs = (C.c_void_p * count)(*[dblobs[i].data_ptr() for i in range(count)])
            blob_fn = lambda: L.check(lib.kzgb_commit_blobs_dev(L.h, dbptrs, lens, count, bxy, binf))
        else:
            blob_fn = lambda: L.check(lib.kzgb_commit_blobs(L.h, bptrs, lens, count, bxy, binf))
        blob_fn()
        if bxy.raw != xy.raw:
            raise SystemExit(f"{wl}: kzgb_commit_blobs disagrees with kzgb_commit_evals")
        rec["commit_blobs_per_s"] = timed(blob_fn, count, args.reps)
    if L.grp:
        rec["group_devices"] = args.group_devices
        rec["group_per_s"] = timed(group, count, args.reps)
    if args.profile:
        rec["profile_kernels_ms"] = profile_call(batch, os.path.join(args.profile, f"commit_polys_{wl}.pt.trace.json"))
    return rec


def run_routes(pkg, args, name):
    """Coefficient-form groups: the selected route against the monomial batched MSM, on a fresh context and with a 2^19
    monomial window table resident."""
    import numpy as np

    out = []
    for resident in (False, True):
        for logn in (9, 10, 11, 12):
            L = Lib(pkg, 1 << 19)
            try:
                if resident:
                    L.check(L.lib.kzgb_srs_precompute(L.h, 1 << 19, 0))
                n, count = 1 << logn, args.routes_count
                _, mont = make_values(L, np.random.default_rng(logn), [n] * count)
                c_ns = (C.c_size_t * count)(*[n] * count)
                ptrs = (C.c_void_p * count)(*[mont[i].data_ptr() for i in range(count)])
                rec = {"routes": f"{count}x2^{logn}", "window_table_2^19": resident, "card": name}
                outs = {}
                for lag in (1, 0):
                    assert L.lib.kzgb_set_option(b"lagrange", lag) == 0
                    xy = C.create_string_buffer(64 * count)
                    fn = lambda: L.check(L.lib.kzgb_commit_coeffs(L.h, ptrs, c_ns, count, xy, None))
                    rec["selected_per_s" if lag else "monomial_per_s"] = timed(fn, count, args.reps)
                    outs[lag] = xy.raw
                assert L.lib.kzgb_set_option(b"lagrange", 1) == 0
                rec["equal"] = outs[0] == outs[1]
                out.append(rec)
                print(json.dumps(rec), flush=True)
            finally:
                assert L.lib.kzgb_set_option(b"lagrange", 1) == 0
                L.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    ap.add_argument("--loop-polys", type=int, default=64, help="entries, sampled across the batch, timed in the loop of the single call")
    ap.add_argument("--ref-count", type=int, default=1024, help="payloads of each size in the reference-shaped workloads")
    ap.add_argument("--group-devices", default=None, help="devices of the group leg (default: every visible GPU)")
    ap.add_argument("--routes", action="store_true", help="time the two coefficient-form group routes instead")
    ap.add_argument("--routes-count", type=int, default=2048)
    ap.add_argument("--profile", default=None, metavar="DIR",
                    help="after timing, one batch call per workload under torch.profiler: its kernel totals are printed "
                         "and its trace written to DIR")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU")
    from __graft_entry__ import load_package

    pkg = load_package()
    name = card()
    print(json.dumps({"card": name, "cpu_count": os.cpu_count(), "cpus_usable": len(os.sched_getaffinity(0)),
                      "visible_gpus": torch.cuda.device_count()}), flush=True)
    if args.routes:
        results = run_routes(pkg, args, name)
    else:
        if args.group_devices is None:
            args.group_devices = ",".join(str(d) for d in range(torch.cuda.device_count()))
        devs = [int(d) for d in args.group_devices.split(",") if d != ""]
        results = []
        wls = args.workloads.split(",")
        # the 2^22 workload needs an SRS of 2^22 points; the others run on 2^19, as the single calls' tests do
        for srs_log, sel in ((19, [w for w in wls if w != "coeffs_8x2^22"]), (22, [w for w in wls if w == "coeffs_8x2^22"])):
            if not sel:
                continue
            L = Lib(pkg, 1 << srs_log, devs)
            try:
                for wl in sel:
                    rec = run_workload(pkg, L, wl, args, name)
                    print(json.dumps(rec), flush=True)
                    results.append(rec)
                    torch.cuda.empty_cache()
            finally:
                L.close()
    if args.out:
        with open(args.out, "a") as f:
            for rec in results:
                f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
