#!/usr/bin/env python3
"""Headline benchmark: blob commits+proofs/s on 2^19-Fr (16 MiB) blobs (BASELINE.json configs[1]).

One step = commit_blob + compute_blob_proof for a batch of B distinct 16 MiB blobs on each GPU
(eval-form IFFT + 2^19-point G1 MSM for the commitment, Fiat-Shamir challenge, barycentric
evaluation + quotient, IFFT + MSM for the proof).  N > 1 shards by blob: every rank runs its own
batch, no collective on the data path ("weak" scaling).

  value : blobs/s with the blob bytes already resident in HBM (kzgb_commit_and_prove_blobs_dev)
  e2e   : the same through the host-buffer C-ABI call (kzgb_commit_and_prove_blobs): pinned host
          blobs, H2D copies and the D2H of every commitment/proof inside the timed region
  roofline : the bucket-accumulation kernel (k_accumulate), achieved Fq multiplications/s against
          the integer-pipe roof measured live (IMAD/s / 136 IMAD per Montgomery multiplication)
  cpu_baseline : the CPU oracle (C++ restatement of the arkworks algorithm) on the box's cores

`--impl reference` times only the CPU oracle (the reference is Rust + arkworks and cannot be
built in this image -- see DESIGN.md) on the same metric/config.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LOG_N = 19
TAU = 2480609854371098259468018140899271569021640719453669963486734696239309822386  # SHA-256("kzg-bn254-b200/tau/v1") mod r
R_MOD = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
FQMUL_PER_MADD = 10  # XYZZ += affine: 8M + 2S (SURVEY.md 8d)
IMAD_PER_FQMUL = 136


def make_blob(n_elems: int, seed: int):
    """D1 'payload' distribution: byte 0 of every 32 B element is 0 (what Blob::from_raw_data yields)."""
    import numpy as np

    rng = np.random.default_rng(seed)
    a = rng.integers(0, 256, size=(n_elems, 32), dtype=np.uint8)
    a[:, 0] = 0
    return a.reshape(-1)


def dump_outputs(out_dir: str, outputs: dict) -> None:
    """Each value is a run of 32-byte compressed G1 points; written as DIR/<name>.npy, float32 of shape (points, 32), one
    byte per element (exact in float32), so the outputs of two builds compare element for element."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, raw in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.frombuffer(raw, dtype=np.uint8).reshape(-1, 32).astype(np.float32))


class ClockSampler(threading.Thread):
    """SM clocks and throttle reasons DURING the timed region.  NVML in-process (nvidia_ml_py: the library nvidia-smi itself
    reads) when importable, the nvidia-smi binary otherwise -- a forked nvidia-smi costs ~0.15 CPU-seconds per call on an 8-GPU
    box, which eight ranks cannot spare while they hash 47 GB/s of transcripts.  Only rank 0 samples, every GPU of the job."""

    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, indices):
        super().__init__(daemon=True)
        self.indices = [indices] if isinstance(indices, int) else list(indices)
        # CUDA ordinals -> what NVML / nvidia-smi address: they enumerate every GPU of the box, whatever CUDA_VISIBLE_DEVICES says
        vis = [t.strip() for t in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if t.strip()]
        self.targets = [vis[i] if i < len(vis) else str(i) for i in self.indices]
        self.rows = []  # (sm_mhz, max_mhz, [reason flags])
        self.stop_flag = False
        self.nvml = None
        try:
            import pynvml

            pynvml.nvmlInit()
            handles = []
            for t in self.targets:
                if t.isdigit():
                    handles.append(pynvml.nvmlDeviceGetHandleByIndex(int(t)))
                else:
                    try:
                        handles.append(pynvml.nvmlDeviceGetHandleByUUID(t))
                    except TypeError:
                        handles.append(pynvml.nvmlDeviceGetHandleByUUID(t.encode()))
            self.handles = handles
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def sample_nvml(self):
        nv = self.nvml
        bits = [nv.nvmlClocksEventReasonHwSlowdown if hasattr(nv, "nvmlClocksEventReasonHwSlowdown") else nv.nvmlClocksThrottleReasonHwSlowdown,
                nv.nvmlClocksEventReasonHwThermalSlowdown if hasattr(nv, "nvmlClocksEventReasonHwThermalSlowdown") else nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                nv.nvmlClocksEventReasonSwThermalSlowdown if hasattr(nv, "nvmlClocksEventReasonSwThermalSlowdown") else nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                nv.nvmlClocksEventReasonSwPowerCap if hasattr(nv, "nvmlClocksEventReasonSwPowerCap") else nv.nvmlClocksThrottleReasonSwPowerCap]
        for h in self.handles:
            sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            try:
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
            except Exception:
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            self.rows.append((sm, mx, [bool(r & b) for b in bits]))

    def sample_smi(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", ",".join(self.targets)],
                             capture_output=True, text=True, timeout=10).stdout.strip()
        for line in out.splitlines():
            r = [x.strip() for x in line.split(",")]
            if len(r) >= 6 and r[0].isdigit() and r[1].isdigit():
                self.rows.append((int(r[0]), int(r[1]), [r[2 + i].lower().startswith("active") for i in range(4)]))

    def run(self):
        while not self.stop_flag:
            try:
                if self.nvml:
                    self.sample_nvml()
                else:
                    self.sample_smi()
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        sm = [r[0] for r in self.rows]
        mx = [r[1] for r in self.rows]
        reasons = sorted({self.NAMES[i] for r in self.rows for i in range(4) if r[2][i]})
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_min_mhz": min(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "gpus_sampled": len(self.indices),
                "source": "NVML in-process (nvidia_ml_py)" if self.nvml else "nvidia-smi"}


def load_oracle_lib():
    path = os.path.join(ROOT, "oracle", "liboracle_cpu.so")
    if not os.path.exists(path):
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")])
    lib = C.CDLL(path)
    lib.ref_hw_threads.restype = C.c_int
    return lib


def cpu_commit_and_prove(olib, blob_bytes: bytes, srs_xy: bytes, threads: int) -> float:
    """One blob through the CPU oracle: commit_blob + compute_blob_proof, Fr-IFFT + MSM form."""
    cm = C.create_string_buffer(64)
    pf = C.create_string_buffer(64)
    t0 = time.perf_counter()
    olib.ref_commit_blob(blob_bytes, C.c_size_t(len(blob_bytes)), srs_xy, threads, 0, cm)
    olib.ref_blob_proof(blob_bytes, C.c_size_t(len(blob_bytes)), cm, srs_xy, threads, 0, pf)
    return time.perf_counter() - t0


def cpu_srs(olib, n: int, threads: int) -> bytes:
    """tau^i * G on the CPU for the reference arm (no GPU involved)."""
    # cheap route: SRS_i = SRS_{i-1} * tau is a scalar mul each; instead build via the oracle MSM-free path:
    from oracle import bn254 as o

    # 2^19 scalar multiplications in pure Python would take minutes; use the C oracle's g1 ops through
    # ref_msm with single-point MSMs batched by thread is also slow.  The reference arm therefore reads
    # a bounded SRS: it benchmarks at the same n but with bases = tau^i G for i < 4096 tiled to n
    # (MSM cost does not depend on the base values).
    small = o.synthetic_srs(4096)
    mont = 1 << 256
    one = b"".join((p[0] * mont % o.P).to_bytes(32, "little") + (p[1] * mont % o.P).to_bytes(32, "little") for p in small)
    return one * (n // 4096)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    olib = load_oracle_lib()
    threads = olib.ref_hw_threads()
    n = 1 << LOG_N
    srs_xy = cpu_srs(olib, n, threads)
    blob = make_blob(n, 1234).tobytes()
    for _ in range(args.warmup if args.warmup < 2 else 1):
        cpu_commit_and_prove(olib, blob, srs_xy, threads)
    times = [cpu_commit_and_prove(olib, blob, srs_xy, threads) for _ in range(args.steps)]
    total = sum(times)
    value = args.steps / total
    line = {
        "impl": "reference", "metric": "blob commits+proofs/s (2^19 Fr, 16 MiB)", "value": value, "unit": "blobs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64 (4x64-bit Montgomery, BN254 Fq/Fr)",
        "data": "synthetic",
        "config": {"workload": "single 16 MiB blob (2^19 Fr): eval-form IFFT + 2^19-point G1 MSM commitment and blob proof", "blobs_per_step": 1,
                   "log_n": LOG_N, "algorithm": "Fr-IFFT + MSM (the cheaper form; the reference's literal G1-IFFT-per-commit path is ~180x slower, see BASELINE.md)"},
        "cpu_baseline": {"value": value, "unit": "blobs/s", "cores": threads, "kind": "port",
                         "sample": "1 blob (2^19 Fr) commit+proof per step; C++ restatement of the arkworks algorithm (oracle/cpu_ref.cpp), "
                                   "MSM threaded over windows as arkworks does, evaluation/quotient with n separate inversions as the reference does"},
        "e2e": {"value": value, "unit": "blobs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--blobs-per-step", type=int, default=64,
                    help="distinct 16 MiB blobs per GPU and step (one C call).  64 = 1 GiB of blobs: deep enough for the library to hash "
                         "transcripts 16 at a time on AVX-512 when a rank has few cores (8 ranks on one host); the 16-blob figure "
                         "of round 1 is reported next to it (batch16)")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-msm-leg", action="store_true", help="skip the config-4 leg (2^26-point MSM by point range) of the default line")
    ap.add_argument("--window-bits", type=int, default=0, help="fixed-base window bits c (0 = the library's choice)")
    ap.add_argument("--option", action="append", default=[], metavar="NAME=VALUE", help="kzgb_set_option before the run (sweeps)")
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c4", "c5"],
                    help="c2 (default, headline): 16 MiB blobs; c3: 1024 x 2^16-Fr blobs sharded by blob; "
                         "c4: 2^26-point MSM sharded by point range; c5: batch-verify RLC over 4096 pairs")
    ap.add_argument("--log-n", type=int, default=0, help="override the problem size of c3/c4/c5")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="c2: write the last timed step's commitments and proofs (every rank's, in rank order; arkworks compressed) "
                         "and the config-4 leg's point (gnark compressed) to DIR as float32 .npy files, one byte per element")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.config != "c2"):
        ap.error("--dump-outputs is implemented for the c2 configuration of the b200 implementation")
    if args.impl == "reference":
        run_reference(args)
        return
    if args.config != "c2":
        import bench_configs

        getattr(bench_configs, "run_" + args.config)(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    from __graft_entry__ import load_package

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))

    pkg = load_package()
    lib = pkg.lib
    for kv in args.option:
        name, _, val = kv.partition("=")
        if lib.kzgb_set_option(name.encode(), int(val)) != 0:
            raise SystemExit(f"unknown option {name}")
    eng = pkg.Engine(local_rank)
    n = 1 << LOG_N
    B = args.blobs_per_step

    # synthetic SRS tau^i G generated on the GPU + fixed-base window tables (one-time setup)
    t_setup = time.perf_counter()
    srs = pkg.SRS.synthetic(n, TAU, engine=eng)
    srs.precompute(n, args.window_bits)
    setup_s = time.perf_counter() - t_setup
    cbits, cwin, ctab = C.c_int(0), C.c_int(0), C.c_size_t(0)
    lib.kzgb_msm_config(eng.h, C.byref(cbits), C.byref(cwin), C.byref(ctab))

    # blobs: pinned host copies (SHA-256 transcript + e2e H2D source) and HBM-resident copies
    host_blobs, dev_blobs = [], []
    for i in range(B):
        hb = torch.from_numpy(make_blob(n, 1000 * rank + i)).pin_memory()
        host_blobs.append(hb)
        dev_blobs.append(hb.to("cuda", non_blocking=False))
    lens = (C.c_size_t * B)(*[n * 32] * B)
    hptr = (C.c_void_p * B)(*[t.data_ptr() for t in host_blobs])
    dptr = (C.c_void_p * B)(*[t.data_ptr() for t in dev_blobs])
    cm = C.create_string_buffer(32 * B)
    pf = C.create_string_buffer(32 * B)

    def step_dev():
        eng.check(lib.kzgb_commit_and_prove_blobs_dev(eng.h, dptr, hptr, lens, B, cm, pf))

    def step_e2e():
        eng.check(lib.kzgb_commit_and_prove_blobs(eng.h, hptr, lens, B, cm, pf))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    import resource

    cpu_used = []  # process CPU seconds (user + system, all threads) of each timed leg on this rank

    def timed(fn, steps):
        ms = C.c_double(0)
        barrier()
        ru0 = resource.getrusage(resource.RUSAGE_SELF)
        w0 = time.perf_counter()
        eng.check(lib.kzgb_timer_begin(eng.h))
        for _ in range(steps):
            fn()
        eng.check(lib.kzgb_timer_end(eng.h, C.byref(ms)))
        wall = (time.perf_counter() - w0) * 1e3
        ru1 = resource.getrusage(resource.RUSAGE_SELF)
        cpu_used.append((ru1.ru_utime - ru0.ru_utime) + (ru1.ru_stime - ru0.ru_stime))
        barrier()
        t = torch.tensor([ms.value, wall], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]), float(t[1])

    for _ in range(args.warmup):
        step_dev()
    lib.kzgb_stats(eng.h, None, None, None, 1)
    sampler = ClockSampler(range(world) if rank == 0 else [])  # one node: the job's GPUs are 0 .. world-1
    if rank == 0:
        sampler.start()
    l0 = eng.launch_count()
    dev_ms, dev_wall = timed(step_dev, args.steps)
    launches = eng.launch_count() - l0
    acc_ms, acc_n, acc_adds = C.c_double(0), C.c_uint64(0), C.c_uint64(0)
    lib.kzgb_stats(eng.h, C.byref(acc_ms), C.byref(acc_n), C.byref(acc_adds), 1)
    out_dev = (cm.raw, pf.raw)

    for _ in range(min(args.warmup, 2)):
        step_e2e()
    e2e_ms, e2e_wall = timed(step_e2e, args.steps)
    sampler.stop_flag = True
    if rank == 0:
        sampler.join(timeout=2)
    assert (cm.raw, pf.raw) == out_dev, "device-resident and host-buffer paths disagree"

    # the same pipeline fed 16 blobs per call (round 1's step; shallow batches leave fill / drain bubbles and cannot use the
    # multi-buffer hash): a few steps, device-resident
    batch16 = None
    if B > 16:
        lens16 = (C.c_size_t * 16)(*[n * 32] * 16)
        hptr16 = (C.c_void_p * 16)(*[t.data_ptr() for t in host_blobs[:16]])
        dptr16 = (C.c_void_p * 16)(*[t.data_ptr() for t in dev_blobs[:16]])
        cm16, pf16 = C.create_string_buffer(32 * 16), C.create_string_buffer(32 * 16)

        def step16():
            eng.check(lib.kzgb_commit_and_prove_blobs_dev(eng.h, dptr16, hptr16, lens16, 16, cm16, pf16))

        for _ in range(2):
            step16()
        ms16, _ = timed(step16, args.steps)
        assert cm16.raw == out_dev[0][: 32 * 16] and pf16.raw == out_dev[1][: 32 * 16]
        batch16 = {"value": world * 16 * args.steps / (ms16 * 1e-3), "unit": "blobs/s", "blobs_per_step_per_gpu": 16,
                   "steps": args.steps, "ms_per_step": ms16 / args.steps}

    # one blob alone through the same call (latency, not throughput): commit -> transcript hash -> proof
    one_ptr = (C.c_void_p * 1)(host_blobs[0].data_ptr())
    one_len = (C.c_size_t * 1)(n * 32)
    cm1, pf1 = C.create_string_buffer(32), C.create_string_buffer(32)
    lat = []
    for _ in range(4):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        eng.check(lib.kzgb_commit_and_prove_blobs(eng.h, one_ptr, one_len, 1, cm1, pf1))
        lat.append((time.perf_counter() - t0) * 1e3)
    single_blob_ms = min(lat[1:])
    assert cm1.raw == out_dev[0][:32] and pf1.raw == out_dev[1][:32]
    outs_dev = [out_dev]
    if args.dump_outputs and world > 1:
        outs_dev = [None] * world
        dist.all_gather_object(outs_dev, out_dev)

    if rank != 0:
        # the other ranks go straight to the config-4 leg (rank 0 joins after its single-GPU roofline measurements)
        del host_blobs, dev_blobs
        eng.close()
        torch.cuda.empty_cache()
        if not args.skip_msm_leg:
            import bench_configs

            margs = argparse.Namespace(**vars(args))
            margs.log_n, margs.skip_cpu_baseline, margs.window_bits = 0, True, 0
            bench_configs.measure_c4(margs, torch, dist, world, rank, local_rank, pkg)
        if world > 1:
            dist.destroy_process_group()
        return

    value = world * B * args.steps / (dev_ms * 1e-3)
    e2e_value = world * B * args.steps / (e2e_ms * 1e-3)

    # integer-pipe roof measured live (dependency-free IMAD chains) and the kernel's achieved rate
    imad = C.c_double(0)
    eng.check(lib.kzgb_microbench(eng.h, 0, C.byref(imad)))
    imadx = C.c_double(0)
    eng.check(lib.kzgb_microbench(eng.h, 2, C.byref(imadx)))
    imadw = C.c_double(0)
    eng.check(lib.kzgb_microbench(eng.h, 1, C.byref(imadw)))
    fqpeak = C.c_double(0)
    eng.check(lib.kzgb_microbench(eng.h, 3, C.byref(fqpeak)))
    peak = imad.value / IMAD_PER_FQMUL / 1e9
    adds_per_launch = acc_adds.value / max(1, acc_n.value)
    avg_acc_ms = acc_ms.value / max(1, acc_n.value)
    # isolated (single stream, nothing else on the GPU) timing of the same kernel
    iso_total, iso_acc = C.c_double(0), C.c_double(0)
    eng.check(lib.kzgb_bench_msm(eng.h, n, 5, C.byref(iso_total), C.byref(iso_acc)))
    achieved_iso = FQMUL_PER_MADD * adds_per_launch / (iso_acc.value * 1e-3) / 1e9 if iso_acc.value else 0.0
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    traffic_src = None
    if os.path.exists(tpath):
        try:
            tj = json.load(open(tpath))
            traffic, traffic_src = tj.get("k_accumulate_dram_bytes_per_launch"), tj.get("source")
        except Exception:
            traffic = None
    # Fr NTT: the batched 2^16 transforms of config 3 (2 GiB, far beyond L2) are the HBM-bound case;
    # the single 16 MiB transform of this config is L2-resident and integer-bound (DESIGN.md 3)
    ntt_ms, ntt1_ms = C.c_double(0), C.c_double(0)
    eng.check(lib.kzgb_bench_ntt(eng.h, 16, 1024, 6, C.byref(ntt_ms)))
    eng.check(lib.kzgb_bench_ntt(eng.h, LOG_N, 1, 20, C.byref(ntt1_ms)))
    hbm_peak = None
    try:
        hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs")
    except Exception:
        pass
    hbm_src = "MEASURED_PEAKS.json hbm_gbs (of measured)" if hbm_peak else "fallback 6650 GB/s (of fallback)"
    hbm_peak = hbm_peak or 6650.0
    ntt_bytes = 64.0 * (1024 << 16)  # algorithmic: one read + one write of every element
    ntt_gbs = ntt_bytes / (ntt_ms.value * 1e-3) / 1e9
    roofline_ntt = {
        "kernel": "k_ntt_pass (Fr inverse/forward NTT, 1024 x 2^16 batched, 2 passes)", "bound": "hbm",
        "achieved": ntt_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": ntt_gbs / hbm_peak, "traffic": None,
        "peak_source": hbm_src, "ms_per_batched_call": ntt_ms.value, "algorithmic_bytes_per_call": ntt_bytes,
        "butterfly_fr_mul_per_s": (1024 << 16) * 8.0 / (ntt_ms.value * 1e-3),
        "single_2p19_ntt_ms": ntt1_ms.value,
        "single_2p19_butterfly_fr_mul_per_s": (1 << LOG_N) * LOG_N / 2.0 / (ntt1_ms.value * 1e-3),
    }
    roofline = {
        "kernel": "k_accumulate (MSM bucket accumulation, XYZZ += affine)", "bound": "integer-pipe (IMAD)",
        "achieved": achieved_iso, "peak": peak, "unit": "GFqmul/s", "frac": achieved_iso / peak if peak else None,
        "traffic": traffic, "traffic_source": traffic_src,
        "launch_ms_isolated": iso_acc.value, "msm_total_ms_isolated": iso_total.value,
        "launch_ms_in_pipeline_overlapping": avg_acc_ms,
        "in_pipeline_note": "inside the timed region the accumulate kernels of the lanes run CONCURRENTLY (about 2 in flight on average, "
                            "scripts/trace_pipeline.py), so their per-launch event times overlap and are not additive; the step-level figure is below",
        "step": {"algorithmic_fqmul_per_step": FQMUL_PER_MADD * acc_adds.value / args.steps,
                 "achieved": FQMUL_PER_MADD * acc_adds.value / (dev_ms * 1e-3) / 1e9,
                 "frac": (FQMUL_PER_MADD * acc_adds.value / (dev_ms * 1e-3) / 1e9) / peak if peak else None,
                 "note": "all point additions of the timed region (exact count read back from the device) x 10 Fq-mul / its duration: "
                         "the fraction of the model roof the WHOLE pipeline runs at, sort / stitch / bucket reduction / evaluation kernels included"},
        "algorithmic_fqmul_per_launch": FQMUL_PER_MADD * adds_per_launch, "point_adds_per_launch": adds_per_launch,
        "executed_note": "algorithmic count (SURVEY 8d): 10 Fq-mul per XYZZ += affine; the kernel executes 10 products and 9 Montgomery reductions (Y3 is one reduction of a difference of two products)",
        "peak_source": "measured live: dependency-free IMAD chains / 136 IMAD per 8x32-bit Montgomery multiplication (SURVEY.md 8d model)",
        "peak_wide_multiply": imadw.value / 132.0 / 1e9, "frac_of_wide_multiply_peak": achieved_iso / (imadw.value / 132.0 / 1e9) if imadw.value else None,
        "peak_wide_multiply_source": "measured live: IMAD.WIDE.U32 issues at half the IMAD rate on sm_100; a multiplication is 128 wide + 8 narrow multiplies",
        "imad_per_s": imad.value, "imad_wide_per_s": imadw.value, "carry_chain_imad_wide_per_s": imadx.value, "fqmul_microbench_per_s": fqpeak.value,
        "hbm_gather_GBps_isolated": adds_per_launch * 64 / (iso_acc.value * 1e-3) / 1e9 if iso_acc.value else None,
    }

    cpu_baseline = None
    if world == 1 and not args.skip_cpu_baseline:
        olib = load_oracle_lib()
        threads = olib.ref_hw_threads()
        xy = C.create_string_buffer(64 * n)
        eng.check(lib.kzgb_srs_get_affine_mont(eng.h, 0, n, xy, None))
        blob0 = host_blobs[0].numpy().tobytes()
        dt = cpu_commit_and_prove(olib, blob0, xy.raw, threads)
        # parity of the timed configuration: CPU oracle vs GPU on the same blob and SRS
        ocm = C.create_string_buffer(64)
        olib.ref_commit_blob(blob0, C.c_size_t(len(blob0)), xy.raw, threads, 0, ocm)
        oc32 = C.create_string_buffer(32)
        lib.kzgb_g1_serialize_compressed(ocm, 0, oc32)
        # the reference's LITERAL eval-form commit (G1-point IFFT of the SRS on every call, kzg.rs:98-100) at
        # n = 2^12, extrapolated by n log n: context only, the baseline value above is the cheaper Fr-IFFT form
        n12 = 1 << 12
        t0 = time.perf_counter()
        olib.ref_commit_blob(blob0[: 32 * n12], C.c_size_t(32 * n12), xy.raw[: 64 * n12], threads, 1, ocm)
        lit12 = time.perf_counter() - t0
        cpu_baseline = {"value": 1.0 / dt, "unit": "blobs/s", "cores": threads, "kind": "port",
                        "sample": "1 blob (2^19 Fr) commit+proof; C++ restatement of the arkworks algorithm (Fr-IFFT + MSM form)",
                        "commitment_matches_gpu": oc32.raw == out_dev[0][:32],
                        "literal_g1_ifft_commit_s_at_2p12": lit12,
                        "literal_g1_ifft_commit_s_at_2p19_extrapolated": lit12 * (n * LOG_N) / (n12 * 12.0)}

    # config-4 leg: the second half of BASELINE's metric ("G1 MSM Mpts/s at 1/2/4/8") on the same line
    msm_leg = None
    del host_blobs, dev_blobs
    eng.close()
    torch.cuda.empty_cache()
    if not args.skip_msm_leg:
        import bench_configs

        margs = argparse.Namespace(**vars(args))
        margs.log_n, margs.skip_cpu_baseline, margs.window_bits = 0, True, 0
        msm_leg = bench_configs.measure_c4(margs, torch, dist, world, rank, local_rank, pkg)

    line = {
        "metric": "blob commits+proofs/s (2^19 Fr, 16 MiB)", "value": value, "unit": "blobs/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u32 (8x32-bit Montgomery limbs, BN254 Fq/Fr)", "data": "synthetic",
        "config": {"workload": "single 16 MiB blob (2^19 Fr): eval-form IFFT + 2^19-point G1 MSM commitment and blob proof",
                   "path": "commit_blob + compute_blob_proof; the eval-form IFFT is the G1 IFFT of the SRS (kzg.rs:98) computed once and kept "
                           "resident as a Lagrange-basis window table, so each commitment / proof is one 2^19-point MSM on the evaluations",
                   "blobs_per_step_per_gpu": B, "log_n": LOG_N, "srs": "tau^i*G, 2^19 points, generated on GPU",
                   "blob_distribution": "D1 payload (byte 0 of each element = 0)", "sharding": "by blob, no collective",
                   "msm_window_bits": cbits.value, "msm_windows": cwin.value,
                   "l2": f"inputs larger than L2: {B * n * 32 >> 20} MiB of blobs + {cwin.value * n * 64 >> 20} MiB Lagrange window table per step"},
        "e2e": {"value": e2e_value, "unit": "blobs/s", "h2d_bytes_per_step": B * n * 32, "d2h_bytes_per_step": B * 2 * 128,
                "ms_per_step": e2e_ms / args.steps, "wall_ms_per_step": e2e_wall / args.steps},
        "gpu_launches": launches, "clocks": sampler.summary(), "roofline": roofline, "roofline_ntt": roofline_ntt,
        "cpu_baseline": cpu_baseline,
        "extra": {"msm_mpts": msm_leg, "batch16": batch16},
        "wall_ms_per_step": dev_wall / args.steps, "setup_s": setup_s,
        "host_cpu_ms_per_blob": {"resident": 1e3 * cpu_used[0] / (B * args.steps), "e2e": 1e3 * cpu_used[1] / (B * args.steps),
                                 "note": "rank 0's process CPU time (user + system, every thread: lanes, SHA-256 pool, driver) per blob inside the "
                                         "timed legs; a 16 MiB transcript alone is 9.2 ms of a SHA-NI core or 4.4 ms of an AVX-512 multi-buffer thread"},
        "single_blob_latency_ms": {"value": single_blob_ms, "note": "one 16 MiB blob through kzgb_commit_and_prove_blobs from host memory; "
                                   "bounded below by the sequential SHA-256 of the 16 MiB Fiat-Shamir transcript on one host core (~9 ms), "
                                   "which overlaps the commitment MSM; GPU work is ~4.5 ms of it"},
    }
    print(json.dumps(line))
    if args.dump_outputs:
        outputs = {"commitments": b"".join(o[0] for o in outs_dev), "proofs": b"".join(o[1] for o in outs_dev)}
        if msm_leg:
            outputs["msm_leg_point"] = bytes.fromhex(msm_leg["result_gnark_be"])
        dump_outputs(args.dump_outputs, outputs)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it (it may be read-only)
    main()
