#!/usr/bin/env python
"""bench.py -- spectrogram frames/sec on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME]
                    [--dump-outputs DIR]

One process per GPU (under torchrun for N > 1: RANK / LOCAL_RANK / WORLD_SIZE from the
environment).  A "step" is one pass of the fused spectrogram path over one rank's shard of
the recording: the N=4096 Hann 50 %-overlap periodogram of a 1-hour 48 kHz synthetic
QRSS/DFCW stream (84 375 frames; 691 MB of float32 samples in, 691 MB of PSD rows out --
both far larger than the 126 MB L2, so no flush is needed between steps).  Ranks are time
shards of an N-hour recording (weak scaling): no data-path collective, torch.distributed is
only used for the barrier and the max-over-ranks of the timings.

value  = frames/s with the samples already resident in HBM (device time, CUDA events on the
         library's stream, max over ranks).
e2e    = the same metric through glfer_gram_run() with pinned HOST buffers: H2D of the samples
         and D2H of the rows inside the timed region, pipelined in chunks on two streams.
roofline = algorithmic bytes (hop*4 + (N/2+1)*4 per frame) / the fused kernel's own duration,
         against the measured HBM copy bandwidth HBM_PEAK_GBS.
cpu_baseline / --impl reference = the reference's own C code (oracle/_ref, float radix-2
         build = what glfer ships) on the host cores, on a bounded sample of the workload.
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FS = 48000
_STDOUT_FD = 1
WORKLOADS = {
    # name: (description, plan kwargs, seconds of signal per rank)
    "metric": ("periodogram N=4096 Hann 50% ovl, 1 h @ 48 kHz per GPU (BASELINE metric config)",
               dict(n=4096, window_type=0, overlap=0.5, sub_mean=True), 3600),
    "c1": ("periodogram N=1024 Hanning 50% ovl (BASELINE configs[0] shape), 1 h @ 48 kHz per GPU",
           dict(n=1024, window_type=0, overlap=0.5, sub_mean=True), 3600),
    "n2048": ("periodogram N=2048 Hanning 50% ovl, 1 h @ 48 kHz per GPU",
              dict(n=2048, window_type=0, overlap=0.5, sub_mean=True), 3600),
    "c2": ("periodogram N=4096 Kaiser 75% ovl + avg.c plain averaging (band 400-1200 Hz, averaged rows band-only), 1 h @ 48 kHz",
           dict(n=4096, window_type=7, overlap=0.75, sub_mean=True, avg_mode=2, avg_depth=4, avg_minbin=34,
                avg_maxbin=102, avg_band_only=True), 3600),
    "c3": ("multitaper N=4096 K'=8 (mtm_k=7) NW=4 50% ovl, 1 h @ 48 kHz",
           dict(n=4096, mode=1, overlap=0.5, sub_mean=True, mtm_w=4.0, mtm_kmax=7), 3600),
    "c4": ("periodogram N=16384 Hann 50% ovl, 3 h @ 48 kHz per GPU (24 h over 8 GPUs)",
           dict(n=16384, window_type=0, overlap=0.5, sub_mean=True), 3 * 3600),
    "c5": ("multitaper N=32768 K'=16 (mtm_k=15) NW=8 50% ovl, 1 h @ 48 kHz per GPU",
           dict(n=32768, mode=1, overlap=0.5, sub_mean=True, mtm_w=8.0, mtm_kmax=15), 3600),
    "odd": ("periodogram N=4096 Hann 90% ovl (hop 409: irregular geometry, general kernel), 20 min @ 48 kHz",
            dict(n=4096, window_type=0, overlap=0.9, sub_mean=True), 1200),
    "lmp": ("LMP detector (lmp.c) N=4096 rectangular 50% ovl, ring of 4 frames, 1 h @ 48 kHz",
            dict(n=4096, mode=3, overlap=0.5, sub_mean=True, lmp_av=4), 3600),
}
# the configurations of BASELINE.json measured inside the default run (compact block `configs` of the line)
CONFIG_BLOCK = ["c1", "c2", "c3", "c5", "lmp"]


# the roofline's peak: read + write bytes of a 4 GiB device-to-device copy over its CUDA-event time, measured on
# one NVIDIA B200 at a 1000 W power limit (three runs of 20 copies: 6659-6662 GB/s)
HBM_PEAK_GBS = 6660.0
HBM_PEAK_SOURCE = "measured: 4 GiB device-to-device copy on one B200 at a 1000 W power limit"


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None
        self.th = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.th = threading.Thread(target=self._read, daemon=True)
        self.th.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "nvidia-smi unavailable"}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [c.strip() for c in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                smax.append(float(f[1]))
                pw.append(float(f[2]))
            except ValueError:
                continue
            for nme, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nme)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "no samples"}
        # "under load": samples in the upper half of the observed power range
        thr = (max(pw) + min(pw)) / 2 if pw else 0
        load = [s for s, p in zip(sm, pw) if p >= thr] or sm
        return {"sm_mhz": float(np.median(load)), "sm_max_mhz": float(max(smax)), "reasons": sorted(reasons),
                "samples": len(sm), "power_w_max": max(pw) if pw else None}


# ----------------------------------------------------------------------------- reference arm
def _ref_worker(args):
    kind, kw, nsamp, reps, seed, libkind = args
    sys.path.insert(0, ROOT)
    from glfer_b200 import synth
    x = synth.tiled_stream(nsamp, fs=FS, block_s=20.0, seed=seed)
    frames = 0
    t = 0.0
    if kind == "reference":
        from oracle import ref_lib as R
        for _ in range(reps):
            if kw.get("mode", 0) == 1:
                dt, nf = R.time_mtm(x, kw["n"], kw["overlap"], kw["mtm_w"], kw["mtm_kmax"], kw.get("sub_mean", True), kind=libkind)
            elif kw.get("mode", 0) == 3:
                t0 = time.perf_counter()
                nf = R.lmp(x, kw["n"], kw["overlap"], kw["lmp_av"], kw.get("sub_mean", True), kind=libkind).shape[0]
                dt = time.perf_counter() - t0
            else:
                dt, nf = R.time_periodogram(x, kw["n"], kw["window_type"], kw["overlap"], kw.get("sub_mean", True), kind=libkind)
            t += dt
            frames += nf
    else:
        from oracle import glfer_oracle as O
        for _ in range(reps):
            t0 = time.perf_counter()
            if kw.get("mode", 0) == 1:
                rows = O.multitaper(x, kw["n"], kw["overlap"], kw["mtm_w"], kw["mtm_kmax"], kw.get("sub_mean", True))
            elif kw.get("mode", 0) == 3:
                rows = O.lmp(x, kw["n"], kw["overlap"], kw["lmp_av"], kw.get("sub_mean", True))
            else:
                rows = O.periodogram(x, kw["n"], kw["window_type"], kw["overlap"], kw.get("sub_mean", True))
            t += time.perf_counter() - t0
            frames += rows.shape[0]
    return frames, t


def cpu_reference_rate(kw, target_s=6.0, cores=None, libkind="f32"):
    """frames/s of the reference's own C implementation with one process per host core
    (mtm.c keeps file-static state, so processes, not threads), each timing the reference
    loop `fft_do; fft_psd` / `mtm_do` over its own copy of a bounded sample.
    libkind: "f32" = gcc -O2 (the autoconf default), "f32_o3" = -O3 -march=x86-64-v3."""
    from oracle import ref_lib as R
    kind = "reference" if R.available(libkind) else "port"
    cores = cores or len(os.sched_getaffinity(0))
    hop = int(kw["n"] * (1.0 - kw["overlap"]))
    # per-core sample: ~2 s of single-core work per repetition at the survey's probe rates
    probe = {1024: 7e4, 4096: 1.7e4, 16384: 2e3, 32768: 9e2}.get(kw["n"], 1e4)
    if kw.get("mode", 0) == 1:
        probe /= 1.6 * (kw["mtm_kmax"] + 2)
    if kind == "port":
        probe *= 0.5
    # bounded per-core buffer (<= 4096 frames), repeated until ~target_s of work per core
    frames_per_rep = max(16, min(int(probe * 2.0), 4096))
    nsamp = frames_per_rep * hop
    reps = max(1, int(round(target_s * probe / frames_per_rep)))
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        t0 = time.perf_counter()
        res = pool.map(_ref_worker, [(kind, kw, nsamp, reps, 100 + i, libkind) for i in range(cores)])
        wall = time.perf_counter() - t0
    frames = sum(r[0] for r in res)
    tmax = max(r[1] for r in res)
    build = {"f32": "gcc -O2", "f32_o3": "gcc -O3 -march=x86-64-v3 (built off-box: -march=native of the build container would not be portable to this host)"}.get(libkind, libkind)
    code = (f"reference float radix-2 build ({build}), fft_do+fft_psd loop" if kind == "reference"
            else "numpy restatement (oracle/glfer_oracle.py): the reference's C build, oracle/_ref, is not present")
    return {"value": frames / tmax, "unit": "frames/s", "cores": cores, "kind": kind,
            "sample": f"{reps} x {frames_per_rep} frames ({nsamp / FS:.0f} s of signal) per core, {cores} core(s) concurrently; "
                      f"{code}; wall {wall:.1f} s",
            "frames": frames, "seconds": tmax}


# ----------------------------------------------------------------------------- main
def pin_to_gpu_numa_node(local_rank: int):
    """Run this process (and place the pinned host buffers it allocates next) on the CPUs of the
    NUMA node the GPU hangs off: with several ranks per box the end-to-end copies otherwise cross
    the socket interconnect.  Returns the previous affinity (restored for the CPU baseline leg)."""
    old = os.sched_getaffinity(0)
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        pr = torch.cuda.get_device_properties(local_rank)
        bus = "%08x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1} & old
        if cpus:
            os.sched_setaffinity(0, cpus)
    except Exception as e:      # no NVML, no topology information: leave the affinity alone
        sys.stderr.write(f"bench.py: NUMA pinning skipped ({e})\n")
    return old


def emit(line: dict) -> None:
    """The one JSON line of the contract, on the real stdout."""
    os.write(_STDOUT_FD, (json.dumps(line) + "\n").encode())


DUMP_BYTES = 64 * 10**6 - 4096         # 64 MB in all, the .npy headers included


def dump_outputs(res: dict, out_dir: str) -> None:
    """Writes the arrays the timed path hands its caller (GramPlan.fetch) as out_dir/<name>.npy in float32 or
    float64, so that two builds can be compared output for output.  When they exceed DUMP_BYTES, every array
    keeps the same frames: a sample drawn with a fixed seed, in frame order."""
    arrays = {k: v if v.dtype in (np.float32, np.float64) else v.astype(np.float64) for k, v in res.items() if v is not None}
    nf = next(iter(arrays.values())).shape[0]
    per_frame = sum(a.nbytes for a in arrays.values()) // max(nf, 1)
    keep = DUMP_BYTES // max(per_frame, 1)
    if nf > keep:
        idx = np.sort(np.random.default_rng(0).choice(nf, keep, replace=False))
        arrays = {k: a[idx] for k, a in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), np.ascontiguousarray(a))


def hop_of(kw):
    return int(kw["n"] * (1.0 - kw["overlap"]))


def roofline_of(kw, nf, gram_s, peak):
    """algorithmic bytes (hop*4 + (N/2+1)*4 per frame, SURVEY 8d) and 5 N log2 N flops per taper over the
    spectrogram kernel's own device time"""
    n, hop, bins = kw["n"], hop_of(kw), kw["n"] // 2 + 1
    ntap = kw["mtm_kmax"] + 1 if kw.get("mode", 0) == 1 else 1
    alg = nf * (hop * 4 + bins * 4)
    fl = nf * ntap * 5 * n * np.log2(n)
    return {"kernel_ms": 1e3 * gram_s, "hbm_gbs": alg / gram_s / 1e9, "frac": alg / gram_s / 1e9 / peak,
            "fp32_tflops_5nlogn": fl / gram_s / 1e12, "algorithmic_bytes_per_launch": int(alg)}


def main():
    global _STDOUT_FD
    # stdout carries exactly one JSON line: anything a library prints there (NCCL's version banner
    # under torchrun, for one) is sent to stderr instead
    sys.stdout.flush()
    _STDOUT_FD = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="metric", choices=sorted(WORKLOADS))
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the `configs` block (the other BASELINE configurations)")
    ap.add_argument("--seconds", type=int, default=0, help="override the seconds of signal per rank")
    ap.add_argument("--kernel-pref", type=int, default=0, help="experiment: 0 auto, 1 general, 2 ring, 3 warp-per-frame, 4 two frames per thread")
    ap.add_argument("--no-submean", action="store_true", help="experiment: opt.autoscale = 0 (no block-mean removal)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (rank 0's shard; "
                         "a fixed, seeded sample of its frames when all of them would exceed 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    desc, kw, seconds = WORKLOADS[args.workload]
    kw = dict(kw)
    if args.no_submean:
        kw["sub_mean"] = False
    if args.seconds:
        seconds = args.seconds
    n = kw["n"]
    hop = hop_of(kw)
    bins = n // 2 + 1
    ntap = kw["mtm_kmax"] + 1 if kw.get("mode", 0) == 1 else 1
    config = {"workload": desc, "n": n, "hop": hop, "window": "Hann" if kw.get("window_type", 5) == 0 else kw.get("window_type"),
              "tapers": ntap, "sub_mean": bool(kw.get("sub_mean", True)), "sample_rate": FS,
              "seconds_per_gpu": seconds, "frames_per_gpu": seconds * FS // hop,
              "parallelism": f"time-sharded x{world}, (N-hop)-sample halo, no collective",
              "l2": "inputs and outputs each > 126 MB L2; no flush between steps"}

    if args.impl == "reference":
        # the reference's CPU implementation on this host; rank 0 alone works
        if rank != 0:
            return
        steps, warm = max(1, args.steps), max(0, args.warmup)
        vals = []
        base = None
        for i in range(warm + steps):
            base = cpu_reference_rate(kw, target_s=4.0)
            if i >= warm:
                vals.append(base)
        frames = sum(v["frames"] for v in vals)
        secs = sum(v["seconds"] for v in vals)
        v = frames / secs
        line = {"impl": "reference", "metric": "spectrogram_frames_per_sec", "value": v, "unit": "frames/s",
                "n_gpus": args.gpus, "steps": steps, "warmup": warm, "ms_per_step": 1e3 * secs / steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic QRSS/DFCW multi-tone + noise, 20 s block tiled", "config": config,
                "samples_per_sec": v * hop,
                "cpu_baseline": {"value": v, "unit": "frames/s", "cores": base["cores"], "kind": base["kind"],
                                 "sample": base["sample"]},
                "e2e": {"value": v, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        emit(line)
        return

    import torch
    import torch.distributed as dist
    from glfer_b200 import api, shard, synth

    if not torch.cuda.is_available() or api.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device (libglfer_b200 has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    affinity0 = pin_to_gpu_numa_node(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v: float) -> float:
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(v: float) -> float:
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    peak, peak_src = HBM_PEAK_GBS, HBM_PEAK_SOURCE

    # this rank's shard of the (world x seconds) recording
    nframes_total = world * seconds * FS // hop
    first, nf = shard.frame_range(nframes_total, world, rank)
    ring = kw.get("lmp_av", 0) if kw.get("mode", 0) == 3 else (kw.get("avg_depth", 0) if kw.get("avg_mode") else 0)
    lo, hi = shard.sample_span(n, hop, first, nf, sub_mean=kw.get("sub_mean", True), avg_depth=ring)
    nsamp = hi - lo
    x_host = api.pinned_empty((nsamp,), np.float32)
    x_host[:] = synth.tiled_stream(nsamp, fs=FS, block_s=20.0, seed=0x5EED + rank)
    if args.kernel_pref:
        api.set_kernel_preference(args.kernel_pref)
    plan = api.GramPlan(device=local_rank, **kw)
    plan.stage(x_host, origin=lo)
    plan.sync()

    # ---- device-resident timing -------------------------------------------------
    # the sampler runs from before the warm-up to the end of the end-to-end region (nvidia-smi
    # needs ~0.1 s to start); "under load" = samples in the upper half of the power range
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(max(3, args.warmup)):
        plan.exec(first, nf, timed=True)
    barrier()
    launches0 = api.kernel_launches()
    step_ms, gram_ms = [], []
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        step_ms.append(plan.exec(first, nf, timed=True))
        gram_ms.append(plan.last_gram_ms())
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = api.kernel_launches() - launches0
    family = api.last_kernel_family()
    if args.dump_outputs and rank == 0:
        dump_outputs(plan.fetch(nf), args.dump_outputs)
    dev_s = max_over_ranks(sum(step_ms) * 1e-3)
    gram_s = sum(gram_ms) * 1e-3 / len(gram_ms)
    value = world * nf * args.steps / dev_s          # all ranks do nf (+-1) frames per step

    # ---- end to end through the host-buffer API -----------------------------------
    e2e = None
    checksum = None
    pcm_host = None
    out_pinned = None
    if not args.no_e2e:
        # one pinned output buffer, re-viewed per configuration
        need = nf * bins * 4
        if not args.no_configs and args.workload == "metric":
            for cname in CONFIG_BLOCK:
                ck = WORKLOADS[cname][1]
                need = max(need, (nsamp // hop_of(ck)) * (ck["n"] // 2 + 1) * 4)
        out_pinned = api.pinned_empty((max(need, 1),), np.uint8)

        def out_view(rows, cols, dtype):
            nbytes = rows * cols * np.dtype(dtype).itemsize
            assert nbytes <= out_pinned.nbytes
            return out_pinned[:nbytes].view(dtype).reshape(rows, cols)

        rows_host = out_view(nf, bins, np.float32)
        out = {"psd": rows_host}
        avg_host = None
        if plan.avg:
            avg_host = api.pinned_empty((nf, plan.avg_cols), np.float32)
            out["avg"] = avg_host
        e2e_steps = max(3, min(args.steps, 8))

        def timed_e2e(fn):
            fn()                                            # warm-up (allocations)
            barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                fn()
            barrier()
            return max_over_ranks(time.perf_counter() - t0)

        e2e_s = timed_e2e(lambda: plan.run(x_host, origin=lo, first_frame=first, nframes=nf, out=out))
        d2h = rows_host.nbytes + (avg_host.nbytes if avg_host is not None else 0)
        e2e = {"value": world * nf * e2e_steps / e2e_s, "unit": "frames/s", "h2d_bytes_per_step": int(x_host.nbytes),
               "d2h_bytes_per_step": int(d2h), "steps": e2e_steps, "ms_per_step": 1e3 * e2e_s / e2e_steps,
               "api": "glfer_gram_run (pinned host buffers, float32 in, float32 rows out, 3-slot chunked pipeline)"}
        checksum = float(rows_host[:: max(1, nf // 97)].sum())
        # the copies alone, same bytes, same buffers' sizes, both directions at once on two streams: what the
        # host <-> device path of this box gives this many ranks, i.e. the ceiling of any end-to-end number
        try:
            hin = torch.empty(x_host.nbytes, dtype=torch.uint8, pin_memory=True)
            hout = torch.empty(d2h, dtype=torch.uint8, pin_memory=True)
            din = torch.empty(x_host.nbytes, dtype=torch.uint8, device="cuda")
            dout = torch.empty(d2h, dtype=torch.uint8, device="cuda")
            s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

            def copies():
                with torch.cuda.stream(s1):
                    din.copy_(hin, non_blocking=True)
                with torch.cuda.stream(s2):
                    hout.copy_(dout, non_blocking=True)
                s1.synchronize()
                s2.synchronize()
            copy_s = timed_e2e(copies)
            e2e["copy_only"] = {"ms_per_step": 1e3 * copy_s / e2e_steps,
                                "gbs_per_gpu_each_way": [x_host.nbytes * e2e_steps / copy_s / 1e9, d2h * e2e_steps / copy_s / 1e9],
                                "frames_per_s_ceiling": world * nf * e2e_steps / copy_s,
                                "note": "cudaMemcpyAsync H2D + D2H of the same byte counts, concurrently, all ranks at once"}
            e2e["fraction_of_copy_ceiling"] = copy_s / e2e_s
            del hin, hout, din, dout
        except Exception as ex:
            e2e["copy_only"] = {"note": f"not measured: {ex}"}
        # the same call with the recording as the 16-bit PCM a WAV file holds (glfer_gram_run_pcm16: the
        # int16 -> float conversion of wav_fmt.c:113 runs on the device, half the bytes go up);
        # reported beside the float32 figure, which stays the headline
        pcm_host = api.pinned_empty((nsamp,), np.int16)
        pcm_host[:] = np.rint(x_host * 32768.0).astype(np.int16)
        pcm_s = timed_e2e(lambda: plan.run(pcm_host, origin=lo, first_frame=first, nframes=nf, out=out))
        e2e["pcm16_input"] = {"value": world * nf * e2e_steps / pcm_s, "unit": "frames/s",
                              "h2d_bytes_per_step": int(pcm_host.nbytes), "d2h_bytes_per_step": int(d2h),
                              "ms_per_step": 1e3 * pcm_s / e2e_steps, "api": "glfer_gram_run_pcm16",
                              "rows_identical_to_float_input": bool(float(rows_host[:: max(1, nf // 97)].sum()) == checksum)}
        # the reference's real end-to-end product is the waterfall: 16-bit PCM of a WAV file in, 8-bit palette
        # indices out (main_window_draw, g_main.c:1186-1229, fixed display range = autoscale off).  The
        # spectrogram kernel writes the levels itself: 2 B/sample up, 1 B/bin down, no float row in HBM.
        if not plan.avg and kw.get("mode", 0) != 3:
            lev_host = out_view(nf, bins, np.uint8)
            disp = dict(log_scale=True, autoscale=False, max_level_db=-20.0, min_level_db=-80.0, thr_level=0.0,
                        out={"levels": lev_host})
            u8_s = timed_e2e(lambda: plan.run_display(pcm_host, origin=lo, first_frame=first, nframes=nf, **disp))
            probe = lev_host[:: max(1, nf // 97)]
            e2e["pcm16_in_u8_out"] = {"value": world * nf * e2e_steps / u8_s, "unit": "frames/s",
                                      "h2d_bytes_per_step": int(pcm_host.nbytes), "d2h_bytes_per_step": int(lev_host.nbytes),
                                      "ms_per_step": 1e3 * u8_s / e2e_steps,
                                      "api": "glfer_gram_run_display_pcm16, fixed display range (levels written by the spectrogram kernel)",
                                      "levels_nonconstant": bool(probe.min() < probe.max())}
            # autoscale (glfer's default): float rows stay in HBM, floor statistics -> AGC recurrence -> levels
            disp["autoscale"] = True
            # (the per-frame display range comes back too: the library stages it through pinned memory)
            au_s = timed_e2e(lambda: plan.run_display(pcm_host, origin=lo, first_frame=first, nframes=nf, **disp))
            e2e["pcm16_in_u8_out_autoscale"] = {"value": world * nf * e2e_steps / au_s, "unit": "frames/s",
                                                "ms_per_step": 1e3 * au_s / e2e_steps,
                                                "api": "glfer_gram_run_display_pcm16, autoscale (compute_floor + AGC + levels on the device)"}

    # ---- the other BASELINE configurations, same process, few steps each ---------------------------
    configs = {}
    if not args.no_configs and args.workload == "metric":
        cfg_steps = 10

        def run_config(name, ckw, cx, corigin, cfirst, cnf, strong_total=None, with_e2e=True):
            p = api.GramPlan(device=local_rank, **ckw)
            p.stage(cx, origin=corigin)
            p.sync()
            for _ in range(3):
                p.exec(cfirst, cnf, timed=True)
            barrier()
            sm, gm = [], []
            for _ in range(cfg_steps):
                sm.append(p.exec(cfirst, cnf, timed=True))
                gm.append(p.last_gram_ms())
            barrier()
            ds = max_over_ranks(sum(sm) * 1e-3)
            gs = max_over_ranks(sum(gm) * 1e-3 / len(gm))
            total = strong_total if strong_total is not None else sum_over_ranks(float(cnf))
            r = {"workload": WORKLOADS[name][0] if name in WORKLOADS else name, "frames_per_step_all_gpus": int(total),
                 "value": total * cfg_steps / ds, "unit": "frames/s", "ms_per_step": 1e3 * ds / cfg_steps,
                 "kernel": api.last_kernel_family(), "steps": cfg_steps}
            r.update(roofline_of(ckw, cnf, gs, peak))
            r["post_kernels_ms"] = max(0.0, r["ms_per_step"] - r["kernel_ms"])
            if with_e2e and out_pinned is not None and cx is x_host:
                o = {"psd": out_view(cnf, p.bins, np.float32)}
                if p.avg:
                    o["avg"] = api.pinned_empty((cnf, p.avg_cols), np.float32)
                p.run(cx, origin=corigin, first_frame=cfirst, nframes=cnf, out=o)
                barrier()
                t0 = time.perf_counter()
                for _ in range(2):
                    p.run(cx, origin=corigin, first_frame=cfirst, nframes=cnf, out=o)
                barrier()
                es = max_over_ranks(time.perf_counter() - t0)
                r["e2e"] = {"value": total * 2 / es, "unit": "frames/s", "ms_per_step": 1e3 * es / 2,
                            "h2d_bytes_per_step": int(cx.nbytes), "d2h_bytes_per_step": int(o["psd"].nbytes + (o["avg"].nbytes if p.avg else 0))}
            p.close()
            return r

        for name in CONFIG_BLOCK:
            cdesc, ckw, csec = WORKLOADS[name]
            ckw = dict(ckw)
            ch = hop_of(ckw)
            # every rank treats its hour of samples as a recording of its own (weak scaling): frames [0, nf)
            cnf = min(len(x_host), csec * FS) // ch
            try:
                configs[name] = run_config(name, ckw, x_host, 0, 0, cnf)
                configs[name]["scaling"] = "weak (one 1-hour recording per GPU)"
            except Exception as ex:
                if world > 1:
                    raise                    # the ranks must not drift apart around the collectives
                configs[name] = {"error": str(ex)}
        # C4: ONE 24-hour 48 kHz recording, N=16384 Hann 50 %, time-sharded over the ranks (STRONG scaling:
        # 506 250 frames in total whatever the number of GPUs), each shard staged at its true 24-hour offset
        try:
            c4kw = dict(WORKLOADS["c4"][1])
            h4 = hop_of(c4kw)
            total4 = 24 * 3600 * FS // h4
            f4, n4 = shard.frame_range(total4, world, rank)
            lo4, hi4 = shard.sample_span(c4kw["n"], h4, f4, n4, sub_mean=True)
            t0 = time.perf_counter()
            x4 = synth.tiled_stream(hi4 - lo4, fs=FS, block_s=20.0, seed=0xC4 + rank)
            gen_s = time.perf_counter() - t0
            r4 = run_config("c4", c4kw, x4, lo4, f4, n4, strong_total=float(total4), with_e2e=False)
            r4["workload"] = "periodogram N=16384 Hann 50% ovl, ONE 24 h @ 48 kHz recording (506 250 frames) time-sharded over all GPUs"
            r4["scaling"] = "strong"
            r4["frames_this_rank"] = int(n4)
            r4["first_sample_this_rank"] = int(lo4)
            r4["host_synthesis_s"] = gen_s
            r4["samples_per_sec"] = r4["value"] * h4
            configs["c4_24h"] = r4
            del x4
        except Exception as ex:
            if world > 1:
                raise
            configs["c4_24h"] = {"error": str(ex)}

    clocks = sampler.stop()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    traffic = None          # DRAM read+write bytes of the kernel per launch, from the committed ncu capture
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            tj = json.load(fh)
        if tj.get("workload") == args.workload and not args.seconds:
            traffic = tj["traffic_bytes_per_launch"]
    except Exception:
        pass
    alg_bytes = nf * (hop * 4 + bins * 4)
    achieved = alg_bytes / gram_s / 1e9
    line = {"metric": "spectrogram_frames_per_sec", "value": value, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": 1e3 * dev_s / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic QRSS/DFCW multi-tone + noise (int16-quantised, /32768), 20 s block tiled to length",
            "config": config, "samples_per_sec": value * hop,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic,
                         "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one ncu --set full capture of this kernel, "
                                           "committed as profiles/traffic.json (not re-measured in this run)",
                         "peak_source": peak_src, "kernel": family,
                         "kernel_ms": 1e3 * gram_s,
                         # kernels after the spectrogram kernel in a step (frame averaging, LMP statistic): not in `achieved`
                         "post_kernels_ms": max(0.0, 1e3 * dev_s / args.steps - 1e3 * gram_s),
                         "algorithmic_bytes_per_launch": alg_bytes,
                         "fp32_flops_per_launch": nf * ntap * 5 * n * int(np.log2(n)),
                         "fp32_tflops_5nlogn": nf * ntap * 5 * n * np.log2(n) / gram_s / 1e12},
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks, "wall_s_timed_region": t_wall,
            "checksum": checksum}
    if configs:
        line["configs"] = configs
    if not args.no_cpu and world == 1:
        os.sched_setaffinity(0, affinity0)           # the baselines use every core of the box
        try:
            line["per_call"] = per_call_leg(api)
        except Exception as e:
            line["per_call"] = {"error": str(e)}
        try:
            cb = cpu_reference_rate(kw, target_s=6.0)
            line["cpu_baseline"] = {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample")}
            one = cpu_reference_rate(kw, target_s=2.0, cores=1)
            line["cpu_baseline"]["single_thread"] = {"value": one["value"], "unit": "frames/s", "sample": one["sample"]}
            from oracle import ref_lib as R
            if R.available("f32_o3"):
                o3 = cpu_reference_rate(kw, target_s=3.0, libkind="f32_o3")
                line["cpu_baseline"]["o3"] = {"value": o3["value"], "unit": "frames/s", "cores": o3["cores"], "sample": o3["sample"]}
        except Exception as e:  # the GPU line must not be lost to a baseline problem
            line.setdefault("cpu_baseline", {"value": None, "unit": "frames/s", "cores": 0, "kind": "reference", "sample": f"failed: {e}"})
    emit(line)
    if world > 1:
        dist.destroy_process_group()


def per_call_leg(api):
    """Latency of the reference's per-hop-block interface on the GPU engine next to the reference C code on
    one host core: microseconds per `fft_do; fft_psd` (and per `mtm_do`) call, one frame per call as
    audio_available() drives it (source.c:130-165)."""
    import ctypes as C
    lib = api.lib()
    res = {}
    rng = np.random.default_rng(1)
    from oracle import ref_lib as R
    for n in (1024, 4096):
        hop = n // 2
        blocks = (rng.standard_normal((300, hop)) * 0.05).astype(np.float32)
        p = api.FftParams()
        p.n, p.window_type, p.overlap, p.a, p.limiter = n, 0, 0.5, 0.0, 0
        lib.glfer_b200_set_autoscale(1)
        lib.glfer_b200_set_first_buffer(1)
        lib.fft_init(C.byref(p))
        psd = np.empty(n // 2 + 1, dtype=np.float32)
        blk = np.empty(hop, dtype=np.float32)
        for i in range(300):
            if i == 100:
                t0 = time.perf_counter()
            blk[:] = blocks[i]
            lib.fft_do(blk.ctypes.data, C.byref(p))
            lib.fft_psd(psd.ctypes.data, None, C.byref(p))
            lib.glfer_b200_set_first_buffer(0)
        us = (time.perf_counter() - t0) / 200 * 1e6
        lib.fft_close(C.byref(p))
        entry = {"gpu_us_per_fft_do_fft_psd": us}
        if R.available("f32"):
            dt, nfr = R.time_periodogram(blocks.reshape(-1), n, 0, 0.5, True)
            entry["reference_cpu_us_per_call_one_core"] = dt / nfr * 1e6
        # the k-block entry of the same interface: 64 hop blocks per call, same sequence semantics
        p = api.FftParams()
        p.n, p.window_type, p.overlap, p.a, p.limiter = n, 0, 0.5, 0.0, 0
        lib.glfer_b200_set_first_buffer(1)
        lib.fft_init(C.byref(p))
        k = 64
        rows = np.empty((k, n // 2 + 1), dtype=np.float32)
        chunk = np.empty((k, hop), dtype=np.float32)
        for i in range(4):
            if i == 1:
                t0 = time.perf_counter()
            chunk[:] = blocks[i * k:(i + 1) * k]
            lib.fft_do_batch(chunk.ctypes.data, k, rows.ctypes.data, C.byref(p))
            lib.glfer_b200_set_first_buffer(0)
        entry["gpu_us_per_block_fft_do_batch_64"] = (time.perf_counter() - t0) / (3 * k) * 1e6
        lib.fft_close(C.byref(p))
        # mtm_do, K' = 8 tapers (NW = 4): one call per hop block
        m = api.MtmParams()
        m.fft.n, m.fft.window_type, m.fft.overlap = n, 5, 0.5
        m.w, m.kmax = 4.0, 7
        lib.glfer_b200_set_first_buffer(1)
        lib.mtm_init(C.byref(m))
        for i in range(150):
            if i == 50:
                t0 = time.perf_counter()
            blk[:] = blocks[i]
            lib.mtm_do(blk.ctypes.data, psd.ctypes.data, None, C.byref(m))
            lib.glfer_b200_set_first_buffer(0)
        entry["gpu_us_per_mtm_do_8_tapers"] = (time.perf_counter() - t0) / 100 * 1e6
        lib.mtm_close(C.byref(m))
        if R.available("f32"):
            dt, nfr = R.time_mtm(blocks[:60].reshape(-1), n, 0.5, 4.0, 7, True)
            entry["reference_cpu_us_per_mtm_do_one_core"] = dt / nfr * 1e6
        res[f"n{n}"] = entry
    res["note"] = "one frame per call is launch-latency bound; fft_do_batch / mtm_do_batch take k hop blocks per call (INTEGRATION.md)"
    return res


if __name__ == "__main__":
    main()
