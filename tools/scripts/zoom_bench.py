"""Zoom spectrogram on one hour of synth.tiled_stream at 48 kHz, n = 4096 (Hann, 50 %), D = 16 / 256 / 1024.

Per D: device time of the decimator (zoom_decim_kernel) and of the frame stage (the general gram_kernel with its
spectrum output + zoom_split_kernel) from torch.profiler with CUDA activities in a run of its own; achieved FP32
FLOP/s of the decimator (4 L flop per decimated output, L = 32 D + 1 taps) and HBM bytes/s of the decimator
(input bytes + 8 B per decimated sample); end-to-end glfer_zoom_run time with pinned buffers for float and int16
input (profiler off, median of 5 after a warm-up).  The GPU name and power limit are read in the same call.

usage: python tools/scripts/zoom_bench.py [--out FILE.json] [--seconds S]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from glfer_b200 import api, synth      # noqa: E402

FS = 48000
N = 4096
DECIMS = (16, 256, 1024)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unavailable"


def kernel_times(plan, x, rows):
    """device time per kernel family in one run of glfer_zoom_run under torch.profiler"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.zeros(1, device="cuda")
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        plan.run(x, out=rows)
        torch.cuda.synchronize()
    t = {"decim_ms": 0.0, "frame_gram_ms": 0.0, "frame_split_ms": 0.0, "h2d_ms": 0.0, "d2h_ms": 0.0, "d2d_ms": 0.0}
    names = set()
    for ev in prof.events():
        if ev.device_type is None or str(ev.device_type).split(".")[-1] != "CUDA":
            continue
        ms = ev.device_time_total / 1e3 if hasattr(ev, "device_time_total") else ev.cuda_time_total / 1e3
        nm = ev.name
        if "zoom_decim_kernel" in nm:
            t["decim_ms"] += ms
        elif "zoom_split_kernel" in nm:
            t["frame_split_ms"] += ms
        elif "gram_kernel" in nm:
            t["frame_gram_ms"] += ms
        elif "HtoD" in nm:
            t["h2d_ms"] += ms
        elif "DtoH" in nm:
            t["d2h_ms"] += ms
        elif "DtoD" in nm:
            t["d2d_ms"] += ms
        else:
            continue
        names.add(nm.split("(")[0])
    t["kernels"] = sorted(names)
    return t


def e2e_ms(plan, x, rows, reps=5):
    plan.run(x, out=rows)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        plan.run(x, out=rows)            # returns after the last download has landed
        ts.append(time.perf_counter() - t0)
    return 1e3 * float(np.median(ts)), 1e3 * float(min(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--seconds", type=float, default=3600.0)
    a = ap.parse_args()
    if api.device_count() < 1:
        raise SystemExit("zoom_bench needs a CUDA device")
    ns = int(a.seconds * FS)
    xs = synth.tiled_stream(ns, fs=FS, block_s=20.0)
    x = api.pinned_empty((ns,), np.float32)
    x[:] = xs
    pcm = api.pinned_empty((ns,), np.int16)
    pcm[:] = np.clip(np.rint(xs * 32768.0), -32768, 32767).astype(np.int16)
    del xs
    res = dict(gpu=gpu_info(), data=f"synth.tiled_stream, {a.seconds:g} s at {FS} Hz ({ns} samples)",
               n=N, window="hann", overlap=0.5, center_hz=800.0, results=[])
    for d in DECIMS:
        p = api.ZoomPlan(n=N, decim=d, window_type=api.HANNING, overlap=0.5, center_hz=800.0, sample_rate=FS)
        nf = p.num_frames(ns)
        rows = api.pinned_empty((nf, N), np.float32)
        md = (ns - 1 - 16 * d) // d + 1
        taps = 32 * d + 1
        r = dict(decim=d, frames=nf, decimated_samples=md, resolution_hz=FS / (d * N))
        r["float_e2e_ms"], r["float_e2e_min_ms"] = e2e_ms(p, x, rows)
        r["int16_e2e_ms"], r["int16_e2e_min_ms"] = e2e_ms(p, pcm, rows)
        kt = kernel_times(p, x, rows)
        r.update(kt)
        flop = 4.0 * taps * md
        r["decim_flop"] = flop
        r["decim_tflops"] = flop / (kt["decim_ms"] * 1e-3) / 1e12 if kt["decim_ms"] > 0 else None
        dbytes = 4.0 * ns + 8.0 * md
        r["decim_hbm_gbs"] = dbytes / (kt["decim_ms"] * 1e-3) / 1e9 if kt["decim_ms"] > 0 else None
        allbytes = dbytes + 4.0 * nf * N
        r["bytes_in_plus_decimated_plus_rows"] = allbytes
        r["float_input_gbs_e2e"] = 4.0 * ns / (r["float_e2e_ms"] * 1e-3) / 1e9
        res["results"].append(r)
        print(json.dumps(r), flush=True)
        p.close()
    res["gpu_after"] = gpu_info()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "results"}))


if __name__ == "__main__":
    main()
