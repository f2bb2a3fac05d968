"""Zoom channel banks on one hour of 48 kHz input: the bank decimator against one zoom_decim_kernel launch per channel,
and a C = 8 bank end to end against eight single-centre plans and against the upload of the input alone.

Kernel A/B (CUDA events, one process, alternated): for real / I/Q x float / int16 input on the device, C launches of
zoom_decim_kernel (glb_launch_zoom_decim[_iq]) against one zoom_bank_decim_kernel launch (glb_launch_zoom_bank_decim)
over every decimated output of the hour, at D = 256 with C = 1, 2, 8, 32 and at D = 16, 1024 with C = 1, 8; median of
the repetitions, the bank's outputs compared bit for bit with the single launches'.  FP32 rate from the FMAs the
polyphase sum needs (33 D taps per output: 2 FMAs per tap real, 4 complex), and the share of the derived floor
(that count at 74 TFLOP/s FP32).  The input (0.35 to 1.4 GB) is larger than L2.

End to end (profiler off, pinned buffers, median of 5, bank / singles / upload alternated): C = 8, D = 256, n = 4096,
Hann, 50 %, rows from real and I/Q float and int16 input, and multitaper K' = 8 rows; the upload is one host-to-device
copy of the same pinned input.  Kernel times of one bank run per case come from torch.profiler in a run of their own.
The GPU name and power limit are read in the same call.

usage: python tools/scripts/zoom_bank_bench.py [--out FILE.json] [--seconds S] [--reps R]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from glfer_b200 import api, synth      # noqa: E402

FS = 48000
FP32_TFLOPS = 74.0          # the derived floor's rate, as DESIGN section 7.2
FORMATS = [("real", "float"), ("real", "int16"), ("iq", "float"), ("iq", "int16")]
KERNEL_CASES = [(256, 1), (256, 2), (256, 8), (256, 32), (16, 1), (16, 8), (1024, 1), (1024, 8)]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unavailable"


def _shim():
    l = api.lib()
    l.glb_launch_zoom_decim.argtypes = [C.c_void_p, C.c_int, C.c_longlong, C.c_longlong, C.c_int, C.c_void_p, C.c_uint,
                                        C.c_longlong, C.c_longlong, C.c_void_p, C.c_void_p]
    l.glb_launch_zoom_decim_iq.argtypes = l.glb_launch_zoom_decim.argtypes
    l.glb_launch_zoom_bank_decim.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_longlong, C.c_longlong, C.c_int, C.c_int,
                                             C.c_void_p, C.POINTER(C.c_uint), C.c_longlong, C.c_longlong, C.c_void_p,
                                             C.c_longlong, C.c_void_p]
    return l


def _ok(rc):
    if rc != 0:
        raise RuntimeError(f"launch failed: {api.last_error()}")


def kernel_ab(l, torch, x_dev, iq, pcm16, ns, decim, nchan, reps):
    """median ms of nchan single launches and of one bank launch, alternated; outputs compared"""
    rng = np.random.default_rng(decim * 100 + nchan)
    taps = torch.from_numpy(rng.standard_normal((nchan, 66 * decim)).astype(np.float32) * 1e-3).cuda()
    steps = (rng.integers(0, 2 ** 32, size=nchan, dtype=np.uint64) * np.uint64(decim)) & np.uint64(0xFFFFFFFF)
    dstep = (C.c_uint * nchan)(*[int(s) for s in steps])
    md = (ns - 1 - 16 * decim) // decim + 1
    y1 = torch.empty((nchan, md, 2), dtype=torch.float32, device="cuda")
    yb = torch.empty((nchan, md, 2), dtype=torch.float32, device="cuda")
    single = l.glb_launch_zoom_decim_iq if iq else l.glb_launch_zoom_decim

    def run_single():
        for c in range(nchan):
            _ok(single(x_dev.data_ptr(), int(pcm16), 0, ns, decim, taps[c].data_ptr(), dstep[c], 0, md,
                       y1[c].data_ptr(), None))

    def run_bank():
        _ok(l.glb_launch_zoom_bank_decim(x_dev.data_ptr(), int(pcm16), int(iq), 0, ns, decim, nchan, taps.data_ptr(),
                                         dstep, 0, md, yb.data_ptr(), md, None))

    def timed(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        return a.elapsed_time(b)

    run_single(); run_bank(); torch.cuda.synchronize()
    ts, tb = [], []
    for r in range(reps):
        if r % 2 == 0:
            ts.append(timed(run_single)); tb.append(timed(run_bank))
        else:
            tb.append(timed(run_bank)); ts.append(timed(run_single))
    same = bool(torch.equal(y1, yb))
    fma = (4 if iq else 2) * 33 * decim * md * nchan
    bank_ms = float(np.median(tb))
    floor_ms = 2.0 * fma / (FP32_TFLOPS * 1e12) * 1e3
    return dict(decim=decim, channels=nchan, outputs_per_channel=md, single_launches_ms=float(np.median(ts)),
                single_spread_ms=[float(min(ts)), float(max(ts))], bank_ms=bank_ms,
                bank_spread_ms=[float(min(tb)), float(max(tb))], bank_over_singles=bank_ms / float(np.median(ts)),
                bank_tflops=2.0 * fma / (bank_ms * 1e-3) / 1e12, floor_ms=floor_ms, bank_share_of_floor=floor_ms / bank_ms,
                bit_identical=same)


def kernel_times(torch, fn):
    """device time per kernel family in one call of fn under torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    t = {"bank_decim_ms": 0.0, "single_decim_ms": 0.0, "frame_ms": 0.0, "h2d_ms": 0.0, "d2h_ms": 0.0, "other_ms": 0.0}
    names = set()
    for ev in prof.events():
        if ev.device_type is None or str(ev.device_type).split(".")[-1] != "CUDA":
            continue
        ms = ev.device_time_total / 1e3 if hasattr(ev, "device_time_total") else ev.cuda_time_total / 1e3
        nm = ev.name
        if "zoom_bank_decim_kernel" in nm:
            t["bank_decim_ms"] += ms
        elif "zoom_decim_kernel" in nm:
            t["single_decim_ms"] += ms
        elif "gram_kernel" in nm or "split_kernel" in nm or "ftest" in nm:
            t["frame_ms"] += ms
        elif "HtoD" in nm:
            t["h2d_ms"] += ms
        elif "DtoH" in nm:
            t["d2h_ms"] += ms
        else:
            t["other_ms"] += ms
        names.add(nm.split("(")[0])
    t["kernels"] = sorted(names)
    return t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--seconds", type=float, default=3600.0)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if api.device_count() < 1:
        raise SystemExit("zoom_bank_bench needs a CUDA device")
    import torch
    torch.zeros(1, device="cuda")
    l = _shim()
    ns = int(a.seconds * FS)
    res = dict(gpu=gpu_info(), data=f"{a.seconds:g} s at {FS} Hz ({ns} samples or complex samples)", kernel=[], e2e=[])

    # host inputs: real from synth.tiled_stream, I/Q a tiled complex stream of the same length
    xs = synth.tiled_stream(ns, fs=FS, block_s=20.0)
    host = {}
    host[("real", "float")] = api.pinned_empty((ns,), np.float32)
    host[("real", "float")][:] = xs
    host[("real", "int16")] = api.pinned_empty((ns,), np.int16)
    host[("real", "int16")][:] = np.clip(np.rint(xs * 32768.0), -32768, 32767).astype(np.int16)
    zq = np.roll(xs, 12345)
    host[("iq", "float")] = api.pinned_empty((ns, 2), np.float32)
    host[("iq", "float")][:, 0] = xs
    host[("iq", "float")][:, 1] = zq
    host[("iq", "int16")] = api.pinned_empty((ns, 2), np.int16)
    host[("iq", "int16")][:] = np.clip(np.rint(host[("iq", "float")] * 32768.0), -32768, 32767).astype(np.int16)
    del xs, zq

    # ---- kernel A/B
    for kind, fmt in FORMATS:
        iq, pcm16 = kind == "iq", fmt == "int16"
        x_dev = torch.from_numpy(host[(kind, fmt)]).cuda()
        for decim, nchan in KERNEL_CASES:
            r = dict(input=f"{kind} {fmt}", **kernel_ab(l, torch, x_dev, iq, pcm16, ns, decim, nchan, a.reps))
            res["kernel"].append(r)
            print(json.dumps(r), flush=True)
        del x_dev
        torch.cuda.empty_cache()

    # ---- end to end, C = 8, D = 256, n = 4096, Hann, 50 %
    centers_real = [600.0, 800.0, 1000.0, 1200.0, 3000.0, 5000.0, 7000.0, 9000.0]
    centers_iq = [-9000.0, -5000.0, -1200.0, -800.0, 800.0, 1200.0, 5000.0, 9000.0]
    cases = [(k, f, False) for k, f in FORMATS] + [("real", "float", True), ("iq", "int16", True)]
    for kind, fmt, mtm in cases:
        iq = kind == "iq"
        centers = centers_iq if iq else centers_real
        kw = dict(n=4096, decim=256, window_type=api.HANNING, overlap=0.5, sample_rate=FS, iq=iq, multitaper=mtm,
                  mtm_w=4.0, mtm_kmax=7)
        bank = api.ZoomPlan(center_hz=centers, **kw)
        singles = [api.ZoomPlan(center_hz=c, **kw) for c in centers]
        x = host[(kind, fmt)]
        nf = bank.num_frames(ns)
        rows = api.pinned_empty((8, nf, 4096), np.float32)
        d_in = torch.empty(x.nbytes, dtype=torch.uint8, device="cuda")
        src = torch.from_numpy(x.reshape(-1).view(np.uint8))

        def run_bank():
            bank.run(x, out=rows)

        def run_singles():
            for c, s in enumerate(singles):
                s.run(x, out=rows[c])

        def upload():
            d_in.copy_(src, non_blocking=True)
            torch.cuda.synchronize()

        fns = dict(bank=run_bank, singles=run_singles, upload=upload)
        for fn in fns.values():
            fn()
        t = {k: [] for k in fns}
        for r in range(5):
            order = list(fns) if r % 2 == 0 else list(fns)[::-1]
            for k in order:
                t0 = time.perf_counter()
                fns[k]()
                t[k].append(1e3 * (time.perf_counter() - t0))
        med = {k: float(np.median(v)) for k, v in t.items()}
        r = dict(input=f"{kind} {fmt}", estimator="multitaper K'=8" if mtm else "periodogram", channels=8, decim=256,
                 n=4096, frames=nf, input_bytes=int(x.nbytes), bank_ms=med["bank"], singles_ms=med["singles"],
                 upload_ms=med["upload"], bank_over_upload=med["bank"] / med["upload"],
                 singles_over_bank=med["singles"] / med["bank"],
                 spread_ms={k: [float(min(v)), float(max(v))] for k, v in t.items()},
                 bank_kernels=kernel_times(torch, run_bank))
        res["e2e"].append(r)
        print(json.dumps(r), flush=True)
        bank.close()
        for s in singles:
            s.close()
        del d_in, src, rows
        torch.cuda.empty_cache()
    res["gpu_after"] = gpu_info()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k not in ("kernel", "e2e")}))


if __name__ == "__main__":
    main()
