"""I/Q spectrogram and I/Q zoom on one hour of synth.iq_stream at 48 kHz (172.8 M complex samples, 1.38 GB as
float: larger than L2).

  * fused I/Q kernel (gram_iq_kernel) against the real ring kernel (gram_ring_kernel) at N = 2n, hop 2h, the same
    window, block means off, over the same floats on the device, n = 2048 and 4096 at 50 %: the two alternate in
    one process, device times from torch.profiler; bytes/s against bench.py's 6660 GB/s roofline constant;
  * the general path (gram_kernel spectrum + zoom_split_kernel) at the same shapes, and at 60 % overlap, where the
    I/Q plan always takes it;
  * the complex decimator beside the real one at D = 16 / 256 / 1024 on the same sample count;
  * end to end IqPlan.run for float and int16 I/Q with pinned buffers (median of 5, profiler off), and the H2D /
    D2H copy totals of one profiled run.
The GPU name and power limit are read in the same call.

usage: python tools/scripts/iq_bench.py [--out FILE.json] [--seconds S] [--reps R]"""
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
ROOFLINE_GBS = 6660.0                  # bench.py: read+write bandwidth of a 4 GiB device copy, B200 at 1000 W


class IqGramArgs(C.Structure):         # include/glb_shim.h glb_iq_gram_args
    _fields_ = [("n", C.c_int), ("hop", C.c_int), ("samples", C.c_void_p), ("origin", C.c_longlong),
                ("count", C.c_longlong), ("taper", C.c_void_p), ("taper_symmetric", C.c_int), ("taper_scale", C.c_float),
                ("first_frame", C.c_longlong), ("nframes", C.c_longlong), ("rows", C.c_void_p), ("tables", C.c_void_p),
                ("scratch", C.c_void_p), ("levels", C.c_void_p), ("levels_stride", C.c_longlong),
                ("level_tables", C.c_void_p), ("levels_log", C.c_int), ("level_lut", C.c_void_p), ("level_min", C.c_float),
                ("level_max", C.c_float), ("level_thr", C.c_float), ("ntapers", C.c_int),
                ("ftest", C.c_void_p), ("ftest_taper", C.c_void_p), ("ftest_u0", C.c_void_p), ("ftest_s", C.c_float)]


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unavailable"


def profile_ms(fn, keys):
    """device time per kernel-name substring (first match wins) of one call of fn under torch.profiler"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    t = {k: 0.0 for k in keys}
    for ev in prof.events():
        if ev.device_type is None or str(ev.device_type).split(".")[-1] != "CUDA":
            continue
        ms = ev.device_time_total / 1e3 if hasattr(ev, "device_time_total") else ev.cuda_time_total / 1e3
        for k in keys:
            if k in ev.name:
                t[k] += ms
                break
    return t


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--seconds", type=float, default=3600.0)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if api.device_count() < 1:
        raise SystemExit("iq_bench needs a CUDA device")
    L = api.lib()
    L.glb_launch_iq_gram.argtypes = [C.POINTER(IqGramArgs), C.c_void_p]
    L.glb_iq_gram_scratch_bytes.argtypes = [C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_int, C.c_int]
    L.glb_iq_gram_scratch_bytes.restype = C.c_longlong
    L.glb_tables_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    L.glb_tables_destroy.argtypes = [C.c_void_p]
    decim_args = [C.c_void_p, C.c_int, C.c_longlong, C.c_longlong, C.c_int, C.c_void_p, C.c_uint, C.c_longlong,
                  C.c_longlong, C.c_void_p, C.c_void_p]
    L.glb_launch_zoom_decim.argtypes = decim_args
    L.glb_launch_zoom_decim_iq.argtypes = decim_args

    ns = int(a.seconds * FS)
    blk = synth.iq_stream_int16(20 * FS, fs=FS, dot_s=1.0)
    pcm = api.pinned_empty((ns, 2), np.int16)
    for i in range(0, ns, len(blk)):
        pcm[i:i + len(blk)] = blk[:ns - i]
    zf = api.pinned_empty((ns, 2), np.float32)
    zf[:] = synth.pcm16_to_float(pcm)
    res = dict(gpu=gpu_info(), data=f"synth.iq_stream_int16 (20 s tiled), {a.seconds:g} s at {FS} Hz ({ns} complex samples)",
               window="hann", roofline_gbs=ROOFLINE_GBS, kernels=[], general=[], decimator=[], e2e=[])
    dev = torch.from_numpy(zf).cuda()                              # the one float buffer both kernels read
    st = torch.cuda.current_stream().cuda_stream

    def iq_launch(n, hop, rows, taper, tables, scratch):
        nf = ns // hop
        g = IqGramArgs(n, hop, dev.data_ptr(), 0, ns, taper.data_ptr(), 1, float(np.float32(1.0 / (2.0 * np.sqrt(2.0 * n)))),
                       0, nf, rows.data_ptr(), tables, scratch)
        api._check(L.glb_launch_iq_gram(C.byref(g), st))

    for n in (2048, 4096):
        hop = n // 2
        nf = ns // hop
        w = api.host_window(n, api.HANNING).astype(np.float64)
        ts = np.float32(1.0 / (2.0 * np.sqrt(2.0 * n)))
        taper = torch.from_numpy(np.repeat((w * float(ts)).astype(np.float32), 2)).cuda()
        tables = C.c_void_p()
        api._check(L.glb_tables_create(2 * n, C.byref(tables)))
        rows = torch.empty((nf, n), dtype=torch.float32, device="cuda")
        real = api.GramPlan(n=2 * n, window_type=api.HANNING, overlap=0.5, sub_mean=False)
        real.stage(zf.reshape(-1))
        assert real.num_frames(2 * ns) == nf
        fi = lambda: iq_launch(n, hop, rows, taper, tables, None)                # noqa: E731
        fr = lambda: real.exec(0, nf)                                            # noqa: E731
        fi(); fr(); torch.cuda.synchronize()
        ti, tr = [], []
        for _ in range(a.reps):
            ti.append(profile_ms(fi, ["gram_iq_kernel"])["gram_iq_kernel"])
            tr.append(profile_ms(fr, ["gram_ring_kernel", "gram_"])["gram_ring_kernel"])
        real.sync()
        bytes_moved = 8.0 * ns + 4.0 * nf * n                               # samples once + rows
        r = dict(n=n, overlap=0.5, frames=nf, iq_kernel_ms=float(np.median(ti)), iq_kernel_ms_all=ti,
                 real_ring_kernel_ms=float(np.median(tr)), real_ring_kernel_ms_all=tr, bytes=bytes_moved)
        r["ratio_iq_over_real"] = r["iq_kernel_ms"] / r["real_ring_kernel_ms"]
        r["iq_gbs"] = bytes_moved / (r["iq_kernel_ms"] * 1e-3) / 1e9
        r["iq_share_of_roofline"] = r["iq_gbs"] / ROOFLINE_GBS
        res["kernels"].append(r)
        print(json.dumps(r), flush=True)
        real.close()
        # general path at the same shape, and the I/Q plan's geometry at 60 % overlap
        for ov in (0.5, 0.6):
            h2 = api.host_hop(n, ov)
            nf2 = ns // h2
            rows2 = torch.empty((nf2, n), dtype=torch.float32, device="cuda") if ov != 0.5 else rows
            api.force_generic_kernel(ov == 0.5)
            try:
                sb = L.glb_iq_gram_scratch_bytes(n, h2, nf2, 0, 1, 0)
                scratch = torch.empty(sb, dtype=torch.uint8, device="cuda")
                fg = lambda: iq_launch(n, h2, rows2, taper, tables, scratch.data_ptr())   # noqa: E731
                fg(); torch.cuda.synchronize()
                tg = [profile_ms(fg, ["gram_kernel", "zoom_split_kernel"]) for _ in range(3)]
            finally:
                api.force_generic_kernel(False)
            g = dict(n=n, overlap=ov, hop=h2, frames=nf2, gram_kernel_ms=float(np.median([t["gram_kernel"] for t in tg])),
                     split_kernel_ms=float(np.median([t["zoom_split_kernel"] for t in tg])))
            g["total_ms"] = g["gram_kernel_ms"] + g["split_kernel_ms"]
            res["general"].append(g)
            print(json.dumps(g), flush=True)
            del scratch, rows2
        del rows, taper
        L.glb_tables_destroy(tables)
        torch.cuda.empty_cache()

    # decimators on the same sample count: real x = I, complex z = (I, Q)
    devr = dev[:, 0].contiguous()
    pcm_dev = torch.from_numpy(pcm).cuda()
    for d in (16, 256, 1024):
        taps = torch.zeros(2 * 33 * d, dtype=torch.float32, device="cuda")
        taps_np = np.zeros(32 * d + 1, np.float32)
        api._check(L.glfer_zoom_taps(d, taps_np.ctypes.data))
        taps[0:2 * (32 * d + 1):2] = torch.from_numpy(taps_np).cuda()
        md = (ns - 1 - 16 * d) // d + 1
        y = torch.empty(2 * md, dtype=torch.float32, device="cuda")
        step = (d * round(800.0 / FS * 2 ** 32)) % (1 << 32)
        fr = lambda: api._check(L.glb_launch_zoom_decim(devr.data_ptr(), 0, 0, ns, d, taps.data_ptr(), step, 0, md, y.data_ptr(), st))  # noqa
        fc = lambda: api._check(L.glb_launch_zoom_decim_iq(dev.data_ptr(), 0, 0, ns, d, taps.data_ptr(), step, 0, md, y.data_ptr(), st))  # noqa
        fs16 = lambda: api._check(L.glb_launch_zoom_decim_iq(pcm_dev.data_ptr(), 1, 0, ns, d, taps.data_ptr(), step, 0, md, y.data_ptr(), st))  # noqa
        fr(); fc(); fs16(); torch.cuda.synchronize()
        tr, tc, t16 = [], [], []
        for _ in range(3):
            tr.append(profile_ms(fr, ["zoom_decim_kernel"])["zoom_decim_kernel"])
            tc.append(profile_ms(fc, ["zoom_decim_kernel"])["zoom_decim_kernel"])
            t16.append(profile_ms(fs16, ["zoom_decim_kernel"])["zoom_decim_kernel"])
        r = dict(decim=d, outputs=md, real_ms=float(np.median(tr)), iq_float_ms=float(np.median(tc)),
                 iq_int16_ms=float(np.median(t16)))
        r["ratio_iq_over_real"] = r["iq_float_ms"] / r["real_ms"]
        r["iq_tflops"] = 8.0 * (32 * d + 1) * md / (r["iq_float_ms"] * 1e-3) / 1e12
        res["decimator"].append(r)
        print(json.dumps(r), flush=True)
    del dev, devr, pcm_dev
    torch.cuda.empty_cache()

    # end to end, pinned buffers
    for n in (2048, 4096):
        p = api.IqPlan(n=n, window_type=api.HANNING, overlap=0.5)
        nf = p.num_frames(ns)
        rows = api.pinned_empty((nf, n), np.float32)
        r = dict(n=n, overlap=0.5, frames=nf, input_float_bytes=8.0 * ns, rows_bytes=4.0 * nf * n)
        for name, src in (("float", zf), ("int16", pcm)):
            p.run(src, out=rows)
            ts = []
            for _ in range(5):
                t0 = time.perf_counter()
                p.run(src, out=rows)
                ts.append(time.perf_counter() - t0)
            r[f"{name}_e2e_ms"] = 1e3 * float(np.median(ts))
            r[f"{name}_e2e_min_ms"] = 1e3 * float(min(ts))
            pt = profile_ms(lambda: p.run(src, out=rows), ["HtoD", "DtoH", "gram_iq_kernel", "pcm16"])
            r[f"{name}_h2d_ms"], r[f"{name}_d2h_ms"] = pt["HtoD"], pt["DtoH"]
            r[f"{name}_kernel_ms"], r[f"{name}_convert_ms"] = pt["gram_iq_kernel"], pt["pcm16"]
            r[f"{name}_e2e_over_max_copy"] = r[f"{name}_e2e_ms"] / max(pt["HtoD"], pt["DtoH"])
        res["e2e"].append(r)
        print(json.dumps(r), flush=True)
        p.close()
    res["gpu_after"] = gpu_info()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(res, fh, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k in ("gpu", "gpu_after", "data")}))


if __name__ == "__main__":
    main()
