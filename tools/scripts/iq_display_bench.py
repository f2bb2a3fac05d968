"""Waterfall output of I/Q and zoom plans on one hour of synth.iq_stream at 48 kHz (172.8 M complex samples).

  * kernel: the level epilogue (gram_iq_kernel<.., LEV = true>, 1 byte per bin) against the float-row gram_iq_kernel,
    n = 2048 and 4096 at 50 %, over the same floats on the device, alternated in one process, device times from
    torch.profiler;
  * end to end, int16 input, pinned buffers, median of 5 with the profiler off: IqPlan.run (float rows, today's
    glfer_iq_run_pcm16) against run_display with a fixed range (fused levels) and with autoscale (rows stay on the
    device: floor statistics -> AGC -> levels); the H2D / D2H copy totals and kernel times of one profiled run each;
  * zoom, D = 256, n = 4096, 50 %: ZoomPlan.run on int16 against run_display with autoscale, the same way.
The GPU name and power limit are read in the same call.

usage: python tools/scripts/iq_display_bench.py [--out FILE.json] [--seconds S] [--reps R]"""
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
GLB_DB_JMIN, GLB_DB_NTHR = -450, 841   # host/glb_host.h


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
    """device time per name substring (first match wins) of one call of fn under torch.profiler"""
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


E2E_KEYS = ["HtoD", "DtoH", "gram_iq_kernel", "pcm16", "floor_stats", "agc_kernel", "levels_kernel", "zoom_decim",
            "gram_kernel", "zoom_split"]


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--seconds", type=float, default=3600.0)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if api.device_count() < 1:
        raise SystemExit("iq_display_bench needs a CUDA device")
    L = api.lib()
    L.glb_launch_iq_gram.argtypes = [C.POINTER(IqGramArgs), C.c_void_p]
    L.glb_tables_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    L.glb_tables_destroy.argtypes = [C.c_void_p]
    L.glb_make_level_tables.argtypes = [C.POINTER(C.c_void_p)]
    L.glb_level_tables_destroy.argtypes = [C.c_void_p]
    L.glb_level_lut.argtypes = [C.c_float, C.c_float, C.c_float, C.c_void_p]
    L.glb_level_lut.restype = None

    ns = int(a.seconds * FS)
    blk = synth.iq_stream_int16(20 * FS, fs=FS, dot_s=1.0)
    pcm = api.pinned_empty((ns, 2), np.int16)
    for i in range(0, ns, len(blk)):
        pcm[i:i + len(blk)] = blk[:ns - i]
    res = dict(gpu=gpu_info(), data=f"synth.iq_stream_int16 (20 s tiled), {a.seconds:g} s at {FS} Hz ({ns} complex samples)",
               window="hann", display="log scale; fixed range -40..-100 dB or autoscale", kernels=[], e2e=[], zoom=[])

    # ---- kernels: level epilogue against float rows on the same device floats
    dev = torch.from_numpy(synth.pcm16_to_float(pcm)).cuda()
    st = torch.cuda.current_stream().cuda_stream
    ltab = C.c_void_p()
    api._check(L.glb_make_level_tables(C.byref(ltab)))
    lut_np = np.empty(GLB_DB_NTHR, np.uint8)
    L.glb_level_lut(-100.0, -40.0, 0.0, lut_np.ctypes.data)
    lut = torch.from_numpy(lut_np).cuda()
    for n in (2048, 4096):
        hop = n // 2
        nf = ns // hop
        w = api.host_window(n, api.HANNING).astype(np.float64)
        ts = np.float32(1.0 / (2.0 * np.sqrt(2.0 * n)))
        taper = torch.from_numpy(np.repeat((w * float(ts)).astype(np.float32), 2)).cuda()
        tables = C.c_void_p()
        api._check(L.glb_tables_create(2 * n, C.byref(tables)))
        rows = torch.empty((nf, n), dtype=torch.float32, device="cuda")
        lev = torch.empty((nf, n), dtype=torch.uint8, device="cuda")

        def launch(levels):
            g = IqGramArgs(n, hop, dev.data_ptr(), 0, ns, taper.data_ptr(), 1, float(ts), 0, nf,
                           None if levels else rows.data_ptr(), tables, None)
            if levels:
                g.levels, g.levels_stride, g.level_tables, g.levels_log = lev.data_ptr(), n, ltab, 1
                g.level_lut, g.level_min, g.level_max, g.level_thr = lut.data_ptr(), -100.0, -40.0, 0.0
            api._check(L.glb_launch_iq_gram(C.byref(g), st))

        launch(False); launch(True); torch.cuda.synchronize()
        tf, tl = [], []
        for _ in range(a.reps):
            tf.append(profile_ms(lambda: launch(False), ["gram_iq_kernel"])["gram_iq_kernel"])
            tl.append(profile_ms(lambda: launch(True), ["gram_iq_kernel"])["gram_iq_kernel"])
        r = dict(n=n, overlap=0.5, frames=nf, float_rows_kernel_ms=float(np.median(tf)), float_rows_kernel_ms_all=tf,
                 levels_kernel_ms=float(np.median(tl)), levels_kernel_ms_all=tl,
                 float_rows_bytes=8.0 * ns + 4.0 * nf * n, levels_bytes=8.0 * ns + 1.0 * nf * n)
        r["ratio_levels_over_float"] = r["levels_kernel_ms"] / r["float_rows_kernel_ms"]
        res["kernels"].append(r)
        print(json.dumps(r), flush=True)
        del rows, lev, taper
        L.glb_tables_destroy(tables)
    L.glb_level_tables_destroy(ltab)
    del dev, lut
    torch.cuda.empty_cache()

    # ---- end to end, int16 I/Q in
    fixed = dict(log_scale=True, autoscale=False, max_level_db=-40.0, min_level_db=-100.0)
    for n in (2048, 4096):
        p = api.IqPlan(n=n, window_type=api.HANNING, overlap=0.5)
        nf = p.num_frames(ns)
        rows = api.pinned_empty((nf, n), np.float32)
        lev = api.pinned_empty((nf, n), np.uint8)
        rng = api.pinned_empty((nf, 2), np.float32)
        runs = {"rows_f32": lambda: p.run(pcm, out=rows),
                "levels_fixed": lambda: p.run_display(pcm, out={"levels": lev}, **fixed),
                "levels_autoscale": lambda: p.run_display(pcm, autoscale=True, out={"levels": lev, "range": rng})}
        r = dict(n=n, overlap=0.5, frames=nf, input_int16_bytes=4.0 * ns, rows_bytes=4.0 * nf * n, levels_bytes=1.0 * nf * n)
        for f in runs.values():
            f()
        ts = {k: [] for k in runs}
        for _ in range(a.reps):                                     # the three alternate
            for k, f in runs.items():
                t0 = time.perf_counter()
                f()
                ts[k].append(1e3 * (time.perf_counter() - t0))
        for k, f in runs.items():
            r[f"{k}_e2e_ms"] = float(np.median(ts[k]))
            r[f"{k}_e2e_ms_all"] = ts[k]
            pt = profile_ms(f, E2E_KEYS)
            r[f"{k}_profile_ms"] = {q: v for q, v in pt.items() if v > 0}
            r[f"{k}_e2e_over_h2d"] = r[f"{k}_e2e_ms"] / pt["HtoD"]
            r[f"{k}_e2e_over_max_copy"] = r[f"{k}_e2e_ms"] / max(pt["HtoD"], pt["DtoH"])
        r["speedup_fixed_over_rows"] = r["rows_f32_e2e_ms"] / r["levels_fixed_e2e_ms"]
        r["speedup_autoscale_over_rows"] = r["rows_f32_e2e_ms"] / r["levels_autoscale_e2e_ms"]
        res["e2e"].append(r)
        print(json.dumps(r), flush=True)
        p.close()
        del rows, lev, rng

    # ---- zoom, real int16 input (the I channel), D = 256
    x = np.ascontiguousarray(pcm[:, 0])
    xp = api.pinned_empty((ns,), np.int16)
    xp[:] = x
    for iq in (False, True):
        p = api.ZoomPlan(n=4096, decim=256, window_type=api.HANNING, overlap=0.5, center_hz=-800.0 if iq else 800.0,
                         sample_rate=FS, iq=iq)
        src = pcm if iq else xp
        nf = p.num_frames(ns)
        rows = api.pinned_empty((nf, 4096), np.float32)
        lev = api.pinned_empty((nf, 4096), np.uint8)
        rng = api.pinned_empty((nf, 2), np.float32)
        runs = {"rows_f32": lambda: p.run(src, out=rows),
                "levels_autoscale": lambda: p.run_display(src, autoscale=True, out={"levels": lev, "range": rng})}
        r = dict(iq=iq, n=4096, decim=256, overlap=0.5, frames=nf, input_int16_bytes=(4.0 if iq else 2.0) * ns)
        for f in runs.values():
            f()
        ts = {k: [] for k in runs}
        for _ in range(a.reps):
            for k, f in runs.items():
                t0 = time.perf_counter()
                f()
                ts[k].append(1e3 * (time.perf_counter() - t0))
        for k, f in runs.items():
            r[f"{k}_e2e_ms"] = float(np.median(ts[k]))
            r[f"{k}_e2e_ms_all"] = ts[k]
            r[f"{k}_profile_ms"] = {q: v for q, v in profile_ms(f, E2E_KEYS).items() if v > 0}
        res["zoom"].append(r)
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
