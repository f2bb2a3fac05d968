"""Multitaper I/Q and zoom plans on one hour of synth.iq_stream at 48 kHz (172.8 M complex samples), 50 % overlap.

  * kernel: the fused multitaper I/Q kernel (gram_iq_mtm_kernel) against the kernel a real GLFER_MODE_MTM plan
    (sub_mean = 0) runs at N = 2n on the same floats with the same K' (gram_ring_kernel<.., MULTI = true, ..>), alternated
    in one process, and the general path (glb_force_generic_kernel: K' spectra + iq_mtm_split_kernel), n = 2048 / 4096
    and K' = 4 / 8; device time of one launch from torch.profiler, median of --reps.  n = 8192 (K' = 8): the fused
    kernel against the general path, the measurement behind the choice of path there.  FLOP/s are counted as
    5 n log2 n K' per frame (one complex FFT of n points per taper); C3's convention, 5 N log2 N K' at the real frame
    length N = 2n, is given too;
  * end to end, pinned buffers, profiler off, median of --reps: IqPlan.run on float and on int16 input and run_display
    with autoscale on int16, n = 2048 / 4096, K' = 4 / 8, against the larger of the H2D / D2H copy totals of one
    profiled run;
  * zoom, D = 256, n = 4096, K' = 8, I/Q int16 input: ZoomPlan.run end to end against its upload.
The GPU name and power limit are read in the same call.

usage: python tools/scripts/iq_mtm_bench.py [--out FILE.json] [--seconds S] [--reps R]"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from glfer_b200 import api, synth      # noqa: E402

FS = 48000
ROOFLINE_GBS = 6660.0                  # bench.py: read+write bandwidth of a 4 GiB device copy, B200 at 1000 W
FP32_TFLOPS = 74.0                     # BASELINE.md §3: derived FP32 rate of the B200 (not measured)
MTM_W = 4.0


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
    """device time per name substring (first match wins) of one call of fn under torch.profiler; key "" = any kernel"""
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
            if k in ev.name and (k or not any(s in ev.name for s in ("Memcpy", "Memset", "HtoD", "DtoH"))):
                t[k] += ms
                break
    return t


E2E_KEYS = ["HtoD", "DtoH", "gram_iq_mtm_kernel", "gram_kernel", "iq_mtm_split", "pcm16", "floor_stats", "agc_kernel",
            "levels_kernel", "zoom_decim"]


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--seconds", type=float, default=3600.0)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if api.device_count() < 1:
        raise SystemExit("iq_mtm_bench needs a CUDA device")
    L = api.lib()
    L.glb_launch_iq_gram.argtypes = [C.POINTER(IqGramArgs), C.c_void_p]
    L.glb_iq_gram_scratch_bytes.argtypes = [C.c_int, C.c_int, C.c_longlong, C.c_int, C.c_int, C.c_int]
    L.glb_iq_gram_scratch_bytes.restype = C.c_longlong
    L.glb_tables_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    L.glb_tables_destroy.argtypes = [C.c_void_p]

    ns = int(a.seconds * FS)
    blk = synth.iq_stream_int16(20 * FS, fs=FS, dot_s=1.0)
    pcm = api.pinned_empty((ns, 2), np.int16)
    for i in range(0, ns, len(blk)):
        pcm[i:i + len(blk)] = blk[:ns - i]
    zf = api.pinned_empty((ns, 2), np.float32)
    zf[:] = synth.pcm16_to_float(pcm)
    res = dict(gpu=gpu_info(), data=f"synth.iq_stream_int16 (20 s tiled), {a.seconds:g} s at {FS} Hz ({ns} complex samples)",
               mtm_w=MTM_W, overlap=0.5, roofline_gbs=ROOFLINE_GBS, fp32_tflops_derived=FP32_TFLOPS,
               flop_convention="5 n log2 n K' per frame (complex FFT of n points per taper); C3: 5 N log2 N K', N = 2n",
               kernels=[], n8192=[], e2e=[], zoom=[])
    dev = torch.from_numpy(zf).cuda()
    st = torch.cuda.current_stream().cuda_stream

    def table(n, k):
        """the plan's device taper table: v_k taper_scale / sqrt(lambda_k) on both floats of a complex sample"""
        t, lam = api.host_dpss(n, MTM_W, k - 1)
        ts = float(np.float32(1.0 / (2.0 * math.sqrt(2.0 * n))))
        tab = np.repeat((t * (ts / np.sqrt(lam))[:, None]).astype(np.float32), 2, axis=1)
        sym = sum(1 << j for j in range(k) if np.array_equal(tab[j], tab[j, ::-1]))
        return torch.from_numpy(np.ascontiguousarray(tab)).cuda(), sym, ts

    def launcher(n, k, rows, generic):
        hop = n // 2
        nf = ns // hop
        tab, sym, ts = table(n, k)
        tables = C.c_void_p()
        api._check(L.glb_tables_create(2 * n, C.byref(tables)))
        api.force_generic_kernel(generic)
        sb = L.glb_iq_gram_scratch_bytes(n, hop, nf, 0, k, 0)
        api.force_generic_kernel(False)
        scratch = torch.empty(max(sb, 4), dtype=torch.uint8, device="cuda")
        g = IqGramArgs(n, hop, dev.data_ptr(), 0, ns, tab.data_ptr(), sym, ts, 0, nf, rows.data_ptr(), tables,
                       scratch.data_ptr() if sb > 0 else None)
        g.ntapers = k

        def run():
            api.force_generic_kernel(generic)
            try:
                api._check(L.glb_launch_iq_gram(C.byref(g), st))
            finally:
                api.force_generic_kernel(False)
        run.keep = (tab, scratch, tables)
        return run

    def flops(n, k, nf, ms):
        return dict(tflops=5.0 * n * math.log2(n) * k * nf / (ms * 1e-3) / 1e12,
                    tflops_c3_convention=5.0 * 2 * n * math.log2(2 * n) * k * nf / (ms * 1e-3) / 1e12)

    # ---- kernels: fused I/Q multitaper against the real multitaper kernel at N = 2n, and the general path
    for n in (2048, 4096):
        hop = n // 2
        nf = ns // hop
        rows = torch.empty((nf, n), dtype=torch.float32, device="cuda")
        for k in (4, 8):
            fi = launcher(n, k, rows, False)
            fg = launcher(n, k, rows, True)
            real = api.GramPlan(n=2 * n, mode=api.MODE_MTM, overlap=0.5, sub_mean=False, mtm_w=MTM_W, mtm_kmax=k - 1)
            real.stage(zf.reshape(-1))
            assert real.num_frames(2 * ns) == nf
            fr = lambda: real.exec(0, nf)                                          # noqa: E731
            fi(); fr(); fg(); torch.cuda.synchronize()
            ti, tr, tg = [], [], []
            for _ in range(a.reps):
                ti.append(profile_ms(fi, [""])[""])
                tr.append(profile_ms(fr, [""])[""])
                tg.append(profile_ms(fg, [""])[""])
            real.sync()
            real.close()
            r = dict(n=n, K=k, frames=nf, iq_mtm_kernel_ms=float(np.median(ti)), iq_mtm_kernel_ms_all=ti,
                     real_mtm_kernel_ms=float(np.median(tr)), real_mtm_kernel_ms_all=tr,
                     general_path_ms=float(np.median(tg)), general_path_ms_all=tg, bytes=8.0 * ns + 4.0 * nf * n)
            r["ratio_iq_over_real"] = r["iq_mtm_kernel_ms"] / r["real_mtm_kernel_ms"]
            r["ratio_general_over_fused"] = r["general_path_ms"] / r["iq_mtm_kernel_ms"]
            r["fused"] = flops(n, k, nf, r["iq_mtm_kernel_ms"])
            r["fused"]["gbs"] = r["bytes"] / (r["iq_mtm_kernel_ms"] * 1e-3) / 1e9
            r["fused"]["share_of_hbm_roofline"] = r["fused"]["gbs"] / ROOFLINE_GBS
            r["fused"]["share_of_fp32_rate"] = r["fused"]["tflops"] / FP32_TFLOPS
            r["fused"]["bound"] = "FP32" if r["fused"]["share_of_fp32_rate"] > r["fused"]["share_of_hbm_roofline"] else "HBM"
            r["real"] = flops(n, k, nf, r["real_mtm_kernel_ms"])
            res["kernels"].append(r)
            print(json.dumps(r), flush=True)
            del fi, fg
        del rows
        torch.cuda.empty_cache()

    # ---- n = 8192: fused against general (the choice of path)
    n, k = 8192, 8
    nf = ns // (n // 2)
    rows = torch.empty((nf, n), dtype=torch.float32, device="cuda")
    fi = launcher(n, k, rows, False)
    fg = launcher(n, k, rows, True)
    fi(); fg(); torch.cuda.synchronize()
    ti, tg, fam = [], [], []
    for _ in range(a.reps):
        ti.append(profile_ms(fi, [""])[""])
        fam.append(api.last_kernel_family())
        tg.append(profile_ms(fg, [""])[""])
    r = dict(n=n, K=k, frames=nf, fused_ms=float(np.median(ti)), fused_ms_all=ti, fused_family=fam[-1],
             general_path_ms=float(np.median(tg)), general_path_ms_all=tg)
    r["ratio_general_over_fused"] = r["general_path_ms"] / r["fused_ms"]
    res["n8192"].append(r)
    print(json.dumps(r), flush=True)
    del fi, fg, rows, dev
    torch.cuda.empty_cache()

    # ---- end to end
    for n in (2048, 4096):
        for k in (4, 8):
            p = api.IqPlan(n=n, overlap=0.5, multitaper=True, mtm_w=MTM_W, mtm_kmax=k - 1)
            nf = p.num_frames(ns)
            rows = api.pinned_empty((nf, n), np.float32)
            lev = api.pinned_empty((nf, n), np.uint8)
            rng = api.pinned_empty((nf, 2), np.float32)
            runs = {"float_rows": lambda: p.run(zf, out=rows),
                    "int16_rows": lambda: p.run(pcm, out=rows),
                    "int16_levels_autoscale": lambda: p.run_display(pcm, autoscale=True, out={"levels": lev, "range": rng})}
            r = dict(n=n, K=k, frames=nf)
            for f in runs.values():
                f()
            ts = {q: [] for q in runs}
            for _ in range(a.reps):
                for q, f in runs.items():
                    t0 = time.perf_counter()
                    f()
                    ts[q].append(1e3 * (time.perf_counter() - t0))
            for q, f in runs.items():
                r[f"{q}_e2e_ms"] = float(np.median(ts[q]))
                r[f"{q}_e2e_ms_all"] = ts[q]
                pt = profile_ms(f, E2E_KEYS)
                r[f"{q}_profile_ms"] = {x: v for x, v in pt.items() if v > 0}
                r[f"{q}_e2e_over_max_copy"] = r[f"{q}_e2e_ms"] / max(pt["HtoD"], pt["DtoH"])
            res["e2e"].append(r)
            print(json.dumps(r), flush=True)
            p.close()
            del rows, lev, rng

    # ---- zoom, D = 256, n = 4096, K' = 8, I/Q int16
    p = api.ZoomPlan(n=4096, decim=256, overlap=0.5, center_hz=-800.0, sample_rate=FS, iq=True, multitaper=True,
                     mtm_w=MTM_W, mtm_kmax=7)
    nf = p.num_frames(ns)
    rows = api.pinned_empty((nf, 4096), np.float32)
    f = lambda: p.run(pcm, out=rows)                                                # noqa: E731
    f()
    ts = []
    for _ in range(a.reps):
        t0 = time.perf_counter()
        f()
        ts.append(1e3 * (time.perf_counter() - t0))
    pt = profile_ms(f, E2E_KEYS)
    r = dict(n=4096, decim=256, K=8, frames=nf, input_int16_bytes=4.0 * ns, e2e_ms=float(np.median(ts)), e2e_ms_all=ts,
             profile_ms={x: v for x, v in pt.items() if v > 0})
    r["e2e_over_h2d"] = r["e2e_ms"] / pt["HtoD"]
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
