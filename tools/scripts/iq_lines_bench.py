"""Harmonic line detection of multitaper I/Q plans (glfer_iq_run_mtm_lines*) on one hour of synth.iq_stream at 48 kHz
(172.8 M complex samples), 50 % overlap, NW = 4, n = 2048 / 4096, K' = 4 / 8, pfa = 1e-3, max_lines = 16, psd on.

  * kernel: device time (torch.profiler, summed over the run's chunks) of ftest_lines_kernel against the F-test kernel
    (gram_iq_ftest_kernel) of the same run and against the HBM floor of one read of the F rows (F bytes over the
    6660 GB/s copy bandwidth measured on this card, DESIGN §7.3), median of --reps; and the all-overflow case
    (pfa = 0.2, max_lines = 4);
  * end to end, pinned buffers, profiler off, median of --reps: lines against F only (glfer_iq_run_mtm_ftest with F rows
    only), float and int16 input, alternated, against the H2D copy total of one profiled run of each;
  * a zoom bank, C = 8, D = 256, n = 4096, K' = 8, I/Q int16: lines against F only, end to end.
The GPU name and power limit are read in the same call.

usage: python tools/scripts/iq_lines_bench.py [--out FILE.json] [--seconds S] [--reps R]"""
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
MTM_W = 4.0
PFA, MAX_LINES = 1e-3, 16
HBM_GBPS = 6660.0                      # copy bandwidth measured on a B200 (DESIGN §7.3)


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


E2E_KEYS = ["HtoD", "DtoH", "ftest_lines_kernel", "gram_iq_ftest_kernel", "pcm16", "zoom_bank_decim"]


def e2e(runs, reps):
    """alternated wall times (median) and one profiled run of each"""
    for f in runs.values():
        f()
    ts = {q: [] for q in runs}
    for _ in range(reps):
        for q, f in runs.items():
            t0 = time.perf_counter()
            f()
            ts[q].append(1e3 * (time.perf_counter() - t0))
    e = {}
    for q, f in runs.items():
        e[f"{q}_e2e_ms"] = float(np.median(ts[q]))
        e[f"{q}_e2e_ms_all"] = ts[q]
        pt = profile_ms(f, E2E_KEYS)
        e[f"{q}_profile_ms"] = {x: v for x, v in pt.items() if v > 0}
        e[f"{q}_e2e_over_upload"] = e[f"{q}_e2e_ms"] / pt["HtoD"]
    return e


def main():
    import torch  # noqa: F401  (CUDA context for the profiler)
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--seconds", type=float, default=3600.0)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if api.device_count() < 1:
        raise SystemExit("iq_lines_bench needs a CUDA device")
    L = api.lib()
    ns = int(a.seconds * FS)
    blk = synth.iq_stream_int16(20 * FS, fs=FS, dot_s=1.0)
    pcm = api.pinned_empty((ns, 2), np.int16)
    for i in range(0, ns, len(blk)):
        pcm[i:i + len(blk)] = blk[:ns - i]
    zf = api.pinned_empty((ns, 2), np.float32)
    zf[:] = synth.pcm16_to_float(pcm)
    res = dict(gpu=gpu_info(), data=f"synth.iq_stream_int16 (20 s tiled), {a.seconds:g} s at {FS} Hz ({ns} complex samples)",
               mtm_w=MTM_W, overlap=0.5, pfa=PFA, max_lines=MAX_LINES, hbm_gbps=HBM_GBPS, kernels=[], e2e=[], bank=None)

    for n in (2048, 4096):
        for k in (4, 8):
            p = api.IqPlan(n=n, overlap=0.5, multitaper=True, mtm_w=MTM_W, mtm_kmax=k - 1)
            nf = p.num_frames(ns)
            ft = api.pinned_empty((nf, n), np.float32)

            def lines_run(src, pfa=PFA, m=MAX_LINES):
                fn = L.glfer_iq_run_mtm_lines_pcm16 if src.dtype == np.int16 else L.glfer_iq_run_mtm_lines
                lc = api.LinesConfig(pfa, m, 0, n)
                cnt = np.empty(nf, np.int32)
                b, lf, lp = (np.empty((nf, m), t) for t in (np.int32, np.float32, np.float32))
                return lambda: api._check(fn(p._h, src.ctypes.data, 0, ns, 0, nf, api.C.byref(lc), cnt.ctypes.data,
                                             b.ctypes.data, lf.ctypes.data, lp.ctypes.data))

            def f_only(src):
                fn = L.glfer_iq_run_mtm_ftest_pcm16 if src.dtype == np.int16 else L.glfer_iq_run_mtm_ftest
                return lambda: api._check(fn(p._h, src.ctypes.data, 0, ns, 0, nf, None, ft.ctypes.data))

            # ---- kernels
            keys = ["ftest_lines_kernel", "gram_iq_ftest_kernel"]
            common, over = lines_run(zf), lines_run(zf, 0.2, 4)
            common(); over()
            tl, tf, to = [], [], []
            for _ in range(a.reps):
                t = profile_ms(common, keys)
                tl.append(t["ftest_lines_kernel"]); tf.append(t["gram_iq_ftest_kernel"])
                to.append(profile_ms(over, keys)["ftest_lines_kernel"])
            fbytes = nf * n * 4
            r = dict(n=n, K=k, frames=nf, f_bytes=fbytes, lines_kernel_ms=float(np.median(tl)), lines_kernel_ms_all=tl,
                     ftest_kernel_ms=float(np.median(tf)), ftest_kernel_ms_all=tf,
                     hbm_floor_ms=fbytes / (HBM_GBPS * 1e9) * 1e3,
                     overflow_lines_kernel_ms=float(np.median(to)), overflow_lines_kernel_ms_all=to)
            r["lines_over_ftest"] = r["lines_kernel_ms"] / r["ftest_kernel_ms"]
            r["lines_over_hbm_floor"] = r["lines_kernel_ms"] / r["hbm_floor_ms"]
            r["target_lines_le_0.10_ftest"] = "met" if r["lines_over_ftest"] <= 0.10 else "not met"
            res["kernels"].append(r)
            print(json.dumps({x: v for x, v in r.items() if not x.endswith("_all")}), flush=True)

            # ---- end to end, lines and F only alternated
            runs = {}
            for name, src in (("float", zf), ("int16", pcm)):
                runs[f"{name}_lines"] = lines_run(src)
                runs[f"{name}_ftest_only"] = f_only(src)
            e = dict(n=n, K=k, frames=nf, **e2e(runs, a.reps))
            e["target_int16_lines_le_1.15_upload"] = "met" if e["int16_lines_e2e_over_upload"] <= 1.15 else "not met"
            e["target_float_lines_le_1.10_upload"] = "met" if e["float_lines_e2e_over_upload"] <= 1.10 else "not met"
            res["e2e"].append(e)
            print(json.dumps({x: v for x, v in e.items() if not x.endswith("_all")}), flush=True)
            p.close()
            del ft

    # ---- zoom bank: C = 8, D = 256, n = 4096, K' = 8, I/Q int16
    centers = [-20000.0 + 5000.0 * c for c in range(8)]
    zb = api.ZoomPlan(n=4096, decim=256, overlap=0.5, center_hz=centers, sample_rate=FS, iq=True, multitaper=True,
                      mtm_w=MTM_W, mtm_kmax=7)
    nf = zb.num_frames(ns)
    zft = api.pinned_empty((8, nf, 4096), np.float32)
    lc = api.LinesConfig(PFA, MAX_LINES, 0, 4096)
    cnt = np.empty((8, nf), np.int32)
    b, lf, lp = (np.empty((8, nf, MAX_LINES), t) for t in (np.int32, np.float32, np.float32))
    runs = {"int16_lines": lambda: api._check(L.glfer_zoom_run_iq_mtm_lines_pcm16(
                zb._h, pcm.ctypes.data, 0, ns, 0, nf, api.C.byref(lc), cnt.ctypes.data, b.ctypes.data, lf.ctypes.data,
                lp.ctypes.data)),
            "int16_ftest_only": lambda: api._check(L.glfer_zoom_run_iq_mtm_ftest_pcm16(
                zb._h, pcm.ctypes.data, 0, ns, 0, nf, None, zft.ctypes.data))}
    e = dict(C=8, decim=256, n=4096, K=8, frames=nf, **e2e(runs, a.reps))
    e["lines_over_ftest_only"] = e["int16_lines_e2e_ms"] / e["int16_ftest_only_e2e_ms"]
    e["target_lines_le_1.03_ftest_only"] = "met" if e["lines_over_ftest_only"] <= 1.03 else "not met"
    res["bank"] = e
    print(json.dumps({x: v for x, v in e.items() if not x.endswith("_all")}), flush=True)
    zb.close()

    res["gpu_after"] = gpu_info()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:               # one line per key and per measured shape
            fh.write("{\n" + ",\n".join(
                f" {json.dumps(k)}: " + ("[\n  " + ",\n  ".join(json.dumps(r) for r in v) + "\n ]"
                                         if isinstance(v, list) else json.dumps(v))
                for k, v in res.items()) + "\n}\n")
    print(json.dumps({k: v for k, v in res.items() if k in ("gpu", "gpu_after", "data")}))


if __name__ == "__main__":
    main()
