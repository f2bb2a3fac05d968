"""Harmonic F-test of multitaper I/Q plans on one hour of synth.iq_stream at 48 kHz (172.8 M complex samples), 50 %
overlap, n = 2048 / 4096, K' = 4 / 8.

  * kernel: device time (torch.profiler, summed over the run's chunks) of the fused F-test kernel
    (gram_iq_ftest_kernel, IqPlan.run_mtm_ftest with F rows only) against the fused multitaper-rows kernel
    (gram_iq_mtm_kernel, IqPlan.run) and against the general path (glb_force_generic_kernel: K' + 1 spectra, the splits
    and the quotient; every kernel but the copies and the int16 conversion), alternated, median of --reps;
  * end to end, pinned buffers, profiler off, median of --reps: rows + F, F only and rows only
    (glfer_iq_run_mtm_ftest[_pcm16]) on float and on int16 input, and glfer_iq_run for reference, against the larger of
    the H2D / D2H copy totals of one profiled run.
The GPU name and power limit are read in the same call.

usage: python tools/scripts/iq_ftest_bench.py [--out FILE.json] [--seconds S] [--reps R]"""
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
            if k in ev.name and (k or not any(s in ev.name for s in ("Memcpy", "Memset", "HtoD", "DtoH", "pcm16"))):
                t[k] += ms
                break
    return t


E2E_KEYS = ["HtoD", "DtoH", "gram_iq_ftest_kernel", "gram_iq_mtm_kernel", "pcm16"]


def main():
    import torch  # noqa: F401  (CUDA context for the profiler)
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--seconds", type=float, default=3600.0)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    if api.device_count() < 1:
        raise SystemExit("iq_ftest_bench needs a CUDA device")
    L = api.lib()
    ns = int(a.seconds * FS)
    blk = synth.iq_stream_int16(20 * FS, fs=FS, dot_s=1.0)
    pcm = api.pinned_empty((ns, 2), np.int16)
    for i in range(0, ns, len(blk)):
        pcm[i:i + len(blk)] = blk[:ns - i]
    zf = api.pinned_empty((ns, 2), np.float32)
    zf[:] = synth.pcm16_to_float(pcm)
    res = dict(gpu=gpu_info(), data=f"synth.iq_stream_int16 (20 s tiled), {a.seconds:g} s at {FS} Hz ({ns} complex samples)",
               mtm_w=MTM_W, overlap=0.5, kernels=[], e2e=[])

    for n in (2048, 4096):
        for k in (4, 8):
            p = api.IqPlan(n=n, overlap=0.5, multitaper=True, mtm_w=MTM_W, mtm_kmax=k - 1)
            nf = p.num_frames(ns)
            rows = api.pinned_empty((nf, n), np.float32)
            ft = api.pinned_empty((nf, n), np.float32)

            def ftest_run(src, fn_f, fn_i, want_rows, want_f):
                fn = fn_i if src.dtype == np.int16 else fn_f
                return lambda: api._check(fn(p._h, src.ctypes.data, 0, ns, 0, nf, rows.ctypes.data if want_rows else None,
                                             ft.ctypes.data if want_f else None))

            f_only = ftest_run(zf, L.glfer_iq_run_mtm_ftest, L.glfer_iq_run_mtm_ftest_pcm16, False, True)
            rows_run = lambda: p.run(zf, out=rows)                                       # noqa: E731

            def general():
                api.force_generic_kernel(True)
                try:
                    f_only()
                finally:
                    api.force_generic_kernel(False)

            # ---- kernels, alternated
            f_only(); rows_run(); general()
            tf, tr, tg = [], [], []
            for _ in range(a.reps):
                tf.append(profile_ms(f_only, ["gram_iq_ftest_kernel"])["gram_iq_ftest_kernel"])
                tr.append(profile_ms(rows_run, ["gram_iq_mtm_kernel"])["gram_iq_mtm_kernel"])
                tg.append(profile_ms(general, [""])[""])
            r = dict(n=n, K=k, frames=nf, ftest_kernel_ms=float(np.median(tf)), ftest_kernel_ms_all=tf,
                     rows_kernel_ms=float(np.median(tr)), rows_kernel_ms_all=tr,
                     general_path_ms=float(np.median(tg)), general_path_ms_all=tg)
            r["ratio_ftest_over_rows"] = r["ftest_kernel_ms"] / r["rows_kernel_ms"]
            r["ratio_general_over_fused"] = r["general_path_ms"] / r["ftest_kernel_ms"]
            res["kernels"].append(r)
            print(json.dumps(r), flush=True)

            # ---- end to end
            runs = {}
            for name, src in (("float", zf), ("int16", pcm)):
                runs[f"{name}_rows_ftest"] = ftest_run(src, L.glfer_iq_run_mtm_ftest, L.glfer_iq_run_mtm_ftest_pcm16, True, True)
                runs[f"{name}_ftest_only"] = ftest_run(src, L.glfer_iq_run_mtm_ftest, L.glfer_iq_run_mtm_ftest_pcm16, False, True)
                runs[f"{name}_rows_only"] = ftest_run(src, L.glfer_iq_run_mtm_ftest, L.glfer_iq_run_mtm_ftest_pcm16, True, False)
                runs[f"{name}_run"] = (lambda s: lambda: p.run(s, out=rows))(src)
            for f in runs.values():
                f()
            ts = {q: [] for q in runs}
            for _ in range(a.reps):
                for q, f in runs.items():
                    t0 = time.perf_counter()
                    f()
                    ts[q].append(1e3 * (time.perf_counter() - t0))
            e = dict(n=n, K=k, frames=nf)
            for q, f in runs.items():
                e[f"{q}_e2e_ms"] = float(np.median(ts[q]))
                e[f"{q}_e2e_ms_all"] = ts[q]
                pt = profile_ms(f, E2E_KEYS)
                e[f"{q}_profile_ms"] = {x: v for x, v in pt.items() if v > 0}
                e[f"{q}_e2e_over_max_copy"] = e[f"{q}_e2e_ms"] / max(pt["HtoD"], pt["DtoH"])
            res["e2e"].append(e)
            print(json.dumps({x: v for x, v in e.items() if not x.endswith("_all")}), flush=True)
            p.close()
            del rows, ft
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
