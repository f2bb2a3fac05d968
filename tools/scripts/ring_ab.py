"""A/B of two builds of the library on the same GPU, alternated, in one call.

    python tools/scripts/ring_ab.py --a glfer_b200/libglfer_b200_plainx2.so --b glfer_b200/libglfer_b200.so \
        --out DIR [--workloads metric,c1] [--reps 5] [--steps 400] [--dump metric,c2,c3,lmp]

Each repetition runs `bench.py --workload W --steps K --no-e2e --no-cpu --no-configs` once with library A and
once with library B (GLFER_B200_LIB), in alternating order, and reads the spectrogram kernel's CUDA-event time
(`roofline.kernel_ms`) and the headline `value`.  It reports, per workload and build, the median and the spread
(min .. max) of kernel_ms, and B's median change against A.  `--dump` workloads are also run once per build with
`--dump-outputs`, and every dumped array of B is compared with A's by exact equality.  The card name, power limit
and SM clocks are read with nvidia-smi in the same call.  Writes DIR/ring_ab.json and prints it."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info() -> dict:
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                             text=True, check=True).stdout.strip().splitlines()[0]
        return dict(zip(q.split(","), [s.strip() for s in out.split(",")]))
    except (OSError, subprocess.CalledProcessError) as e:
        return {"error": str(e)}


def bench(lib: str, workload: str, steps: int, warmup: int, dump: str | None = None) -> dict:
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--steps", str(steps),
           "--warmup", str(warmup), "--no-e2e", "--no-cpu", "--no-configs"]
    if dump:
        cmd += ["--dump-outputs", dump]
    env = dict(os.environ, GLFER_B200_LIB=os.path.abspath(lib))
    res = subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=ROOT)
    if res.returncode != 0:
        raise RuntimeError(f"bench.py failed ({lib}, {workload}):\n{res.stderr[-4000:]}")
    line = [ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1]
    d = json.loads(line)
    return {"kernel_ms": d["roofline"]["kernel_ms"], "value": d["value"]}


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--a", required=True, help="library A (reference build)")
    ap.add_argument("--b", required=True, help="library B (candidate build)")
    ap.add_argument("--out", required=True)
    ap.add_argument("--workloads", default="metric,c1")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--dump", default="", help="workloads whose outputs are compared between the builds")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    libs = {"A": args.a, "B": args.b}
    result = {"gpu_before": gpu_info(), "libs": libs, "steps": args.steps, "reps": args.reps, "workloads": {}}
    for w in [s for s in args.workloads.split(",") if s]:
        runs = {"A": [], "B": []}
        for rep in range(args.reps):
            for k in (("A", "B") if rep % 2 == 0 else ("B", "A")):
                runs[k].append(bench(libs[k], w, args.steps, args.warmup))
        entry = {}
        for k in ("A", "B"):
            ms = [r["kernel_ms"] for r in runs[k]]
            entry[k] = {"kernel_ms": ms, "median_ms": statistics.median(ms), "min_ms": min(ms), "max_ms": max(ms),
                        "value_median": statistics.median(r["value"] for r in runs[k])}
        entry["B_vs_A_kernel_ms"] = entry["B"]["median_ms"] / entry["A"]["median_ms"] - 1.0
        entry["B_vs_A_value"] = entry["B"]["value_median"] / entry["A"]["value_median"] - 1.0
        result["workloads"][w] = entry
        print(w, json.dumps(entry), flush=True)
    result["identical_outputs"] = {}
    for w in [s for s in args.dump.split(",") if s]:
        dirs = {k: os.path.join(args.out, f"dump_{w}_{k}") for k in libs}
        for k in libs:
            bench(libs[k], w, 1, 1, dump=dirs[k])
        names = sorted(os.listdir(dirs["A"]))
        same = names == sorted(os.listdir(dirs["B"])) and all(
            np.array_equal(np.load(os.path.join(dirs["A"], n)), np.load(os.path.join(dirs["B"], n))) for n in names)
        result["identical_outputs"][w] = {"arrays": names, "array_equal": bool(same)}
        print(w, "outputs identical:", same, names, flush=True)
    result["gpu_after"] = gpu_info()
    with open(os.path.join(args.out, "ring_ab.json"), "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps(result, indent=1))
    return 0 if all(v["array_equal"] for v in result["identical_outputs"].values()) else 1


if __name__ == "__main__":
    sys.exit(main())
