"""Build recipe for libglfer_b200.so (CUDA kernels for sm_100a + C host layer), in-tree.

`python -m glfer_b200.build` or glfer_b200.build.build().  nvcc cross-compiles without a
GPU; the resulting .so travels to the GPU box with the repository snapshot."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
LIB = os.path.join(HERE, "libglfer_b200.so")
LIB_FFTW = os.path.join(HERE, "libglfer_b200_fftw.so")      # fft_params_t in the reference's FFTW (double) layout
OBJ = os.path.join(HERE, "_build")

# (source, tag, extra flags): gram_part.cu is compiled once per subset of FFT sizes, in parallel
CU_UNITS = ([("csrc/gram_kernels.cu", "", []), ("csrc/gram_big.cu", "", []), ("csrc/zoom.cu", "", []), ("csrc/iq.cu", "", [])]
            + [("csrc/gram_part.cu", f".p{k}", [f"-DGLB_PART={k}"]) for k in range(4)])
C_SOURCES = ["host/window.c", "host/dpss.c", "host/gram.c", "host/dropin.c", "host/wav.c", "host/levels.c",
             "host/zoom.c", "host/iq.c", "host/display.c"]
HEADERS = ["csrc/fft_core.cuh", "csrc/fft_wpf.cuh", "csrc/fft_big.cuh", "csrc/levels.cuh", "csrc/avg_frame.cuh", "csrc/twiddle_consts.cuh", "csrc/gram_common.cuh", "csrc/iq_core.cuh", "csrc/tables.hpp", "host/glb_host.h", "../include/glb_shim.h", "../include/fft.h",
           "../include/mtm.h", "../include/avg.h", "../include/lmp.h", "../include/glfer_b200.h"]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]
# no -march=native / -ffast-math: the window tables must round exactly like the reference's
C_FLAGS = ["-O2", "-fPIC", "-std=gnu11", "-Wall", "-Wno-unused-function", "-pthread"]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target: str, deps: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def _run(cmd: list[str], log: str | None = None) -> None:
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if log:
        with open(log, "w") as fh:
            fh.write(" ".join(cmd) + "\n" + res.stdout)
    if res.returncode != 0:
        sys.stderr.write(res.stdout)
        raise RuntimeError("build step failed: " + " ".join(cmd))


def _compile_cu(nvcc: str, extra: list[str], tag: str, force: bool, hdrs: list[str], verbose: bool) -> list[str]:
    """All CUDA translation units (in parallel); returns the object files."""
    from concurrent.futures import ThreadPoolExecutor
    jobs, objs = [], []
    for src, part, flags in CU_UNITS:
        s = os.path.join(HERE, src)
        o = os.path.join(OBJ, os.path.basename(src) + part + (f".{tag}" if tag else "") + ".o")
        objs.append(o)
        if force or _stale(o, [s] + hdrs):
            if verbose:
                print("nvcc", src, " ".join(flags))
            jobs.append(([nvcc] + NVCC_FLAGS + extra + flags + ["-c", s, "-o", o], o + ".log"))
    if jobs:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as ex:
            for fut in [ex.submit(_run, cmd, log) for cmd, log in jobs]:
                fut.result()
    return objs


def build_variant(tag: str, extra_nvcc: list[str]) -> str:
    """Experiment helper: a second library with extra nvcc flags (e.g. another register
    target), selected at run time with GLFER_B200_LIB=<path>."""
    build()
    nvcc = _nvcc()
    hdrs = [os.path.join(HERE, h) for h in HEADERS] + [os.path.abspath(__file__)]
    objs = _compile_cu(nvcc, extra_nvcc, tag, True, hdrs, False)
    objs += [os.path.join(OBJ, os.path.basename(src) + ".o") for src in C_SOURCES]
    out = os.path.join(HERE, f"libglfer_b200_{tag}.so")
    _run([nvcc, "-shared", "-o", out] + objs + ["-Xcompiler", "-pthread", "-lm", "-lpthread"])
    return out


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    hdrs = [os.path.join(HERE, h) for h in HEADERS] + [os.path.abspath(__file__)]
    nvcc = _nvcc()
    objs = _compile_cu(nvcc, [], "", force, hdrs, verbose)
    for src in C_SOURCES:
        s = os.path.join(HERE, src)
        o = os.path.join(OBJ, os.path.basename(src) + ".o")
        if force or _stale(o, [s] + hdrs):
            if verbose:
                print("gcc", src)
            _run(["gcc"] + C_FLAGS + ["-c", s, "-o", o])
        objs.append(o)
    if force or _stale(LIB, objs):
        if verbose:
            print("link", LIB)
        # nvcc links the static CUDA runtime: the .so depends on libcuda only at run time
        _run([nvcc, "-shared", "-o", LIB] + objs + ["-Xcompiler", "-pthread", "-lm", "-lpthread"])
    # the same library for callers built WITH FFTW (HAVE_LIBRFFTW): fft_params_t starts with the plan and its
    # buffers are doubles (reference fft.h:36-48); only the per-call layer depends on the layout
    fobjs = []
    for o in objs:
        if os.path.basename(o) == "dropin.c.o":
            s = os.path.join(HERE, "host/dropin.c")
            fo = os.path.join(OBJ, "dropin.c.fftw.o")
            if force or _stale(fo, [s] + hdrs):
                if verbose:
                    print("gcc host/dropin.c -DGLFER_FFTW_LAYOUT")
                _run(["gcc"] + C_FLAGS + ["-DGLFER_FFTW_LAYOUT", "-c", s, "-o", fo])
            fobjs.append(fo)
        else:
            fobjs.append(o)
    if force or _stale(LIB_FFTW, fobjs):
        if verbose:
            print("link", LIB_FFTW)
        _run([nvcc, "-shared", "-o", LIB_FFTW] + fobjs + ["-Xcompiler", "-pthread", "-lm", "-lpthread"])
    return LIB


def build_tools(force: bool = False) -> str:
    """The headless harness (tools/glfer_headless.c) against the product library."""
    build(force=False)
    out = os.path.join(ROOT, "tools", "glfer_headless")
    src = os.path.join(ROOT, "tools", "glfer_headless.c")
    if os.path.exists(src) and (force or _stale(out, [src, LIB])):
        _run(["gcc", "-O2", "-std=gnu11", "-I", os.path.join(ROOT, "include"), src, "-o", out,
              "-L", HERE, "-lglfer_b200", "-Wl,-rpath," + HERE, "-lm"])
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
