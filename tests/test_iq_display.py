"""Waterfall output of I/Q and zoom plans (glfer_iq_run_display*, glfer_zoom_run_display*).

CPU: the pixel addressing of the I/Q kernel's level epilogue, thread by thread (tests/emu/emu_iq_levels.cpp).
GPU: the levels equal main_window_draw's mapping (oracle.display_levels, pinned to the reference GUI) of the plan's
own rows, bit for bit -- fixed range on every fused geometry and on the general path, fused against two-pass,
int16 against float input; autoscale across several chunks, chained through agc_state, for the I/Q plan and both
zoom plans; RGB through the palette; and the argument checks."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from oracle import glfer_oracle as O  # noqa: E402

FS = 48000
HANNING, KAISER = 0, 7
FUSED_N = (32, 64, 128, 256, 512, 1024, 2048, 4096, 8192)
FUSED_OV = (0.0, 0.5, 0.75, 0.875, 0.9375)


@pytest.fixture(scope="module")
def dapi():
    from glfer_b200 import build
    build.build()
    from glfer_b200 import api
    if api.device_count() < 1:
        pytest.fail("no CUDA device visible: the display GPU tests need a B200 (no CPU fallback exists)")
    return api


def _iq_int16(count, seed=0x5EED):
    from glfer_b200 import synth
    return synth.iq_stream_int16(count, fs=FS, seed=seed, dot_s=0.5)


def _fixed_displays(rows):
    """three fixed displays whose range cuts through the rows' levels: log, log with a threshold, linear"""
    db = 10 * np.log10(np.maximum(rows.astype(np.float64), 1e-30))
    lo, hi = float(np.floor(np.percentile(db, 5))), float(np.ceil(np.percentile(db, 99.5)))
    return (dict(log_scale=True, max_level_db=hi, min_level_db=lo, thr_level=0.0),
            dict(log_scale=True, max_level_db=hi, min_level_db=lo, thr_level=12.5),
            dict(log_scale=False, max_level_db=hi, min_level_db=lo - 10.0, thr_level=0.0))


def _oracle(rows, overlap, disp, autoscale, first_frame=0, agc_state=(0.0, 0.0)):
    return O.display_levels(rows, rows, overlap, disp.get("log_scale", True), autoscale, disp.get("max_level_db", -20.0),
                            disp.get("min_level_db", -80.0), disp.get("thr_level", 0.0), first_frame, agc_state)


# ------------------------------------------------------------------------------------------------ CPU
def test_iq_level_pixel_addressing_emulation(tmp_path):
    """every pixel written once, pixel of bin k = n - 1 - ((k + n/2) mod n), a warp's byte stores consecutive"""
    exe = str(tmp_path / "emu_iq_levels")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "emu", "emu_iq_levels.cpp")],
                   check=True)
    res = subprocess.run([exe], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout
    rows = [[int(v) for v in ln.split()] for ln in res.stdout.strip().splitlines()]
    assert [r[0] for r in rows] == list(FUSED_N)
    assert all(r[1:] == [0, 0, 0] for r in rows), res.stdout


# ------------------------------------------------------------------------------------------------ GPU: fixed range
FIXED = ([(n, ov, False) for n in FUSED_N for ov in FUSED_OV]
         + [(1024, 0.6, False), (16384, 0.5, False), (2048, 0.5, True)])


@pytest.mark.gpu
@pytest.mark.parametrize("n,overlap,forced", FIXED)
def test_iq_fixed_range_levels(dapi, n, overlap, forced):
    p = dapi.IqPlan(n=n, window_type=KAISER, overlap=overlap)
    nframes = 24
    pcm = _iq_int16(p.required_span(0, nframes)[1], seed=n)
    from glfer_b200 import synth
    z = synth.pcm16_to_float(pcm)
    fused_geo = not forced and n <= 8192 and overlap in FUSED_OV
    dapi.force_generic_kernel(forced)
    try:
        rows = p.run(z)
        for disp in _fixed_displays(rows):
            dapi.set_fused_levels(True)
            n0 = dapi.kernel_launches()
            fused = p.run_display(z, autoscale=False, **disp)["levels"]
            n_fused = dapi.kernel_launches() - n0
            fam = dapi.last_kernel_family()
            dapi.set_fused_levels(False)
            n0 = dapi.kernel_launches()
            two = p.run_display(z, autoscale=False, **disp)["levels"]
            n_two = dapi.kernel_launches() - n0
            dapi.set_fused_levels(True)
            want = _oracle(rows, overlap, disp, False)[0]
            assert np.array_equal(fused, want), (disp, int((fused != want).sum()))
            assert np.array_equal(two, want), disp
            assert np.array_equal(dapi.map_levels(rows, **disp), want), disp
            assert fused.min() < fused.max()
            if fused_geo:
                assert fam.startswith("gram_ring_kernel"), fam
                assert n_fused < n_two, (n_fused, n_two)
            # int16 in, the same bytes
            assert np.array_equal(p.run_display(pcm, autoscale=False, **disp)["levels"], fused), disp
    finally:
        dapi.force_generic_kernel(False)
        dapi.set_fused_levels(True)


# ------------------------------------------------------------------------------------------------ GPU: autoscale
def _check_autoscale(plan, z, overlap, nframes, log_scale, split):
    rows = plan.run(z, nframes=nframes)
    d = plan.run_display(z, nframes=nframes, log_scale=log_scale, autoscale=True)
    lev, rng, state = _oracle(rows, overlap, dict(log_scale=log_scale), True)
    assert np.array_equal(d["levels"], lev), int((d["levels"] != lev).sum())
    assert np.array_equal(d["range"], rng)
    assert tuple(float(v) for v in d["agc_state"]) == state
    assert lev.min() < lev.max()
    # two calls chained through agc_state equal one call
    a = plan.run_display(z, nframes=split, log_scale=log_scale, autoscale=True)
    b = plan.run_display(z, first_frame=split, nframes=nframes - split, log_scale=log_scale, autoscale=True,
                         agc_state=a["agc_state"])
    assert np.array_equal(np.concatenate([a["levels"], b["levels"]]), d["levels"])
    assert np.array_equal(np.concatenate([a["range"], b["range"]]), d["range"])


@pytest.mark.gpu
@pytest.mark.parametrize("n,overlap,nframes,log_scale", [(4096, 0.5, 5000, True),      # three chunks, wide rows
                                                          (4096, 0.75, 300, False),
                                                          (1024, 0.5, 3000, True),
                                                          (8192, 0.875, 200, True),
                                                          (16384, 0.5, 60, True)])      # general path
def test_iq_autoscale_levels(dapi, n, overlap, nframes, log_scale):
    from glfer_b200 import synth
    p = dapi.IqPlan(n=n, window_type=HANNING, overlap=overlap)
    z = synth.pcm16_to_float(_iq_int16(p.required_span(0, nframes)[1], seed=11))
    _check_autoscale(p, z, overlap, nframes, log_scale, nframes // 3 + 1)


@pytest.mark.gpu
@pytest.mark.parametrize("iq,n,overlap,nframes", [(False, 4096, 0.5, 600), (True, 4096, 0.5, 400),
                                                  (False, 1024, 0.75, 300), (True, 1024, 0.0, 100)])
def test_zoom_autoscale_levels(dapi, iq, n, overlap, nframes):
    """several chunks (~32 MiB of input each) of a zoom at D = 16, real and I/Q"""
    from glfer_b200 import synth
    p = dapi.ZoomPlan(n=n, decim=16, window_type=HANNING, overlap=overlap, center_hz=-1000.0 if iq else 1000.0,
                      sample_rate=FS, iq=iq)
    span = p.required_span(0, nframes)[1]
    if iq:
        x = synth.pcm16_to_float(_iq_int16(span, seed=5))
    else:
        x = synth.qrss_stream(span, fs=FS, dot_s=0.5)
    _check_autoscale(p, x, overlap, nframes, True, nframes // 2 + 1)
    # int16 in, the same bytes
    pcm = _iq_int16(span, seed=5) if iq else synth.qrss_stream_int16(span, fs=FS, dot_s=0.5)
    assert np.array_equal(p.run_display(pcm, nframes=nframes)["levels"], p.run_display(x, nframes=nframes)["levels"])


# ------------------------------------------------------------------------------------------------ GPU: RGB
@pytest.mark.gpu
def test_rgb_is_the_palette_of_the_levels(dapi):
    from glfer_b200 import synth
    pal = dapi.palette(7)
    p = dapi.IqPlan(n=2048, window_type=HANNING, overlap=0.5)
    z = synth.pcm16_to_float(_iq_int16(p.required_span(0, 40)[1]))
    rows = p.run(z)
    for disp in (dict(autoscale=True), dict(autoscale=False, **_fixed_displays(rows)[0])):
        d = p.run_display(z, colortab=pal, want_rgb=True, **disp)
        assert np.array_equal(d["rgb"], pal[d["levels"]])
        assert np.array_equal(d["levels"], _oracle(rows, 0.5, disp, disp["autoscale"])[0])
    q = dapi.ZoomPlan(n=512, decim=16, window_type=HANNING, overlap=0.5, center_hz=-800.0, sample_rate=FS, iq=True)
    zq = synth.pcm16_to_float(_iq_int16(q.required_span(0, 30)[1]))
    d = q.run_display(zq, colortab=pal, want_rgb=True)
    assert np.array_equal(d["rgb"], pal[d["levels"]])
    assert np.array_equal(d["levels"], _oracle(q.run(zq), 0.5, {}, True)[0])


# ------------------------------------------------------------------------------------------------ GPU: argument checks
@pytest.mark.gpu
def test_display_argument_checks(dapi):
    lib = dapi.lib()
    iqp = dapi.IqPlan(n=256, window_type=HANNING, overlap=0.5)
    real = dapi.ZoomPlan(n=256, decim=16, center_hz=800.0, sample_rate=FS)
    zq = dapi.ZoomPlan(n=256, decim=16, center_hz=-800.0, sample_rate=FS, iq=True)
    nf = 4
    levels = np.empty((nf, 256), np.uint8)
    rgb = np.empty((nf, 256, 3), np.uint8)
    pal = dapi.palette(0)
    auto = dapi.DisplayConfig(1, 1, -20.0, -80.0, 0.0, None)
    fixed = dapi.DisplayConfig(1, 0, -20.0, -80.0, 0.0, None)
    hi = max(real.required_span(0, nf + 2)[1], iqp.required_span(0, nf + 2)[1])
    x = np.zeros(2 * hi, np.float32)
    pcm = np.zeros(2 * hi, np.int16)
    state = np.zeros(2, np.float32)
    cases = [(lib.glfer_iq_run_display, iqp), (lib.glfer_iq_run_display_pcm16, iqp),
             (lib.glfer_zoom_run_display, real), (lib.glfer_zoom_run_display_pcm16, real),
             (lib.glfer_zoom_run_display_iq, zq), (lib.glfer_zoom_run_display_iq_pcm16, zq)]
    for fn, plan in cases:
        buf = pcm if fn.__name__.endswith("pcm16") else x
        ok = fn(plan._h, buf.ctypes.data, 0, hi, 0, nf, C.byref(auto), None, levels.ctypes.data, None, None)
        assert ok == 0, (fn.__name__, dapi.last_error())
        # autoscale from a later frame without the carried state
        assert fn(plan._h, buf.ctypes.data, 0, hi, 1, nf, C.byref(auto), None, levels.ctypes.data, None, None) == -2
        assert fn(plan._h, buf.ctypes.data, 0, hi, 1, nf, C.byref(auto), state.ctypes.data, levels.ctypes.data, None,
                  None) == 0
        # RGB without a palette
        assert fn(plan._h, buf.ctypes.data, 0, hi, 0, nf, C.byref(fixed), None, levels.ctypes.data, rgb.ctypes.data,
                  None) == -2
        # input that does not cover the required span
        lo_, hi_ = plan.required_span(2, nf)
        assert fn(plan._h, buf.ctypes.data, 0, hi_ - 1, 2, nf, C.byref(fixed), None, levels.ctypes.data, None,
                  None) == -2
        assert fn(plan._h, buf.ctypes.data, max(lo_, 0) + 1, hi_, 2, nf, C.byref(fixed), None, levels.ctypes.data, None,
                  None) == -2
    # the zoom's real entry points reject I/Q plans, and the reverse
    for fn, plan, buf in ((lib.glfer_zoom_run_display, zq, x), (lib.glfer_zoom_run_display_pcm16, zq, pcm),
                          (lib.glfer_zoom_run_display_iq, real, x), (lib.glfer_zoom_run_display_iq_pcm16, real, pcm)):
        assert fn(plan._h, buf.ctypes.data, 0, hi, 0, nf, C.byref(fixed), None, levels.ctypes.data, None, None) == -2
    d = dapi.DisplayConfig(1, 0, -20.0, -80.0, 0.0, pal.ctypes.data)
    assert lib.glfer_iq_run_display(iqp._h, x.ctypes.data, 0, hi, 0, nf, C.byref(d), None, levels.ctypes.data,
                                    rgb.ctypes.data, None) == 0
