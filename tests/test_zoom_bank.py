"""Zoom channel banks (glfer_zoom_plan_create_bank[_mtm]): C centres of one config decimated together.

CPU: the argument checks that precede every device call.  GPU: every channel of a bank is bit-identical to a
single-centre zoom plan at its centre -- rows, multitaper rows, F rows, display levels, RGB, display range and the
carried AGC state -- for real and I/Q input, float and int16, over decimations, sizes, overlaps and channel counts;
runs of several chunks, split calls and origins beyond 2^32 agree with one call; two channels against the float64
oracles; the launches per chunk do not grow with C; and the entry points' rejections."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from parity import assert_psd_close  # noqa: E402
from test_zoom import oracle  # noqa: E402
from test_iq_mtm import zoom_frames, mtm_rows  # noqa: E402

FS = 48000.0
HANNING, RECTANGULAR, KAISER = 0, 5, 7
EINVAL = -2


@pytest.fixture(scope="module")
def bapi():
    from glfer_b200 import build
    build.build()
    from glfer_b200 import api
    return api


@pytest.fixture(scope="module")
def bgpu(bapi):
    if bapi.device_count() < 1:
        pytest.fail("no CUDA device visible: the zoom bank GPU tests need a B200 (no CPU fallback exists)")
    return bapi


def _input(count, iq, pcm16, seed):
    """a test stream of `count` (complex) samples in the format of the plan's entry points"""
    rng = np.random.default_rng(seed)
    if pcm16:
        return rng.integers(-20000, 20000, size=(count, 2) if iq else count, dtype=np.int16)
    if iq:
        return (0.3 * rng.standard_normal(2 * count)).astype(np.float32).view(np.complex64)
    from glfer_b200 import synth
    return synth.qrss_stream(count, fs=int(FS), seed=seed, dot_s=0.5)


def _singles(api, centers, **kw):
    return [api.ZoomPlan(center_hz=float(c), **kw) for c in centers]


# ------------------------------------------------------------------------------------------------ CPU
def _cfg(api, **kw):
    c = api.ZoomConfig()
    api.lib().glfer_zoom_config_default(C.byref(c))
    for k, v in kw.items():
        setattr(c, k, v)
    return c


def test_bank_validation_precedes_device_calls(bapi):
    lib = bapi.lib()
    cfg = _cfg(bapi, n=256, decim=16)
    h = C.c_void_p()
    ok = np.array([800.0, 1200.0], np.float64)
    cases = [
        (ok.ctypes.data, 0, 0, "channels"), (ok.ctypes.data, 33, 0, "channels"), (None, 2, 0, "null"),
        (np.array([800.0, -1.0]).ctypes.data, 2, 0, "centre"), (np.array([FS / 2 + 1.0]).ctypes.data, 1, 0, "centre"),
        (np.array([-FS / 2 - 1.0, 0.0]).ctypes.data, 2, 1, "I/Q centre"), (np.array([np.nan]).ctypes.data, 1, 1, "centre"),
    ]
    keep = [ok]
    for ptr, nchan, iq, msg in cases:
        assert lib.glfer_zoom_plan_create_bank(C.byref(cfg), ptr, nchan, iq, C.byref(h)) == EINVAL
        assert msg in bapi.last_error(), bapi.last_error()
        assert not h.value
        assert lib.glfer_zoom_plan_create_bank_mtm(C.byref(cfg), ptr, nchan, iq, 4.0, 3, C.byref(h)) == EINVAL
        assert msg in bapi.last_error(), bapi.last_error()
    # the bounds themselves pass validation: what follows is the device (absent on a CPU-only machine)
    edges = np.array([0.0, FS / 2] * 16, np.float64)
    for ptr, nchan, iq in ((edges.ctypes.data, 32, 0), (np.array([-FS / 2, FS / 2]).ctypes.data, 2, 1)):
        rc = lib.glfer_zoom_plan_create_bank(C.byref(cfg), ptr, nchan, iq, C.byref(h))
        if rc == 0:
            assert lib.glfer_zoom_channels(h) == nchan
            lib.glfer_zoom_plan_destroy(h)
            h = C.c_void_p()
        else:
            assert "no CUDA device" in bapi.last_error(), bapi.last_error()
    del keep


# ------------------------------------------------------------------------------------------------ GPU
BITS = [
    # iq, pcm16, multitaper, decim, n, overlap, centres
    (False, False, False, 2, 32, 0.0, [0.0, 800.0, FS / 2]),
    (False, True, False, 7, 64, 0.75, [800.0, 800.0, 10.0, 1234.5, 0.0, FS / 2, 23999.0, 800.0]),
    (False, False, False, 1024, 2048, 0.5, [700.0]),
    (False, True, True, 256, 16384, 0.75, [800.0, 1000.0, FS / 2]),
    (False, False, True, 16, 1024, 0.5, [float(c) for c in np.linspace(0.0, FS / 2, 32)]),
    (True, False, False, 16, 1024, 0.5, [-FS / 2, FS / 2, 0.0, -1234.5, 800.0, 800.0, 5000.0, -7.25]),
    (True, True, False, 256, 4096, 0.5, [float(c) for c in np.linspace(-3000.0, 3000.0, 32)]),
    (True, False, True, 1024, 256, 0.0, [-800.0, 0.0, 800.0, -FS / 2, FS / 2, 1.5, -1.5, 800.0]),
    (True, True, True, 7, 128, 0.75, [-1234.5]),
    (True, False, False, 2, 16384, 0.0, [-FS / 2, 100.0, FS / 2]),
]


@pytest.mark.gpu
@pytest.mark.parametrize("iq,pcm16,mtm,decim,n,overlap,centers", BITS)
def test_bank_channels_are_single_plans(bgpu, iq, pcm16, mtm, decim, n, overlap, centers):
    kw = dict(n=n, decim=decim, window_type=KAISER if decim == 7 else HANNING, overlap=overlap, sample_rate=FS, iq=iq,
              multitaper=mtm, mtm_kmax=3)
    bank = bgpu.ZoomPlan(center_hz=centers, **kw)
    assert bank.channels == len(centers)
    nframes = 5 if n >= 4096 else 11
    x = _input(bank.required_span(0, nframes)[1], iq, pcm16, seed=decim * 7 + n)
    rows = bank.run(x)
    assert rows.shape == (len(centers), nframes, n)
    singles = _singles(bgpu, centers, **kw)
    np.testing.assert_array_equal(bank.centers_hz(), [s.center_hz() for s in singles])
    assert bank.center_hz() == singles[0].center_hz()
    for c, s in enumerate(singles):
        assert np.array_equal(rows[c], s.run(x)), c
    if mtm:
        f = bank.run_mtm_ftest(x)
        assert np.array_equal(f["psd"], rows)
        for c, s in enumerate(singles):
            assert np.array_equal(f["ftest"][c], s.run_mtm_ftest(x, want_psd=False)["ftest"], equal_nan=True), c


@pytest.mark.gpu
@pytest.mark.parametrize("iq,pcm16,mtm,decim,n,overlap,nframes", [
    (False, False, False, 16, 1024, 0.5, 40), (True, True, True, 64, 512, 0.75, 60), (False, True, True, 7, 64, 0.0, 30)])
def test_bank_display_is_single_plans(bgpu, iq, pcm16, mtm, decim, n, overlap, nframes):
    centers = [-900.0, 0.0, 900.0, 900.0] if iq else [0.0, 900.0, 900.0, 3000.0]
    kw = dict(n=n, decim=decim, overlap=overlap, sample_rate=FS, iq=iq, multitaper=mtm, mtm_kmax=3)
    bank = bgpu.ZoomPlan(center_hz=centers, **kw)
    singles = _singles(bgpu, centers, **kw)
    x = _input(bank.required_span(0, nframes)[1], iq, pcm16, seed=11)
    pal = bgpu.palette(7)
    for log_scale in (True, False):
        fixed = dict(log_scale=log_scale, autoscale=False, max_level_db=-10.0, min_level_db=-90.0, thr_level=0.1)
        d = bank.run_display(x, colortab=pal, want_rgb=True, **fixed)
        assert d["levels"].shape == (len(centers), nframes, n) and d["rgb"].shape == (len(centers), nframes, n, 3)
        for c, s in enumerate(singles):
            e = s.run_display(x, colortab=pal, want_rgb=True, **fixed)
            assert np.array_equal(d["levels"][c], e["levels"]) and np.array_equal(d["rgb"][c], e["rgb"]), c
        d = bank.run_display(x, log_scale=log_scale, autoscale=True, colortab=pal, want_rgb=True)
        assert d["range"].shape == (len(centers), nframes, 2) and d["agc_state"].shape == (len(centers), 2)
        split = nframes // 3 + 1
        a = bank.run_display(x, nframes=split, log_scale=log_scale, autoscale=True)
        b = bank.run_display(x, first_frame=split, nframes=nframes - split, log_scale=log_scale, autoscale=True,
                             agc_state=a["agc_state"])
        assert np.array_equal(np.concatenate([a["levels"], b["levels"]], axis=1), d["levels"])
        assert np.array_equal(np.concatenate([a["range"], b["range"]], axis=1), d["range"])
        assert np.array_equal(b["agc_state"], d["agc_state"])
        for c, s in enumerate(singles):
            e = s.run_display(x, log_scale=log_scale, autoscale=True, colortab=pal, want_rgb=True)
            assert np.array_equal(d["levels"][c], e["levels"]), c
            assert np.array_equal(d["rgb"][c], e["rgb"]), c
            assert np.array_equal(d["range"][c], e["range"]), c
            assert np.array_equal(d["agc_state"][c], e["agc_state"]), c


@pytest.mark.gpu
@pytest.mark.parametrize("iq,nframes", [(False, 5000), (True, 2500)])
def test_bank_chunks_and_split_calls(bgpu, iq, nframes):
    # ~32 MiB of input per chunk: 2048 (real) or 1024 (I/Q) frames here, so three chunks and two device-side carries
    centers = [-800.0, 350.0, 800.0] if iq else [0.0, 350.0, 800.0]
    kw = dict(n=64, decim=256, window_type=HANNING, overlap=0.75, sample_rate=FS, iq=iq)
    bank = bgpu.ZoomPlan(center_hz=centers, **kw)
    x = _input(bank.required_span(0, nframes)[1], iq, False, seed=3)
    whole = bank.run(x)
    parts = [bank.run(x, first_frame=a, nframes=min(1000, nframes - a)) for a in range(0, nframes, 1000)]
    assert np.array_equal(np.concatenate(parts, axis=1), whole)
    for c, s in enumerate(_singles(bgpu, centers, **kw)):
        assert np.array_equal(whole[c], s.run(x)), c
    lo, hi = bank.required_span(7, 23)
    part = bank.run(np.ascontiguousarray(x[lo:hi]), origin=lo, first_frame=7, nframes=23)
    assert np.array_equal(part, whole[:, 7:30])


@pytest.mark.gpu
@pytest.mark.parametrize("iq", [False, True])
def test_bank_frames_beyond_sample_2_pow_32(bgpu, iq):
    n, decim = 1024, 16
    centers = [-800.0, 800.0] if iq else [800.0, 6000.0]
    kw = dict(n=n, decim=decim, window_type=HANNING, overlap=0.5, sample_rate=FS, iq=iq)
    bank = bgpu.ZoomPlan(center_hz=centers, **kw)
    first = ((1 << 32) + 12345) // (bank.hop * decim) + 3
    nframes = 8
    lo, hi = bank.required_span(first, nframes)
    assert lo > (1 << 32)
    x = _input(hi - lo, iq, False, seed=7)
    got = bank.run(x, origin=lo, first_frame=first, nframes=nframes)
    for c, s in enumerate(_singles(bgpu, centers, **kw)):
        assert np.array_equal(got[c], s.run(x, origin=lo, first_frame=first, nframes=nframes)), c
    a = bank.run(x, origin=lo, first_frame=first, nframes=3)
    lo2 = bank.required_span(first + 3, nframes - 3)[0]
    b = bank.run(np.ascontiguousarray(x[lo2 - lo:]), origin=lo2, first_frame=first + 3, nframes=nframes - 3)
    assert np.array_equal(np.concatenate([a, b], axis=1), got)


@pytest.mark.gpu
def test_bank_oracle_parity(bgpu):
    n, decim, nframes = 1024, 16, 12
    centers = [800.0, 6000.0]
    bank = bgpu.ZoomPlan(n=n, decim=decim, window_type=HANNING, overlap=0.5, center_hz=centers, sample_rate=FS)
    x = _input(bank.required_span(0, nframes)[1], False, False, seed=5)
    got = bank.run(x)
    for c, fc in enumerate(centers):
        ref = oracle(bgpu, x, 0, n, decim, HANNING, 0.5, fc, 0, nframes)
        assert_psd_close(got[c], ref, f"bank channel {c} at {fc} Hz")
    # I/Q multitaper bank against the multitaper oracle of the decimated frames
    centers = [-1234.5, 2000.0]
    bank = bgpu.ZoomPlan(n=256, decim=decim, overlap=0.5, center_hz=centers, sample_rate=FS, iq=True, multitaper=True,
                         mtm_kmax=3)
    z = _input(bank.required_span(0, nframes)[1], True, False, seed=6)
    got = bank.run(z)
    tapers, lam = bank.tapers()
    for c, fc in enumerate(centers):
        frames = zoom_frames(bgpu, z, 0, 256, decim, 0.5, fc, 0, nframes)
        assert_psd_close(got[c], mtm_rows(frames, tapers, lam), f"I/Q multitaper bank channel {c} at {fc} Hz")


@pytest.mark.gpu
@pytest.mark.parametrize("mtm", [False, True])
def test_bank_launches_do_not_grow_with_channels(bgpu, mtm):
    kw = dict(n=512, decim=64, overlap=0.5, sample_rate=FS, iq=True, multitaper=mtm, mtm_kmax=7)
    one = bgpu.ZoomPlan(center_hz=[800.0], **kw)
    eight = bgpu.ZoomPlan(center_hz=[float(c) for c in np.linspace(-4000.0, 4000.0, 8)], **kw)
    nframes = 3000                                   # two chunks
    z = _input(one.required_span(0, nframes)[1], True, True, seed=9)
    counts = []
    for p in (one, eight, one, eight):
        k0 = bgpu.kernel_launches()
        p.run(z)
        counts.append(bgpu.kernel_launches() - k0)
    assert counts[0] == counts[1] == counts[2] == counts[3], counts


@pytest.mark.gpu
def test_bank_entry_points_and_queries(bgpu):
    lib = bgpu.lib()
    with pytest.raises(bgpu.GlferError):
        bgpu.ZoomPlan(center_hz=[])
    with pytest.raises(bgpu.GlferError):
        bgpu.ZoomPlan(center_hz=[800.0] * 33)
    with pytest.raises(bgpu.GlferError):
        bgpu.ZoomPlan(center_hz=[800.0, -800.0])
    with pytest.raises(bgpu.GlferError):
        bgpu.ZoomPlan(center_hz=[800.0, FS], iq=True)
    real = bgpu.ZoomPlan(n=256, decim=16, center_hz=[800.0, 900.0], sample_rate=FS)
    iq = bgpu.ZoomPlan(n=256, decim=16, center_hz=[-800.0, 900.0], sample_rate=FS, iq=True, multitaper=True)
    assert real.channels == 2 and lib.glfer_zoom_channels(real._h) == 2
    assert np.isnan(lib.glfer_zoom_channel_center_hz(real._h, 2)) and np.isnan(lib.glfer_zoom_channel_center_hz(real._h, -1))
    assert bgpu.ZoomPlan(n=256, decim=16, center_hz=800.0).channels == 1
    hi = real.required_span(0, 2)[1]
    x = np.zeros(2 * hi, np.float32)
    pcm = np.zeros(2 * hi, np.int16)
    rows = np.empty((2, 2, 256), np.float32)
    levels = np.empty((2, 2, 256), np.uint8)
    disp = bgpu.DisplayConfig(1, 1, -20.0, -80.0, 0.0, None)
    for fn, plan, buf in ((lib.glfer_zoom_run, iq, x), (lib.glfer_zoom_run_pcm16, iq, pcm),
                          (lib.glfer_zoom_run_iq, real, x), (lib.glfer_zoom_run_iq_pcm16, real, pcm)):
        assert fn(plan._h, buf.ctypes.data, 0, hi, 0, 2, rows.ctypes.data) == EINVAL
    for fn, plan, buf in ((lib.glfer_zoom_run_display, iq, x), (lib.glfer_zoom_run_display_iq_pcm16, real, pcm)):
        assert fn(plan._h, buf.ctypes.data, 0, hi, 0, 2, C.byref(disp), None, levels.ctypes.data, None, None) == EINVAL
    for fn, plan, buf in ((lib.glfer_zoom_run_mtm_ftest, iq, x), (lib.glfer_zoom_run_iq_mtm_ftest, real, x)):
        assert fn(plan._h, buf.ctypes.data, 0, hi, 0, 2, rows.ctypes.data, None) == EINVAL
