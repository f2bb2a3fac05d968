"""Multitaper I/Q and zoom plans (glfer_iq_plan_create_mtm, glfer_zoom_plan_create[_iq]_mtm).

CPU: the argument checks, which reject a plan before any device is touched.  GPU: rows against a float64
restatement of the contract in include/glfer_b200.h, built from the plan's own tapers, on the fused and the general
path; the tapers against the real multitaper plan's and the oracle's DPSS; the I/Q row of (x, 0) against the real
multitaper row of x; the variance reduction on white noise; bit-identical rows under splitting, chunking, int16 input,
a stereo WAV and origins beyond 2^32; the zoom's parity, real-against-I/Q identity and chunking; the waterfall against
the oracle's display mapping of the plan's own rows; and the zoom's entry-point checks."""
import ctypes as C
import math
import os
import sys

import numpy as np
import pytest
from scipy.signal import upfirdn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from oracle import glfer_oracle as O  # noqa: E402
from parity import assert_psd_close  # noqa: E402

FS = 48000.0
HANNING = 0


@pytest.fixture(scope="module")
def mapi():
    from glfer_b200 import build
    build.build()
    from glfer_b200 import api
    return api


@pytest.fixture(scope="module")
def mgpu(mapi):
    if mapi.device_count() < 1:
        pytest.fail("no CUDA device visible: the multitaper I/Q GPU tests need a B200 (no CPU fallback exists)")
    return mapi


def _iq(n, seed=0x5EED):
    from glfer_b200 import synth
    return synth.iq_stream(n, fs=int(FS), seed=seed, dot_s=0.5)


def _step(center, fs=FS):
    v = center / fs * 2.0 ** 32
    return int(math.copysign(math.floor(abs(v) + 0.5), v)) % (1 << 32)        # llround, modulo 2^32


def mtm_rows(frames, tapers, lam):
    """the contract's row of each complex frame: sum_k |FFT(v_k z_f)|^2 / (n lambda_k), fft-shifted"""
    n = frames.shape[1]
    acc = np.zeros(frames.shape)
    for v, la in zip(tapers, lam):
        acc += np.abs(np.fft.fft(v[None, :] * frames, axis=1)) ** 2 / (n * la)
    return np.fft.fftshift(acc, axes=1)


def iq_frames(z, origin, n, hop, first_frame, nframes):
    """frame f = z[f hop - (n - hop) .. f hop + hop), zeros before sample 0 (tests/test_iq.py's gathering)"""
    s0 = (first_frame + np.arange(nframes, dtype=np.int64)) * hop - (n - hop)
    idx = s0[:, None] + np.arange(n, dtype=np.int64)[None, :]
    seg = np.zeros(idx.shape, dtype=np.complex128)
    ok = idx >= 0
    seg[ok] = z[idx[ok] - origin].astype(np.complex128)
    return seg


def zoom_frames(api, z, origin, n, decim, overlap, center, first_frame, nframes):
    """the decimated frames of the zoom contract with complex x (tests/test_iq.py's decimation, signed step)"""
    h = api.zoom_taps(decim).astype(np.float64)
    K = 16 * decim
    hop = api.host_hop(n, overlap)
    step = np.uint64(_step(center))
    m_lo = first_frame * hop - (n - hop)
    m0 = max(m_lo, 0)
    m_hi = (first_frame + nframes) * hop
    a, b = m0 * decim - K, (m_hi - 1) * decim + K + 1
    idx = np.arange(a, b, dtype=np.int64)
    xs = np.zeros(b - a, dtype=np.complex128)
    ok = idx >= 0
    xs[ok] = z[idx[ok] - origin].astype(np.complex128)
    ph = ((np.where(ok, idx, 0).astype(np.uint64) * step) & np.uint64(0xFFFFFFFF)).astype(np.float64) / 2.0 ** 32
    v = xs * np.exp(-2j * np.pi * ph)
    y = upfirdn(h, v, 1, decim)[2 * K // decim: 2 * K // decim + (m_hi - m0)]
    yfull = np.zeros(m_hi - m_lo, dtype=np.complex128)
    yfull[m0 - m_lo:] = y
    s = (first_frame + np.arange(nframes)) * hop - (n - hop) - m_lo
    return np.stack([yfull[q:q + n] for q in s])


def _fused(n, hop):
    return n <= 8192 and (n - hop) % hop == 0 and any(hop == (n // 16) << s for s in range(5))


# ------------------------------------------------------------------------------------------------ CPU
def test_mtm_argument_checks(mapi):
    """mtm_kmax outside 0..31, mtm_w not > 0 and a non-positive DPSS eigenvalue are rejected before any device use"""
    bad = [dict(mtm_kmax=-1), dict(mtm_kmax=32), dict(mtm_w=0.0), dict(mtm_w=-1.0), dict(mtm_w=float("nan")),
           dict(n=64, mtm_w=1.0, mtm_kmax=31)]
    _, lam = mapi.host_dpss(64, 1.0, 31)
    assert (lam <= 0).any()                                        # the last pair has a non-positive eigenvalue
    for kw in bad:
        args = dict(n=256, mtm_w=4.0, mtm_kmax=7)
        args.update(kw)
        for make in (lambda a: mapi.IqPlan(multitaper=True, **a),
                     lambda a: mapi.ZoomPlan(decim=16, multitaper=True, **a),
                     lambda a: mapi.ZoomPlan(decim=16, center_hz=-800.0, iq=True, multitaper=True, **a)):
            with pytest.raises(mapi.GlferError):
                make(args)
            assert "mtm" in mapi.last_error() or "eigenvalue" in mapi.last_error(), mapi.last_error()


# ------------------------------------------------------------------------------------------------ GPU: I/Q parity
KW = [(1, 4.0), (4, 2.5), (4, 4.0), (8, 2.5), (8, 4.0), (16, 2.5), (16, 4.0), (1, 2.5)]
PARITY = [(n, ov) for n in (32, 256, 1024, 2048, 4096, 8192, 16384) for ov in (0.0, 0.5, 0.75, 0.6)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,overlap", PARITY)
def test_iq_mtm_oracle_parity(mgpu, n, overlap):
    nframes = 6 if n >= 8192 else 12
    for kp, w in KW:
        p = mgpu.IqPlan(n=n, overlap=overlap, multitaper=True, mtm_w=w, mtm_kmax=kp - 1)
        z = _iq(p.required_span(0, nframes)[1], seed=n + kp)
        tapers, lam = p.tapers()
        ref = mtm_rows(iq_frames(z, 0, n, p.hop, 0, nframes), tapers, lam)
        fused = _fused(n, p.hop)
        for forced in ([False, True] if fused else [True]):
            mgpu.force_generic_kernel(forced)
            try:
                got = p.run(z)
                fam = mgpu.last_kernel_family()
            finally:
                mgpu.force_generic_kernel(False)
            assert fam.startswith("gram_kernel" if forced or not fused else "gram_ring_kernel"), fam
            assert_psd_close(got, ref, f"iq mtm n={n} ov={overlap} K'={kp} NW={w} general={forced}")
        p.close()


# ------------------------------------------------------------------------------------------------ GPU: tapers
@pytest.mark.gpu
@pytest.mark.parametrize("n,w,kmax", [(256, 4.0, 7), (1024, 2.5, 3), (4096, 4.0, 15), (512, 3.0, 0)])
def test_tapers_are_the_real_plans(mgpu, n, w, kmax):
    real = mgpu.GramPlan(n=n, mode=mgpu.MODE_MTM, overlap=0.5, mtm_w=w, mtm_kmax=kmax)
    tr, lr = real.tapers()
    plans = [mgpu.IqPlan(n=n, multitaper=True, mtm_w=w, mtm_kmax=kmax),
             mgpu.ZoomPlan(n=n, decim=16, multitaper=True, mtm_w=w, mtm_kmax=kmax),
             mgpu.ZoomPlan(n=n, decim=16, center_hz=-800.0, iq=True, multitaper=True, mtm_w=w, mtm_kmax=kmax)]
    for p in plans:
        t, lam = p.tapers()
        assert t.shape == (kmax + 1, n) and lam.shape == (kmax + 1,)
        assert np.array_equal(t, tr) and np.array_equal(lam, lr)
    tb, lb = O.gl_dpss(n, w, kmax)                                 # tolerances of tests/test_host.py
    assert np.allclose(lr, lb, rtol=1e-9, atol=1e-15)
    sgn = np.sign(np.sum(tr * tb, axis=1))
    assert np.max(np.abs(tr * sgn[:, None] - tb)) < 1e-7
    # periodogram plans have no tapers to report
    for p in (mgpu.IqPlan(n=n), mgpu.ZoomPlan(n=n, decim=16), mgpu.ZoomPlan(n=n, decim=16, center_hz=-800.0, iq=True)):
        with pytest.raises(mgpu.GlferError):
            p.tapers()


# ------------------------------------------------------------------------------------------------ GPU: estimator
@pytest.mark.gpu
@pytest.mark.parametrize("n,overlap,w,kmax", [(1024, 0.5, 4.0, 7), (4096, 0.75, 2.5, 3), (256, 0.0, 4.0, 15)])
def test_iq_row_of_real_input_is_the_real_multitaper_row(mgpu, n, overlap, w, kmax):
    from glfer_b200 import synth
    real = mgpu.GramPlan(n=n, mode=mgpu.MODE_MTM, overlap=overlap, sub_mean=False, mtm_w=w, mtm_kmax=kmax)
    q = mgpu.IqPlan(n=n, overlap=overlap, multitaper=True, mtm_w=w, mtm_kmax=kmax)
    nframes = 20
    x = synth.qrss_stream(q.required_span(0, nframes)[1], fs=int(FS), dot_s=0.5)
    rr = real.run(x)["psd"][:nframes].astype(np.float64)
    rq = q.run(np.stack([x, np.zeros_like(x)], axis=1)).astype(np.float64)
    k = np.arange(n // 2 + 1)
    assert_psd_close(rq[:, (n // 2 + k) % n], rr, "iq (x, 0) against the real multitaper row")
    assert_psd_close(rq[:, (n // 2 - k) % n], rq[:, (n // 2 + k) % n], "mirror symmetry about n/2")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1024, 4096])
def test_multitaper_cuts_the_variance_of_white_noise(mgpu, n):
    rng = np.random.default_rng(5)
    nframes = 64
    per = mgpu.IqPlan(n=n, window_type=HANNING, overlap=0.5)
    mtm = mgpu.IqPlan(n=n, overlap=0.5, multitaper=True, mtm_w=4.0, mtm_kmax=7)
    span = per.required_span(0, nframes)[1]
    z = (rng.standard_normal(span) + 1j * rng.standard_normal(span)).astype(np.complex64)
    rp = per.run(z)[2:].astype(np.float64)                         # past the zero history
    rm = mtm.run(z)[2:].astype(np.float64)

    def spread(r):
        return float(np.mean(r.std(axis=1) / r.mean(axis=1)))
    assert spread(rm) <= 0.5 * spread(rp), (spread(rm), spread(rp))
    # the level the header states: sum_k 1 / lambda_k against the window's energy
    _, lam = mtm.tapers()
    w = mgpu.host_window(n, HANNING).astype(np.float64)
    want_db = 10 * np.log10(np.sum(1.0 / lam) / np.sum(w * w))
    got_db = 10 * np.log10(rm.mean() / rp.mean())
    assert abs(got_db - want_db) < 0.3, (got_db, want_db)


# ------------------------------------------------------------------------------------------------ GPU: invariance
@pytest.mark.gpu
@pytest.mark.parametrize("n,overlap", [(1024, 0.5), (1024, 0.6), (4096, 0.75)])
def test_iq_mtm_split_and_pcm16_are_bit_identical(mgpu, n, overlap):
    from glfer_b200 import synth
    p = mgpu.IqPlan(n=n, overlap=overlap, multitaper=True, mtm_w=4.0, mtm_kmax=7)
    nframes = 40
    pcm = synth.iq_stream_int16(p.required_span(0, nframes)[1], fs=int(FS), dot_s=0.5)
    zf = synth.pcm16_to_float(pcm)
    whole = p.run(zf)
    assert whole.shape == (nframes, n)
    assert np.array_equal(p.run(np.ascontiguousarray(zf).view(np.complex64)[:, 0]), whole)
    assert np.array_equal(p.run(pcm), whole)
    parts = []
    for a, b in ((0, 1), (1, 7), (7, 23), (23, 40)):
        lo, hi = p.required_span(a, b - a)
        lo = max(lo, 0)
        parts.append(p.run(np.ascontiguousarray(zf[lo:hi]), origin=lo, first_frame=a, nframes=b - a))
    assert np.array_equal(np.concatenate(parts), whole)


@pytest.mark.gpu
@pytest.mark.parametrize("overlap", [0.5, 0.6])
def test_iq_mtm_run_longer_than_a_chunk(mgpu, overlap):
    p = mgpu.IqPlan(n=1024, overlap=overlap, multitaper=True, mtm_w=4.0, mtm_kmax=3)
    nframes = (5 << 21) // p.hop
    z = _iq(p.required_span(0, nframes)[1], seed=3)
    big = p.run(z)
    step = nframes // 4 + 1
    parts = [p.run(z, first_frame=a, nframes=min(step, nframes - a)) for a in range(0, nframes, step)]
    assert np.array_equal(np.concatenate(parts), big)


@pytest.mark.gpu
def test_iq_mtm_stereo_wav(mgpu, tmp_path):
    from glfer_b200 import synth
    p = mgpu.IqPlan(n=2048, overlap=0.5, multitaper=True, mtm_w=4.0, mtm_kmax=7)
    nframes = 30
    pcm = synth.iq_stream_int16(p.required_span(0, nframes)[1], fs=int(FS), dot_s=0.5)
    path = str(tmp_path / "iq.wav")
    synth.write_wav16(path, pcm.reshape(-1), int(FS), channels=2)
    want = p.run(pcm)
    lib = mgpu.lib()
    wav = mgpu.Wav()
    assert lib.glfer_wav_load(path.encode(), C.byref(wav)) == 0
    try:
        rows = np.empty((nframes, 2048), np.float32)
        mgpu._check(lib.glfer_iq_run_pcm16(p._h, wav.data, 0, wav.nsamples // 2, 0, nframes, rows.ctypes.data))
    finally:
        lib.glfer_wav_free(C.byref(wav))
    assert np.array_equal(rows, want)


@pytest.mark.gpu
@pytest.mark.parametrize("forced", [False, True])
def test_iq_mtm_frames_beyond_sample_2_pow_32(mgpu, forced):
    n, overlap = 2048, 0.75
    p = mgpu.IqPlan(n=n, overlap=overlap, multitaper=True, mtm_w=4.0, mtm_kmax=7)
    first = ((1 << 32) + 12345) // p.hop + 3
    nframes = 8
    lo, hi = p.required_span(first, nframes)
    assert lo > (1 << 32)
    z = _iq(hi - lo, seed=7)
    mgpu.force_generic_kernel(forced)
    try:
        got = p.run(z, origin=lo, first_frame=first, nframes=nframes)
    finally:
        mgpu.force_generic_kernel(False)
    tapers, lam = p.tapers()
    assert_psd_close(got, mtm_rows(iq_frames(z, lo, n, p.hop, first, nframes), tapers, lam), "iq mtm beyond 2^32")


# ------------------------------------------------------------------------------------------------ GPU: zoom
@pytest.mark.gpu
@pytest.mark.parametrize("decim,center,kmax", [(d, c, k) for d in (16, 256) for c in (-1234.5, 800.0) for k in (3, 7)])
def test_iq_mtm_zoom_oracle_parity(mgpu, decim, center, kmax):
    n = 256
    p = mgpu.ZoomPlan(n=n, decim=decim, overlap=0.5, center_hz=center, sample_rate=FS, iq=True, multitaper=True,
                      mtm_w=4.0, mtm_kmax=kmax)
    nframes = 10
    z = _iq(p.required_span(0, nframes)[1])
    tapers, lam = p.tapers()
    ref = mtm_rows(zoom_frames(mgpu, z, 0, n, decim, 0.5, center, 0, nframes), tapers, lam)
    assert_psd_close(p.run(z), ref, f"iq mtm zoom D={decim} c={center} K'={kmax + 1}")


@pytest.mark.gpu
@pytest.mark.parametrize("center", [0.0, 800.0, FS / 2])
def test_mtm_zoom_of_real_input_is_the_real_mtm_zoom(mgpu, center):
    from glfer_b200 import synth
    kw = dict(n=512, decim=16, overlap=0.75, center_hz=center, sample_rate=FS, multitaper=True, mtm_w=4.0, mtm_kmax=7)
    r = mgpu.ZoomPlan(**kw)
    q = mgpu.ZoomPlan(iq=True, **kw)
    nframes = 20
    x = synth.qrss_stream(r.required_span(0, nframes)[1], fs=int(FS), dot_s=0.5)
    want = r.run(x)
    assert np.array_equal(q.run(np.stack([x, np.zeros_like(x)], axis=1)), want)
    pcm = synth.qrss_stream_int16(len(x), fs=int(FS), dot_s=0.5)
    assert np.array_equal(q.run(np.stack([pcm, np.zeros_like(pcm)], axis=1)), r.run(pcm))
    # the real multitaper zoom against the contract, x as (x, 0)
    tapers, lam = r.tapers()
    ref = mtm_rows(zoom_frames(mgpu, x.astype(np.complex128), 0, 512, 16, 0.75, center, 0, nframes), tapers, lam)
    assert_psd_close(want, ref, f"real mtm zoom c={center}")


@pytest.mark.gpu
def test_iq_mtm_zoom_chunking_and_pcm16(mgpu):
    from glfer_b200 import synth
    p = mgpu.ZoomPlan(n=1024, decim=64, overlap=0.75, center_hz=-800.0, sample_rate=FS, iq=True, multitaper=True,
                      mtm_w=4.0, mtm_kmax=7)
    nframes = 40
    pcm = synth.iq_stream_int16(p.required_span(0, nframes)[1], fs=int(FS), dot_s=0.5)
    zf = synth.pcm16_to_float(pcm)
    whole = p.run(zf)
    assert np.array_equal(p.run(pcm), whole)
    parts = []
    for a, b in ((0, 1), (1, 7), (7, 23), (23, 40)):
        lo, hi = p.required_span(a, b - a)
        lo = max(lo, 0)
        parts.append(p.run(np.ascontiguousarray(zf[lo:hi]), origin=lo, first_frame=a, nframes=b - a))
    assert np.array_equal(np.concatenate(parts), whole)
    # runs of several chunks (~32 MiB of input each) against runs of their parts
    q = mgpu.ZoomPlan(n=64, decim=256, overlap=0.75, center_hz=-3000.0, sample_rate=FS, iq=True, multitaper=True,
                      mtm_w=2.5, mtm_kmax=3)
    zl = _iq(q.required_span(0, 3000)[1], seed=3)
    big = q.run(zl)
    parts = [q.run(zl, first_frame=a, nframes=min(1000, 3000 - a)) for a in range(0, 3000, 1000)]
    assert np.array_equal(np.concatenate(parts), big)


@pytest.mark.gpu
def test_mtm_zoom_entry_points(mgpu):
    lib = mgpu.lib()
    real = mgpu.ZoomPlan(n=256, decim=16, center_hz=800.0, sample_rate=FS, multitaper=True)
    iq = mgpu.ZoomPlan(n=256, decim=16, center_hz=-800.0, sample_rate=FS, iq=True, multitaper=True)
    hi = real.required_span(0, 2)[1]
    x = np.zeros(2 * hi, np.float32)
    pcm = np.zeros(2 * hi, np.int16)
    rows = np.empty((2, 256), np.float32)
    levels = np.empty((2, 256), np.uint8)
    disp = mgpu.DisplayConfig(1, 1, -20.0, -80.0, 0.0, None)
    for fn, plan, buf in ((lib.glfer_zoom_run, iq, x), (lib.glfer_zoom_run_pcm16, iq, pcm),
                          (lib.glfer_zoom_run_iq, real, x), (lib.glfer_zoom_run_iq_pcm16, real, pcm)):
        assert fn(plan._h, buf.ctypes.data, 0, hi, 0, 2, rows.ctypes.data) == -2
    for fn, plan, buf in ((lib.glfer_zoom_run_display, iq, x), (lib.glfer_zoom_run_display_pcm16, iq, pcm),
                          (lib.glfer_zoom_run_display_iq, real, x), (lib.glfer_zoom_run_display_iq_pcm16, real, pcm)):
        assert fn(plan._h, buf.ctypes.data, 0, hi, 0, 2, C.byref(disp), None, levels.ctypes.data, None, None) == -2


# ------------------------------------------------------------------------------------------------ GPU: display
def _oracle(rows, overlap, disp, autoscale, first_frame=0, agc_state=(0.0, 0.0)):
    return O.display_levels(rows, rows, overlap, disp.get("log_scale", True), autoscale, disp.get("max_level_db", -20.0),
                            disp.get("min_level_db", -80.0), disp.get("thr_level", 0.0), first_frame, agc_state)


def _fixed(rows, log_scale):
    db = 10 * np.log10(np.maximum(rows.astype(np.float64), 1e-30))
    lo, hi = float(np.floor(np.percentile(db, 5))), float(np.ceil(np.percentile(db, 99.5)))
    return dict(log_scale=log_scale, max_level_db=hi, min_level_db=lo if log_scale else lo - 10.0, thr_level=0.0)


def _check_display(api, plan, z, overlap, nframes):
    rows = plan.run(z, nframes=nframes)
    pal = api.palette(7)
    for log_scale in (True, False):
        # fixed range
        disp = _fixed(rows, log_scale)
        d = plan.run_display(z, nframes=nframes, autoscale=False, colortab=pal, want_rgb=True, **disp)
        want = _oracle(rows, overlap, disp, False)[0]
        assert np.array_equal(d["levels"], want), int((d["levels"] != want).sum())
        assert np.array_equal(d["rgb"], pal[d["levels"]])
        assert want.min() < want.max()
        # autoscale, and two calls chained through agc_state against one
        d = plan.run_display(z, nframes=nframes, log_scale=log_scale, autoscale=True, colortab=pal, want_rgb=True)
        lev, rng, state = _oracle(rows, overlap, dict(log_scale=log_scale), True)
        assert np.array_equal(d["levels"], lev), int((d["levels"] != lev).sum())
        assert np.array_equal(d["range"], rng)
        assert tuple(float(v) for v in d["agc_state"]) == state
        assert np.array_equal(d["rgb"], pal[d["levels"]])
        split = nframes // 3 + 1
        a = plan.run_display(z, nframes=split, log_scale=log_scale, autoscale=True)
        b = plan.run_display(z, first_frame=split, nframes=nframes - split, log_scale=log_scale, autoscale=True,
                             agc_state=a["agc_state"])
        assert np.array_equal(np.concatenate([a["levels"], b["levels"]]), d["levels"])
        assert np.array_equal(np.concatenate([a["range"], b["range"]]), d["range"])


@pytest.mark.gpu
@pytest.mark.parametrize("n,overlap,nframes", [(2048, 0.5, 3000), (1024, 0.6, 200), (16384, 0.5, 40)])
def test_iq_mtm_display(mgpu, n, overlap, nframes):
    from glfer_b200 import synth
    p = mgpu.IqPlan(n=n, overlap=overlap, multitaper=True, mtm_w=4.0, mtm_kmax=7)
    z = synth.pcm16_to_float(synth.iq_stream_int16(p.required_span(0, nframes)[1], fs=int(FS), seed=11, dot_s=0.5))
    _check_display(mgpu, p, z, overlap, nframes)
    # int16 in, the same bytes
    pcm = synth.iq_stream_int16(p.required_span(0, nframes)[1], fs=int(FS), seed=11, dot_s=0.5)
    assert np.array_equal(p.run_display(pcm, nframes=nframes)["levels"], p.run_display(z, nframes=nframes)["levels"])


@pytest.mark.gpu
@pytest.mark.parametrize("iq", [False, True])
def test_mtm_zoom_display(mgpu, iq):
    from glfer_b200 import synth
    p = mgpu.ZoomPlan(n=1024, decim=16, overlap=0.75, center_hz=-1000.0 if iq else 1000.0, sample_rate=FS, iq=iq,
                      multitaper=True, mtm_w=4.0, mtm_kmax=7)
    nframes = 300
    span = p.required_span(0, nframes)[1]
    if iq:
        z = synth.pcm16_to_float(synth.iq_stream_int16(span, fs=int(FS), seed=5, dot_s=0.5))
    else:
        z = synth.qrss_stream(span, fs=int(FS), dot_s=0.5)
    _check_display(mgpu, p, z, 0.75, nframes)
