"""Complex (I/Q) input: the I/Q spectrogram (glfer_iq_*) and the I/Q zoom (glfer_zoom_*_iq).

CPU: the fused kernel's passes and epilogue emulated thread by thread (tests/emu/emu_iq.cpp).  GPU: rows against a
float64 restatement of the contracts in include/glfer_b200.h on both the fused and the general path, two-sided
placement and level, bit-identical invariance under splitting / chunking / int16 input / a stereo WAV, origins
beyond 2^32, the frame arithmetic and the argument checks; for the zoom, parity at negative and positive centres,
real input as (x, 0) bit-identical to the real zoom, negative-frequency selectivity and the entry-point checks."""
import ctypes as C
import math
import os
import subprocess
import sys

import numpy as np
import pytest
from scipy.signal import upfirdn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from parity import assert_psd_close  # noqa: E402

FS = 48000.0
HANNING, RECTANGULAR, KAISER = 0, 5, 7


@pytest.fixture(scope="module")
def iapi():
    from glfer_b200 import build
    build.build()
    from glfer_b200 import api
    return api


@pytest.fixture(scope="module")
def igpu(iapi):
    if iapi.device_count() < 1:
        pytest.fail("no CUDA device visible: the I/Q GPU tests need a B200 (no CPU fallback exists)")
    return iapi


def _iq(n, seed=0x5EED):
    from glfer_b200 import synth
    return synth.iq_stream(n, fs=int(FS), seed=seed, dot_s=0.5)


def _window(api, n, wt):
    return np.ones(n) if wt == RECTANGULAR else api.host_window(n, wt).astype(np.float64)


def iq_oracle(api, z, origin, n, wt, overlap, first_frame, nframes):
    """float64 restatement: frame f = z[f hop - (n - hop) .. f hop + hop), zeros before sample 0,
    rows |FFT(w z_f)|^2 / n, fft-shifted"""
    hop = api.host_hop(n, overlap)
    w = _window(api, n, wt)
    s0 = (first_frame + np.arange(nframes, dtype=np.int64)) * hop - (n - hop)
    idx = s0[:, None] + np.arange(n, dtype=np.int64)[None, :]
    seg = np.zeros(idx.shape, dtype=np.complex128)
    ok = idx >= 0
    seg[ok] = z[idx[ok] - origin].astype(np.complex128)
    return np.fft.fftshift(np.abs(np.fft.fft(w * seg, axis=1)) ** 2, axes=1) / n


def _step(center, fs=FS):
    v = center / fs * 2.0 ** 32
    return int(math.copysign(math.floor(abs(v) + 0.5), v)) % (1 << 32)        # llround, modulo 2^32


def zoom_oracle(api, z, origin, n, decim, wt, overlap, center, first_frame, nframes):
    """float64 restatement of the zoom contract with complex x (tests/test_zoom.py's, signed step)"""
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
    w = _window(api, n, wt)
    rows = np.empty((nframes, n))
    for f in range(nframes):
        s = (first_frame + f) * hop - (n - hop) - m_lo
        rows[f] = np.fft.fftshift(np.abs(np.fft.fft(w * yfull[s:s + n])) ** 2) / n
    return rows


def _fused_geometry(api, n, overlap):
    hop = api.host_hop(n, overlap)
    return n <= 8192 and (n - hop) % hop == 0 and any(hop == (n // 16) << s for s in range(5))


# ------------------------------------------------------------------------------------------------ CPU
def test_iq_kernel_emulation(tmp_path):
    """the fused kernel's passes and epilogue on the CPU, n = 32 .. 8192: rows against a long-double DFT, and every
    row position written exactly once at the fft-shifted index; accuracy as the real path's at the same size"""
    exe = str(tmp_path / "emu_iq")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "emu", "emu_iq.cpp")], check=True)
    res = subprocess.run([exe], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout
    rows = [ln.split() for ln in res.stdout.strip().splitlines()]
    assert [int(r[0]) for r in rows] == [32, 64, 128, 256, 512, 1024, 2048, 4096, 8192]
    assert all(int(r[2]) == 0 for r in rows), res.stdout
    # emu_fft.cpp holds the real path to 1e-4 relative at or above the 1e-6 floor, on the same inputs
    assert all(float(r[1]) <= 1e-4 for r in rows), res.stdout


# ------------------------------------------------------------------------------------------------ GPU: spectrogram
PARITY = [(n, wt, ov) for n in (32, 1024, 2048, 4096, 8192, 16384) for wt in (HANNING, KAISER, RECTANGULAR)
          for ov in (0.0, 0.5, 0.75, 0.6)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,wt,overlap", PARITY)
def test_iq_oracle_parity(igpu, n, wt, overlap):
    p = igpu.IqPlan(n=n, window_type=wt, overlap=overlap)
    nframes = 6 if n >= 8192 else 12
    z = _iq(p.required_span(0, nframes)[1])
    assert p.num_frames(len(z)) == nframes
    ref = iq_oracle(igpu, z, 0, n, wt, overlap, 0, nframes)
    fused = _fused_geometry(igpu, n, overlap)
    paths = [False, True] if fused else [True]
    for forced in paths:
        igpu.force_generic_kernel(forced)
        try:
            got = p.run(z)
            fam = igpu.last_kernel_family()
        finally:
            igpu.force_generic_kernel(False)
        assert fam.startswith("gram_kernel" if forced or not fused else "gram_ring_kernel"), fam
        st = assert_psd_close(got, ref, f"iq n={n} w={wt} ov={overlap} general={forced}")
        print(f"n={n} w={wt} ov={overlap} {fam}: max rel above floor={st['max_rel_above_floor']:.2e}")


@pytest.mark.gpu
@pytest.mark.parametrize("n,k1,k2", [(1024, 100, 230), (4096, 1500, 37), (16384, 5000, 6001)])
def test_iq_two_sided_placement(igpu, n, k1, k2):
    p = igpu.IqPlan(n=n, window_type=HANNING, overlap=0.5)
    nframes = 4
    s = np.arange(p.required_span(0, nframes + 2)[1], dtype=np.float64)
    a1, a2 = 0.3, 0.1
    z = (a1 * np.exp(-2j * np.pi * k1 * s / n + 0.2j) + a2 * np.exp(2j * np.pi * k2 * s / n - 1.0j)).astype(np.complex64)
    rows = p.run(z)[2:].astype(np.float64)                        # frames past the zero history
    w = _window(igpu, n, HANNING)
    for amp, b, mirror in ((a1, n // 2 - k1, n // 2 + k1), (a2, n // 2 + k2, n // 2 - k2)):
        want = amp ** 2 * w.sum() ** 2 / n
        assert np.abs(10 * np.log10(rows[:, b] / want)).max() <= 0.01
        lo, hi = max(b - 3, 0), min(b + 4, n)
        assert (rows[:, lo:hi].argmax(axis=1) == b - lo).all()
        assert 10 * np.log10(rows[:, mirror].max() / rows[:, b].min()) <= -90.0


@pytest.mark.gpu
@pytest.mark.parametrize("n,overlap", [(1024, 0.5), (1024, 0.6)])
def test_iq_split_and_pcm16_are_bit_identical(igpu, n, overlap):
    from glfer_b200 import synth
    p = igpu.IqPlan(n=n, window_type=KAISER, overlap=overlap)
    nframes = 40
    pcm = synth.iq_stream_int16(p.required_span(0, nframes)[1], fs=int(FS), dot_s=0.5)
    zf = synth.pcm16_to_float(pcm)                                 # float32 [count, 2]
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
    # origins before the span's start, odd ones too: the samples before the span are not read
    lo, hi = p.required_span(9, 5)
    for o in (lo - 1, lo - 2, lo - 3):
        assert np.array_equal(p.run(np.ascontiguousarray(zf[o:hi + 5]), origin=o, first_frame=9, nframes=5), whole[9:14])


@pytest.mark.gpu
@pytest.mark.parametrize("overlap", [0.5, 0.6])
def test_iq_run_longer_than_a_chunk(igpu, overlap):
    """a run the library splits into chunks of ~32 MiB of input (4 Mi complex samples) against runs of its parts"""
    p = igpu.IqPlan(n=1024, window_type=HANNING, overlap=overlap)
    nframes = (5 << 21) // p.hop
    z = _iq(p.required_span(0, nframes)[1], seed=3)
    big = p.run(z)
    step = nframes // 4 + 1
    parts = [p.run(z, first_frame=a, nframes=min(step, nframes - a)) for a in range(0, nframes, step)]
    assert np.array_equal(np.concatenate(parts), big)


@pytest.mark.gpu
@pytest.mark.parametrize("forced", [False, True])
def test_iq_frames_beyond_sample_2_pow_32(igpu, forced):
    n, overlap = 2048, 0.75
    p = igpu.IqPlan(n=n, window_type=HANNING, overlap=overlap)
    first = ((1 << 32) + 12345) // p.hop + 3
    nframes = 8
    lo, hi = p.required_span(first, nframes)
    assert lo > (1 << 32)
    z = _iq(hi - lo, seed=7)
    igpu.force_generic_kernel(forced)
    try:
        got = p.run(z, origin=lo, first_frame=first, nframes=nframes)
    finally:
        igpu.force_generic_kernel(False)
    assert_psd_close(got, iq_oracle(igpu, z, lo, n, HANNING, overlap, first, nframes), "iq beyond 2^32")


@pytest.mark.gpu
def test_iq_stereo_wav(igpu, tmp_path):
    from glfer_b200 import synth
    p = igpu.IqPlan(n=2048, window_type=HANNING, overlap=0.5)
    nframes = 30
    pcm = synth.iq_stream_int16(p.required_span(0, nframes)[1], fs=int(FS), dot_s=0.5)
    path = str(tmp_path / "iq.wav")
    synth.write_wav16(path, pcm.reshape(-1), int(FS), channels=2)
    want = p.run(pcm)
    lib = igpu.lib()
    wav = igpu.Wav()
    assert lib.glfer_wav_load(path.encode(), C.byref(wav)) == 0
    try:
        assert wav.channels == 2 and wav.bits == 16 and wav.nsamples == pcm.size
        rows = np.empty((nframes, 2048), np.float32)
        igpu._check(lib.glfer_iq_run_pcm16(p._h, wav.data, 0, wav.nsamples // 2, 0, nframes, rows.ctypes.data))
    finally:
        lib.glfer_wav_free(C.byref(wav))
    assert np.array_equal(rows, want)


@pytest.mark.gpu
@pytest.mark.parametrize("n,overlap", [(1024, 0.5), (64, 0.75), (32, 0.0), (4096, 0.6)])
def test_iq_frame_arithmetic(igpu, n, overlap):
    p = igpu.IqPlan(n=n, window_type=HANNING, overlap=overlap)
    hop = igpu.host_hop(n, overlap)
    assert p.hop == hop and p.bins == n
    for S in (0, 1, hop - 1, hop, hop + 1, 10 ** 7 + 3):
        assert p.num_frames(S) == S // hop
    for first, cnt in ((0, 1), (0, 5), (3, 2), (100, 9)):
        assert p.required_span(first, cnt) == (first * hop - (n - hop), (first + cnt) * hop)
    z = _iq(p.required_span(2, 2)[1])
    lo, hi = p.required_span(2, 2)
    with pytest.raises(igpu.GlferError):                          # samples do not cover the frames
        p.run(np.ascontiguousarray(z[max(lo, 0) + 1:hi]), origin=max(lo, 0) + 1, first_frame=2, nframes=2)
    with pytest.raises(igpu.GlferError):
        p.run(np.ascontiguousarray(z[:hi - 1]), first_frame=2, nframes=2)


@pytest.mark.gpu
def test_iq_invalid_configs_are_rejected(igpu):
    for kw in (dict(n=16), dict(n=1000), dict(n=32768), dict(window_type=8), dict(overlap=1.0), dict(device=10 ** 6)):
        with pytest.raises(igpu.GlferError):
            igpu.IqPlan(**kw)


# ------------------------------------------------------------------------------------------------ GPU: zoom
ZPARITY = [(d, c) for d in (2, 16, 256) for c in (-FS / 2, -1234.5, 0.0, 800.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("decim,center", ZPARITY)
def test_iq_zoom_oracle_parity(igpu, decim, center):
    n = 256
    p = igpu.ZoomPlan(n=n, decim=decim, window_type=HANNING, overlap=0.5, center_hz=center, sample_rate=FS, iq=True)
    nframes = 10
    z = _iq(p.required_span(0, nframes)[1])
    assert p.num_frames(len(z)) == nframes
    s = _step(center)
    assert p.center_hz() == (s - (1 << 32) if s >= 1 << 31 else s) * FS / 2 ** 32
    got = p.run(z)
    ref = zoom_oracle(igpu, z, 0, n, decim, HANNING, 0.5, center, 0, nframes)
    assert_psd_close(got, ref, f"iq zoom D={decim} c={center}")


@pytest.mark.gpu
@pytest.mark.parametrize("center", [0.0, 800.0, 6000.0, FS / 2])
def test_iq_zoom_of_real_input_is_the_real_zoom(igpu, center):
    from glfer_b200 import synth
    kw = dict(n=512, decim=16, window_type=KAISER, overlap=0.75, center_hz=center, sample_rate=FS)
    r = igpu.ZoomPlan(**kw)
    q = igpu.ZoomPlan(iq=True, **kw)
    nframes = 20
    x = synth.qrss_stream(r.required_span(0, nframes)[1], fs=int(FS), dot_s=0.5)
    zx = np.stack([x, np.zeros_like(x)], axis=1)
    assert np.array_equal(q.run(zx), r.run(x))
    pcm = synth.qrss_stream_int16(len(x), fs=int(FS), dot_s=0.5)
    assert np.array_equal(q.run(np.stack([pcm, np.zeros_like(pcm)], axis=1)), r.run(pcm))


@pytest.mark.gpu
@pytest.mark.parametrize("decim", [16, 256])
def test_iq_zoom_negative_frequency_selectivity(igpu, decim):
    n, c = 1024, 1234.5
    below = igpu.ZoomPlan(n=n, decim=decim, window_type=KAISER, overlap=0.5, center_hz=-c, sample_rate=FS, iq=True)
    above = igpu.ZoomPlan(n=n, decim=decim, window_type=KAISER, overlap=0.5, center_hz=c, sample_rate=FS, iq=True)
    res = FS / (decim * n)
    k0 = 37
    f_tone = below.center_hz() + k0 * res
    nframes = 4
    s = np.arange(below.required_span(0, nframes + 2)[1], dtype=np.float64)
    z = (0.5 * np.exp(2j * np.pi * f_tone / FS * s)).astype(np.complex64)
    rb = below.run(z)[2:]
    ra = above.run(z)[2:]
    assert (rb.argmax(axis=1) == n // 2 + k0).all()
    assert 10 * np.log10(ra.max() / rb.max()) <= -95.0, 10 * np.log10(ra.max() / rb.max())


@pytest.mark.gpu
def test_iq_zoom_chunking_pcm16_and_range(igpu):
    from glfer_b200 import synth
    p = igpu.ZoomPlan(n=1024, decim=64, window_type=KAISER, overlap=0.75, center_hz=-800.0, sample_rate=FS, iq=True)
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
    q = igpu.ZoomPlan(n=64, decim=256, window_type=HANNING, overlap=0.75, center_hz=-3000.0, sample_rate=FS, iq=True)
    zl = _iq(q.required_span(0, 3000)[1], seed=3)
    big = q.run(zl)
    parts = [q.run(zl, first_frame=a, nframes=min(1000, 3000 - a)) for a in range(0, 3000, 1000)]
    assert np.array_equal(np.concatenate(parts), big)
    # beyond 2^32
    r = igpu.ZoomPlan(n=1024, decim=16, window_type=HANNING, overlap=0.5, center_hz=-800.0, sample_rate=FS, iq=True)
    first = ((1 << 32) + 12345) // (r.hop * 16) + 3
    lo, hi = r.required_span(first, 8)
    assert lo > (1 << 32)
    z = _iq(hi - lo, seed=7)
    got = r.run(z, origin=lo, first_frame=first, nframes=8)
    assert_psd_close(got, zoom_oracle(igpu, z, lo, 1024, 16, HANNING, 0.5, -800.0, first, 8), "iq zoom beyond 2^32")


@pytest.mark.gpu
def test_iq_zoom_entry_points_and_centre_range(igpu):
    lib = igpu.lib()
    real = igpu.ZoomPlan(n=256, decim=16, center_hz=800.0, sample_rate=FS)
    iq = igpu.ZoomPlan(n=256, decim=16, center_hz=-800.0, sample_rate=FS, iq=True)
    hi = real.required_span(0, 2)[1]
    x = np.zeros(2 * hi, np.float32)
    pcm = np.zeros(2 * hi, np.int16)
    rows = np.empty((2, 256), np.float32)
    for fn, plan, buf in ((lib.glfer_zoom_run, iq, x), (lib.glfer_zoom_run_pcm16, iq, pcm),
                          (lib.glfer_zoom_run_iq, real, x), (lib.glfer_zoom_run_iq_pcm16, real, pcm)):
        assert fn(plan._h, buf.ctypes.data, 0, hi, 0, 2, rows.ctypes.data) == -2
    for c in (-FS / 2 - 0.5, FS / 2 + 0.5):
        with pytest.raises(igpu.GlferError):
            igpu.ZoomPlan(n=256, decim=16, center_hz=c, sample_rate=FS, iq=True)
    for c in (-FS / 2, FS / 2):
        assert igpu.ZoomPlan(n=256, decim=16, center_hz=c, sample_rate=FS, iq=True).center_hz() == -FS / 2
    with pytest.raises(igpu.GlferError):
        igpu.ZoomPlan(n=256, decim=16, center_hz=-1.0, sample_rate=FS)
