"""Zoom spectrogram (glfer_zoom_*): the low-pass design on the host, and on the GPU the rows against a float64
restatement of the contract in include/glfer_b200.h, tone level and placement, alias rejection, invariance
under chunking / input format / origins beyond 2^32, frame arithmetic and argument checks."""
import os
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
def zapi():
    from glfer_b200 import build
    build.build()
    from glfer_b200 import api
    return api


@pytest.fixture(scope="module")
def zgpu(zapi):
    if zapi.device_count() < 1:
        pytest.fail("no CUDA device visible: the zoom GPU tests need a B200 (no CPU fallback exists)")
    return zapi


def _stream(n, seed=0x5EED):
    from glfer_b200 import synth
    return synth.qrss_stream(n, fs=int(FS), seed=seed, dot_s=0.5)


def _step(center, fs=FS):
    return int(np.floor(center / fs * 2.0 ** 32 + 0.5))        # llround of a non-negative value


def _window(api, n, wt):
    return np.ones(n) if wt == RECTANGULAR else api.host_window(n, wt).astype(np.float64)


def oracle(api, x, origin, n, decim, wt, overlap, center, first_frame, nframes, fs=FS):
    """float64 restatement: y[m] = sum_l h[l] x[mD - l] e^{-2 pi i phi(mD - l)} with the exact integer phase of the
    absolute index, frames of n complex samples at glb_hop(n, overlap), rows |FFT(w y_f)|^2 / n, fft-shifted."""
    h = api.zoom_taps(decim).astype(np.float64)
    K = 16 * decim
    hop = api.host_hop(n, overlap)
    step = np.uint64(_step(center, fs))
    m_lo = first_frame * hop - (n - hop)
    m0 = max(m_lo, 0)
    m_hi = (first_frame + nframes) * hop
    a, b = m0 * decim - K, (m_hi - 1) * decim + K + 1            # stream span of y[m0 .. m_hi)
    idx = np.arange(a, b, dtype=np.int64)
    xs = np.zeros(b - a)
    ok = idx >= 0
    xs[ok] = x[idx[ok] - origin].astype(np.float64)
    ph = ((np.where(ok, idx, 0).astype(np.uint64) * step) & np.uint64(0xFFFFFFFF)).astype(np.float64) / 2.0 ** 32
    v = xs * np.exp(-2j * np.pi * ph)
    y = upfirdn(h, v, 1, decim)[2 * K // decim: 2 * K // decim + (m_hi - m0)]
    yfull = np.zeros(m_hi - m_lo, dtype=np.complex128)
    yfull[m0 - m_lo:] = y
    w = _window(api, n, wt)
    rows = np.empty((nframes, n))
    for f in range(nframes):
        s = (first_frame + f) * hop - (n - hop) - m_lo
        z = np.fft.fft(w * yfull[s:s + n])
        rows[f] = np.fft.fftshift(np.abs(z) ** 2) / n
    return rows


def _samples_for(plan, nframes):
    """a stream just long enough for nframes frames"""
    return plan.required_span(0, nframes)[1]


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("decim", [2, 7, 64, 1024])
def test_zoom_taps_design(zapi, decim):
    h = zapi.zoom_taps(decim)
    assert h.dtype == np.float32 and h.shape == (32 * decim + 1,)
    assert np.array_equal(h.view(np.uint32), h[::-1].view(np.uint32))
    hd = h.astype(np.float64)
    assert abs(hd.sum() - 1.0) <= 1e-6
    nfft = 1 << int(np.ceil(np.log2(16 * len(h))))
    H = np.abs(np.fft.rfft(hd, nfft))
    f = np.arange(len(H)) / nfft                                  # cycles per input sample
    pb = 20 * np.log10(H[f <= 0.4 / decim])
    assert pb.max() <= 0.001 and pb.min() >= -0.001, (pb.min(), pb.max())
    assert 20 * np.log10(H[f >= 0.6 / decim].max()) <= -95.0


def test_zoom_taps_reject_bad_decimation(zapi):
    for d in (0, 1, 1025):
        with pytest.raises(zapi.GlferError):
            zapi.zoom_taps(d)


# ------------------------------------------------------------------------------------------------ GPU
PARITY = [
    # decim, n, window, overlap, centre
    (2, 32, HANNING, 0.0, 0.0),
    (2, 1024, KAISER, 0.5, 800.0),
    (2, 16384, RECTANGULAR, 0.75, FS / 2 - 10.0),
    (16, 32, RECTANGULAR, 0.5, 800.0),
    (16, 1024, HANNING, 0.75, FS / 2 - 3.3),
    (16, 16384, KAISER, 0.0, 0.0),
    (256, 32, KAISER, 0.75, FS / 2),
    (256, 1024, RECTANGULAR, 0.0, 800.0),
    (256, 16384, HANNING, 0.5, 800.0),
]


@pytest.mark.gpu
@pytest.mark.parametrize("decim,n,wt,overlap,center", PARITY)
def test_zoom_oracle_parity(zgpu, decim, n, wt, overlap, center):
    p = zgpu.ZoomPlan(n=n, decim=decim, window_type=wt, overlap=overlap, center_hz=center, sample_rate=FS)
    nframes = 6 if n == 16384 else 12
    x = _stream(_samples_for(p, nframes))
    assert p.num_frames(len(x)) == nframes
    got = p.run(x)
    ref = oracle(zgpu, x, 0, n, decim, wt, overlap, center, 0, nframes)
    st = assert_psd_close(got, ref, f"zoom D={decim} n={n} w={wt} ov={overlap} c={center}")
    print(f"D={decim} n={n}: frac(rel<=1e-4)={st['frac_1e4']:.5f} max rel above floor={st['max_rel_above_floor']:.2e}")


@pytest.mark.gpu
@pytest.mark.parametrize("decim,n,wt", [(16, 1024, HANNING), (256, 4096, KAISER), (64, 512, RECTANGULAR)])
def test_zoom_tone_level_and_placement(zgpu, decim, n, wt):
    center = 1234.5
    p = zgpu.ZoomPlan(n=n, decim=decim, window_type=wt, overlap=0.5, center_hz=center, sample_rate=FS)
    res = FS / (decim * n)
    k0 = int(0.3 * FS / decim / res)                               # inside the clean span
    f_tone = p.center_hz() + k0 * res
    amp = 0.25
    nframes = 4
    t = np.arange(_samples_for(p, nframes + 2), dtype=np.float64)
    x = (amp * np.cos(2 * np.pi * f_tone / FS * t + 0.4)).astype(np.float32)
    rows = p.run(x)[2:]                                            # frames past the zero history
    w = _window(zgpu, n, wt)
    want = amp ** 2 / 4 * w.sum() ** 2 / n
    assert (rows.argmax(axis=1) == n // 2 + k0).all()
    assert np.abs(10 * np.log10(rows.max(axis=1) / want)).max() <= 0.01


@pytest.mark.gpu
@pytest.mark.parametrize("decim", [16, 256])
def test_zoom_alias_rejection(zgpu, decim):
    n, center = 1024, 6000.0
    p = zgpu.ZoomPlan(n=n, decim=decim, window_type=KAISER, overlap=0.5, center_hz=center, sample_rate=FS)
    nframes = 4
    t = np.arange(_samples_for(p, nframes + 2), dtype=np.float64)

    def peak(f):
        x = (0.5 * np.cos(2 * np.pi * f / FS * t)).astype(np.float32)
        return p.run(x)[2:].max()

    inband = peak(p.center_hz() + 0.1 * FS / decim)
    alias = peak(p.center_hz() + 0.7 * FS / decim)
    assert 10 * np.log10(alias / inband) <= -95.0, 10 * np.log10(alias / inband)


@pytest.mark.gpu
def test_zoom_chunking_and_pcm16_are_bit_identical(zgpu):
    from glfer_b200 import synth
    p = zgpu.ZoomPlan(n=1024, decim=64, window_type=KAISER, overlap=0.75, center_hz=800.0, sample_rate=FS)
    nframes = 40
    pcm = synth.qrss_stream_int16(_samples_for(p, nframes), fs=int(FS), dot_s=0.5)
    x = synth.pcm16_to_float(pcm)
    whole = p.run(x)
    assert whole.shape == (nframes, 1024)
    parts = []
    for a, b in ((0, 1), (1, 7), (7, 23), (23, 40)):
        lo, hi = p.required_span(a, b - a)
        lo = max(lo, 0)
        parts.append(p.run(np.ascontiguousarray(x[lo:hi]), origin=lo, first_frame=a, nframes=b - a))
    assert np.array_equal(np.concatenate(parts), whole)
    assert np.array_equal(p.run(pcm), whole)
    # a run the library splits into chunks of ~32 MiB of input (2048 frames here): the n - hop decimated samples
    # a chunk shares with the previous one are carried on the device, not recomputed
    q = zgpu.ZoomPlan(n=64, decim=256, window_type=HANNING, overlap=0.75, center_hz=800.0, sample_rate=FS)
    xl = _stream(q.required_span(0, 5000)[1], seed=3)
    big = q.run(xl)
    assert big.shape[0] == 5000
    parts = [q.run(xl, first_frame=a, nframes=min(1000, 5000 - a)) for a in range(0, 5000, 1000)]
    assert np.array_equal(np.concatenate(parts), big)


@pytest.mark.gpu
def test_zoom_frames_beyond_sample_2_pow_32(zgpu):
    n, decim, center = 1024, 16, 800.0
    p = zgpu.ZoomPlan(n=n, decim=decim, window_type=HANNING, overlap=0.5, center_hz=center, sample_rate=FS)
    first = ((1 << 32) + 12345) // (p.hop * decim) + 3
    nframes = 8
    lo, hi = p.required_span(first, nframes)
    assert lo > (1 << 32)
    x = _stream(hi - lo, seed=7)
    got = p.run(x, origin=lo, first_frame=first, nframes=nframes)
    ref = oracle(zgpu, x, lo, n, decim, HANNING, 0.5, center, first, nframes)
    assert_psd_close(got, ref, "zoom beyond 2^32")


@pytest.mark.gpu
@pytest.mark.parametrize("decim,n,overlap", [(16, 1024, 0.5), (7, 64, 0.75), (256, 32, 0.0)])
def test_zoom_frame_arithmetic(zgpu, decim, n, overlap):
    p = zgpu.ZoomPlan(n=n, decim=decim, window_type=HANNING, overlap=overlap, center_hz=100.0, sample_rate=FS)
    K = 16 * decim
    hop = zgpu.host_hop(n, overlap)
    assert p.hop == hop and p.bins == n
    for S in (0, 1, K, K + 1, K + decim * hop, K + decim * hop + 1, 10 ** 7 + 3):
        md = 0 if S - 1 - K < 0 else (S - 1 - K) // decim + 1
        assert p.num_frames(S) == md // hop, S
    for first, cnt in ((0, 1), (0, 5), (3, 2), (100, 9)):
        lo, hi = p.required_span(first, cnt)
        assert lo == (first * hop - (n - hop)) * decim - K
        assert hi == ((first + cnt) * hop - 1) * decim + K + 1
        assert p.num_frames(hi) >= first + cnt and p.num_frames(hi - 1) < first + cnt
    assert p.required_span(0, 1)[0] < 0
    assert abs(p.center_hz() - round(100.0 / FS * 2 ** 32) * FS / 2 ** 32) < 1e-9
    x = _stream(p.required_span(2, 2)[1])
    lo, hi = p.required_span(2, 2)
    with pytest.raises(zgpu.GlferError):                          # samples do not cover the frames
        p.run(np.ascontiguousarray(x[max(lo, 0) + 1:hi]), origin=max(lo, 0) + 1, first_frame=2, nframes=2)


@pytest.mark.gpu
def test_zoom_invalid_configs_are_rejected(zgpu):
    bad = (dict(n=16), dict(n=1000), dict(n=32768), dict(decim=1), dict(decim=1025), dict(window_type=8),
           dict(window_type=-1), dict(overlap=1.0), dict(center_hz=-1.0), dict(center_hz=24000.5),
           dict(sample_rate=0.0), dict(device=10 ** 6))
    for kw in bad:
        with pytest.raises(zgpu.GlferError):
            zgpu.ZoomPlan(**kw)
