"""Thomson's harmonic F-test of multitaper I/Q and zoom plans (glfer_iq_run_mtm_ftest*, glfer_zoom_run[_iq]_mtm_ftest*).

CPU: the fused kernel's F-test epilogue emulated thread by thread (tests/emu/emu_iq_ftest.cpp).  GPU: F rows against a
float64 restatement of the contract in include/glfer_b200.h built from the plan's own tapers, on the fused and the
general path, with rows bit-identical to run(); the I/Q F-test of (x, 0) against the real plan's F-test of x, and the
real zoom's against the I/Q zoom's; the F(2, 2K' - 2) null distribution on white noise and the detection of a weak
line; bit-identical F rows under splitting, chunking, int16 input, a stereo WAV, origins beyond 2^32 and zoom
chunking; and the entry points' rejections."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_iq_mtm import iq_frames, zoom_frames, _fused  # noqa: E402

FS = 48000.0
FUSED_N = [32, 64, 128, 256, 512, 1024, 2048, 4096, 8192]


@pytest.fixture(scope="module")
def fapi():
    from glfer_b200 import build
    build.build()
    from glfer_b200 import api
    return api


@pytest.fixture(scope="module")
def fgpu(fapi):
    if fapi.device_count() < 1:
        pytest.fail("no CUDA device visible: the F-test GPU tests need a B200 (no CPU fallback exists)")
    return fapi


def _iq(n, seed=0x5EED):
    from glfer_b200 import synth
    return synth.iq_stream(n, fs=int(FS), seed=seed, dot_s=0.5)


def ftest_rows(frames, tapers):
    """the contract's F of each complex frame, fft-shifted, in float64"""
    u0 = tapers.sum(axis=1)
    s = float(np.sum(u0 * u0))
    hn = (u0 @ tapers) / s
    mu = np.fft.fft(hn[None, :] * frames, axis=1)
    den = np.zeros(frames.shape)
    for v, u in zip(tapers, u0):
        den += np.abs(np.fft.fft(v[None, :] * frames, axis=1) - mu * u) ** 2
    return np.fft.fftshift((len(tapers) - 1) * np.abs(mu) ** 2 * s / den, axes=1)


def assert_f_close(got, ref, what, med=2e-6, p99=1e-4, mx=2e-3):
    """median / p99 / max relative error on the finite bins.  The real F-test's bounds, except the max: on a B200 the
    median stays near 3e-7 and the p99 near 3e-6 at every shape, but the worst bin of the largest shapes (n = 8192 fused
    and n = 16384 general, K' = 4 / 16) reaches 1.0e-3 .. 1.4e-3, on bins where |mu| is far below the row's level and
    F is near 0"""
    ok = np.isfinite(ref) & (ref > 0)
    assert np.isfinite(got[ok]).all(), what
    rel = np.abs(got[ok].astype(np.float64) - ref[ok]) / ref[ok]
    stats = (float(np.median(rel)), float(np.percentile(rel, 99)), float(rel.max()))
    assert stats[0] < med and stats[1] < p99 and stats[2] < mx, (what, stats)


# ------------------------------------------------------------------------------------------------ CPU
def test_iq_ftest_epilogue_emulation(tmp_path):
    """the F-test epilogue on the CPU, n = 32 .. 8192: F against a long-double DFT restatement, rows against the
    tapered powers, every row position written exactly once"""
    exe = str(tmp_path / "emu_iq_ftest")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "emu", "emu_iq_ftest.cpp")],
                   check=True)
    res = subprocess.run([exe], capture_output=True, text=True)
    assert res.returncode == 0, res.stdout
    rows = [ln.split() for ln in res.stdout.strip().splitlines()]
    assert [int(r[0]) for r in rows] == FUSED_N
    assert all(int(r[3]) == 0 for r in rows), res.stdout
    assert all(float(r[1]) <= 1e-3 and float(r[2]) <= 1e-4 for r in rows), res.stdout


# ------------------------------------------------------------------------------------------------ GPU: parity
KW = [(2, 4.0), (4, 2.5), (4, 4.0), (8, 2.5), (8, 4.0), (16, 2.5), (16, 4.0), (2, 2.5)]
PARITY = [(n, ov) for n in (32, 256, 1024, 2048, 4096, 8192, 16384) for ov in (0.0, 0.5, 0.75, 0.6)]


@pytest.mark.gpu
@pytest.mark.parametrize("n,overlap", PARITY)
def test_iq_ftest_oracle_parity(fgpu, n, overlap):
    """F against the float64 contract on the fused and the forced general path; rows array_equal to run()'s"""
    nframes = 6 if n >= 8192 else 12
    for kp, w in KW:
        p = fgpu.IqPlan(n=n, overlap=overlap, multitaper=True, mtm_w=w, mtm_kmax=kp - 1)
        z = _iq(p.required_span(0, nframes)[1], seed=n + kp)
        tapers, _ = p.tapers()
        ref = ftest_rows(iq_frames(z, 0, n, p.hop, 0, nframes), tapers)
        fused = _fused(n, p.hop)
        for forced in ([False, True] if fused else [True]):
            fgpu.force_generic_kernel(forced)
            try:
                got = p.run_mtm_ftest(z)
                fam = fgpu.last_kernel_family()
                rows = p.run(z)
                only_f = p.run_mtm_ftest(z, want_psd=False)["ftest"]
                only_rows = p.run_mtm_ftest(z, want_ftest=False)["psd"]
            finally:
                fgpu.force_generic_kernel(False)
            assert fam.startswith("gram_kernel" if forced or not fused else "gram_ring_kernel"), fam
            what = f"iq ftest n={n} ov={overlap} K'={kp} NW={w} general={forced}"
            assert_f_close(got["ftest"], ref, what)
            assert np.array_equal(got["psd"], rows), what
            assert np.array_equal(only_f, got["ftest"]), what
            assert np.array_equal(only_rows, rows), what
        p.close()


# ------------------------------------------------------------------------------------------------ GPU: real input
@pytest.mark.gpu
@pytest.mark.parametrize("n,overlap,w,kmax", [(1024, 0.5, 4.0, 7), (4096, 0.75, 2.5, 3), (256, 0.0, 4.0, 15)])
def test_iq_ftest_of_real_input_is_the_real_ftest(fgpu, n, overlap, w, kmax):
    from glfer_b200 import synth
    real = fgpu.GramPlan(n=n, mode=fgpu.MODE_MTM, overlap=overlap, sub_mean=False, mtm_w=w, mtm_kmax=kmax, mtm_ftest=True)
    q = fgpu.IqPlan(n=n, overlap=overlap, multitaper=True, mtm_w=w, mtm_kmax=kmax)
    nframes = 20
    x = synth.qrss_stream(q.required_span(0, nframes)[1], fs=int(FS), dot_s=0.5)
    fr = real.run_mtm_ftest(x)["ftest"][:nframes].astype(np.float64)
    fq = q.run_mtm_ftest(np.stack([x, np.zeros_like(x)], axis=1))["ftest"]
    j = np.arange(1, n // 2)
    assert_f_close(fq[:, n // 2 + j], fr[:, j], "iq (x, 0) against the real F-test", med=2e-5, p99=1e-3, mx=1e-2)
    assert_f_close(fq[:, n // 2 - j], fq[:, n // 2 + j].astype(np.float64), "mirror symmetry about n/2",
                   med=2e-5, p99=1e-3, mx=1e-2)


@pytest.mark.gpu
@pytest.mark.parametrize("center", [0.0, 800.0, FS / 2])
def test_real_zoom_ftest_is_the_iq_zoom_ftest(fgpu, center):
    from glfer_b200 import synth
    kw = dict(n=512, decim=16, overlap=0.75, center_hz=center, sample_rate=FS, multitaper=True, mtm_w=4.0, mtm_kmax=7)
    r = fgpu.ZoomPlan(**kw)
    q = fgpu.ZoomPlan(iq=True, **kw)
    nframes = 20
    x = synth.qrss_stream(r.required_span(0, nframes)[1], fs=int(FS), dot_s=0.5)
    want = r.run_mtm_ftest(x)
    got = q.run_mtm_ftest(np.stack([x, np.zeros_like(x)], axis=1))
    assert np.array_equal(got["ftest"], want["ftest"]) and np.array_equal(got["psd"], want["psd"])
    assert np.array_equal(want["psd"], r.run(x))
    pcm = synth.qrss_stream_int16(len(x), fs=int(FS), dot_s=0.5)
    assert np.array_equal(q.run_mtm_ftest(np.stack([pcm, np.zeros_like(pcm)], axis=1))["ftest"],
                          r.run_mtm_ftest(pcm)["ftest"])
    tapers, _ = r.tapers()
    ref = ftest_rows(zoom_frames(fgpu, x.astype(np.complex128), 0, 512, 16, 0.75, center, 0, nframes), tapers)
    assert_f_close(want["ftest"], ref, f"real zoom ftest c={center}")


@pytest.mark.gpu
@pytest.mark.parametrize("decim,center,kmax", [(16, -1234.5, 3), (256, 800.0, 7)])
def test_iq_zoom_ftest_oracle_parity(fgpu, decim, center, kmax):
    n = 256
    p = fgpu.ZoomPlan(n=n, decim=decim, overlap=0.5, center_hz=center, sample_rate=FS, iq=True, multitaper=True,
                      mtm_w=4.0, mtm_kmax=kmax)
    nframes = 10
    z = _iq(p.required_span(0, nframes)[1])
    tapers, _ = p.tapers()
    got = p.run_mtm_ftest(z)
    assert np.array_equal(got["psd"], p.run(z))
    assert_f_close(got["ftest"], ftest_rows(zoom_frames(fgpu, z, 0, n, decim, 0.5, center, 0, nframes), tapers),
                   f"iq zoom ftest D={decim} c={center} K'={kmax + 1}")


# ------------------------------------------------------------------------------------------------ GPU: statistics
@pytest.mark.gpu
@pytest.mark.parametrize("kp", [4, 8])
def test_ftest_null_distribution_on_white_noise(fgpu, kp):
    from scipy import stats
    n, nframes = 1024, 160
    p = fgpu.IqPlan(n=n, overlap=0.0, multitaper=True, mtm_w=4.0, mtm_kmax=kp - 1)
    rng = np.random.default_rng(kp)
    span = p.required_span(0, nframes)[1]
    z = (rng.standard_normal(span) + 1j * rng.standard_normal(span)).astype(np.complex64)
    f = p.run_mtm_ftest(z, want_psd=False)["ftest"][1:].astype(np.float64).ravel()
    assert f.size >= 100_000
    d = stats.kstest(f, stats.f(2, 2 * kp - 2).cdf).statistic
    assert d < 0.02, d


@pytest.mark.gpu
def test_ftest_detects_a_weak_line_on_a_zoom_bin(fgpu):
    from scipy import stats
    n, decim, center, kp = 512, 16, 800.0, 8
    p = fgpu.ZoomPlan(n=n, decim=decim, overlap=0.0, center_hz=center, sample_rate=FS, iq=True, multitaper=True,
                      mtm_w=4.0, mtm_kmax=kp - 1)
    nframes = 60
    span = p.required_span(0, nframes)[1]
    rng = np.random.default_rng(9)
    bin_off = 10
    f_tone = p.center_hz() + bin_off * FS / (decim * n)
    t = np.arange(span)
    z = (0.1 * np.exp(2j * np.pi * f_tone / FS * t)
         + rng.standard_normal(span) + 1j * rng.standard_normal(span)).astype(np.complex64)
    f = p.run_mtm_ftest(z, want_psd=False)["ftest"][2:, n // 2 + bin_off]
    thr = stats.f(2, 2 * kp - 2).ppf(0.9999)
    assert np.mean(f > thr) >= 0.95, (np.mean(f > thr), thr, np.median(f))


# ------------------------------------------------------------------------------------------------ GPU: invariance
@pytest.mark.gpu
@pytest.mark.parametrize("n,overlap", [(1024, 0.5), (1024, 0.6), (4096, 0.75)])
def test_iq_ftest_split_and_pcm16_are_bit_identical(fgpu, n, overlap):
    from glfer_b200 import synth
    p = fgpu.IqPlan(n=n, overlap=overlap, multitaper=True, mtm_w=4.0, mtm_kmax=7)
    nframes = 40
    pcm = synth.iq_stream_int16(p.required_span(0, nframes)[1], fs=int(FS), dot_s=0.5)
    zf = synth.pcm16_to_float(pcm)
    whole = p.run_mtm_ftest(zf)["ftest"]
    assert whole.shape == (nframes, n)
    assert np.array_equal(p.run_mtm_ftest(np.ascontiguousarray(zf).view(np.complex64)[:, 0])["ftest"], whole)
    assert np.array_equal(p.run_mtm_ftest(pcm)["ftest"], whole)
    parts = []
    for a, b in ((0, 1), (1, 7), (7, 23), (23, 40)):
        lo, hi = p.required_span(a, b - a)
        lo = max(lo, 0)
        parts.append(p.run_mtm_ftest(np.ascontiguousarray(zf[lo:hi]), origin=lo, first_frame=a, nframes=b - a)["ftest"])
    assert np.array_equal(np.concatenate(parts), whole)


@pytest.mark.gpu
@pytest.mark.parametrize("overlap", [0.5, 0.6])
def test_iq_ftest_run_longer_than_a_chunk(fgpu, overlap):
    p = fgpu.IqPlan(n=1024, overlap=overlap, multitaper=True, mtm_w=4.0, mtm_kmax=3)
    nframes = (5 << 21) // p.hop
    z = _iq(p.required_span(0, nframes)[1], seed=3)
    big = p.run_mtm_ftest(z)
    assert np.array_equal(big["psd"], p.run(z))
    step = nframes // 4 + 1
    parts = [p.run_mtm_ftest(z, first_frame=a, nframes=min(step, nframes - a))["ftest"] for a in range(0, nframes, step)]
    assert np.array_equal(np.concatenate(parts), big["ftest"])


@pytest.mark.gpu
def test_iq_ftest_stereo_wav(fgpu, tmp_path):
    from glfer_b200 import synth
    p = fgpu.IqPlan(n=2048, overlap=0.5, multitaper=True, mtm_w=4.0, mtm_kmax=7)
    nframes = 30
    pcm = synth.iq_stream_int16(p.required_span(0, nframes)[1], fs=int(FS), dot_s=0.5)
    path = str(tmp_path / "iq.wav")
    synth.write_wav16(path, pcm.reshape(-1), int(FS), channels=2)
    want = p.run_mtm_ftest(pcm)["ftest"]
    lib = fgpu.lib()
    wav = fgpu.Wav()
    assert lib.glfer_wav_load(path.encode(), C.byref(wav)) == 0
    try:
        ft = np.empty((nframes, 2048), np.float32)
        fgpu._check(lib.glfer_iq_run_mtm_ftest_pcm16(p._h, wav.data, 0, wav.nsamples // 2, 0, nframes, None,
                                                     ft.ctypes.data))
    finally:
        lib.glfer_wav_free(C.byref(wav))
    assert np.array_equal(ft, want)


@pytest.mark.gpu
@pytest.mark.parametrize("forced", [False, True])
def test_iq_ftest_frames_beyond_sample_2_pow_32(fgpu, forced):
    n, overlap = 2048, 0.75
    p = fgpu.IqPlan(n=n, overlap=overlap, multitaper=True, mtm_w=4.0, mtm_kmax=7)
    first = ((1 << 32) + 12345) // p.hop + 3
    nframes = 8
    lo, hi = p.required_span(first, nframes)
    assert lo > (1 << 32)
    z = _iq(hi - lo, seed=7)
    fgpu.force_generic_kernel(forced)
    try:
        got = p.run_mtm_ftest(z, origin=lo, first_frame=first, nframes=nframes)["ftest"]
    finally:
        fgpu.force_generic_kernel(False)
    tapers, _ = p.tapers()
    assert_f_close(got, ftest_rows(iq_frames(z, lo, n, p.hop, first, nframes), tapers), "iq ftest beyond 2^32")


@pytest.mark.gpu
def test_iq_zoom_ftest_chunking_and_pcm16(fgpu):
    from glfer_b200 import synth
    p = fgpu.ZoomPlan(n=1024, decim=64, overlap=0.75, center_hz=-800.0, sample_rate=FS, iq=True, multitaper=True,
                      mtm_w=4.0, mtm_kmax=7)
    nframes = 40
    pcm = synth.iq_stream_int16(p.required_span(0, nframes)[1], fs=int(FS), dot_s=0.5)
    zf = synth.pcm16_to_float(pcm)
    whole = p.run_mtm_ftest(zf)["ftest"]
    assert np.array_equal(p.run_mtm_ftest(pcm)["ftest"], whole)
    parts = []
    for a, b in ((0, 1), (1, 7), (7, 23), (23, 40)):
        lo, hi = p.required_span(a, b - a)
        lo = max(lo, 0)
        parts.append(p.run_mtm_ftest(np.ascontiguousarray(zf[lo:hi]), origin=lo, first_frame=a, nframes=b - a)["ftest"])
    assert np.array_equal(np.concatenate(parts), whole)
    # runs of several chunks (~32 MiB of input each) against runs of their parts
    q = fgpu.ZoomPlan(n=64, decim=256, overlap=0.75, center_hz=-3000.0, sample_rate=FS, iq=True, multitaper=True,
                      mtm_w=2.5, mtm_kmax=3)
    zl = _iq(q.required_span(0, 3000)[1], seed=3)
    big = q.run_mtm_ftest(zl)
    assert np.array_equal(big["psd"], q.run(zl))
    parts = [q.run_mtm_ftest(zl, first_frame=a, nframes=min(1000, 3000 - a))["ftest"] for a in range(0, 3000, 1000)]
    assert np.array_equal(np.concatenate(parts), big["ftest"])


# ------------------------------------------------------------------------------------------------ GPU: rejections
@pytest.mark.gpu
def test_ftest_entry_point_rejections(fgpu):
    lib = fgpu.lib()
    n = 256
    iqp = fgpu.IqPlan(n=n, overlap=0.5)                                    # periodogram
    iq1 = fgpu.IqPlan(n=n, overlap=0.5, multitaper=True, mtm_kmax=0)       # K' = 1
    iqm = fgpu.IqPlan(n=n, overlap=0.5, multitaper=True)
    zr = fgpu.ZoomPlan(n=n, decim=16, center_hz=800.0, sample_rate=FS, multitaper=True)
    zq = fgpu.ZoomPlan(n=n, decim=16, center_hz=-800.0, sample_rate=FS, iq=True, multitaper=True)
    zp = fgpu.ZoomPlan(n=n, decim=16, center_hz=-800.0, sample_rate=FS, iq=True)
    z1 = fgpu.ZoomPlan(n=n, decim=16, center_hz=800.0, sample_rate=FS, multitaper=True, mtm_kmax=0)
    hi = zr.required_span(0, 2)[1]
    x = np.zeros(2 * hi, np.float32)
    pcm = np.zeros(2 * hi, np.int16)
    rows = np.empty((2, n), np.float32)
    ft = np.empty((2, n), np.float32)
    R, F = rows.ctypes.data, ft.ctypes.data
    iq_fns = ((lib.glfer_iq_run_mtm_ftest, x), (lib.glfer_iq_run_mtm_ftest_pcm16, pcm))
    for fn, buf in iq_fns:
        assert fn(iqm._h, buf.ctypes.data, 0, hi, 0, 2, R, F) == 0
        assert fn(iqp._h, buf.ctypes.data, 0, hi, 0, 2, R, F) == -2            # periodogram plan
        assert fn(iq1._h, buf.ctypes.data, 0, hi, 0, 2, R, F) == -2            # K' = 1
        assert fn(iqm._h, buf.ctypes.data, 0, hi, 0, 2, None, None) == -2      # no output
        assert fn(iqm._h, buf.ctypes.data, 0, iqm.required_span(0, 2)[1] - 1, 0, 2, R, F) == -2   # short input
    for fn, plan, other, buf in ((lib.glfer_zoom_run_mtm_ftest, zr, zq, x), (lib.glfer_zoom_run_mtm_ftest_pcm16, zr, zq, pcm),
                                 (lib.glfer_zoom_run_iq_mtm_ftest, zq, zr, x),
                                 (lib.glfer_zoom_run_iq_mtm_ftest_pcm16, zq, zr, pcm)):
        assert fn(plan._h, buf.ctypes.data, 0, hi, 0, 2, R, F) == 0
        assert fn(other._h, buf.ctypes.data, 0, hi, 0, 2, R, F) == -2          # real entry, I/Q plan or the reverse
        assert fn(plan._h, buf.ctypes.data, 0, hi, 0, 2, None, None) == -2
        assert fn(plan._h, buf.ctypes.data, 0, hi - 1, 0, 2, R, F) == -2
    assert lib.glfer_zoom_run_iq_mtm_ftest(zp._h, x.ctypes.data, 0, hi, 0, 2, R, F) == -2   # periodogram zoom
    assert lib.glfer_zoom_run_mtm_ftest(z1._h, x.ctypes.data, 0, hi, 0, 2, R, F) == -2      # K' = 1
