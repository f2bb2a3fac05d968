"""Harmonic line detection of multitaper I/Q and zoom plans (glfer_*_run_mtm_lines*, glfer_ftest_threshold).

The selection is exact on given floats, so every GPU test runs run_mtm_ftest on the same plan and call, applies the numpy
restatement of the selection rule (select_lines) to its F and P rows and asserts array_equal for count, bin, ftest and
psd.  CPU: the threshold against scipy's F(2, 2K' - 2), its rejections, and the restatement against a per-bin loop on
hand-built rows (plateaus, wrap-around, NaN and inf, ties at the cap, ranges that exclude a peak).  GPU: exactness on
the fused and the general path, real and I/Q zoom, a bank, int16 input, chunked and split runs, frames beyond 2^32,
optional outputs, caps that overflow, narrow ranges and silence; the count on white noise and a weak zoom line; the
launch count and the entry points' rejections."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_iq_mtm import _fused  # noqa: E402

FS = 48000.0


@pytest.fixture(scope="module")
def lapi():
    from glfer_b200 import build
    build.build()
    from glfer_b200 import api
    return api


@pytest.fixture(scope="module")
def lgpu(lapi):
    if lapi.device_count() < 1:
        pytest.fail("no CUDA device visible: the line detection GPU tests need a B200 (no CPU fallback exists)")
    return lapi


def select_lines(F, P, thr, max_lines, bin_range=None):
    """the contract's selection on F rows [..., nframes, n] (and P rows of the same shape, or None): dict(count, bin,
    ftest, psd) as the *_run_mtm_lines entries return them"""
    F = np.asarray(F, np.float32)
    lead, n = F.shape[:-1], F.shape[-1]
    lo, hi = (0, n) if bin_range is None else bin_range
    f2 = F.reshape(-1, n)
    p2 = None if P is None else np.asarray(P, np.float32).reshape(-1, n)
    with np.errstate(invalid="ignore"):
        cand = (f2 > np.float32(thr)) & (f2 > np.roll(f2, 1, axis=1)) & (f2 >= np.roll(f2, -1, axis=1))
    cand[:, :lo] = False
    cand[:, hi:] = False
    count = cand.sum(axis=1).astype(np.int32)
    b = np.full((len(f2), max_lines), -1, np.int32)
    ft = np.zeros((len(f2), max_lines), np.float32)
    ps = np.zeros((len(f2), max_lines), np.float32)
    for r in np.nonzero(count)[0]:
        js = np.nonzero(cand[r])[0]
        if len(js) > max_lines:
            js = np.sort(js[np.lexsort((js, -f2[r, js]))[:max_lines]])
        b[r, :len(js)] = js
        ft[r, :len(js)] = f2[r, js]
        if p2 is not None:
            ps[r, :len(js)] = p2[r, js]
    return dict(count=count.reshape(lead), bin=b.reshape(lead + (max_lines,)), ftest=ft.reshape(lead + (max_lines,)),
                psd=ps.reshape(lead + (max_lines,)) if P is not None else None)


def brute_lines(row, thr, max_lines, lo, hi):
    """one row, bin by bin with Python floats: (count, selected bins in ascending order)"""
    n = len(row)
    cands = []
    for j in range(lo, hi):
        v, left, right = float(row[j]), float(row[(j - 1) % n]), float(row[(j + 1) % n])
        if v > thr and v > left and v >= right:
            cands.append(j)
    chosen = cands
    if len(cands) > max_lines:
        chosen = sorted(sorted(cands, key=lambda j: (-float(row[j]), j))[:max_lines])
    return len(cands), chosen


def assert_lines_equal(got, want, what):
    for key in ("count", "bin", "ftest", "psd"):
        if want.get(key) is None or got.get(key) is None:
            continue
        g, w = got[key], want[key]
        assert g.shape == w.shape, (what, key, g.shape, w.shape)
        eq = np.array_equal(g.view(np.int32), w.view(np.int32)) if g.dtype == np.float32 else np.array_equal(g, w)
        assert eq, (what, key, int(np.sum(g != w)))


def _iq(n, seed=0x5EED):
    from glfer_b200 import synth
    return synth.iq_stream(n, fs=int(FS), seed=seed, dot_s=0.5)


def _check_plan(api, plan, z, thr_pfa, max_lines, bin_range=None, what="", **kw):
    """lines of plan on z against the restatement on run_mtm_ftest of the same call; returns the lines"""
    ref = plan.run_mtm_ftest(z, **kw)
    kp = plan.mtm_kmax + 1
    thr = api.ftest_threshold(kp, thr_pfa)
    got = plan.run_mtm_lines(z, pfa=thr_pfa, max_lines=max_lines, bin_range=bin_range, **kw)
    assert_lines_equal(got, select_lines(ref["ftest"], ref["psd"], thr, max_lines, bin_range), what)
    return got


# ------------------------------------------------------------------------------------------------ CPU
def test_threshold_against_scipy(lapi):
    from scipy import stats
    for kp in (2, 4, 8, 16, 32):
        for e in range(2, 10):
            pfa = 10.0 ** -e
            thr = lapi.ftest_threshold(kp, pfa)
            ref = stats.f(2, 2 * kp - 2).isf(pfa)
            assert abs(thr - ref) / ref <= 1e-6, (kp, pfa, thr, ref)
            assert thr == float(np.float32(thr))


def test_threshold_rejections(lapi):
    import ctypes as C
    for kp, pfa in ((1, 1e-3), (0, 1e-3), (8, 0.0), (8, 1.0), (8, -0.1), (8, 2.0), (8, float("nan"))):
        with pytest.raises(lapi.GlferError):
            lapi.ftest_threshold(kp, pfa)
    assert lapi.lib().glfer_ftest_threshold(8, 1e-3, None) == -2
    t = C.c_float()
    assert lapi.lib().glfer_ftest_threshold(8, 1e-3, C.byref(t)) == 0 and t.value > 1.0


def _hand_rows():
    nan, inf = np.float32("nan"), np.float32("inf")
    rows = [
        [9, 1, 1, 5, 5, 5, 1, 7, 7, 2, 3, 9, 1, 8, 2, 9],     # plateaus, one across the wrap (j = 15, 0)
        [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16],  # wraps: j = 15 beats j = 0
        [16, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 1],  # wraps: j = 0 beats j = 15 (and 14 peaks)
        [nan, 5, 1, 6, nan, 2, inf, 3, 4, nan, 4, 1, 3, 3, 3, 2],  # NaN and inf
        [5, 1, 5, 1, 5, 1, 5, 1, 4, 1, 5, 1, 5, 1, 5, 1],     # ties at the cap
        [2, 3, 2, 3, 2, 3, 2, 3, 2, 3, 2, 3, 2, 3, 2, 3],     # every other bin a line
        [0] * 16,
        [nan] * 16,
        [7] * 16,                                              # one plateau over the whole row: no left edge
    ]
    return np.array(rows, np.float32)


@pytest.mark.parametrize("max_lines", [1, 2, 3, 4, 16])
@pytest.mark.parametrize("bin_range", [(0, 16), (1, 15), (4, 5), (5, 8), (13, 16), (0, 1)])
def test_restatement_against_a_per_bin_loop(max_lines, bin_range):
    rows = _hand_rows()
    P = np.arange(rows.size, dtype=np.float32).reshape(rows.shape) + 0.5
    thr = 1.5
    got = select_lines(rows, P, thr, max_lines, bin_range)
    for r, row in enumerate(rows):
        cnt, js = brute_lines(row, thr, max_lines, *bin_range)
        assert got["count"][r] == cnt, (r, bin_range)
        assert list(got["bin"][r, :len(js)]) == js and (got["bin"][r, len(js):] == -1).all(), (r, bin_range, js)
        assert np.array_equal(got["ftest"][r, :len(js)], row[js]) and (got["ftest"][r, len(js):] == 0).all()
        assert np.array_equal(got["psd"][r, :len(js)], P[r, js]) and (got["psd"][r, len(js):] == 0).all()


def test_restatement_hand_cases():
    rows = _hand_rows()
    full = select_lines(rows, None, 1.5, 16)
    assert list(full["bin"][0][:full["count"][0]]) == [3, 7, 11, 13, 15]         # plateaus: the leftmost bin, cyclically
    assert list(full["bin"][1][:full["count"][1]]) == [15]
    assert list(full["bin"][2][:full["count"][2]]) == [0, 14]
    assert list(full["bin"][3][:full["count"][3]]) == [6, 12]                    # NaN never wins, nor beats a NaN; inf wins
    assert full["count"][6] == 0 and full["count"][7] == 0 and full["count"][8] == 0
    cap = select_lines(rows, None, 1.5, 3)
    assert cap["count"][4] == 8 and list(cap["bin"][4]) == [0, 2, 4]             # ties at 5 go to the smaller j
    # a peak outside the range is not reported even though its neighbour inside is smaller
    assert list(select_lines(rows, None, 1.5, 16, (1, 3))["bin"][0][:1]) == [-1]
    assert list(select_lines(rows, None, 1.5, 16, (12, 15))["bin"][0][:2]) == [13, -1]


# ------------------------------------------------------------------------------------------------ GPU: exactness
@pytest.mark.gpu
@pytest.mark.parametrize("n", [32, 256, 2048, 8192, 16384])
@pytest.mark.parametrize("overlap", [0.5, 0.6])
def test_iq_lines_exact(lgpu, n, overlap):
    p = lgpu.IqPlan(n=n, overlap=overlap, multitaper=True, mtm_w=4.0, mtm_kmax=3)
    nframes = 6 if n >= 8192 else 24
    z = _iq(p.required_span(0, nframes)[1], seed=n)
    fused = _fused(n, p.hop)
    for forced in ([False, True] if fused else [True]):
        lgpu.force_generic_kernel(forced)
        try:
            for pfa, m in ((1e-2, 16), (0.2, 4)):
                what = f"iq n={n} ov={overlap} general={forced} pfa={pfa} M={m}"
                got = _check_plan(lgpu, p, z, pfa, m, what=what)
                assert got["count"].sum() > 0, what
                for wf, wp in ((False, True), (True, False), (False, False)):
                    part = p.run_mtm_lines(z, pfa=pfa, max_lines=m, want_ftest=wf, want_psd=wp)
                    assert np.array_equal(part["count"], got["count"]) and np.array_equal(part["bin"], got["bin"]), what
                    assert (part["ftest"] is None) != wf and (part["psd"] is None) != wp
                    if wf:
                        assert np.array_equal(part["ftest"], got["ftest"]), what
                    if wp:
                        assert np.array_equal(part["psd"], got["psd"]), what
        finally:
            lgpu.force_generic_kernel(False)
    p.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n,max_lines,pfa", [(2048, 1, 0.2), (2048, 16, 0.2), (8192, 1024, 0.5), (256, 1024, 0.2)])
def test_iq_lines_top_k(lgpu, n, max_lines, pfa):
    """caps that most frames overflow: the radix select and the tie rule on the device"""
    p = lgpu.IqPlan(n=n, overlap=0.5, multitaper=True, mtm_w=2.5, mtm_kmax=1)
    nframes = 8 if n >= 8192 else 30
    rng = np.random.default_rng(n + max_lines)
    span = p.required_span(0, nframes)[1]
    z = (rng.standard_normal(span) + 1j * rng.standard_normal(span)).astype(np.complex64)
    got = _check_plan(lgpu, p, z, pfa, max_lines, what=f"top-k n={n} M={max_lines}")
    if max_lines < 1024 or n >= 8192:
        assert np.mean(got["count"] > max_lines) > 0.5, got["count"]


@pytest.mark.gpu
def test_lines_ties_on_the_device(lgpu):
    """ties of F at the cap on the device: a frame of tones at exact bin centres of equal amplitude repeats the same F
    values on bins of the same pattern; whatever ties arise, the restatement decides them the same way"""
    n = 256
    p = lgpu.IqPlan(n=n, overlap=0.0, multitaper=True, mtm_w=4.0, mtm_kmax=3)
    t = np.arange(p.required_span(0, 10)[1])
    z = np.zeros(len(t), np.complex64)
    for k in range(-120, 120, 24):
        z += np.exp(2j * np.pi * k * t / n).astype(np.complex64)
    for m in (1, 3, 5):
        _check_plan(lgpu, p, z, 0.2, m, what=f"tones M={m}")


@pytest.mark.gpu
@pytest.mark.parametrize("iq", [False, True])
def test_zoom_lines_exact(lgpu, iq):
    from glfer_b200 import synth
    p = lgpu.ZoomPlan(n=512, decim=16, overlap=0.75, center_hz=-800.0 if iq else 800.0, sample_rate=FS, iq=iq,
                      multitaper=True, mtm_w=4.0, mtm_kmax=7)
    nframes = 30
    span = p.required_span(0, nframes)[1]
    x = _iq(span, seed=11) if iq else synth.qrss_stream(span, fs=int(FS), dot_s=0.5)
    for m, pfa, rng in ((16, 1e-2, None), (4, 0.2, None), (16, 1e-2, (56, 456))):
        _check_plan(lgpu, p, x, pfa, m, rng, what=f"zoom iq={iq} M={m} range={rng}")
    pcm = synth.iq_stream_int16(span, fs=int(FS), dot_s=0.5) if iq else synth.qrss_stream_int16(span, fs=int(FS), dot_s=0.5)
    _check_plan(lgpu, p, pcm, 1e-2, 16, what=f"zoom pcm16 iq={iq}")


@pytest.mark.gpu
@pytest.mark.parametrize("iq", [False, True])
def test_bank_lines_are_the_single_plans(lgpu, iq):
    from glfer_b200 import synth
    centers = [-1500.0, 700.0, 2300.5] if iq else [600.0, 1500.0, 2300.5]
    kw = dict(n=256, decim=32, overlap=0.5, sample_rate=FS, iq=iq, multitaper=True, mtm_w=4.0, mtm_kmax=5)
    bank = lgpu.ZoomPlan(center_hz=centers, **kw)
    nframes = 40
    span = bank.required_span(0, nframes)[1]
    x = synth.iq_stream_int16(span, fs=int(FS), dot_s=0.5) if iq else synth.qrss_stream_int16(span, fs=int(FS), dot_s=0.5)
    got = _check_plan(lgpu, bank, x, 1e-2, 8, what=f"bank iq={iq}")
    assert got["count"].shape == (3, nframes) and got["bin"].shape == (3, nframes, 8)
    for c, fc in enumerate(centers):
        single = lgpu.ZoomPlan(center_hz=fc, **kw)
        one = single.run_mtm_lines(x, pfa=1e-2, max_lines=8)
        for key in ("count", "bin", "ftest", "psd"):
            assert np.array_equal(one[key], got[key][c]), (c, key)
        single.close()


@pytest.mark.gpu
@pytest.mark.parametrize("overlap", [0.5, 0.6])
def test_iq_lines_chunks_splits_and_pcm16(lgpu, overlap):
    from glfer_b200 import synth
    p = lgpu.IqPlan(n=1024, overlap=overlap, multitaper=True, mtm_w=4.0, mtm_kmax=3)
    nframes = (5 << 21) // p.hop                             # several ~32 MiB chunks
    pcm = synth.iq_stream_int16(p.required_span(0, nframes)[1], fs=int(FS), dot_s=0.5)
    zf = synth.pcm16_to_float(pcm)
    whole = _check_plan(lgpu, p, zf, 1e-3, 16, what=f"chunked ov={overlap}")
    assert_lines_equal(p.run_mtm_lines(pcm, pfa=1e-3, max_lines=16), whole, "pcm16")
    step = nframes // 3 + 7
    parts = [p.run_mtm_lines(zf, pfa=1e-3, max_lines=16, first_frame=a, nframes=min(step, nframes - a))
             for a in range(0, nframes, step)]
    for key in ("count", "bin", "ftest", "psd"):
        assert np.array_equal(np.concatenate([q[key] for q in parts]), whole[key]), key


@pytest.mark.gpu
def test_zoom_lines_chunked_bank(lgpu):
    """a bank run of several chunks against runs of its parts"""
    centers = [-3000.0, 1000.0]
    q = lgpu.ZoomPlan(n=64, decim=256, overlap=0.75, center_hz=centers, sample_rate=FS, iq=True, multitaper=True,
                      mtm_w=2.5, mtm_kmax=3)
    z = _iq(q.required_span(0, 3000)[1], seed=3)
    whole = _check_plan(lgpu, q, z, 1e-2, 4, what="chunked bank")
    parts = [q.run_mtm_lines(z, pfa=1e-2, max_lines=4, first_frame=a, nframes=min(1000, 3000 - a))
             for a in range(0, 3000, 1000)]
    for key in ("count", "bin", "ftest", "psd"):
        assert np.array_equal(np.concatenate([r[key] for r in parts], axis=1), whole[key]), key


@pytest.mark.gpu
@pytest.mark.parametrize("forced", [False, True])
def test_iq_lines_beyond_sample_2_pow_32(lgpu, forced):
    p = lgpu.IqPlan(n=2048, overlap=0.75, multitaper=True, mtm_w=4.0, mtm_kmax=7)
    first = ((1 << 32) + 12345) // p.hop + 3
    nframes = 8
    lo, hi = p.required_span(first, nframes)
    assert lo > (1 << 32)
    z = _iq(hi - lo, seed=7)
    lgpu.force_generic_kernel(forced)
    try:
        got = _check_plan(lgpu, p, z, 1e-2, 16, what=f"beyond 2^32 general={forced}", origin=lo, first_frame=first,
                          nframes=nframes)
    finally:
        lgpu.force_generic_kernel(False)
    assert got["count"].sum() > 0


@pytest.mark.gpu
def test_lines_narrow_range_and_silence(lgpu):
    n = 1024
    p = lgpu.IqPlan(n=n, overlap=0.5, multitaper=True, mtm_w=4.0, mtm_kmax=7)
    nframes = 20
    z = _iq(p.required_span(0, nframes)[1], seed=5)
    for rng in ((500, 530), (0, 1), (n - 1, n), (127, 129)):
        _check_plan(lgpu, p, z, 0.2, 4, rng, what=f"range {rng}")
    quiet = np.zeros(len(z), np.complex64)
    got = p.run_mtm_lines(quiet, pfa=0.5, max_lines=8)
    assert (got["count"] == 0).all() and (got["bin"] == -1).all()
    assert (got["ftest"] == 0).all() and (got["psd"] == 0).all()
    assert np.isnan(p.run_mtm_ftest(quiet, want_psd=False)["ftest"]).all()
    zq = lgpu.ZoomPlan(n=256, decim=16, center_hz=800.0, sample_rate=FS, multitaper=True)
    assert (zq.run_mtm_lines(np.zeros(zq.required_span(0, 5)[1], np.float32), pfa=0.5)["count"] == 0).all()


# ------------------------------------------------------------------------------------------------ GPU: statistics
@pytest.mark.gpu
def test_lines_on_white_noise_stay_below_the_false_alarm_count(lgpu):
    """local maxima above the threshold are a subset of the exceedances, whose expected number is pfa n frames; on a
    B200 the count comes to roughly a third of that (neighbouring F bins are correlated over the taper bandwidth)"""
    n, kp, pfa, nframes = 1024, 8, 1e-3, 400
    p = lgpu.IqPlan(n=n, overlap=0.0, multitaper=True, mtm_w=4.0, mtm_kmax=kp - 1)
    rng = np.random.default_rng(42)
    span = p.required_span(0, nframes)[1]
    z = (rng.standard_normal(span) + 1j * rng.standard_normal(span)).astype(np.complex64)
    got = p.run_mtm_lines(z, pfa=pfa, max_lines=16)
    expected = pfa * n * (nframes - 1)
    total = int(got["count"][1:].sum())
    assert total <= 1.2 * expected, (total, expected)        # 1.2: some 4 standard deviations of a Poisson count
    f = p.run_mtm_ftest(z, want_psd=False)["ftest"][1:]
    assert total <= int((f > lgpu.ftest_threshold(kp, pfa)).sum())


@pytest.mark.gpu
def test_lines_report_a_weak_zoom_line(lgpu):
    """the weak line of test_ftest_detects_a_weak_line_on_a_zoom_bin, reported at its bin in >= 95 % of the frames"""
    n, decim, center, kp = 512, 16, 800.0, 8
    p = lgpu.ZoomPlan(n=n, decim=decim, overlap=0.0, center_hz=center, sample_rate=FS, iq=True, multitaper=True,
                      mtm_w=4.0, mtm_kmax=kp - 1)
    nframes = 60
    span = p.required_span(0, nframes)[1]
    rng = np.random.default_rng(9)
    bin_off = 10
    f_tone = p.center_hz() + bin_off * FS / (decim * n)
    t = np.arange(span)
    z = (0.1 * np.exp(2j * np.pi * f_tone / FS * t)
         + rng.standard_normal(span) + 1j * rng.standard_normal(span)).astype(np.complex64)
    got = p.run_mtm_lines(z, pfa=1e-4, max_lines=16, bin_range=(n // 2 - int(0.4 * n), n // 2 + int(0.4 * n)))
    hit = (got["bin"][2:] == n // 2 + bin_off).any(axis=1)
    assert hit.mean() >= 0.95, (hit.mean(), got["count"][2:])


# ------------------------------------------------------------------------------------------------ GPU: launches, rejections
@pytest.mark.gpu
@pytest.mark.parametrize("nchan", [1, 8])
def test_lines_launch_count(lgpu, nchan):
    """a lines run launches what the F-only run launches plus one kernel per chunk, whatever the number of channels"""
    centers = [-4000.0 + 1000.0 * c for c in range(nchan)]
    p = lgpu.ZoomPlan(n=256, decim=64, overlap=0.5, center_hz=centers if nchan > 1 else centers[0], sample_rate=FS,
                      iq=True, multitaper=True, mtm_w=4.0, mtm_kmax=3)
    chunk = (32 << 20) // (p.hop * 64 * 8)
    nframes = 2 * chunk + 5                                   # three chunks
    z = _iq(p.required_span(0, nframes)[1], seed=1)
    q = lgpu.IqPlan(n=1024, overlap=0.5, multitaper=True, mtm_w=4.0, mtm_kmax=3)
    qchunk = (32 << 20) // (q.hop * 8)
    zq = _iq(q.required_span(0, qchunk + 3)[1], seed=2)
    for plan, x, chunks in ((p, z, 3), (q, zq, 2)):
        if plan is q and nchan > 1:
            continue
        for want_psd in (False, True):
            plan.run_mtm_ftest(x, want_psd=want_psd)
            a = lgpu.kernel_launches()
            plan.run_mtm_ftest(x, want_psd=want_psd)
            f_only = lgpu.kernel_launches() - a
            a = lgpu.kernel_launches()
            plan.run_mtm_lines(x, want_psd=want_psd)
            lines = lgpu.kernel_launches() - a
            assert lines == f_only + chunks, (want_psd, lines, f_only, chunks)


@pytest.mark.gpu
def test_lines_entry_point_rejections(lgpu):
    import ctypes as C
    lib = lgpu.lib()
    n = 256
    iqp = lgpu.IqPlan(n=n, overlap=0.5)                                    # periodogram
    iq1 = lgpu.IqPlan(n=n, overlap=0.5, multitaper=True, mtm_kmax=0)       # K' = 1
    iqm = lgpu.IqPlan(n=n, overlap=0.5, multitaper=True)
    zr = lgpu.ZoomPlan(n=n, decim=16, center_hz=800.0, sample_rate=FS, multitaper=True)
    zq = lgpu.ZoomPlan(n=n, decim=16, center_hz=-800.0, sample_rate=FS, iq=True, multitaper=True)
    zp = lgpu.ZoomPlan(n=n, decim=16, center_hz=-800.0, sample_rate=FS, iq=True)
    z1 = lgpu.ZoomPlan(n=n, decim=16, center_hz=800.0, sample_rate=FS, multitaper=True, mtm_kmax=0)
    hi = zr.required_span(0, 2)[1]
    x = np.zeros(2 * hi, np.float32)
    pcm = np.zeros(2 * hi, np.int16)
    cnt = np.empty(2, np.int32)
    b = np.empty((2, 1024), np.int32)
    ft = np.empty((2, 1024), np.float32)
    ps = np.empty((2, 1024), np.float32)
    CN, B, F, P = cnt.ctypes.data, b.ctypes.data, ft.ctypes.data, ps.ctypes.data
    good = lgpu.LinesConfig(1e-3, 16, 0, n)
    bad = [lgpu.LinesConfig(0.0, 16, 0, n), lgpu.LinesConfig(1.0, 16, 0, n), lgpu.LinesConfig(float("nan"), 16, 0, n),
           lgpu.LinesConfig(1e-3, 0, 0, n), lgpu.LinesConfig(1e-3, 1025, 0, n), lgpu.LinesConfig(1e-3, 16, -1, n),
           lgpu.LinesConfig(1e-3, 16, 5, 5), lgpu.LinesConfig(1e-3, 16, 6, 5), lgpu.LinesConfig(1e-3, 16, 0, n + 1)]

    def common(fn, plan, buf, span):
        g = C.byref(good)
        assert fn(plan._h, buf.ctypes.data, 0, span, 0, 2, g, CN, B, F, P) == 0
        assert fn(plan._h, buf.ctypes.data, 0, span, 0, 2, g, CN, B, None, None) == 0
        assert fn(plan._h, buf.ctypes.data, 0, span, 0, 2, None, CN, B, F, P) == -2          # lc NULL
        assert fn(plan._h, buf.ctypes.data, 0, span, 0, 2, g, None, B, F, P) == -2          # line_count NULL
        assert fn(plan._h, buf.ctypes.data, 0, span, 0, 2, g, CN, None, F, P) == -2         # line_bin NULL
        assert fn(plan._h, None, 0, span, 0, 2, g, CN, B, F, P) == -2                       # samples NULL
        assert fn(plan._h, buf.ctypes.data, 0, span - 1, 0, 2, g, CN, B, F, P) == -2        # short input
        assert fn(plan._h, buf.ctypes.data, 0, span, 0, -1, g, CN, B, F, P) == -2           # negative frame range
        for lc in bad:
            assert fn(plan._h, buf.ctypes.data, 0, span, 0, 2, C.byref(lc), CN, B, F, P) == -2, (
                lc.pfa, lc.max_lines, lc.bin_lo, lc.bin_hi)

    for fn, buf in ((lib.glfer_iq_run_mtm_lines, x), (lib.glfer_iq_run_mtm_lines_pcm16, pcm)):
        common(fn, iqm, buf, iqm.required_span(0, 2)[1])
        g = C.byref(good)
        assert fn(iqp._h, buf.ctypes.data, 0, hi, 0, 2, g, CN, B, F, P) == -2          # periodogram plan
        assert fn(iq1._h, buf.ctypes.data, 0, hi, 0, 2, g, CN, B, F, P) == -2          # K' = 1
        assert fn(None, buf.ctypes.data, 0, hi, 0, 2, g, CN, B, F, P) == -2
    for fn, plan, other, buf in ((lib.glfer_zoom_run_mtm_lines, zr, zq, x), (lib.glfer_zoom_run_mtm_lines_pcm16, zr, zq, pcm),
                                 (lib.glfer_zoom_run_iq_mtm_lines, zq, zr, x),
                                 (lib.glfer_zoom_run_iq_mtm_lines_pcm16, zq, zr, pcm)):
        common(fn, plan, buf, hi)
        assert fn(other._h, buf.ctypes.data, 0, hi, 0, 2, C.byref(good), CN, B, F, P) == -2   # real entry, I/Q plan or the reverse
    assert lib.glfer_zoom_run_iq_mtm_lines(zp._h, x.ctypes.data, 0, hi, 0, 2, C.byref(good), CN, B, F, P) == -2
    assert lib.glfer_zoom_run_mtm_lines(z1._h, x.ctypes.data, 0, hi, 0, 2, C.byref(good), CN, B, F, P) == -2
    with pytest.raises(lgpu.GlferError):
        iqm.run_mtm_lines(np.zeros(hi, np.complex64), pfa=1e-3, max_lines=2000)
