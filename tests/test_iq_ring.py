"""The fused I/Q ring kernels in their steady state (gram_iq_kernel with float rows and with levels, gram_iq_mtm_kernel,
gram_iq_ftest_kernel), against the float64 restatements of tests/test_iq.py, test_iq_mtm.py, test_iq_ftest.py and
test_iq_display.py.

The launch policy gives short runs one frame per frame group, so without a cap the ring's frame loop never passes its
first iteration: the mbarrier waits of later frames and their phase parity, the request of the next block, the slot
rotation and its wrap, TMA refilling slots the prologue zero-filled, the ragged last group and the inactive groups of a
partly filled CTA.  api.set_ring_groups(c) caps the group count, so that every group holds at least 2 nb + 2 frames
(nb = n / hop ring slots: every slot refilled at least twice, both parities waited on).

  A  every fused geometry (n = 32 .. 8192, overlap 0 .. 93.75 %) x every fused kernel, c = 1, 3 and G + 1 (G frame
     groups per CTA): oracle parity, and rows, F rows and levels bit-identical across c and to the uncapped launch.
  B  frame origins in the steady state: the stream start, a partial zero history, far from 0, an odd origin.
  C  the launch policy itself on a run of two chunks, with several frames per group.
  D  all 8 window types on one fused geometry and on the general path.

The launcher declines none of these geometries: its shared-memory gate (227 KiB) is met everywhere, the largest case
being the F-test at n = 8192 (one frame group of 137 KiB, 8 KiB of mid-pass twiddles and 68 KiB of mu columns:
213 KiB; the ring takes 8 n bytes at every overlap), and one CTA always fits an SM, so every case asserts the ring
kernel family."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from parity import assert_psd_close  # noqa: E402
from test_iq import iq_oracle  # noqa: E402
from test_iq_display import _fixed_displays, _oracle  # noqa: E402
from test_iq_ftest import assert_f_close, ftest_rows  # noqa: E402
from test_iq_mtm import iq_frames, mtm_rows  # noqa: E402

pytestmark = pytest.mark.gpu

FS = 48000
KAISER = 7
FUSED_N = (32, 64, 128, 256, 512, 1024, 2048, 4096, 8192)
FUSED_OV = (0.0, 0.5, 0.75, 0.875, 0.9375)
VARIANTS = ("rows", "levels", "mtm", "ftest")
RING = "gram_ring_kernel"


@pytest.fixture(scope="module")
def rapi():
    from glfer_b200 import build
    build.build()
    from glfer_b200 import api
    if api.device_count() < 1:
        pytest.fail("no CUDA device visible: the I/Q ring tests need a B200 (no CPU fallback exists)")
    try:
        yield api
    finally:
        api.set_ring_groups(0)
        api.force_generic_kernel(False)
        api.set_fused_levels(True)


def _iq(count, seed):
    from glfer_b200 import synth
    return synth.iq_stream(count, fs=FS, seed=seed, dot_s=0.5)


def _cdiv(a, b):
    return -(-a // b)


def _groups_per_cta(n):
    """Geo<n>::G: 128 threads of n / 16 threads per frame group, one group from n = 2048 on"""
    return max(1, 2048 // n)


def _frames_for(nb, cs):
    """the least frame count with >= 2 nb + 2 frames in every group at each cap c, a ragged last group (c > 1) and
    exactly c groups in use"""
    need = 2 * nb + 2
    nf = max(cs) * need
    while not all(_cdiv(nf, c) >= need and (c == 1 or nf % _cdiv(nf, c) != 0) and _cdiv(nf, _cdiv(nf, c)) == c
                  for c in cs):
        nf += 1
    return nf


def _capped(api, c, fn):
    """fn() with the fused launches capped at c frame groups (0: the launch policy); returns (result, kernel family,
    frames per group of the last fused launch)"""
    api.set_ring_groups(c)
    try:
        out = fn()
        return out, api.last_kernel_family(), api.last_frames_per_group()
    finally:
        api.set_ring_groups(0)


def _plan(api, n, overlap, variant, kp=3, window_type=KAISER):
    if variant in ("rows", "levels"):
        return api.IqPlan(n=n, window_type=window_type, overlap=overlap)
    return api.IqPlan(n=n, overlap=overlap, multitaper=True, mtm_w=4.0, mtm_kmax=kp - 1)


def _display(api, p, z, fused_levels, disp, **kw):
    api.set_fused_levels(fused_levels)
    try:
        return p.run_display(z, autoscale=False, **disp, **kw)["levels"]
    finally:
        api.set_fused_levels(True)


# ------------------------------------------------------------------------------------------------ A: capped groups
CASES_A = ([(n, ov, v, 3 if v in ("mtm", "ftest") else 1) for n in FUSED_N for ov in FUSED_OV for v in VARIANTS]
           + [(256, ov, v, 16) for ov in FUSED_OV for v in ("mtm", "ftest")])


@pytest.mark.parametrize("n,overlap,variant,kp", CASES_A)
def test_capped_groups_match_the_oracle(rapi, n, overlap, variant, kp):
    api = rapi
    p = _plan(api, n, overlap, variant, kp)
    hop = p.hop
    nb = n // hop
    cs = sorted({1, 3, _groups_per_cta(n) + 1})
    nf = _frames_for(nb, cs)
    z = _iq(p.required_span(0, nf)[1], seed=n + 17 * nb + kp)
    what = f"n={n} ov={overlap} {variant} K'={kp} nframes={nf}"
    if variant in ("rows", "levels"):
        ref = iq_oracle(api, z, 0, n, KAISER, overlap, 0, nf)
    else:
        frames = iq_frames(z, 0, n, hop, 0, nf)
        tapers, lam = p.tapers()
        ref = mtm_rows(frames, tapers, lam)
        fref = ftest_rows(frames, tapers) if variant == "ftest" else None
        del frames

    base, fam, _ = _capped(api, 0, lambda: p.run(z))
    assert fam.startswith(RING), (what, fam)
    assert_psd_close(base, ref, what + " uncapped")
    if variant == "ftest":
        fbase, fam, _ = _capped(api, 0, lambda: p.run_mtm_ftest(z))
        assert fam.startswith(RING), (what, fam)
        assert_f_close(fbase["ftest"], fref, what + " uncapped")
        assert np.array_equal(fbase["psd"], base), what

    for c in cs:
        wc = f"{what} c={c}"
        rows, fam, fpg = _capped(api, c, lambda: p.run(z))
        assert fam.startswith(RING), (wc, fam)
        assert fpg == _cdiv(nf, c), (wc, fpg)
        assert_psd_close(rows, ref, wc)
        assert np.array_equal(rows, base), wc                     # a frame's row does not depend on its place
        if variant == "ftest":
            got, fam, fpg = _capped(api, c, lambda: p.run_mtm_ftest(z))
            assert fam.startswith(RING) and fpg == _cdiv(nf, c), (wc, fam, fpg)
            assert_f_close(got["ftest"], fref, wc)
            assert np.array_equal(got["psd"], rows), wc
            assert np.array_equal(got["ftest"], fbase["ftest"]), wc
        elif variant == "levels":
            for disp in _fixed_displays(base):
                want = _oracle(base, overlap, disp, False)[0]
                assert want.min() < want.max(), disp
                fused, fam, fpg = _capped(api, c, lambda: _display(api, p, z, True, disp))
                assert fam.startswith(RING) and fpg == _cdiv(nf, c), (wc, disp, fam, fpg)
                assert np.array_equal(fused, want), (wc, disp, int((fused != want).sum()))
                two, fam, fpg = _capped(api, c, lambda: _display(api, p, z, False, disp))
                assert fam.startswith(RING) and fpg == _cdiv(nf, c), (wc, disp, fam, fpg)
                assert np.array_equal(two, want), (wc, disp, int((two != want).sum()))
    p.close()


# ------------------------------------------------------------------------------------------------ B: frame origins
def _start(n, hop, nb, nf, start):
    """(first_frame, origin, sample count) of a run of nf frames from the given start"""
    first = {"zero": 0, "half": nb // 2, "far": 1_000_003, "odd_origin": 3 * nb + 1}[start]
    lo, hi = first * hop - (n - hop), (first + nf) * hop
    origin = {"zero": 0, "half": 0, "far": lo, "odd_origin": lo - 1}[start]
    return first, origin, hi - origin


@pytest.mark.parametrize("start", ("zero", "half", "far", "odd_origin"))
@pytest.mark.parametrize("variant", ("rows", "ftest"))
@pytest.mark.parametrize("overlap", (0.875, 0.9375))
@pytest.mark.parametrize("n", (64, 1024, 8192))
def test_frame_origins_in_the_steady_state(rapi, n, overlap, variant, start):
    """zero: the prologue's zero-filled slots are refilled by TMA later in the group; half: a partial zero history;
    far: every block from TMA; odd_origin: an odd origin one sample before the frames' first sample (lo is even on
    every fused geometry, the hops being even), so the staged copy starts one complex sample into the caller's
    buffer"""
    api = rapi
    p = _plan(api, n, overlap, variant)
    hop = p.hop
    nb = n // hop
    nf = 2 * nb + 3
    first, origin, count = _start(n, hop, nb, nf, start)
    z = _iq(count, seed=n + nb + len(start))
    what = f"n={n} ov={overlap} {variant} start={start} first={first} origin={origin}"
    if variant == "rows":
        got, fam, fpg = _capped(api, 1, lambda: p.run(z, origin=origin, first_frame=first, nframes=nf))
        assert fam.startswith(RING) and fpg == nf, (what, fam, fpg)
        assert_psd_close(got, iq_oracle(api, z, origin, n, KAISER, overlap, first, nf), what)
    else:
        got, fam, fpg = _capped(api, 1, lambda: p.run_mtm_ftest(z, origin=origin, first_frame=first, nframes=nf))
        assert fam.startswith(RING) and fpg == nf, (what, fam, fpg)
        frames = iq_frames(z, origin, n, hop, first, nf)
        tapers, lam = p.tapers()
        assert_f_close(got["ftest"], ftest_rows(frames, tapers), what)
        assert_psd_close(got["psd"], mtm_rows(frames, tapers, lam), what)
    p.close()


# ------------------------------------------------------------------------------------------------ C: launch policy
SLICE = 512                                                       # oracle frames at a time (host memory)
F_FLOOR = 1e-6


def _assert_f_close_long(got, ref, what):
    """assert_f_close on the bins with F >= F_FLOOR, and an absolute error below 2e-3 F_FLOOR under it.  F is
    proportional to |mu|^2, whose float32 error is absolute (about 3e-7 of the row's level): where F ~ 1e-7 (|mu| some
    3e-4 of its mean) that is a relative error of ~2e-3.  The 12 short frames of the other F-tests hold no such bin;
    the 50 M bins of a two-chunk run at n = 4096 hold a few (2.4e-3 measured on a B200, at median 2.7e-7 and p99
    2.7e-6).  At F_FLOOR itself the rounding is ~6e-4 relative, inside assert_f_close's bound."""
    ok = np.isfinite(ref) & (ref > 0)
    big = ok & (ref >= F_FLOOR)
    assert_f_close(got[big], ref[big], what)
    small = ok & ~big
    assert np.isfinite(got[small]).all(), what
    err = np.abs(got[small].astype(np.float64) - ref[small])
    assert err.size == 0 or err.max() < 2e-3 * F_FLOOR, (what, int(small.sum()), float(err.max()))


@pytest.mark.parametrize("variant", VARIANTS)
def test_launch_policy_on_a_run_of_two_chunks(rapi, variant):
    """n = 4096 at 87.5 %: chunks of 8192 frames (~32 MiB of input), the second one of 4099, each launch with several
    frames per group under the uncapped policy"""
    api = rapi
    n, overlap = 4096, 0.875
    p = _plan(api, n, overlap, variant)
    hop = p.hop
    nf = 8192 + 4099
    z = _iq(p.required_span(0, nf)[1], seed=41)
    what = f"n={n} ov={overlap} {variant} nframes={nf}"
    if variant in ("mtm", "ftest"):
        tapers, lam = p.tapers()
    if variant == "ftest":
        out, fam, fpg = _capped(api, 0, lambda: p.run_mtm_ftest(z))
        rows, ft = out["psd"], out["ftest"]
    else:
        rows, fam, fpg = _capped(api, 0, lambda: p.run(z))
    assert fam.startswith(RING) and fpg >= 4, (what, fam, fpg)
    for a in range(0, nf, SLICE):
        k = min(SLICE, nf - a)
        ws = f"{what} frames {a}..{a + k}"
        if variant in ("rows", "levels"):
            assert_psd_close(rows[a:a + k], iq_oracle(api, z, 0, n, KAISER, overlap, a, k), ws)
            continue
        frames = iq_frames(z, 0, n, hop, a, k)
        assert_psd_close(rows[a:a + k], mtm_rows(frames, tapers, lam), ws)
        if variant == "ftest":
            _assert_f_close_long(ft[a:a + k], ftest_rows(frames, tapers), ws)
    if variant == "levels":
        for disp in _fixed_displays(rows):
            fused, fam, fpg = _capped(api, 0, lambda: _display(api, p, z, True, disp))
            assert fam.startswith(RING) and fpg >= 4, (what, disp, fam, fpg)
            want = _oracle(rows, overlap, disp, False)[0]
            assert np.array_equal(fused, want), (what, disp, int((fused != want).sum()))
    p.close()


# ------------------------------------------------------------------------------------------------ D: windows
@pytest.mark.parametrize("forced", [False, True])
@pytest.mark.parametrize("wt", range(8))
def test_every_window_type(rapi, wt, forced):
    """the eight windows at n = 512, 87.5 %: the fused kernel with one frame group, and the general path"""
    api = rapi
    n, overlap = 512, 0.875
    p = _plan(api, n, overlap, "rows", window_type=wt)
    nb = n // p.hop
    nf = 2 * nb + 3
    z = _iq(p.required_span(0, nf)[1], seed=100 + wt)
    api.force_generic_kernel(forced)
    try:
        got, fam, fpg = _capped(api, 1, lambda: p.run(z))
    finally:
        api.force_generic_kernel(False)
    what = f"n={n} ov={overlap} window={wt} general={forced}"
    if forced:
        assert fam.startswith("gram_kernel"), (what, fam)
    else:
        assert fam.startswith(RING) and fpg == nf, (what, fam, fpg)
    assert_psd_close(got, iq_oracle(api, z, 0, n, wt, overlap, 0, nf), what)
    p.close()
