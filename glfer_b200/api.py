"""ctypes binding of libglfer_b200.so for the tests and bench.py.

Thin on purpose: every call goes straight to the C-ABI entry points declared in
include/glfer_b200.h, include/fft.h, include/mtm.h and include/avg.h.  There is no
Python (or CPU) implementation behind it: if the library is missing or no CUDA device is
present the calls raise."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GLFER_B200_LIB") or os.path.join(HERE, "libglfer_b200.so")

MODE_FFT, MODE_MTM = 0, 1
MODE_LMP = 3                           # glfer.h:45 MODE_LMP
NO_AVG, AVG_SUMAVG, AVG_PLAIN, AVG_SUMEXTREME = 0, 1, 2, 3
HANNING, BLACKMAN, GAUSSIAN, WELCH, BARTLETT, RECTANGULAR, HAMMING, KAISER = range(8)


class GlferError(RuntimeError):
    pass


class GramConfig(C.Structure):
    _fields_ = [("mode", C.c_int), ("n", C.c_int), ("window_type", C.c_int), ("overlap", C.c_float),
                ("a", C.c_float), ("limiter", C.c_int), ("sub_mean", C.c_int), ("mtm_w", C.c_float),
                ("mtm_kmax", C.c_int), ("avg_mode", C.c_int), ("avg_depth", C.c_int), ("avg_minbin", C.c_int),
                ("avg_maxbin", C.c_int), ("avg_max0", C.c_int), ("avg_peakbin_init", C.c_int),
                ("scale_db", C.c_int), ("device", C.c_int), ("lmp_av", C.c_int), ("avg_band_only", C.c_int),
                ("mtm_ftest", C.c_int), ("zero_history", C.c_int)]


class FftParams(C.Structure):          # include/fft.h (reference fft.h:51-63)
    _fields_ = [("inbuf_audio", C.POINTER(C.c_float)), ("inbuf_fft", C.POINTER(C.c_float)),
                ("outbuf", C.POINTER(C.c_float)), ("n", C.c_int), ("window", C.POINTER(C.c_float)),
                ("window_type", C.c_int), ("overlap", C.c_float), ("a", C.c_float), ("limiter", C.c_int),
                ("sub_mean", C.c_int)]


class MtmParams(C.Structure):          # include/mtm.h (reference mtm.h:36-44)
    _fields_ = [("fft", FftParams), ("window", C.POINTER(C.POINTER(C.c_double))), ("sig", C.POINTER(C.c_double)),
                ("w", C.c_float), ("kmax", C.c_int)]


class LmpParams(C.Structure):          # include/lmp.h (reference lmp.h:37-46)
    _fields_ = [("fft", FftParams), ("avg", C.c_int), ("window", C.POINTER(C.POINTER(C.c_double))),
                ("sig", C.POINTER(C.c_double)), ("w", C.c_float), ("kmax", C.c_int)]


class AvgData(C.Structure):            # include/avg.h (reference avg.h:28-36)
    _fields_ = [("avgwidth", C.c_int), ("avgdepth", C.c_int), ("effdepth", C.c_int), ("avg", C.POINTER(C.c_double)),
                ("cum", C.POINTER(C.c_double)), ("avgarray", C.POINTER(C.POINTER(C.c_double)))]


class DisplayConfig(C.Structure):      # include/glfer_b200.h glfer_display_config
    _fields_ = [("log_scale", C.c_int), ("autoscale", C.c_int), ("max_level_db", C.c_float),
                ("min_level_db", C.c_float), ("thr_level", C.c_float), ("colortab", C.c_void_p)]


class ZoomConfig(C.Structure):       # include/glfer_b200.h glfer_zoom_config
    _fields_ = [("n", C.c_int), ("decim", C.c_int), ("window_type", C.c_int), ("overlap", C.c_float),
                ("center_hz", C.c_double), ("sample_rate", C.c_double), ("device", C.c_int)]


class IqConfig(C.Structure):         # include/glfer_b200.h glfer_iq_config
    _fields_ = [("n", C.c_int), ("window_type", C.c_int), ("overlap", C.c_float), ("device", C.c_int)]


class LinesConfig(C.Structure):      # include/glfer_b200.h glfer_lines_config
    _fields_ = [("pfa", C.c_double), ("max_lines", C.c_int), ("bin_lo", C.c_int), ("bin_hi", C.c_int)]


class Wav(C.Structure):
    _fields_ = [("sample_rate", C.c_int), ("bits", C.c_int), ("channels", C.c_int), ("nsamples", C.c_longlong),
                ("data", C.c_void_p)]


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GlferError(f"{LIB_PATH} is missing: run `python -m glfer_b200.build` (no fallback exists)")
        l = C.CDLL(LIB_PATH)
        l.glfer_b200_last_error.restype = C.c_char_p
        l.glfer_b200_host_alloc.restype = C.c_void_p
        l.glfer_b200_host_alloc.argtypes = [C.c_size_t]
        l.glfer_b200_host_free.argtypes = [C.c_void_p]
        l.glfer_b200_kernel_launches.restype = C.c_ulonglong
        l.glfer_gram_plan_create.argtypes = [C.POINTER(GramConfig), C.POINTER(C.c_void_p)]
        l.glfer_gram_plan_destroy.argtypes = [C.c_void_p]
        l.glfer_gram_hop.argtypes = [C.c_void_p]
        l.glfer_gram_bins.argtypes = [C.c_void_p]
        l.glfer_gram_avg_cols.argtypes = [C.c_void_p]
        l.glfer_gram_num_frames.argtypes = [C.c_void_p, C.c_longlong]
        l.glfer_gram_num_frames.restype = C.c_longlong
        l.glfer_gram_required_span.argtypes = [C.c_void_p, C.c_longlong, C.c_longlong, C.POINTER(C.c_longlong),
                                               C.POINTER(C.c_longlong)]
        l.glfer_gram_required_span.restype = None
        l.glfer_gram_window.argtypes = [C.c_void_p, C.c_void_p]
        l.glfer_gram_tapers.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        run_args = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_longlong, C.c_longlong,
                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        l.glfer_gram_run.argtypes = run_args
        l.glfer_gram_run_pcm16.argtypes = run_args
        l.glfer_gram_run_mtm_ftest.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_longlong, C.c_longlong,
                                               C.c_void_p, C.c_void_p]
        l.glfer_gram_stage.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong]
        l.glfer_gram_stage_pcm16.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong]
        l.glfer_gram_exec.argtypes = [C.c_void_p, C.c_longlong, C.c_longlong, C.POINTER(C.c_float)]
        l.glfer_gram_sync.argtypes = [C.c_void_p]
        l.glfer_gram_last_gram_ms.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        l.glfer_gram_fetch.argtypes = [C.c_void_p] + [C.c_void_p] * 5
        disp_args = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_longlong, C.c_longlong,
                     C.POINTER(DisplayConfig), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        l.glfer_gram_run_display.argtypes = disp_args
        l.glfer_gram_run_display_pcm16.argtypes = disp_args
        l.glfer_gram_run_sharded.argtypes = [C.POINTER(GramConfig), C.c_int, C.POINTER(C.c_int), C.c_void_p,
                                             C.c_longlong] + [C.c_void_p] * 5
        l.glfer_gram_shard_range.argtypes = [C.c_longlong, C.c_int, C.c_int, C.POINTER(C.c_longlong),
                                             C.POINTER(C.c_longlong)]
        l.glfer_gram_shard_range.restype = None
        l.glfer_wav_load.argtypes = [C.c_char_p, C.POINTER(Wav)]
        l.glfer_wav_free.argtypes = [C.POINTER(Wav)]
        l.glfer_wav_select_channel.argtypes = [C.POINTER(Wav), C.c_int]
        l.glfer_wav_num_frames.argtypes = [C.c_void_p, C.POINTER(Wav)]
        l.glfer_wav_num_frames.restype = C.c_longlong
        l.glfer_gram_run_wav.argtypes = [C.c_void_p, C.POINTER(Wav)] + [C.c_void_p] * 5
        # zoom spectrogram
        l.glfer_zoom_plan_create.argtypes = [C.POINTER(ZoomConfig), C.POINTER(C.c_void_p)]
        l.glfer_zoom_plan_destroy.argtypes = [C.c_void_p]
        l.glfer_zoom_hop.argtypes = [C.c_void_p]
        l.glfer_zoom_bins.argtypes = [C.c_void_p]
        l.glfer_zoom_center_hz.argtypes = [C.c_void_p]
        l.glfer_zoom_center_hz.restype = C.c_double
        l.glfer_zoom_num_frames.argtypes = [C.c_void_p, C.c_longlong]
        l.glfer_zoom_num_frames.restype = C.c_longlong
        l.glfer_zoom_required_span.argtypes = [C.c_void_p, C.c_longlong, C.c_longlong, C.POINTER(C.c_longlong),
                                               C.POINTER(C.c_longlong)]
        l.glfer_zoom_required_span.restype = None
        zoom_args = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_longlong, C.c_longlong, C.c_void_p]
        l.glfer_zoom_run.argtypes = zoom_args
        l.glfer_zoom_run_pcm16.argtypes = zoom_args
        l.glfer_zoom_taps.argtypes = [C.c_int, C.c_void_p]
        l.glfer_zoom_plan_create_iq.argtypes = [C.POINTER(ZoomConfig), C.POINTER(C.c_void_p)]
        l.glfer_zoom_run_iq.argtypes = zoom_args
        l.glfer_zoom_plan_create_bank.argtypes = [C.POINTER(ZoomConfig), C.c_void_p, C.c_int, C.c_int,
                                                  C.POINTER(C.c_void_p)]
        l.glfer_zoom_plan_create_bank_mtm.argtypes = [C.POINTER(ZoomConfig), C.c_void_p, C.c_int, C.c_int, C.c_float,
                                                      C.c_int, C.POINTER(C.c_void_p)]
        l.glfer_zoom_channels.argtypes = [C.c_void_p]
        l.glfer_zoom_channel_center_hz.argtypes = [C.c_void_p, C.c_int]
        l.glfer_zoom_channel_center_hz.restype = C.c_double
        l.glfer_zoom_run_iq_pcm16.argtypes = zoom_args
        # I/Q spectrogram
        l.glfer_iq_plan_create.argtypes = [C.POINTER(IqConfig), C.POINTER(C.c_void_p)]
        l.glfer_iq_plan_destroy.argtypes = [C.c_void_p]
        l.glfer_iq_hop.argtypes = [C.c_void_p]
        l.glfer_iq_bins.argtypes = [C.c_void_p]
        l.glfer_iq_num_frames.argtypes = [C.c_void_p, C.c_longlong]
        l.glfer_iq_num_frames.restype = C.c_longlong
        l.glfer_iq_required_span.argtypes = [C.c_void_p, C.c_longlong, C.c_longlong, C.POINTER(C.c_longlong),
                                             C.POINTER(C.c_longlong)]
        l.glfer_iq_required_span.restype = None
        l.glfer_iq_plan_create_mtm.argtypes = [C.POINTER(IqConfig), C.c_float, C.c_int, C.POINTER(C.c_void_p)]
        l.glfer_zoom_plan_create_mtm.argtypes = [C.POINTER(ZoomConfig), C.c_float, C.c_int, C.POINTER(C.c_void_p)]
        l.glfer_zoom_plan_create_iq_mtm.argtypes = [C.POINTER(ZoomConfig), C.c_float, C.c_int, C.POINTER(C.c_void_p)]
        l.glfer_iq_tapers.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        l.glfer_zoom_tapers.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        l.glfer_iq_run.argtypes = zoom_args
        l.glfer_iq_run_pcm16.argtypes = zoom_args
        for name in ("glfer_iq_run_mtm_ftest", "glfer_iq_run_mtm_ftest_pcm16", "glfer_zoom_run_mtm_ftest",
                     "glfer_zoom_run_mtm_ftest_pcm16", "glfer_zoom_run_iq_mtm_ftest", "glfer_zoom_run_iq_mtm_ftest_pcm16"):
            getattr(l, name).argtypes = zoom_args + [C.c_void_p]
        for name in ("glfer_iq_run_mtm_lines", "glfer_iq_run_mtm_lines_pcm16", "glfer_zoom_run_mtm_lines",
                     "glfer_zoom_run_mtm_lines_pcm16", "glfer_zoom_run_iq_mtm_lines", "glfer_zoom_run_iq_mtm_lines_pcm16"):
            getattr(l, name).argtypes = zoom_args[:-1] + [C.POINTER(LinesConfig)] + [C.c_void_p] * 4
        l.glfer_ftest_threshold.argtypes = [C.c_int, C.c_double, C.POINTER(C.c_float)]
        for name in ("glfer_iq_run_display", "glfer_iq_run_display_pcm16", "glfer_zoom_run_display",
                     "glfer_zoom_run_display_pcm16", "glfer_zoom_run_display_iq", "glfer_zoom_run_display_iq_pcm16"):
            getattr(l, name).argtypes = disp_args
        # per-call interface
        l.fft_init.argtypes = [C.POINTER(FftParams)]
        l.fft_do.argtypes = [C.c_void_p, C.POINTER(FftParams)]
        l.fft_psd.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(FftParams)]
        l.fft_close.argtypes = [C.POINTER(FftParams)]
        l.fft_do_batch.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(FftParams)]
        l.mtm_do_batch.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(MtmParams)]
        l.prepare_audio.argtypes = [C.c_void_p, C.POINTER(FftParams)]
        l.compute_window.argtypes = [C.POINTER(FftParams)]
        l.compute_floor.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                    C.POINTER(C.c_float), C.POINTER(C.c_uint)]
        l.mtm_init.argtypes = [C.POINTER(MtmParams)]
        l.mtm_do.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(MtmParams)]
        l.mtm_close.argtypes = [C.POINTER(MtmParams)]
        l.alloc_avg.argtypes = [C.POINTER(AvgData), C.c_int, C.c_int]
        l.init_avg.argtypes = [C.POINTER(AvgData)]
        l.delete_avg.argtypes = [C.POINTER(AvgData)]
        for name in ("update_avg_plain", "update_avg_sumextreme", "update_avg_sumavg"):
            getattr(l, name).restype = C.c_double
        l.update_avg_plain.argtypes = [C.POINTER(AvgData), C.c_int, C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int)]
        l.update_avg_sumextreme.argtypes = [C.POINTER(AvgData), C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                            C.POINTER(C.c_int)]
        l.update_avg_sumavg.argtypes = [C.POINTER(AvgData), C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                        C.POINTER(C.c_int), C.POINTER(C.c_double)]
        # host-side table generators (no device needed)
        l.glb_window_table.argtypes = [C.c_int, C.c_int, C.c_void_p]
        l.glb_window_table.restype = None
        l.glb_dpss.argtypes = [C.c_int, C.c_double, C.c_int, C.c_void_p, C.c_void_p]
        l.glb_hop.argtypes = [C.c_int, C.c_float]
        l.glfer_b200_map_levels.argtypes = [C.c_void_p, C.c_longlong, C.c_int, C.POINTER(DisplayConfig), C.c_void_p,
                                            C.c_void_p, C.c_int]
        l.glfer_b200_set_fused_levels.argtypes = [C.c_int]
        l.glfer_b200_set_fused_levels.restype = None
        l.glfer_palette.argtypes = [C.c_int, C.c_void_p]
        l.glb_short_db_f.argtypes = [C.c_float]
        l.glb_force_generic_kernel.argtypes = [C.c_int]
        l.glb_force_generic_kernel.restype = None
        l.glb_set_kernel_preference.argtypes = [C.c_int]
        l.glb_set_kernel_preference.restype = None
        l.glb_set_ring_groups.argtypes = [C.c_int]
        l.glb_set_ring_groups.restype = None
        l.glb_last_frames_per_group.restype = C.c_int
        _lib = l
    return _lib


def last_error() -> str:
    return lib().glfer_b200_last_error().decode(errors="replace")


def _check(rc: int) -> None:
    if rc != 0:
        raise GlferError(f"libglfer_b200 error {rc}: {last_error()}")


def device_count() -> int:
    return lib().glfer_b200_device_count()


def kernel_launches() -> int:
    return int(lib().glfer_b200_kernel_launches())


KERNEL_FAMILIES = {0: "none", 1: "gram_kernel (general)", 2: "gram_ring_kernel (TMA ring)", 3: "gram_wpf_kernel (warp per frame)",
                   4: "gram_pair_kernel (two frames per thread)", 5: "gram_big_kernel (32 points per thread)"}


def last_kernel_family() -> str:
    """Family of the last spectrogram kernel the library launched."""
    return KERNEL_FAMILIES.get(int(lib().glb_last_kernel_family()), "?")


def _ptr(a):
    return None if a is None else a.ctypes.data


class _PinnedBuffer:
    """Owner of one glfer_b200_host_alloc block; numpy views keep it alive through their base."""

    def __init__(self, nbytes: int):
        self.nbytes = max(int(nbytes), 1)
        self.ptr = lib().glfer_b200_host_alloc(self.nbytes)
        if not self.ptr:
            raise GlferError("pinned allocation failed: " + last_error())
        self.__array_interface__ = {"shape": (self.nbytes,), "typestr": "|u1", "data": (self.ptr, False), "version": 3}

    def __del__(self):
        try:
            if self.ptr:
                lib().glfer_b200_host_free(self.ptr)
                self.ptr = None
        except Exception:
            pass


def pinned_empty(shape, dtype) -> np.ndarray:
    """numpy array over pinned host memory from glfer_b200_host_alloc; the memory is freed when the
    last view of the array is collected (the owner object is the base of every view)."""
    dtype = np.dtype(dtype)
    count = int(np.prod(shape))
    owner = _PinnedBuffer(count * dtype.itemsize)
    raw = np.asarray(owner)                       # base -> owner
    return raw[:count * dtype.itemsize].view(dtype).reshape(shape)


def make_config(n=1024, window_type=KAISER, overlap=0.0, mode=MODE_FFT, sub_mean=True, a=0.0, limiter=0,
                mtm_w=4.0, mtm_kmax=7, avg_mode=NO_AVG, avg_depth=4, avg_minbin=0, avg_maxbin=0, avg_max0=0,
                avg_peakbin_init=0, scale_db=False, device=0, lmp_av=4, avg_band_only=False, mtm_ftest=False,
                zero_history=False) -> GramConfig:
    return GramConfig(mode, n, window_type, overlap, a, limiter, int(sub_mean), mtm_w, mtm_kmax, avg_mode, avg_depth,
                      avg_minbin, avg_maxbin, avg_max0, avg_peakbin_init, int(scale_db), device, lmp_av,
                      int(avg_band_only), int(mtm_ftest), int(zero_history))


class GramPlan:
    """glfer_gram_plan: batch counterpart of fft_init/mtm_init (+ alloc_avg)."""

    def __init__(self, **kw):
        self.cfg = make_config(**kw)
        self._h = C.c_void_p()
        _check(lib().glfer_gram_plan_create(C.byref(self.cfg), C.byref(self._h)))
        self.n = self.cfg.n
        self.hop = lib().glfer_gram_hop(self._h)
        self.bins = lib().glfer_gram_bins(self._h)
        self.avg = self.cfg.avg_mode != NO_AVG
        self.avg_cols = lib().glfer_gram_avg_cols(self._h)

    def close(self):
        if self._h:
            lib().glfer_gram_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def num_frames(self, nsamples: int) -> int:
        return int(lib().glfer_gram_num_frames(self._h, nsamples))

    def required_span(self, first_frame: int, nframes: int):
        lo, hi = C.c_longlong(), C.c_longlong()
        lib().glfer_gram_required_span(self._h, first_frame, nframes, C.byref(lo), C.byref(hi))
        return lo.value, hi.value

    def window(self) -> np.ndarray:
        w = np.empty(self.n, dtype=np.float32)
        _check(lib().glfer_gram_window(self._h, w.ctypes.data))
        return w

    def tapers(self):
        k = self.cfg.mtm_kmax + 1
        t = np.empty((k, self.n), dtype=np.float64)
        lam = np.empty(k, dtype=np.float64)
        _check(lib().glfer_gram_tapers(self._h, t.ctypes.data, lam.ctypes.data))
        return t, lam

    def _outs(self, nframes, want_psd, out=None):
        out = out or {}
        psd = out.get("psd") if "psd" in out else (np.empty((nframes, self.bins), np.float32) if want_psd else None)
        avg = ret = pk = var = None
        if self.avg:
            avg = out.get("avg") if "avg" in out else np.empty((nframes, self.avg_cols), np.float32)
            # (the library stages these small per-frame outputs through pinned memory of its own: plain arrays do
            # not stall the chunk pipeline; allocating pinned memory per call would cost ~100 ms per array)
            ret = out.get("ret") if "ret" in out else np.empty((nframes,), np.float64)
            pk = out.get("peakbin") if "peakbin" in out else np.empty((nframes,), np.int32)
            var = out.get("variance") if "variance" in out else np.empty((nframes,), np.float64)
        return psd, avg, ret, pk, var

    def run(self, samples: np.ndarray, origin: int = 0, first_frame: int = 0, nframes: int | None = None,
            want_psd: bool = True, out: dict | None = None):
        """glfer_gram_run: host buffers in and out.  Returns dict(psd, avg, ret, peakbin, variance)."""
        pcm = samples.dtype == np.int16
        if not pcm:
            assert samples.dtype == np.float32
        assert samples.flags["C_CONTIGUOUS"]
        if nframes is None:
            nframes = (origin + len(samples)) // self.hop - first_frame
        psd, avg, ret, pk, var = self._outs(nframes, want_psd, out)
        fn = lib().glfer_gram_run_pcm16 if pcm else lib().glfer_gram_run
        _check(fn(self._h, samples.ctypes.data, origin, len(samples), first_frame, nframes, _ptr(psd), _ptr(avg),
                  _ptr(ret), _ptr(pk), _ptr(var)))
        return dict(psd=psd, avg=avg, ret=ret, peakbin=pk, variance=var)

    def run_mtm_ftest(self, samples: np.ndarray, origin: int = 0, first_frame: int = 0, nframes: int | None = None):
        """glfer_gram_run_mtm_ftest: multitaper rows and the harmonic F-test rows (plan with mtm_ftest=True)."""
        assert samples.dtype == np.float32 and samples.flags["C_CONTIGUOUS"]
        if nframes is None:
            nframes = (origin + len(samples)) // self.hop - first_frame
        psd = np.empty((nframes, self.bins), np.float32)
        ft = np.empty((nframes, self.bins), np.float32)
        _check(lib().glfer_gram_run_mtm_ftest(self._h, samples.ctypes.data, origin, len(samples), first_frame, nframes,
                                              psd.ctypes.data, ft.ctypes.data))
        return dict(psd=psd, ftest=ft)

    def stage(self, samples: np.ndarray, origin: int = 0):
        assert samples.flags["C_CONTIGUOUS"]
        if samples.dtype == np.int16:
            _check(lib().glfer_gram_stage_pcm16(self._h, samples.ctypes.data, origin, len(samples)))
        else:
            assert samples.dtype == np.float32
            _check(lib().glfer_gram_stage(self._h, samples.ctypes.data, origin, len(samples)))

    def exec(self, first_frame: int, nframes: int, timed: bool = False):
        ms = C.c_float(0.0)
        _check(lib().glfer_gram_exec(self._h, first_frame, nframes, C.byref(ms) if timed else None))
        return ms.value if timed else None

    def last_gram_ms(self) -> float:
        ms = C.c_float(0.0)
        _check(lib().glfer_gram_last_gram_ms(self._h, C.byref(ms)))
        return ms.value

    def sync(self):
        _check(lib().glfer_gram_sync(self._h))

    def fetch(self, nframes: int, want_psd: bool = True):
        psd, avg, ret, pk, var = self._outs(nframes, want_psd)
        _check(lib().glfer_gram_fetch(self._h, _ptr(psd), _ptr(avg), _ptr(ret), _ptr(pk), _ptr(var)))
        return dict(psd=psd, avg=avg, ret=ret, peakbin=pk, variance=var)

    def run_display(self, samples: np.ndarray, log_scale=True, autoscale=True, max_level_db=-20.0, min_level_db=-80.0,
                    thr_level=0.0, colortab: np.ndarray | None = None, origin: int = 0, first_frame: int = 0,
                    nframes: int | None = None, agc_state: np.ndarray | None = None, want_rgb: bool = False,
                    out: dict | None = None, want_range: bool = True):
        """glfer_gram_run_display: rows -> 8-bit levels (and RGB) as main_window_draw maps them.
        out: optional pre-allocated (pinned) "levels" array -- a download of rows into pageable memory blocks the
        host thread and with it the chunk pipeline (the small "range" output is staged by the library)."""
        pcm = samples.dtype == np.int16
        assert samples.flags["C_CONTIGUOUS"] and (pcm or samples.dtype == np.float32)
        if nframes is None:
            nframes = (origin + len(samples)) // self.hop - first_frame
        out = out or {}
        levels = out.get("levels") if "levels" in out else np.empty((nframes, self.bins), np.uint8)
        rgb = np.empty((nframes, self.bins, 3), np.uint8) if want_rgb else None
        rng = None
        if autoscale and want_range:
            rng = out.get("range") if "range" in out else np.empty((nframes, 2), np.float32)
        if colortab is not None:
            colortab = np.ascontiguousarray(colortab, dtype=np.uint8)
            assert colortab.size == 768
        dc = DisplayConfig(int(log_scale), int(autoscale), max_level_db, min_level_db, thr_level,
                           colortab.ctypes.data if colortab is not None else None)
        state = agc_state if agc_state is not None else np.zeros(2, np.float32)
        fn = lib().glfer_gram_run_display_pcm16 if pcm else lib().glfer_gram_run_display
        _check(fn(self._h, samples.ctypes.data, origin, len(samples), first_frame, nframes, C.byref(dc), state.ctypes.data,
                  _ptr(levels), _ptr(rgb), _ptr(rng)))
        return dict(levels=levels, rgb=rgb, range=rng, agc_state=state)

    def run_wav(self, path: str, want_psd: bool = True, channel: int | None = None):
        """glfer_gram_run_wav; channel: keep one channel of a multi-channel file (an extension -- the reference, and
        the default here, feed the interleaved samples to the estimator as they are)."""
        wav = Wav()
        _check(lib().glfer_wav_load(path.encode(), C.byref(wav)))
        try:
            if channel is not None:
                _check(lib().glfer_wav_select_channel(C.byref(wav), channel))
            nframes = int(lib().glfer_wav_num_frames(self._h, C.byref(wav)))
            psd, avg, ret, pk, var = self._outs(nframes, want_psd)
            _check(lib().glfer_gram_run_wav(self._h, C.byref(wav), _ptr(psd), _ptr(avg), _ptr(ret), _ptr(pk), _ptr(var)))
            return dict(psd=psd, avg=avg, ret=ret, peakbin=pk, variance=var, sample_rate=wav.sample_rate,
                        bits=wav.bits)
        finally:
            lib().glfer_wav_free(C.byref(wav))


def _run_display(fn, handle, ptr, count, bins, nframes, log_scale, autoscale, max_level_db, min_level_db, thr_level,
                 colortab, origin, first_frame, agc_state, want_rgb, out, want_range, lead=()):
    """one *_run_display call of an I/Q or zoom plan, with the keywords and outputs of GramPlan.run_display; lead: (C,)
    for a zoom bank, whose outputs and agc_state carry a leading channel axis"""
    out = out or {}
    nc = int(np.prod(lead, dtype=np.int64))
    levels = out.get("levels") if "levels" in out else np.empty(lead + (nframes, bins), np.uint8)
    assert levels.dtype == np.uint8 and levels.size >= nc * nframes * bins
    rgb = np.empty(lead + (nframes, bins, 3), np.uint8) if want_rgb else None
    rng = None
    if autoscale and want_range:
        rng = out.get("range") if "range" in out else np.empty(lead + (nframes, 2), np.float32)
    if colortab is not None:
        colortab = np.ascontiguousarray(colortab, dtype=np.uint8)
        assert colortab.size == 768
    dc = DisplayConfig(int(log_scale), int(autoscale), max_level_db, min_level_db, thr_level,
                       colortab.ctypes.data if colortab is not None else None)
    state = agc_state if agc_state is not None else np.zeros(lead + (2,), np.float32)
    _check(fn(handle, ptr, origin, count, first_frame, nframes, C.byref(dc), state.ctypes.data, _ptr(levels), _ptr(rgb),
              _ptr(rng)))
    return dict(levels=levels, rgb=rgb, range=rng, agc_state=state)


def _iq_samples(iq: np.ndarray):
    """(pointer, complex sample count, pcm16) of an I/Q array: 1-D complex64 (its memory is already interleaved,
    no copy), float32 [count, 2] or int16 [count, 2] (I, Q)"""
    assert iq.flags["C_CONTIGUOUS"], "I/Q samples must be C-contiguous"
    if iq.dtype == np.complex64 and iq.ndim == 1:
        return iq.ctypes.data, len(iq), False
    assert iq.ndim == 2 and iq.shape[1] == 2 and iq.dtype in (np.float32, np.int16), \
        "I/Q samples: complex64 [count], float32 [count, 2] or int16 [count, 2]"
    return iq.ctypes.data, iq.shape[0], iq.dtype == np.int16


def _tapers(fn, h, k, n):
    k = max(k, 1)
    t = np.empty((k, n), dtype=np.float64)
    lam = np.empty(k, dtype=np.float64)
    _check(fn(h, t.ctypes.data, lam.ctypes.data))
    return t, lam


class ZoomPlan:
    """glfer_zoom_plan: mix center_hz to DC, low-pass and decimate by `decim`, complex FFT frames of n points.
    Rows hold n bins in frequency order, bin j at center_hz() + (j - n/2) * sample_rate / (decim * n).
    iq=True: complex (I/Q) input (glfer_zoom_plan_create_iq), centre in [-sample_rate/2, sample_rate/2].
    multitaper=True: rows of K' = mtm_kmax + 1 DPSS tapers of NW = mtm_w (glfer_zoom_plan_create[_iq]_mtm; window_type
    is ignored).
    center_hz a sequence: a channel bank (glfer_zoom_plan_create_bank[_mtm]), one channel per centre; run,
    run_mtm_ftest, run_mtm_lines and run_display then return arrays with a leading channel axis, (C, nframes, ...), and run_display
    takes and returns agc_state of shape (C, 2)."""

    def __init__(self, n=4096, decim=256, window_type=HANNING, overlap=0.0, center_hz=800.0, sample_rate=48000.0,
                 device=0, iq=False, multitaper=False, mtm_w=4.0, mtm_kmax=7):
        self.bank = np.ndim(center_hz) > 0
        centers = np.ascontiguousarray(center_hz, dtype=np.float64).reshape(-1)
        self.cfg = ZoomConfig(n, decim, window_type, overlap, 0.0 if self.bank else center_hz, sample_rate, device)
        self._h = C.c_void_p()
        self.iq = iq
        self.multitaper = multitaper
        self.mtm_kmax = mtm_kmax
        if self.bank and multitaper:
            _check(lib().glfer_zoom_plan_create_bank_mtm(C.byref(self.cfg), centers.ctypes.data, len(centers), int(iq),
                                                         mtm_w, mtm_kmax, C.byref(self._h)))
        elif self.bank:
            _check(lib().glfer_zoom_plan_create_bank(C.byref(self.cfg), centers.ctypes.data, len(centers), int(iq),
                                                     C.byref(self._h)))
        elif multitaper:
            create = lib().glfer_zoom_plan_create_iq_mtm if iq else lib().glfer_zoom_plan_create_mtm
            _check(create(C.byref(self.cfg), mtm_w, mtm_kmax, C.byref(self._h)))
        else:
            create = lib().glfer_zoom_plan_create_iq if iq else lib().glfer_zoom_plan_create
            _check(create(C.byref(self.cfg), C.byref(self._h)))
        self.n = n
        self.decim = decim
        self.hop = lib().glfer_zoom_hop(self._h)
        self.bins = lib().glfer_zoom_bins(self._h)
        self.channels = lib().glfer_zoom_channels(self._h)
        self._lead = (self.channels,) if self.bank else ()

    def close(self):
        if self._h:
            lib().glfer_zoom_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def center_hz(self) -> float:
        """the actual centre, step * sample_rate / 2**32 (channel 0's of a bank)"""
        return float(lib().glfer_zoom_center_hz(self._h))

    def centers_hz(self) -> np.ndarray:
        """the actual centre of every channel, float64 [C]"""
        return np.array([lib().glfer_zoom_channel_center_hz(self._h, c) for c in range(self.channels)], np.float64)

    def num_frames(self, nsamples: int) -> int:
        return int(lib().glfer_zoom_num_frames(self._h, nsamples))

    def required_span(self, first_frame: int, nframes: int):
        lo, hi = C.c_longlong(), C.c_longlong()
        lib().glfer_zoom_required_span(self._h, first_frame, nframes, C.byref(lo), C.byref(hi))
        return lo.value, hi.value

    def taps(self) -> np.ndarray:
        return zoom_taps(self.decim)

    def tapers(self):
        """glfer_zoom_tapers: (tapers [K'][n], lambda [K']) as float64, before scaling (multitaper plans only)"""
        return _tapers(lib().glfer_zoom_tapers, self._h, self.mtm_kmax + 1 if self.multitaper else 1, self.n)

    def run(self, samples: np.ndarray, origin: int = 0, first_frame: int = 0, nframes: int | None = None,
            out: np.ndarray | None = None) -> np.ndarray:
        """glfer_zoom_run / glfer_zoom_run_pcm16 (int16 samples): rows [nframes][n] ([C][nframes][n] for a bank).
        out: optional pre-allocated (e.g. pinned) rows.  An I/Q plan takes the formats of IqPlan.run."""
        if self.iq:
            ptr, count, pcm = _iq_samples(samples)
            if nframes is None:
                nframes = self.num_frames(origin + count) - first_frame
            rows = out if out is not None else np.empty(self._lead + (nframes, self.bins), np.float32)
            assert rows.dtype == np.float32 and rows.size >= self.channels * nframes * self.bins
            fn = lib().glfer_zoom_run_iq_pcm16 if pcm else lib().glfer_zoom_run_iq
            _check(fn(self._h, ptr, origin, count, first_frame, nframes, rows.ctypes.data))
            return rows
        pcm = samples.dtype == np.int16
        assert samples.flags["C_CONTIGUOUS"] and (pcm or samples.dtype == np.float32)
        if nframes is None:
            nframes = self.num_frames(origin + len(samples)) - first_frame
        rows = out if out is not None else np.empty(self._lead + (nframes, self.bins), np.float32)
        assert rows.dtype == np.float32 and rows.size >= self.channels * nframes * self.bins
        fn = lib().glfer_zoom_run_pcm16 if pcm else lib().glfer_zoom_run
        _check(fn(self._h, samples.ctypes.data, origin, len(samples), first_frame, nframes, rows.ctypes.data))
        return rows

    def run_mtm_ftest(self, samples: np.ndarray, origin: int = 0, first_frame: int = 0, nframes: int | None = None,
                      want_psd: bool = True, want_ftest: bool = True):
        """glfer_zoom_run[_iq]_mtm_ftest[_pcm16]: the multitaper rows and the harmonic F-test rows, [nframes][n] each
        (None when not wanted), of a multitaper plan.  Input formats of run."""
        if self.iq:
            ptr, count, pcm = _iq_samples(samples)
            fn = lib().glfer_zoom_run_iq_mtm_ftest_pcm16 if pcm else lib().glfer_zoom_run_iq_mtm_ftest
        else:
            pcm = samples.dtype == np.int16
            assert samples.flags["C_CONTIGUOUS"] and (pcm or samples.dtype == np.float32)
            ptr, count = samples.ctypes.data, len(samples)
            fn = lib().glfer_zoom_run_mtm_ftest_pcm16 if pcm else lib().glfer_zoom_run_mtm_ftest
        if nframes is None:
            nframes = self.num_frames(origin + count) - first_frame
        return _run_ftest(fn, self._h, ptr, origin, count, first_frame, nframes, self.bins, want_psd, want_ftest,
                          self._lead)

    def run_mtm_lines(self, samples: np.ndarray, pfa: float = 1e-3, max_lines: int = 16, bin_range=None,
                      origin: int = 0, first_frame: int = 0, nframes: int | None = None, want_ftest: bool = True,
                      want_psd: bool = True):
        """glfer_zoom_run[_iq]_mtm_lines[_pcm16]: the harmonic lines of each frame, selected on the device from the F rows
        of run_mtm_ftest at the F(2, 2K' - 2) threshold of pfa.  Keywords and outputs of IqPlan.run_mtm_lines, with the
        bank's leading channel axis.  Input formats of run."""
        if self.iq:
            ptr, count, pcm = _iq_samples(samples)
            fn = lib().glfer_zoom_run_iq_mtm_lines_pcm16 if pcm else lib().glfer_zoom_run_iq_mtm_lines
        else:
            pcm = samples.dtype == np.int16
            assert samples.flags["C_CONTIGUOUS"] and (pcm or samples.dtype == np.float32)
            ptr, count = samples.ctypes.data, len(samples)
            fn = lib().glfer_zoom_run_mtm_lines_pcm16 if pcm else lib().glfer_zoom_run_mtm_lines
        if nframes is None:
            nframes = self.num_frames(origin + count) - first_frame
        return _run_lines(fn, self._h, ptr, origin, count, first_frame, nframes, self.bins, pfa, max_lines, bin_range,
                          want_ftest, want_psd, self._lead)

    def run_display(self, samples: np.ndarray, log_scale=True, autoscale=True, max_level_db=-20.0, min_level_db=-80.0,
                    thr_level=0.0, colortab: np.ndarray | None = None, origin: int = 0, first_frame: int = 0,
                    nframes: int | None = None, agc_state: np.ndarray | None = None, want_rgb: bool = False,
                    out: dict | None = None, want_range: bool = True):
        """glfer_zoom_run_display*: the plan's rows -> 8-bit levels (and RGB) as main_window_draw maps them, pixel i =
        bin n - 1 - i.  Keywords and outputs of GramPlan.run_display; an I/Q plan takes the formats of IqPlan.run."""
        if self.iq:
            ptr, count, pcm = _iq_samples(samples)
            fn = lib().glfer_zoom_run_display_iq_pcm16 if pcm else lib().glfer_zoom_run_display_iq
        else:
            pcm = samples.dtype == np.int16
            assert samples.flags["C_CONTIGUOUS"] and (pcm or samples.dtype == np.float32)
            ptr, count = samples.ctypes.data, len(samples)
            fn = lib().glfer_zoom_run_display_pcm16 if pcm else lib().glfer_zoom_run_display
        if nframes is None:
            nframes = self.num_frames(origin + count) - first_frame
        return _run_display(fn, self._h, ptr, count, self.bins, nframes, log_scale, autoscale, max_level_db, min_level_db,
                            thr_level, colortab, origin, first_frame, agc_state, want_rgb, out, want_range, self._lead)


class IqPlan:
    """glfer_iq_plan: two-sided spectrogram of complex (I/Q) input.  Rows hold n bins, bin j at
    (j - n/2) * sample_rate / n (DC at n/2): |FFT(w z_f)|^2 / n, fft-shifted.
    multitaper=True: rows of K' = mtm_kmax + 1 DPSS tapers of NW = mtm_w (glfer_iq_plan_create_mtm; window_type is
    ignored)."""

    def __init__(self, n=4096, window_type=HANNING, overlap=0.5, device=0, multitaper=False, mtm_w=4.0, mtm_kmax=7):
        self.cfg = IqConfig(n, window_type, overlap, device)
        self._h = C.c_void_p()
        self.multitaper = multitaper
        self.mtm_kmax = mtm_kmax
        if multitaper:
            _check(lib().glfer_iq_plan_create_mtm(C.byref(self.cfg), mtm_w, mtm_kmax, C.byref(self._h)))
        else:
            _check(lib().glfer_iq_plan_create(C.byref(self.cfg), C.byref(self._h)))
        self.n = n
        self.hop = lib().glfer_iq_hop(self._h)
        self.bins = lib().glfer_iq_bins(self._h)

    def close(self):
        if self._h:
            lib().glfer_iq_plan_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def num_frames(self, nsamples: int) -> int:
        return int(lib().glfer_iq_num_frames(self._h, nsamples))

    def required_span(self, first_frame: int, nframes: int):
        lo, hi = C.c_longlong(), C.c_longlong()
        lib().glfer_iq_required_span(self._h, first_frame, nframes, C.byref(lo), C.byref(hi))
        return lo.value, hi.value

    def tapers(self):
        """glfer_iq_tapers: (tapers [K'][n], lambda [K']) as float64, before scaling (multitaper plans only)"""
        return _tapers(lib().glfer_iq_tapers, self._h, self.mtm_kmax + 1 if self.multitaper else 1, self.n)

    def run(self, iq: np.ndarray, origin: int = 0, first_frame: int = 0, nframes: int | None = None,
            out: np.ndarray | None = None) -> np.ndarray:
        """glfer_iq_run / glfer_iq_run_pcm16: rows [nframes][n] of complex64 [count], float32 [count, 2] or int16
        [count, 2] I/Q samples (origin and count in complex samples).  out: optional pre-allocated (e.g. pinned)
        rows."""
        ptr, count, pcm = _iq_samples(iq)
        if nframes is None:
            nframes = self.num_frames(origin + count) - first_frame
        rows = out if out is not None else np.empty((nframes, self.bins), np.float32)
        assert rows.dtype == np.float32 and rows.size >= nframes * self.bins
        fn = lib().glfer_iq_run_pcm16 if pcm else lib().glfer_iq_run
        _check(fn(self._h, ptr, origin, count, first_frame, nframes, rows.ctypes.data))
        return rows

    def run_mtm_ftest(self, iq: np.ndarray, origin: int = 0, first_frame: int = 0, nframes: int | None = None,
                      want_psd: bool = True, want_ftest: bool = True):
        """glfer_iq_run_mtm_ftest / _pcm16: the multitaper rows and the harmonic F-test rows, [nframes][n] each (None
        when not wanted), of a multitaper plan.  Input formats of run."""
        ptr, count, pcm = _iq_samples(iq)
        if nframes is None:
            nframes = self.num_frames(origin + count) - first_frame
        fn = lib().glfer_iq_run_mtm_ftest_pcm16 if pcm else lib().glfer_iq_run_mtm_ftest
        return _run_ftest(fn, self._h, ptr, origin, count, first_frame, nframes, self.bins, want_psd, want_ftest)

    def run_mtm_lines(self, iq: np.ndarray, pfa: float = 1e-3, max_lines: int = 16, bin_range=None, origin: int = 0,
                      first_frame: int = 0, nframes: int | None = None, want_ftest: bool = True, want_psd: bool = True):
        """glfer_iq_run_mtm_lines / _pcm16: the harmonic lines of each frame, selected on the device from the F rows of
        run_mtm_ftest at the F(2, 2K' - 2) threshold of pfa (ftest_threshold), searched over row positions
        bin_range = (lo, hi) (None: the whole row).  Returns dict(count [nframes] int32, bin [nframes][max_lines] int32,
        ftest and psd [nframes][max_lines] float32, None when not wanted); unused slots hold bin -1 and 0.0.  Input
        formats of run."""
        ptr, count, pcm = _iq_samples(iq)
        if nframes is None:
            nframes = self.num_frames(origin + count) - first_frame
        fn = lib().glfer_iq_run_mtm_lines_pcm16 if pcm else lib().glfer_iq_run_mtm_lines
        return _run_lines(fn, self._h, ptr, origin, count, first_frame, nframes, self.bins, pfa, max_lines, bin_range,
                          want_ftest, want_psd)

    def run_display(self, iq: np.ndarray, log_scale=True, autoscale=True, max_level_db=-20.0, min_level_db=-80.0,
                    thr_level=0.0, colortab: np.ndarray | None = None, origin: int = 0, first_frame: int = 0,
                    nframes: int | None = None, agc_state: np.ndarray | None = None, want_rgb: bool = False,
                    out: dict | None = None, want_range: bool = True):
        """glfer_iq_run_display / _pcm16: the plan's rows -> 8-bit levels (and RGB) as main_window_draw maps them,
        pixel i = row position n - 1 - i.  Input formats of IqPlan.run; keywords and outputs of GramPlan.run_display."""
        ptr, count, pcm = _iq_samples(iq)
        if nframes is None:
            nframes = self.num_frames(origin + count) - first_frame
        fn = lib().glfer_iq_run_display_pcm16 if pcm else lib().glfer_iq_run_display
        return _run_display(fn, self._h, ptr, count, self.bins, nframes, log_scale, autoscale, max_level_db, min_level_db,
                            thr_level, colortab, origin, first_frame, agc_state, want_rgb, out, want_range)


def _run_ftest(fn, h, ptr, origin, count, first_frame, nframes, bins, want_psd, want_ftest, lead=()):
    psd = np.empty(lead + (nframes, bins), np.float32) if want_psd else None
    ft = np.empty(lead + (nframes, bins), np.float32) if want_ftest else None
    _check(fn(h, ptr, origin, count, first_frame, nframes, _ptr(psd), _ptr(ft)))
    return dict(psd=psd, ftest=ft)


def _run_lines(fn, h, ptr, origin, count, first_frame, nframes, bins, pfa, max_lines, bin_range, want_ftest, want_psd,
               lead=()):
    lo, hi = (0, bins) if bin_range is None else bin_range
    lc = LinesConfig(pfa, max_lines, lo, hi)
    m = max(int(max_lines), 0)
    cnt = np.empty(lead + (nframes,), np.int32)
    b = np.empty(lead + (nframes, m), np.int32)
    ft = np.empty(lead + (nframes, m), np.float32) if want_ftest else None
    psd = np.empty(lead + (nframes, m), np.float32) if want_psd else None
    _check(fn(h, ptr, origin, count, first_frame, nframes, C.byref(lc), cnt.ctypes.data, b.ctypes.data, _ptr(ft),
              _ptr(psd)))
    return dict(count=cnt, bin=b, ftest=ft, psd=psd)


def ftest_threshold(ntapers: int, pfa: float) -> float:
    """glfer_ftest_threshold: the F(2, 2K' - 2) threshold of a per-bin false-alarm probability pfa; needs no device"""
    thr = C.c_float()
    _check(lib().glfer_ftest_threshold(int(ntapers), float(pfa), C.byref(thr)))
    return float(thr.value)


def zoom_taps(decim: int) -> np.ndarray:
    """glfer_zoom_taps: the zoom low-pass h[l], l = -K..K (K = 16 decim), as float32; needs no device"""
    h = np.empty(32 * decim + 1 if 2 <= decim <= 1024 else 1, dtype=np.float32)   # the library rejects other values
    _check(lib().glfer_zoom_taps(decim, h.ctypes.data))
    return h


def run_sharded(samples: np.ndarray, ndev: int, devices=None, want_psd: bool = True, **kw):
    """glfer_gram_run_sharded: one host thread per device inside this process."""
    cfg = make_config(**kw)
    hop = lib().glb_hop(cfg.n, cfg.overlap)
    nframes = len(samples) // hop
    bins = cfg.n // 2 + 1
    psd = np.empty((nframes, bins), np.float32) if want_psd else None
    avg = ret = pk = var = None
    if cfg.avg_mode != NO_AVG:
        avg = np.empty((nframes, cfg.avg_maxbin - cfg.avg_minbin if cfg.avg_band_only else bins), np.float32)
        ret = np.empty(nframes, np.float64)
        pk = np.empty(nframes, np.int32)
        var = np.empty(nframes, np.float64)
    devs = (C.c_int * ndev)(*devices) if devices is not None else None
    _check(lib().glfer_gram_run_sharded(C.byref(cfg), ndev, devs, samples.ctypes.data, len(samples), _ptr(psd),
                                        _ptr(avg), _ptr(ret), _ptr(pk), _ptr(var)))
    return dict(psd=psd, avg=avg, ret=ret, peakbin=pk, variance=var)


def shard_range(nframes: int, ndev: int, g: int):
    a, b = C.c_longlong(), C.c_longlong()
    lib().glfer_gram_shard_range(nframes, ndev, g, C.byref(a), C.byref(b))
    return a.value, b.value


def host_window(n: int, window_type: int) -> np.ndarray:
    w = np.empty(n, dtype=np.float32)
    lib().glb_window_table(n, window_type, w.ctypes.data)
    return w


def host_dpss(n: int, nw: float, kmax: int):
    t = np.empty((kmax + 1, n), dtype=np.float64)
    lam = np.empty(kmax + 1, dtype=np.float64)
    rc = lib().glb_dpss(n, float(np.float32(nw)), kmax, t.ctypes.data, lam.ctypes.data)
    if rc != 0:
        raise GlferError("glb_dpss failed")
    return t, lam


def map_levels(rows: np.ndarray, log_scale=True, max_level_db=-20.0, min_level_db=-80.0, thr_level=0.0,
               display_range: np.ndarray | None = None, device: int = 0) -> np.ndarray:
    """glfer_b200_map_levels: main_window_draw's level mapping on given rows (fixed levels, or a
    (display_max, display_min) pair per row)."""
    rows = np.ascontiguousarray(rows, dtype=np.float32)
    nrows, nbins = rows.shape
    out = np.empty((nrows, nbins), dtype=np.uint8)
    dc = DisplayConfig(int(log_scale), 0, max_level_db, min_level_db, thr_level, None)
    rng = None if display_range is None else np.ascontiguousarray(display_range, dtype=np.float32)
    _check(lib().glfer_b200_map_levels(rows.ctypes.data, nrows, nbins, C.byref(dc), _ptr(rng), out.ctypes.data, device))
    return out


def set_fused_avg(on: bool) -> None:
    """True = frame averaging inside the spectrogram kernel where possible (default False: measured slower)"""
    lib().glfer_b200_set_fused_avg(int(on))


def set_fused_levels(on: bool) -> None:
    """testing aid: False = display levels always mapped in a second pass over float rows"""
    lib().glfer_b200_set_fused_levels(int(on))


def palette(p: int) -> np.ndarray:
    """glfer_palette: the 256 RGB triplets of set_palette (g_main.c:649-762)"""
    tab = np.empty((256, 3), dtype=np.uint8)
    _check(lib().glfer_palette(p, tab.ctypes.data))
    return tab


def force_generic_kernel(on: bool) -> None:
    """testing aid: run the general kernel where the TMA ring kernel would be chosen"""
    lib().glb_force_generic_kernel(int(on))


def set_ring_groups(groups: int) -> None:
    """testing aid: groups > 0 replaces the frame-group count of fused I/Q launches (at most one group per frame), so
    that a short run holds several frames per group; 0 (the default) restores the launch policy"""
    lib().glb_set_ring_groups(int(groups))


def last_frames_per_group() -> int:
    """testing aid: frames per group of the last fused I/Q launch"""
    return int(lib().glb_last_frames_per_group())


def set_kernel_preference(pref: int) -> None:
    """0 automatic, 1 general kernel, 2 TMA ring kernel, 3 warp-per-frame kernel"""
    lib().glb_set_kernel_preference(pref)


def host_hop(n: int, overlap: float) -> int:
    return lib().glb_hop(n, overlap)
