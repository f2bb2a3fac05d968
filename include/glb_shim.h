/* glb_shim.h -- the thin C-ABI CUDA shim under the C host layer.
 *
 * Internal boundary of libglfer_b200.so: plain pointers and sizes only, no C++ or
 * framework types.  The C host layer (glfer_b200/host/ *.c) never includes CUDA headers; every
 * device operation goes through these entry points, implemented in
 * glfer_b200/csrc/gram_kernels.cu.  All functions return 0 on success, a negative
 * GLB_E* code otherwise, and record a message retrievable with glb_last_error().
 */
#ifndef GLB_SHIM_H
#define GLB_SHIM_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GLB_OK 0
#define GLB_ECUDA (-1)     /* a CUDA runtime call failed */
#define GLB_EINVAL (-2)    /* invalid argument (e.g. unsupported FFT size) */
#define GLB_ENOMEM (-3)
#define GLB_ENODEV (-4)    /* no CUDA device: the library has no CPU fallback */

const char *glb_last_error(void);
void glb_set_error(const char *msg);

/* devices, memory, streams, events */
int glb_device_count(int *count);
int glb_set_device(int dev);
int glb_sm_count(int dev, int *sms);
int glb_malloc(void **dptr, size_t bytes);
int glb_free(void *dptr);
int glb_memset(void *dptr, int value, size_t bytes, void *stream);
int glb_host_alloc(void **hptr, size_t bytes);      /* pinned */
int glb_host_free(void *hptr);
int glb_memcpy_h2d(void *dst, const void *src, size_t bytes, void *stream);  /* async when stream != NULL */
int glb_memcpy_d2h(void *dst, const void *src, size_t bytes, void *stream);
int glb_memcpy_d2d(void *dst, const void *src, size_t bytes, void *stream);
int glb_stream_create(void **stream);
int glb_stream_destroy(void *stream);
int glb_stream_sync(void *stream);
int glb_stream_wait_event(void *stream, void *event);
int glb_device_sync(void);
int glb_event_create(void **event);
int glb_event_destroy(void *event);
int glb_event_record(void *event, void *stream);
int glb_event_sync(void *event);
int glb_event_elapsed_ms(void *start, void *stop, float *ms);

/* FFT constant tables (twiddles + real-FFT split factors) for frame length n, on
 * the current device.  n must be a power of two, 32 <= n <= 32768. */
int glb_fft_supported(int n);
int glb_tables_create(int n, void **tables);
int glb_tables_destroy(void *tables);

/* One launch of the fused spectrogram kernel: frames [first_frame, first_frame +
 * nframes) of the stream, frame f = stream samples [f*hop - n_ov, f*hop + hop). */
typedef struct {
  int n;                       /* frame length N */
  int hop;                     /* new samples per frame */
  const float *samples;        /* device: stream samples [origin, origin + count) */
  long long origin;            /* stream index of samples[0] (may be negative-free: >= 0) */
  long long count;             /* samples resident; stream indices outside [0,..) and outside the buffer read as 0 */
  const float *tapers;         /* device: [ntapers][n] floats, pre-scaled (see host layer) */
  int ntapers;                 /* 1 = periodogram, K' = kmax+1 for multitaper */
  const float *block_means;    /* device: mean of hop block b at [b - means_first_block], or NULL */
  long long means_first_block;
  int fused_mean;              /* 1: block means computed inside the kernel (needs glb_gram_fused_mean_ok) */
  float ra9mb_a;               /* > 0: x / (a + x^2) before the taper (fft.c:127-136) */
  int limiter;                 /* 1: sign(v) |v|^0.1 after the taper (fft.c:151-156) */
  int zero_history;            /* 1: the first n - hop samples of every frame read as 0 (first_buffer stuck TRUE) */
  float taper_scale;           /* the scale folded into tapers (needed by limiter / spectrum output) */
  long long first_frame;
  long long nframes;
  float *rows;                 /* device out: [nframes][row_stride] PSD, or NULL */
  long long row_stride;
  int rows_db;                 /* 1: write 10*log10(psd) */
  float *spectrum;             /* device out: [nframes][n/2+1] (re,im) pairs, or NULL (periodogram only) */
  const void *tables;          /* from glb_tables_create(n) */
  int groups_hint;             /* 0 = auto: resident frame-groups per launch */
  const void *fused_avg;       /* glb_avg_args * or NULL: the sliding frame averaging of the launch's frames done by the
                                  spectrogram kernel itself (band-only float rows; needs glb_gram_fused_avg_ok; its
                                  first_frame / nframes must be the launch's, psd is ignored) */
  int general_only;            /* 1: general kernel whatever the geometry (plain global loads: the per-call layer hands
                                  it pinned HOST memory, which every device access reaches over PCIe) */
  /* fused display mapping (main_window_draw, g_main.c:1186-1229): 8-bit palette indices written by the
     spectrogram kernel itself, beside or instead of the float rows; pixel i of a row shows bin n/2 - i */
  unsigned char *levels;       /* device out: [nframes][levels_stride], or NULL */
  long long levels_stride;
  const void *level_tables;    /* from glb_level_tables_create() */
  int levels_log;              /* 1: SCALE_LOG / SCALE_LOG_MAX0 (integer-truncated dB), 0: linear */
  const unsigned char *level_lut;   /* device: level of every integer dB value (fixed display range, log scales) or NULL */
  float level_min, level_max;  /* display_min / display_max (dB in the log scales); used when level_lut == NULL */
  float level_thr;             /* opt.thr_level / 100 */
  int taper_symmetric;         /* 1: ntapers == 1 and tapers[i] == tapers[n - 1 - i] bit for bit (checked by the host layer
                                  on the table it uploads): lets a kernel keep half of it in shared memory */
} glb_gram_args;

/* host-computed tables of the display mapping on the current device: dB thresholds as floats and doubles
 * (host/levels.c: GLB_DB_NTHR entries each) */
int glb_level_tables_create(const float *thr_f, const double *thr_d, int count, void **tables);
int glb_level_tables_destroy(void *tables);

int glb_launch_gram(const glb_gram_args *a, void *stream);
/* the in-kernel block-mean removal covers hop = (n/16) << s, s = 0..4, with (n - hop) a
 * multiple of hop (0 %, 50 %, 75 %, 87.5 %, 93.75 % overlap); other geometries use
 * glb_launch_block_means + block_means */
int glb_gram_fused_mean_ok(int n, int hop);
/* fused averaging is available when the launch runs on the TMA ring kernel with one frame group per CTA
 * (n = 4096 or 8192, regular hop) and the band history [depth][maxbin - minbin] fits 2 KB of shared memory */
int glb_gram_fused_avg_ok(int n, int hop, int depth, int band);
/* testing aid: 1 = always use the general kernel (the TMA ring kernel is chosen automatically
 * for the regular geometries) */
void glb_force_generic_kernel(int on);
/* 0 = automatic choice, 1 = general kernel, 2 = TMA ring kernel, 3 = warp-per-frame kernel, 4 = two frames per
 * thread, 5 = 32-points-per-thread kernel (N = 16384 / 32768; what the automatic choice takes there),
 * 6 = automatic, but the 32-point kernel never pairs two frame groups per CTA (A/B measurements)
 * (a preference: launches a family cannot serve fall through to the next one) */
void glb_set_kernel_preference(int pref);

/* mean of every complete hop block: means[b - first_block] = mean(stream[b*hop, (b+1)*hop)) */
int glb_launch_block_means(const float *samples, long long origin, long long count, int hop,
                           long long first_block, long long nblocks, float *means, void *stream);

/* int16 PCM -> float exactly as wav_fmt.c:113 ((float) s / 32768) */
int glb_launch_pcm16_to_float(const short *pcm, float *out, long long count, void *stream);
/* uint8 PCM -> float as wav_fmt.c:108 (((float) b - 128) / 128) */
int glb_launch_pcm8_to_float(const unsigned char *pcm, float *out, long long count, void *stream);

/* Sliding per-bin frame averaging (avg.c:108-298) over PSD rows resident on the device. */
typedef struct {
  int mode;                    /* avgmode_t: 1 sumavg, 2 plain, 3 sumextreme */
  int depth;
  int minbin, maxbin;
  int max0;
  int nbins;                   /* bins written per output row (N/2+1) */
  const float *psd;            /* device: row of frame g at psd + (g - psd_first_frame) * psd_stride */
  long long psd_first_frame;
  long long psd_stride;
  int psd_ring_rows;           /* > 0: psd is a ring, frame g lives in row g % psd_ring_rows */
  long long first_frame;       /* global (since alloc_avg) index of the first output frame */
  long long nframes;
  int out_double;              /* 0: float rows, 1: double rows */
  void *avg_rows;              /* device out [nframes][out_stride] */
  long long out_stride;
  int rows_db;                 /* 1: 10*log10 of the averaged row (float rows only) */
  double *ret;                 /* device out [nframes]: the function's return value */
  int *peak_cand;              /* device out [nframes]: bin written to *peakbin, or -1 if not written */
  double *variance;            /* device out [nframes] (sumavg) or NULL */
  int peakbin_init;            /* caller's *peakbin before the first frame */
  int *unresolved;             /* device counter: frames whose variance needed an unknown carried peakbin */
  int sequential;              /* 1: one CTA walks all frames in order (exact carry; slow) */
  int band_only;               /* 1: output rows hold bins [minbin, maxbin) only (column j = bin minbin + j); no 1e-15 fill */
} glb_avg_args;

int glb_launch_avg(const glb_avg_args *a, void *stream);
/* The per-bin statistic of the LMP estimator (lmp_do, lmp.c:131-160) over rectangular-window PSD
 * rows resident on the device: for output frame f the ring psdbufl[j], j = 0..nl-1, is the row
 * of the latest frame g <= f with g % nl == j (zeros when there is none yet, lmp.c:86-93); mean
 * and variance over the ring in double, in slot order, then the detector formula, stored to
 * float, 1e-3 where <= 1e-3, bin 0 = 1e-3.
 * psd_ring_rows > 0: psd is the ring itself (row j at psd + j * psd_stride; per-call interface). */
int glb_launch_lmp(const float *psd, long long psd_first_frame, long long psd_stride, int psd_ring_rows, int nbins,
                   long long first_frame, long long nframes, int nl, int rows_db, float *out, long long out_stride,
                   void *stream);

/* peakbin[f] = peak_cand[f] >= 0 ? peak_cand[f] : peakbin[f-1], peakbin[-1] = init */
int glb_launch_peak_carry(const int *peak_cand, int *peakbin, long long nframes, int init, void *stream);

/* PSD and phase of one half-complex spectrum (fft_psd, fft.c:203-226): hc[k] = Re X[k],
 * hc[n-k] = Im X[k]; psd / phase may be NULL; all device pointers. */
int glb_launch_halfcomplex_psd(const float *hc, int n, float *psd, float *phase, void *stream);

/* Per-row statistics of compute_floor (fft.c:240-294): stats[row] = { sig = largest bin,
 * floor = (sum of the lowest n - (int)(0.95 n) bins) / 0.05 / n, peak value, peak bin (as
 * float) }.  nbins <= 16385.  stats: [nrows][4] floats. */
int glb_launch_floor_stats(const float *rows, long long stride, int nbins, long long nrows, float *stats,
                           void *stream);

/* Display mapping of main_window_draw (g_main.c:1109-1229).  stats: [nframes][4] from
 * glb_launch_floor_stats; state[2] = (display_max_lvl, display_min_lvl) carried between calls;
 * range: [nframes][2] (display_max, display_min) per frame (dB in the log scales). */
int glb_launch_agc(const float *stats, long long nframes, long long first_frame, float overlap, int log_scale,
                   float *state, float *range, void *stream);
/* rows -> 8-bit levels (pixel i = bin nbins-1-i) and optional RGB through a 256-entry palette.
 * range: device, per frame (autoscale); or fixed_range[2] = (display_max, display_min): HOST values for all
 * frames, with the optional device look-up table level_lut (log scales). */
int glb_launch_levels(const float *rows, long long stride, int nbins, long long nframes, const float *range,
                      const float *fixed_range, int log_scale, float thr, const void *level_tables,
                      const unsigned char *level_lut, const unsigned char *colortab, unsigned char *levels,
                      unsigned char *rgb, void *stream);

/* Harmonic F-test (mtm.c:204-233) from the complex spectra of one chunk of frames: spec = [ntapers + 1][nframes][nbins]
 * (re, im) pairs, plane 0 = mu (the hn-weighted frame), plane 1 + j = y_j.  u0: device, [ntapers] doubles. */
int glb_launch_ftest(const float *spec, long long nframes, int nbins, int n, int ntapers, const double *u0,
                     double sum_u0_sqr, float *ftest, long long stride, void *stream);

/* Zoom spectrogram (glfer_b200/csrc/zoom.cu) and I/Q spectrogram (glfer_b200/csrc/iq.cu).
 * Decimator: y[m - m_first] = e^{-2 pi i (m dstep mod 2^32) / 2^32} sum_{j=0..32 decim} taps[j] x[m decim - 16 decim + j]
 * for m in [m_first, m_first + m_count); taps: device, [33 decim] (re, im) pairs, zero past index 32 decim;
 * dstep = decim * phase step mod 2^32.  x (float, or int16 PCM when pcm16 = 1, converted as wav_fmt.c:113) holds
 * stream samples [origin, origin + count); indices outside read as 0.  y: device, (re, im) pairs. */
int glb_launch_zoom_decim(const void *x, int pcm16, long long origin, long long count, int decim, const void *taps,
                          unsigned dstep, long long m_first, long long m_count, void *y, void *stream);
/* rows[f][j] = |Z_f[(j + nz/2) mod nz]|^2 / nz, with Z_f the complex FFT recovered from spec = [nframes][nz + 1]
 * (re, im) pairs, the real FFT of frame f's interleaved (re, im) samples as 2 nz real points */
int glb_launch_zoom_split(const void *spec, int nz, long long nframes, float *rows, void *stream);
/* Decimator of complex input: as glb_launch_zoom_decim with x the complex stream, interleaved (I, Q) floats, or
 * (I, Q) int16 PCM when pcm16 = 1; origin and count in complex samples.  Per tap the sum runs
 *     ar = fma(tr, ur, ar); ar = fma(-ti, ui, ar); ai = fma(ti, ur, ai); ai = fma(tr, ui, ai),
 * so with Q = 0 every output is bit-identical to glb_launch_zoom_decim's of I. */
int glb_launch_zoom_decim_iq(const void *x, int pcm16, long long origin, long long count, int decim, const void *taps,
                             unsigned dstep, long long m_first, long long m_count, void *y, void *stream);
/* Bank decimator: glb_launch_zoom_decim (iq = 0) or glb_launch_zoom_decim_iq (iq = 1) for nchan channels
 * (1..GLB_ZOOM_MAX_CHANNELS) of the same x in one launch: taps [nchan][33 decim] (re, im) pairs on the device,
 * dstep [nchan] on the host, channel c's outputs at y + c y_stride (complex samples; y_stride >= m_count when
 * nchan > 1).  Each input sample is loaded and converted once per tile for a group of up to 8 channels.  Every output
 * of channel c is bit-identical to the single-channel decimator's with taps + c 33 decim and dstep[c]: the same lane
 * partials over the same phases, taps in the same order, summed in the same order. */
#define GLB_ZOOM_MAX_CHANNELS 32
int glb_launch_zoom_bank_decim(const void *x, int pcm16, int iq, long long origin, long long count, int decim,
                               int nchan, const void *taps, const unsigned *dstep, long long m_first, long long m_count,
                               void *y, long long y_stride, void *stream);

/* Rows of complex frames (I/Q spectrogram, zoom frame stage) of an interleaved (I, Q) stream z:
 *     rows[f - first_frame][j] = |sum_i w[i] z[f hop - (n - hop) + i] e^{-2 pi i (j - n/2) i / n}|^2 / n
 * The taper holds w[i] taper_scale on both floats of complex sample i, with taper_scale = (float) (1 / (2 sqrt(2 n)))
 * (the fused kernel folds 1 / (n taper_scale^2) = 8 into its epilogue).
 * Multitaper (ntapers = K' > 1): taper points at [K'][2n] floats, taper k holding v_k[i] taper_scale / sqrt(lambda_k) on
 * both floats of complex sample i, and the row is the sum over k = 0..K'-1, in that order, of the rows of each taper. */
typedef struct {
  int n;                       /* complex frame length: power of two, 32..16384 */
  int hop;                     /* complex samples per frame */
  const float *samples;        /* device: interleaved (I, Q) of complex samples [origin, origin + count) */
  long long origin, count;     /* complex samples; indices < 0 read as 0 */
  const float *taper;          /* device: [2n] floats, or [ntapers][2n] */
  int taper_symmetric;         /* bit k: taper k satisfies taper[i] == taper[2n - 1 - i] bit for bit (one taper: 0 or 1) */
  float taper_scale;
  long long first_frame, nframes;
  float *rows;                 /* device out: [nframes][n] */
  const void *tables;          /* glb_tables_create(2 n) */
  void *scratch;               /* device: glb_iq_gram_scratch_bytes() bytes, or NULL when that is 0 */
  /* display levels of a fixed range instead of rows (main_window_draw, g_main.c:1186-1229; fields as glb_gram_args):
     pixel i of a row shows row position n - 1 - i.  Exactly one of rows and levels is set. */
  unsigned char *levels;       /* device out: [nframes][levels_stride], levels_stride = n */
  long long levels_stride;
  const void *level_tables;    /* from glb_level_tables_create() */
  int levels_log;              /* 1: integer-truncated dB, 0: linear */
  const unsigned char *level_lut;   /* device: level of every integer dB value (log scales) or NULL */
  float level_min, level_max;  /* display_min / display_max (dB in the log scales) */
  float level_thr;             /* opt.thr_level / 100 */
  int ntapers;                 /* 0 or 1: periodogram; K' = 2..32: multitaper (no levels: GLB_EINVAL) */
  /* Thomson's harmonic F-test of a multitaper launch (include/glfer_b200.h, glfer_iq_run_mtm_ftest):
       F[f][j] = (K' - 1) |mu(j)|^2 S / sum_k |y_k(j) - mu(j) U0_k|^2
     with mu the transform of the frame under hn and y_k under the unit-energy taper v_k.  Rows may then be NULL. */
  float *ftest;                /* device out: [nframes][n] F rows, or NULL */
  const float *ftest_taper;    /* device: [2n] floats, hn[i] taper_scale on both floats of complex sample i */
  const float *ftest_u0;       /* device: [ntapers] float pairs (U0_k, sqrt(lambda_k)) */
  float ftest_s;               /* S = sum_k U0_k^2 */
} glb_iq_gram_args;
/* The one entry of the I/Q spectrogram: the fused kernel (iq.cu, regular geometry n = 32..8192, hop = (n/16) << s
 * with n - hop a multiple of hop; needs an even origin, a 16-byte aligned samples pointer and samples that cover
 * every frame's blocks) or, for any other launch or under glb_force_generic_kernel(1), the general path below.
 * With levels the fused kernel maps the powers in its epilogue; the general path writes rows into scratch and
 * maps them with glb_launch_levels. */
int glb_launch_iq_gram(const glb_iq_gram_args *a, void *stream);
/* device scratch glb_launch_iq_gram needs for nframes frames (0 when the fused kernel serves the geometry);
 * levels: 1 when the launch writes levels (the general path then also holds the float rows); ntapers as in the
 * arguments (the general path reuses one spectrum plane for all tapers, so the size does not grow with it);
 * ftest: 1 when the launch writes F rows (the general path then also holds the mu and den planes) */
long long glb_iq_gram_scratch_bytes(int n, int hop, long long nframes, int levels, int ntapers, int ftest);
/* testing aids of the fused I/Q kernels: groups > 0 replaces the number of frame groups the launch policy picks
 * (still at most one per frame), so that a short run puts several frames into each group and exercises the ring's
 * steady state; 0, the default, restores the policy.  Occupancy, shared memory and the kernel choice are unchanged. */
void glb_set_ring_groups(int groups);
/* frames per group of the last fused I/Q launch */
int glb_last_frames_per_group(void);
/* the general path: the general spectrogram kernel's spectrum output on the 2n-float frames (into scratch, at
 * least nframes (n + 1) (re, im) pairs), then glb_launch_zoom_split; multitaper: that spectrum once per taper, each
 * followed by a split that stores (taper 0) or adds (the others) its powers into the rows.  F-test: scratch holds
 * nframes 3 n more floats; the hn spectrum is split first into the mu plane ([nframes][n] (re, im) pairs behind
 * the spectrum), each taper's split also adds its residual to the den plane ([nframes][n] floats behind mu), and a
 * last kernel forms F */
int glb_launch_iq_gram_general(const glb_iq_gram_args *a, void *stream);
/* device scratch glb_launch_iq_gram_general needs for nframes frames: the spectrum, then the float rows (levels = 1,
 * the two-pass levels of glb_launch_iq_gram) or the mu and den planes (ftest = 1) */
long long glb_iq_gram_general_scratch_bytes(int n, long long nframes, int levels, int ftest);

/* Harmonic lines of nframes F rows (glfer_b200/csrc/lines.cu; include/glfer_b200.h, glfer_iq_run_mtm_lines): one launch
 * for nchan channels laid as the frame stage lays them, channel c's frame i at row c crows + i of ftest (and of rows,
 * the multitaper rows, needed only for line_psd), rows of n floats at a stride of `stride` floats.  Bin j of
 * [bin_lo, bin_hi) is a candidate when F[j] > thr, F[j] > F[(j - 1) mod n] and F[j] >= F[(j + 1) mod n]; count[o] is
 * the number of candidates of output frame o = c nframes + i, and slots 0 .. min(count, max_lines) - 1 of bin / line_ftest
 * / line_psd ([nchan nframes][max_lines]) hold all of them, or the max_lines largest by (F, -j), in ascending j; the
 * other slots hold -1 / 0.0f / 0.0f.  line_ftest and line_psd may be NULL.  n a power of two in 32..16384, max_lines
 * 1..1024. */
int glb_launch_ftest_lines(const float *ftest, const float *rows, int n, long long stride, long long nframes, int nchan,
                           long long crows, float thr, int max_lines, int bin_lo, int bin_hi, int *count, int *bin,
                           float *line_ftest, float *line_psd, void *stream);

/* counters */
unsigned long long glb_kernel_launches(void);
/* family of the last spectrogram kernel launched: 1 general, 2 TMA ring (or its I/Q form, gram_iq_kernel), 3 warp-per-frame,
 * 4 two frames per thread, 5 32 points per thread */
int glb_last_kernel_family(void);

#ifdef __cplusplus
}
#endif
#endif
