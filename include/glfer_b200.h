/* glfer_b200.h -- batched spectrogram extension of the estimator interface.
 *
 * The reference computes one frame per call (fft_do / mtm_do / update_avg_*, called from
 * audio_available(), source.c:130-165).  A GPU launch per hop block is latency bound, so
 * the library adds a batched entry point that a file source or a headless harness calls
 * once per recording (or per time shard).  Its results equal the sequence of per-call
 * results of the reference loop:
 *     for each hop block f:  fft_do; fft_psd   (or mtm_do);   [update_avg_*]
 * with glfer.first_buffer TRUE on block 0 only: frame f covers stream samples
 * [f*hop - (N-hop), f*hop + hop) with zeros before the stream start (fft.c:98-113), block
 * means removed per hop block when sub_mean (fft.c:86-96), averaging warm-up and the
 * effdepth+1 divisor counted from frame 0 (avg.c:116-156).
 *
 * All functions return 0 on success or a negative GLFER_E* code; glfer_b200_last_error()
 * returns the message.  There is no CPU fallback: without a CUDA device plan creation
 * fails with GLFER_ENODEV.
 */
#ifndef GLFER_B200_H
#define GLFER_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GLFER_OK 0
#define GLFER_ECUDA (-1)
#define GLFER_EINVAL (-2)
#define GLFER_ENOMEM (-3)
#define GLFER_ENODEV (-4)

/* estimator mode: values of the reference's mode enum (glfer.h:47) */
#define GLFER_MODE_FFT 0
#define GLFER_MODE_MTM 1
#define GLFER_MODE_LMP 3   /* MODE_LMP: rectangular periodogram ring -> per-bin detector statistic (lmp.c) */
/* averaging mode: values of avgmode_t (glfer.h:53-55) */
#define GLFER_NO_AVG 0
#define GLFER_AVG_SUMAVG 1
#define GLFER_AVG_PLAIN 2
#define GLFER_AVG_SUMEXTREME 3

typedef struct {
  int mode;            /* GLFER_MODE_FFT | GLFER_MODE_MTM | GLFER_MODE_LMP */
  int n;               /* FFT size (opt.data_block_size): power of two, 32..32768 */
  int window_type;     /* fft.h window enum; ignored for MTM (forced rectangular, source.c:344) */
  float overlap;       /* opt.data_blocks_overlap; hop = (int)(n * (1.0 - overlap)) (fft.c:70) */
  float a;             /* opt.limiter_a, RA9MB parameter; <= 0 disables */
  int limiter;         /* opt.enable_limiter */
  int sub_mean;        /* opt.autoscale as latched by fft_init (fft.c:186) */
  float mtm_w;         /* opt.mtm_w (N*W) */
  int mtm_kmax;        /* opt.mtm_k: kmax + 1 tapers are used */
  int avg_mode;        /* GLFER_NO_AVG ... */
  int avg_depth;       /* opt.avgsamples */
  int avg_minbin;      /* (int)(opt.min_avgband / binsize) (g_main.c:1145) */
  int avg_maxbin;
  int avg_max0;        /* scale_type is *_MAX0 (g_main.c:1148-1151) */
  int avg_peakbin_init;/* the caller's peakbin before frame 0 */
  int scale_db;        /* 1: rows are 10*log10(value) (g_main.c:1191-1199) */
  int device;          /* CUDA device ordinal */
  int lmp_av;          /* opt.lmp_av: rows in the LMP ring (>= 2); the "psd" rows of an LMP plan are the
                          statistic of lmp_do; window forced rectangular (source.c:395), RA9MB / limiter
                          do not reach the spectrum (lmp.c:112-114); no frame averaging in this mode */
  int avg_band_only;   /* 1: averaged rows hold the band only, [nframes][avg_maxbin - avg_minbin] (column j = bin
                          avg_minbin + j).  The reference fills the rest of avg[] with the constant 1e-15
                          (avg.c:152-153); writing and shipping that constant is most of the cost of the averaging
                          pass when the band is a few dozen bins out of thousands */
  int mtm_ftest;       /* 1 (MTM plans): also prepare Thomson's harmonic F-test, which mtm_do computes into a file-static
                          nothing reads (mtm.c:59,165-174,204-210,222-233); rows through glfer_gram_run_mtm_ftest() */
  int zero_history;    /* 1: glfer.first_buffer stays TRUE, i.e. prepare_audio zeroes the N-hop history on EVERY
                          frame (fft.c:99-108).  That is what the reference GUI does with opt.autoscale == 0:
                          first_buffer is cleared only inside `if (opt.autoscale)` (g_main.c:1111-1120).
                          0 (default): TRUE on block 0 only, the sequence a sane caller drives */
} glfer_gram_config;

typedef struct glfer_gram_plan glfer_gram_plan;

const char *glfer_b200_last_error(void);
int glfer_b200_device_count(void);
/* pinned host memory for fast transfers (optional; any host pointer is accepted) */
void *glfer_b200_host_alloc(size_t bytes);
void glfer_b200_host_free(void *p);
/* kernels launched by this process so far */
unsigned long long glfer_b200_kernel_launches(void);

void glfer_gram_config_default(glfer_gram_config *cfg);     /* the defaults of glfer.c:238-279 */
int glfer_gram_plan_create(const glfer_gram_config *cfg, glfer_gram_plan **plan);
void glfer_gram_plan_destroy(glfer_gram_plan *plan);

int glfer_gram_hop(const glfer_gram_plan *plan);
int glfer_gram_bins(const glfer_gram_plan *plan);                       /* n/2 + 1 */
int glfer_gram_avg_cols(const glfer_gram_plan *plan);                   /* columns of an averaged row: bins, or the band (avg_band_only) */
long long glfer_gram_num_frames(const glfer_gram_plan *plan, long long nsamples);  /* nsamples / hop */
/* stream span [lo, hi) the frames [first_frame, first_frame + nframes) read (lo may be
 * negative: indices < 0 are the zero history) */
void glfer_gram_required_span(const glfer_gram_plan *plan, long long first_frame, long long nframes,
                              long long *lo, long long *hi);
/* window / taper tables as the estimator uses them (unit energy, before internal scaling) */
int glfer_gram_window(const glfer_gram_plan *plan, float *window /* [n] */);
int glfer_gram_tapers(const glfer_gram_plan *plan, double *tapers /* [kmax+1][n] */, double *lambda /* [kmax+1] */);

/* ---- one call, host buffers in and out (transfers pipelined with the kernels) ----
 * samples points at stream index `origin`, `count` samples long, and must cover
 * glfer_gram_required_span() clipped to [0, inf).  Any output pointer may be NULL.
 *   psd_rows [nframes][bins]   PSD (or dB when scale_db)
 *   avg_rows [nframes][bins]   averaged rows (avg_mode != GLFER_NO_AVG)
 *   avg_ret / avg_peakbin / avg_variance [nframes]: return value, *peakbin, *variance of
 *   update_avg_* after each frame. */
int glfer_gram_run(glfer_gram_plan *plan, const float *samples, long long origin, long long count,
                   long long first_frame, long long nframes, float *psd_rows, float *avg_rows,
                   double *avg_ret, int *avg_peakbin, double *avg_variance);
/* same, 16-bit PCM input converted on the device as wav_fmt.c:113 does */
int glfer_gram_run_pcm16(glfer_gram_plan *plan, const short *pcm, long long origin, long long count,
                         long long first_frame, long long nframes, float *psd_rows, float *avg_rows,
                         double *avg_ret, int *avg_peakbin, double *avg_variance);

/* Multitaper rows plus the harmonic F-test of every frame (plan created with mtm_ftest = 1):
 *   ftest[f][i] = kmax |mu(i)|^2 sum_U0_sqr / sum_j |y_j(i) - mu(i) U0_j|^2        (mtm.c:204-233)
 * with mu = FFT(frame * hn), hn = sum_j U0_j v_j / sum_U0_sqr, U0_j = sum_i v_j[i] (mtm.c:78-84,125-136).  As in the
 * reference the DC bin uses real parts only and, for even n, ftest[f][n/2] = num / 0 (inf, or nan for a zero
 * numerator).  Either output may be NULL. */
int glfer_gram_run_mtm_ftest(glfer_gram_plan *plan, const float *samples, long long origin, long long count,
                             long long first_frame, long long nframes, float *psd_rows, float *ftest_rows);

/* ---- device-resident path: stage once, execute many times, fetch when wanted ---- */
int glfer_gram_stage(glfer_gram_plan *plan, const float *samples, long long origin, long long count);
int glfer_gram_stage_pcm16(glfer_gram_plan *plan, const short *pcm, long long origin, long long count);
/* frames [first_frame, first_frame + nframes) from the staged samples into device rows;
 * returns after the work is queued.  kernel_ms (may be NULL) receives the device time of
 * the launch sequence measured with CUDA events on the plan's stream (this call then
 * waits for completion). */
int glfer_gram_exec(glfer_gram_plan *plan, long long first_frame, long long nframes, float *kernel_ms);
/* device time of the fused spectrogram kernel alone in the last glfer_gram_exec that was
 * given a non-NULL kernel_ms (the other launches are block means / averaging) */
int glfer_gram_last_gram_ms(glfer_gram_plan *plan, float *ms);
int glfer_gram_sync(glfer_gram_plan *plan);
int glfer_gram_fetch(glfer_gram_plan *plan, float *psd_rows, float *avg_rows, double *avg_ret,
                     int *avg_peakbin, double *avg_variance);

/* ---- display mapping: what main_window_draw does with a row (g_main.c:1109-1229) ----
 * compute_floor statistics -> AGC of the display range (autoscale) or fixed dB levels ->
 * level = 10*log10 (through the reference's `short` level buffer: integer dB) or linear ->
 * 8-bit palette index with threshold and clipping, pixel i = bin bins-1-i -> optional RGB.
 * The rows shown are the averaged rows when the plan averages, else the PSD rows. */
typedef struct {
  int log_scale;          /* opt.scale_type is SCALE_LOG or SCALE_LOG_MAX0 (g_main.c:1132,1191) */
  int autoscale;          /* opt.autoscale (g_main.c:1111) */
  float max_level_db;     /* opt.max_level_db / opt.min_level_db, used when !autoscale (g_main.c:1126-1128) */
  float min_level_db;
  float thr_level;        /* opt.thr_level, percent (g_main.c:1098) */
  const unsigned char *colortab;   /* 256 RGB triplets (set_palette, g_main.c:651-762) or NULL */
} glfer_display_config;
/* levels [nframes][bins] and/or rgb [nframes][bins][3]; display_range [nframes][2] (max, min)
 * when autoscale (optional).  agc_state [2] = (display_max_lvl, display_min_lvl): in when
 * first_frame > 0, out always (lets time shards chain the recurrence); may be NULL for runs
 * that start at frame 0. */
int glfer_gram_run_display(glfer_gram_plan *plan, const float *samples, long long origin, long long count,
                           long long first_frame, long long nframes, const glfer_display_config *dc,
                           float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range);
int glfer_gram_run_display_pcm16(glfer_gram_plan *plan, const short *pcm, long long origin, long long count,
                                 long long first_frame, long long nframes, const glfer_display_config *dc,
                                 float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range);

/* The level mapping alone on caller-provided rows (host memory): rows [nrows][nbins] -> levels [nrows][nbins],
 * pixel i of a row = bin nbins-1-i.  range: [nrows][2] = (display_max, display_min) per row as main_window_draw
 * holds them (dB in the log scales), or NULL for the fixed levels of dc (dc->autoscale is ignored). */
int glfer_b200_map_levels(const float *rows, long long nrows, int nbins, const glfer_display_config *dc,
                          const float *range, unsigned char *levels, int device);
/* per-call interface (fft_do / mtm_do / lmp_do): 1 (default) = the frame is read from, and the results are written
 * to, pinned host memory by the kernel itself (no copy-engine round trips); 0 = staged through device buffers */
void glfer_b200_set_zero_copy(int on);
/* 0 (default) = frame averaging as a second pass over the PSD rows; 1 = fused into the spectrogram kernel where it
 * can be (avg_band_only plans, N = 4096 / 8192, regular overlap, band history <= 2 KB): bit-identical rows, but
 * measured slower on B200 (1.31 ms against 0.82 + 0.20 ms on BASELINE config C2), so it is opt-in */
void glfer_b200_set_fused_avg(int on);
/* testing aid: 0 = glfer_gram_run_display and glfer_iq_run_display always map the levels in a second pass over float
 * rows; 1 (default) = with a fixed display range and no averaging the spectrogram kernel writes the 8-bit levels itself */
void glfer_b200_set_fused_levels(int on);
/* the palettes of set_palette (g_main.c:649-762; glfer.h:47: 0 HSV, 1 THRESH, 2 COOL, 3 HOT, 4 BW, 5 BONE,
 * 6 COPPER, 7 OTD): 256 RGB triplets into tab[768] */
int glfer_palette(int palette, unsigned char *tab);

/* ---- time-sharded multi-GPU run inside one process (one host thread per device) ----
 * Frames [0, nframes) are split into ndev contiguous ranges; device g gets samples
 * [F_g*hop - halo, F_{g+1}*hop) (halo = N - hop, plus (depth-1) frames when averaging);
 * no inter-GPU communication.  devices == NULL means 0..ndev-1. */
int glfer_gram_run_sharded(const glfer_gram_config *cfg, int ndev, const int *devices, const float *samples,
                           long long nsamples, float *psd_rows, float *avg_rows, double *avg_ret,
                           int *avg_peakbin, double *avg_variance);
/* the shard arithmetic on its own: frame range of shard g of ndev */
void glfer_gram_shard_range(long long nframes, int ndev, int g, long long *first, long long *count);

/* ---- WAV source (wav_fmt.c:45-121 semantics, LP64-safe) ---- */
typedef struct {
  int sample_rate;
  int bits;             /* 8 or 16 */
  int channels;
  long long nsamples;   /* samples in the data chunk (channels not de-interleaved, as the reference) */
  void *data;           /* raw PCM as read */
} glfer_wav;
int glfer_wav_load(const char *path, glfer_wav *wav);
/* extension (the reference treats a stereo file's interleaved samples as one channel): keep one channel, in place */
int glfer_wav_select_channel(glfer_wav *wav, int channel);
void glfer_wav_free(glfer_wav *wav);
/* spectrogram of a WAV exactly as `glfer -f file` would see it block by block, including
 * the stale tail of a short final read (wav_fmt.c:102-119).  Returns frames via *nframes;
 * psd_rows must hold glfer_wav_num_frames() rows. */
long long glfer_wav_num_frames(const glfer_gram_plan *plan, const glfer_wav *wav);
int glfer_gram_run_wav(glfer_gram_plan *plan, const glfer_wav *wav, float *psd_rows, float *avg_rows,
                       double *avg_ret, int *avg_peakbin, double *avg_variance);

/* ---- zoom spectrogram: sub-hertz bins around a chosen frequency ----
 * The stream is mixed by the centre frequency to DC (phase phi(n) = (n step mod 2^32) / 2^32, exact from the
 * absolute sample index, step = llround(center_hz / sample_rate 2^32)), low-passed by a 32 D + 1 tap Kaiser
 * windowed sinc (glfer_zoom_taps) and decimated by D:
 *     y[m] = sum_{l=-K..K} h[l] x[mD - l] e^{-2 pi i phi(mD - l)},  K = 16 D,  x[n < 0] = 0,  y[m < 0] = 0.
 * Frames of n complex samples at hop glb_hop(n, overlap) cover y[f hop - (n - hop), f hop + hop); a row is
 *     P[f][j] = |sum_i w[i] y_f[i] e^{-2 pi i (j - n/2) i / n}|^2 / n,   j = 0..n-1,
 * with w the spectrogram window of that size (rectangular: all ones).  Bin j is at
 * center + (j - n/2) sample_rate / (D n); the clean span is |f - center| <= 0.4 sample_rate / D. */
typedef struct {
  int n;               /* complex FFT size: power of two, 32..16384 */
  int decim;           /* decimation D: 2..1024 */
  int window_type;     /* fft.h window enum */
  float overlap;       /* hop = (int)(n * (1.0 - overlap)), as the spectrogram */
  double center_hz;    /* 0 <= center_hz <= sample_rate / 2 */
  double sample_rate;
  int device;          /* CUDA device ordinal */
} glfer_zoom_config;

typedef struct glfer_zoom_plan glfer_zoom_plan;

void glfer_zoom_config_default(glfer_zoom_config *cfg);
int glfer_zoom_plan_create(const glfer_zoom_config *cfg, glfer_zoom_plan **plan);
void glfer_zoom_plan_destroy(glfer_zoom_plan *plan);
int glfer_zoom_hop(const glfer_zoom_plan *plan);
int glfer_zoom_bins(const glfer_zoom_plan *plan);                       /* n */
double glfer_zoom_center_hz(const glfer_zoom_plan *plan);               /* step sample_rate / 2^32 */
/* frames of a stream of nsamples samples: floor(Md / hop), Md = number of m >= 0 with mD + K <= nsamples - 1 */
long long glfer_zoom_num_frames(const glfer_zoom_plan *plan, long long nsamples);
/* stream span [lo, hi) the frames [first_frame, first_frame + nframes) read (lo may be negative: indices < 0 are
 * the zero history) */
void glfer_zoom_required_span(const glfer_zoom_plan *plan, long long first_frame, long long nframes,
                              long long *lo, long long *hi);
/* samples point at stream index `origin`, `count` samples long, and must cover glfer_zoom_required_span()
 * clipped to [0, inf).  rows: [nframes][n] */
int glfer_zoom_run(glfer_zoom_plan *plan, const float *samples, long long origin, long long count,
                   long long first_frame, long long nframes, float *rows);
int glfer_zoom_run_pcm16(glfer_zoom_plan *plan, const short *pcm, long long origin, long long count,
                         long long first_frame, long long nframes, float *rows);
/* the low-pass filter h[l], l = -K..K, as taps[l + K] (32 decim + 1 floats); host only, needs no device */
int glfer_zoom_taps(int decim, float *taps);

/* ---- complex (I/Q) input: SDR baseband recordings ----
 * An I/Q stream is interleaved: iq[2s] is I and iq[2s + 1] is Q of complex sample s, z[s] = I + iQ; origin and
 * count are in complex samples.  The pcm16 forms take the data chunk of a 16-bit stereo WAV exactly as
 * glfer_wav_load returns it (I on the left channel, Q on the right), with count = wav.nsamples / 2; samples are
 * converted as the mono reader does ((float) s / 32768).  Frequencies are relative to the recording's centre (the
 * receiver's dial frequency): negative below it, positive above. */

/* I/Q zoom: the zoom above with complex x, no mirror image.  The centre may be anywhere in
 * [-sample_rate / 2, sample_rate / 2]; step = (uint32) llround(center_hz / sample_rate 2^32), modulo 2^32, and
 * glfer_zoom_center_hz of an I/Q plan reads the step as a signed 32-bit value.  The clean span is again
 * |f - center| <= 0.4 sample_rate / D.  Real entry points reject I/Q plans and the reverse (GLFER_EINVAL). */
int glfer_zoom_plan_create_iq(const glfer_zoom_config *cfg, glfer_zoom_plan **plan);
int glfer_zoom_run_iq(glfer_zoom_plan *plan, const float *iq, long long origin, long long count,
                      long long first_frame, long long nframes, float *rows);
int glfer_zoom_run_iq_pcm16(glfer_zoom_plan *plan, const short *iq, long long origin, long long count,
                            long long first_frame, long long nframes, float *rows);

/* I/Q spectrogram: two-sided rows of complex FFT frames at the full sample rate.  Frame f covers complex samples
 * [f hop - (n - hop), f hop + hop) (samples before index 0 are zero) and its row is
 *     P[f][j] = |sum_i w[i] z[f hop - (n - hop) + i] e^{-2 pi i (j - n/2) i / n}|^2 / n,   j = 0..n-1,
 * so bin j lies at (j - n/2) sample_rate / n and DC is at j = n/2.  No block-mean removal, RA9MB or limiter;
 * glfer_iq_run_display gives the waterfall's pixels directly. */
typedef struct {
  int n;               /* complex FFT size: power of two, 32..16384 */
  int window_type;     /* fft.h window enum (rectangular: all ones, as the zoom) */
  float overlap;       /* hop = (int)(n * (1.0 - overlap)), as the spectrogram */
  int device;          /* CUDA device ordinal */
} glfer_iq_config;

typedef struct glfer_iq_plan glfer_iq_plan;

void glfer_iq_config_default(glfer_iq_config *cfg);
int glfer_iq_plan_create(const glfer_iq_config *cfg, glfer_iq_plan **plan);
void glfer_iq_plan_destroy(glfer_iq_plan *plan);
int glfer_iq_hop(const glfer_iq_plan *plan);
int glfer_iq_bins(const glfer_iq_plan *plan);                           /* n */
long long glfer_iq_num_frames(const glfer_iq_plan *plan, long long nsamples);   /* nsamples / hop */
/* complex-sample span [lo, hi) the frames [first_frame, first_frame + nframes) read (lo may be negative) */
void glfer_iq_required_span(const glfer_iq_plan *plan, long long first_frame, long long nframes,
                            long long *lo, long long *hi);
/* iq points at complex sample `origin`, `count` complex samples long, and must cover glfer_iq_required_span()
 * clipped to [0, inf).  rows: [nframes][n] */
int glfer_iq_run(glfer_iq_plan *plan, const float *iq, long long origin, long long count,
                 long long first_frame, long long nframes, float *rows);
int glfer_iq_run_pcm16(glfer_iq_plan *plan, const short *iq, long long origin, long long count,
                       long long first_frame, long long nframes, float *rows);

/* ---- multitaper I/Q and zoom plans ----
 * Thomson's multitaper estimator on the complex frames of an I/Q or zoom plan.  Frame f is the plan's frame above
 * (complex samples [f hop - (n - hop), f hop + hop) of z, or of the decimated y for a zoom, zeros before index 0),
 * and its row is
 *     P[f][j] = sum_{k=0..K'-1} |sum_i v_k[i] z_f[i] e^{-2 pi i (j - n/2) i / n}|^2 / (n lambda_k),   j = 0..n-1,
 * K' = mtm_kmax + 1, with v_k, lambda_k = glb_dpss(n, mtm_w, mtm_kmax): the unit-energy DPSS tapers and eigenvalues
 * that a real GLFER_MODE_MTM plan of the same n uses (NW = mtm_w as gl_dpss takes it).  The weights are 1 / lambda_k,
 * not normalised, as mtm_do weighs them (mtm.c:214-219): an I/Q multitaper row of (x, 0) is the real multitaper row
 * of x on its positive half.  So on white noise a multitaper row sits about 10 log10(sum_k 1 / lambda_k) dB above the
 * periodogram row of the same n (the tapers and the spectrogram windows all have unit energy; the rectangular window,
 * all ones, has energy n instead): +9.3 dB at NW = 4, K' = 8 (sum_k 1 / lambda_k = 8.51), +23.8 dB at NW = 2.5,
 * K' = 8, where the last tapers have small eigenvalues.  A fixed display range chosen for periodogram rows must move
 * up by that much.
 * Rows are fft-shifted as before (DC at n/2; zoom bin j at centre + (j - n/2) sample_rate / (D n)); window_type is
 * ignored, everything else in the config means what it means above.  GLFER_EINVAL for mtm_kmax outside 0..31, mtm_w
 * not > 0, or a DPSS eigenvalue that is not positive.  Every run, run_display and query entry point serves these
 * plans unchanged (run_display maps the multitaper rows), and the zoom's real and I/Q entry points keep rejecting
 * each other's plans. */
int glfer_iq_plan_create_mtm(const glfer_iq_config *cfg, float mtm_w, int mtm_kmax, glfer_iq_plan **plan);
int glfer_zoom_plan_create_mtm(const glfer_zoom_config *cfg, float mtm_w, int mtm_kmax, glfer_zoom_plan **plan);
int glfer_zoom_plan_create_iq_mtm(const glfer_zoom_config *cfg, float mtm_w, int mtm_kmax, glfer_zoom_plan **plan);
/* the plan's tapers [mtm_kmax + 1][n] and eigenvalues [mtm_kmax + 1] before scaling; GLFER_EINVAL on a periodogram plan */
int glfer_iq_tapers(const glfer_iq_plan *plan, double *tapers, double *lambda);
int glfer_zoom_tapers(const glfer_zoom_plan *plan, double *tapers, double *lambda);

/* ---- zoom channel banks: several centres of one recording ----
 * A bank is a zoom plan with C channels: C centre frequencies that share one config (n, decim, window, overlap, sample
 * rate, device), real (iq = 0) or I/Q (iq = 1) input, periodogram or multitaper (mtm_w, mtm_kmax as
 * glfer_zoom_plan_create_mtm).  cfg->center_hz is ignored; centers_hz[c], c = 0..nchan-1, is validated as the
 * single-centre constructors validate center_hz ([0, sample_rate / 2] real, [-sample_rate / 2, sample_rate / 2] I/Q);
 * duplicates are allowed; nchan in 1..32.  All of this is checked before any device call (GLFER_EINVAL).
 * Each run uploads the input once and decimates it for every channel in one kernel.  Every zoom run, run_display,
 * mtm_ftest and query entry point serves banks with its own signature; per-channel outputs are stacked on a leading
 * axis: rows, F rows and levels [C][nframes][n], RGB [C][nframes][n][3], display_range [C][nframes][2], agc_state
 * [C][2] (one AGC recurrence per channel).  The required span, hop, bins and frame count do not depend on the centre.
 * A plan from the single-centre constructors has C = 1, and with C = 1 every layout is the one above.
 * Channel c of a bank is bit-identical to a single-centre zoom plan at centers_hz[c] with the same config: rows, F
 * rows, levels, RGB, display range and AGC state, for every input format and estimator. */
int glfer_zoom_plan_create_bank(const glfer_zoom_config *cfg, const double *centers_hz, int nchan, int iq,
                                glfer_zoom_plan **plan);
int glfer_zoom_plan_create_bank_mtm(const glfer_zoom_config *cfg, const double *centers_hz, int nchan, int iq,
                                    float mtm_w, int mtm_kmax, glfer_zoom_plan **plan);
int glfer_zoom_channels(const glfer_zoom_plan *plan);                      /* C; 1 for the single-centre constructors */
/* as glfer_zoom_center_hz, of channel c (NaN outside 0..C-1); glfer_zoom_center_hz is channel 0's */
double glfer_zoom_channel_center_hz(const glfer_zoom_plan *plan, int c);

/* Thomson's harmonic F-test of multitaper I/Q and zoom plans (real and I/Q zoom).  Frame f is the plan's complex frame
 * z_f above (I/Q samples, or the decimated y of a zoom), v_k and lambda_k the plan's tapers (glfer_iq_tapers /
 * glfer_zoom_tapers), K' = mtm_kmax + 1, and
 *     U0_k = sum_i v_k[i],   S = sum_k U0_k^2,   hn[i] = sum_k U0_k v_k[i] / S
 * built exactly as a real GLFER_MODE_MTM plan with mtm_ftest = 1 builds them (U0 in double, S and hn through float
 * accumulators, mtm.c:78-84,123-136).  For every row position j = 0..n-1 (fft-shifted, DC at n/2, as the rows):
 *     y_k(j) = sum_i v_k[i] z_f[i] e^{-2 pi i (j - n/2) i / n}     (the unit-energy taper, not weighted by 1 / lambda_k)
 *     mu(j)  = sum_i hn[i] z_f[i] e^{-2 pi i (j - n/2) i / n}
 *     F[f][j] = (K' - 1) |mu(j)|^2 S / sum_k |y_k(j) - mu(j) U0_k|^2
 * Every bin of a complex frame is complex: none of the real F-test's DC and Nyquist special cases, the denominator is
 * accumulated at every position.  For I/Q input (x, 0), F at row position n/2 + j is the real plan's F-test of x at bin
 * j, 1 <= j < n/2.  On white complex Gaussian noise F follows the F(2, 2K' - 2) distribution, so a threshold has a
 * stated false-alarm rate.  The division follows IEEE rules: an all-zero frame gives 0 / 0 = NaN.
 * Each call returns the rows (bit-identical to glfer_iq_run / glfer_zoom_run* of the same frames) and/or the F rows,
 * [nframes][n] each; either pointer may be NULL, not both.  Every multitaper I/Q or zoom plan serves them.  GLFER_EINVAL
 * for a periodogram plan, K' < 2 (no degrees of freedom), both outputs NULL, input that does not cover the plan's
 * required span, and (zoom) a real entry point with an I/Q plan or the reverse. */
int glfer_iq_run_mtm_ftest(glfer_iq_plan *plan, const float *iq, long long origin, long long count,
                           long long first_frame, long long nframes, float *rows, float *ftest);
int glfer_iq_run_mtm_ftest_pcm16(glfer_iq_plan *plan, const short *iq, long long origin, long long count,
                                 long long first_frame, long long nframes, float *rows, float *ftest);
int glfer_zoom_run_mtm_ftest(glfer_zoom_plan *plan, const float *samples, long long origin, long long count,
                             long long first_frame, long long nframes, float *rows, float *ftest);
int glfer_zoom_run_mtm_ftest_pcm16(glfer_zoom_plan *plan, const short *pcm, long long origin, long long count,
                                   long long first_frame, long long nframes, float *rows, float *ftest);
int glfer_zoom_run_iq_mtm_ftest(glfer_zoom_plan *plan, const float *iq, long long origin, long long count,
                                long long first_frame, long long nframes, float *rows, float *ftest);
int glfer_zoom_run_iq_mtm_ftest_pcm16(glfer_zoom_plan *plan, const short *iq, long long origin, long long count,
                                      long long first_frame, long long nframes, float *rows, float *ftest);

/* ---- harmonic line detection of multitaper I/Q and zoom plans ----
 * Threshold of the harmonic F-test at a per-bin false-alarm probability pfa under the null, F(2, 2K' - 2):
 *     P(F > x) = (1 + x / (K' - 1))^-(K' - 1)   =>   x = (K' - 1) expm1(-log(pfa) / (K' - 1)),
 * computed in double and rounded to float.  Host only, needs no device.  GLFER_EINVAL for ntapers < 2, pfa outside
 * (0, 1) or thr NULL. */
int glfer_ftest_threshold(int ntapers, double pfa, float *thr);

typedef struct {
  double pfa;          /* per-bin false-alarm probability, 0 < pfa < 1 -> thr = glfer_ftest_threshold(K', pfa) */
  int max_lines;       /* slots per frame, 1..1024 */
  int bin_lo, bin_hi;  /* row positions searched, 0 <= bin_lo < bin_hi <= n (a zoom's clean span is about n/2 +- 0.4 n) */
} glfer_lines_config;

/* The lines of each frame, selected on the device from the F rows, which never leave it.  F[f][j] and P[f][j] are the
 * F row and the row that the *_run_mtm_ftest entry of the same input form returns for the same plan and call (on the
 * same path: fused or general, glb_force_generic_kernel alike).
 *   Candidates: bin j in [bin_lo, bin_hi) of frame f with F[j] > thr, F[j] > F[(j - 1) mod n] and F[j] >= F[(j + 1)
 *   mod n], all float comparisons; the neighbours are cyclic and read from the whole row, also outside the range.  One
 *   bin per peak, the leftmost of a plateau.  IEEE rules apply: a NaN bin is never a candidate and never beats a
 *   neighbour (an all-zero frame, F = 0 / 0 = NaN, has no lines); an infinite F can be a line.
 *   line_count[f]: the number of candidates, also when it exceeds max_lines (the frame was truncated).
 *   Selected: every candidate when count <= max_lines, otherwise the max_lines candidates with the largest F, ties to
 *   the smaller j.  They are stored in ascending j in slots 0 .. min(count, max_lines) - 1: line_bin[f][s] = j,
 *   line_ftest[f][s] = F[f][j], line_psd[f][s] = P[f][j], the same floats bit for bit; the other slots hold bin -1, F
 *   0.0f and psd 0.0f.
 *   Layouts: line_count [nframes], the others [nframes][max_lines]; a bank adds a leading channel axis ([C][nframes],
 *   [C][nframes][max_lines]) and channel c is bit-identical to a single-centre plan at its centre.  line_count and
 *   line_bin are required; line_ftest and line_psd may be NULL (without line_psd no rows are formed on the device).
 *   The outputs are staged in pinned memory of the plan, so pageable arrays do not stall the chunk pipeline.
 * GLFER_EINVAL for everything the *_mtm_ftest entries reject, and for lc NULL, pfa outside (0, 1), max_lines outside
 * 1..1024, a bin range outside 0 <= bin_lo < bin_hi <= n, and line_count or line_bin NULL; all checked before any
 * device call.
 * Not covered: the sub-bin frequency and the complex amplitude (mu) of a line, and line detection of real
 * GLFER_MODE_MTM plans, whose F-test has DC and Nyquist special cases (inf at n/2). */
int glfer_iq_run_mtm_lines(glfer_iq_plan *plan, const float *iq, long long origin, long long count,
                           long long first_frame, long long nframes, const glfer_lines_config *lc, int *line_count,
                           int *line_bin, float *line_ftest, float *line_psd);
int glfer_iq_run_mtm_lines_pcm16(glfer_iq_plan *plan, const short *iq, long long origin, long long count,
                                 long long first_frame, long long nframes, const glfer_lines_config *lc,
                                 int *line_count, int *line_bin, float *line_ftest, float *line_psd);
int glfer_zoom_run_mtm_lines(glfer_zoom_plan *plan, const float *samples, long long origin, long long count,
                             long long first_frame, long long nframes, const glfer_lines_config *lc, int *line_count,
                             int *line_bin, float *line_ftest, float *line_psd);
int glfer_zoom_run_mtm_lines_pcm16(glfer_zoom_plan *plan, const short *pcm, long long origin, long long count,
                                   long long first_frame, long long nframes, const glfer_lines_config *lc,
                                   int *line_count, int *line_bin, float *line_ftest, float *line_psd);
int glfer_zoom_run_iq_mtm_lines(glfer_zoom_plan *plan, const float *iq, long long origin, long long count,
                                long long first_frame, long long nframes, const glfer_lines_config *lc,
                                int *line_count, int *line_bin, float *line_ftest, float *line_psd);
int glfer_zoom_run_iq_mtm_lines_pcm16(glfer_zoom_plan *plan, const short *iq, long long origin, long long count,
                                      long long first_frame, long long nframes, const glfer_lines_config *lc,
                                      int *line_count, int *line_bin, float *line_ftest, float *line_psd);

/* ---- display output of I/Q and zoom plans ----
 * The waterfall of the plan's own rows, as glfer_gram_run_display gives it for real audio: levels, rgb, agc_state
 * and display_range as there, and exactly main_window_draw's mapping (g_main.c:1109-1229) of the rows that
 * glfer_iq_run / glfer_zoom_run* compute.  Both the floor statistics and the row shown are the plan's row (these
 * plans do not average); pixel i of a row is row position n - 1 - i, the highest frequency first; the AGC's first
 * frame divides by the plan's overlap.  agc_state chains the recurrence between calls and time shards.  GLFER_EINVAL
 * for autoscale from first_frame > 0 without agc_state, RGB without a palette, input that does not cover the
 * plan's required span, and (zoom) a real entry point with an I/Q plan or the reverse.
 * The I/Q centre -- the receiver's LO leakage, at row position n/2 -- is a bin like any other: a strong spike there
 * can be the row's largest bin and so set the AGC's upper level, as it would in the reference's mapping.
 * Periodogram I/Q plans with a fixed range and no RGB compute the levels in the spectrogram kernel itself (no float
 * row is stored); the other cases, multitaper plans always, map device rows, and only the levels (or RGB) and the
 * range cross PCIe. */
int glfer_iq_run_display(glfer_iq_plan *plan, const float *iq, long long origin, long long count,
                         long long first_frame, long long nframes, const glfer_display_config *dc,
                         float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range);
int glfer_iq_run_display_pcm16(glfer_iq_plan *plan, const short *iq, long long origin, long long count,
                               long long first_frame, long long nframes, const glfer_display_config *dc,
                               float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range);
int glfer_zoom_run_display(glfer_zoom_plan *plan, const float *samples, long long origin, long long count,
                           long long first_frame, long long nframes, const glfer_display_config *dc,
                           float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range);
int glfer_zoom_run_display_pcm16(glfer_zoom_plan *plan, const short *pcm, long long origin, long long count,
                                 long long first_frame, long long nframes, const glfer_display_config *dc,
                                 float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range);
int glfer_zoom_run_display_iq(glfer_zoom_plan *plan, const float *iq, long long origin, long long count,
                              long long first_frame, long long nframes, const glfer_display_config *dc,
                              float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range);
int glfer_zoom_run_display_iq_pcm16(glfer_zoom_plan *plan, const short *iq, long long origin, long long count,
                                    long long first_frame, long long nframes, const glfer_display_config *dc,
                                    float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range);

/* ---- hidden inputs of the per-call interface (fft.c:99,186: globals `glfer`, `opt`) ----
 * When the host program defines `opt` and `glfer` (as glfer.c:56-62 does) the per-call
 * functions read them.  Otherwise these setters provide the two values. */
void glfer_b200_set_autoscale(int autoscale);
void glfer_b200_set_first_buffer(int first_buffer);

#ifdef __cplusplus
}
#endif
#endif
