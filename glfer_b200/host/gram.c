/* gram.c -- batched spectrogram plans: the C host layer over the CUDA shim.
 *
 * A plan is the batch counterpart of fft_init()/mtm_init() + alloc_avg(): it owns the
 * window / DPSS taper tables (built on the host in double, uploaded once as floats with the
 * PSD normalisation folded in), the FFT constant tables and two "slots" of device
 * buffers with their own streams, so that glfer_gram_run() can overlap the upload of one
 * chunk of the recording with the kernels and the download of the previous one.
 *
 * Folded scaling.  fft_psd divides |X|^2 by N (fft.c:212-216) and mtm_do divides each
 * eigen-spectrum by lambda_k (mtm.c:215).  The real-FFT split in the kernel produces
 * 2 X[k]; multiplying the taper by s = 1 / (2 sqrt(N)) (and by 1 / sqrt(lambda_k) for
 * multitaper) makes |2 s X|^2 the PSD sample itself, so the kernel epilogue is a bare
 * re^2 + im^2.
 */
#include <math.h>
#include <pthread.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "glb_host.h"

/* chunks in flight (stream + device buffers each).  Two overlap H2D / kernels / D2H of a plain run; the autoscale
   display chain (floor statistics -> AGC recurrence -> levels, ~0.25 ms of dependent kernels per chunk between the
   copies) needs a third to stay PCIe-bound: 8.9 -> 7.0 ms per hour of signal (four: 7.4 ms). */
#ifndef NSLOT
#define NSLOT 3
#endif

typedef struct {
  void *stream;
  void *ev0, *ev1, *ev2, *ev3;
  int time_gram;        /* record ev2/ev3 around the gram kernel */
  float *d_samples;     /* staged stream span */
  size_t samples_cap;   /* floats */
  long long s_origin, s_count;
  short *d_pcm;
  size_t pcm_cap;       /* shorts */
  float *d_means;
  size_t means_cap;
  float *d_psd;         /* [halo + nframes][bins] */
  size_t psd_cap;       /* floats */
  float *d_avg;
  size_t avg_cap;
  double *d_ret, *d_var;
  int *d_cand, *d_peak, *d_unres;
  size_t scal_cap;      /* frames */
  long long out_first, out_nframes, out_halo;
  glb_display_slot disp;  /* display mapping */
} slot_t;

struct glfer_gram_plan {
  glfer_gram_config cfg;
  int hop, bins, ntapers;
  int avg_cols;         /* columns of an averaged row: bins, or the band when cfg.avg_band_only */
  float taper_scale;
  float *h_window;      /* unit-energy window as compute_window leaves it */
  double *h_tapers;     /* MTM: [ntapers][n] */
  double *h_lambda;
  float *d_tapers;
  int taper_sym;        /* periodogram: the uploaded table is mirror-symmetric bit for bit */
  void *tables;
  slot_t slot[NSLOT];
  int *d_cand_all, *d_peak_all;   /* whole-run *peakbin candidates / carried values */
  size_t cand_all_cap;
  glb_display disp;     /* display mapping */
  /* harmonic F-test (mtm_ftest): hn and the unit-energy tapers scaled for the spectrum output, U0 */
  float *d_ftapers;     /* [ntapers + 1][n] */
  double *d_u0;
  double sum_u0_sqr;
  float *d_fspec, *d_ftest;
  size_t fspec_cap, ftest_cap;
  void *h_scal;         /* pinned staging of the small per-frame outputs (ret / variance / peakbin) */
  size_t h_scal_cap;
};

/* what a display run asks of exec_slot: levels written by the spectrogram kernel itself */
typedef struct {
  int log_scale;
  float dmin, dmax, thr;
} fused_levels;

/* Frame averaging inside the spectrogram kernel exists and is bit-identical to the two-pass form, but it is
   OFF by default: measured on B200 (C2: N=4096 Kaiser 75 %, depth 4, band of 68 bins, 168 750 frames) the
   fused kernel takes 1.31 ms against 0.82 ms + 0.20 ms in two passes -- the averaging of a frame is a
   ~5 000-cycle chain of double-precision reductions on one warp that sits on the frame group's critical
   path, while the stand-alone kernel runs the same chains on every warp of the chip at once. */
static int g_fused_avg = 0;
void glfer_b200_set_fused_avg(int on) { g_fused_avg = on; }
static int g_fused_levels = 1;
/* testing aid: 0 = always map levels in a second pass over float rows */
void glfer_b200_set_fused_levels(int on) { g_fused_levels = on; }
int glb_host_fused_levels(void) { return g_fused_levels; }

static __thread char g_msg[512];

const char *glfer_b200_last_error(void)
{
  return g_msg[0] ? g_msg : glb_last_error();
}

static int fail(int code, const char *msg)
{
  snprintf(g_msg, sizeof g_msg, "%s", msg);
  return code;
}

static int shim(int rc)
{
  if (rc != GLB_OK) snprintf(g_msg, sizeof g_msg, "%s", glb_last_error());
  return rc;   /* GLB_E* and GLFER_E* share values */
}

int glb_host_fail(int code, const char *msg) { return fail(code, msg); }
int glb_host_shim(int rc) { return shim(rc); }
void glb_host_clear_error(void) { g_msg[0] = 0; }

int glfer_b200_device_count(void)
{
  int c = 0;
  if (glb_device_count(&c) != GLB_OK) return 0;
  return c;
}

void *glfer_b200_host_alloc(size_t bytes)
{
  void *p = NULL;
  if (shim(glb_host_alloc(&p, bytes)) != 0) return NULL;
  return p;
}

void glfer_b200_host_free(void *p) { glb_host_free(p); }

unsigned long long glfer_b200_kernel_launches(void) { return glb_kernel_launches(); }

/* hop exactly as prepare_audio computes it (fft.c:70): double product, truncated */
int glb_hop(int n, float overlap)
{
  int n_eff = n * (1.0 - overlap);
  return n_eff;
}

void glfer_gram_config_default(glfer_gram_config *c)
{
  memset(c, 0, sizeof *c);
  c->mode = GLFER_MODE_FFT;
  c->n = 1024;                 /* glfer.c:238-279 */
  c->window_type = KAISER_WINDOW;
  c->overlap = 0.0f;
  c->a = 0.0f;
  c->limiter = 0;
  c->sub_mean = 1;             /* opt.autoscale = 1 */
  c->mtm_w = 4.0f;
  c->mtm_kmax = 7;
  c->avg_mode = GLFER_NO_AVG;
  c->avg_depth = 4;
  c->avg_minbin = 0;
  c->avg_maxbin = 0;
  c->device = 0;
  c->lmp_av = 4;               /* glfer.c:252 */
}

int glb_plan_sub_mean(const glfer_gram_plan *p) { return p->cfg.sub_mean; }
int glfer_gram_hop(const glfer_gram_plan *p) { return p->hop; }
int glfer_gram_bins(const glfer_gram_plan *p) { return p->bins; }
int glfer_gram_avg_cols(const glfer_gram_plan *p) { return p->avg_cols; }
long long glfer_gram_num_frames(const glfer_gram_plan *p, long long nsamples) { return nsamples / p->hop; }

static long long halo_frames(const glfer_gram_plan *p, long long first_frame)
{
  long long h = 0;
  if (p->cfg.mode == GLFER_MODE_LMP) h = p->cfg.lmp_av - 1;          /* the ring of lmp.c:86-93 */
  else if (p->cfg.avg_mode != GLFER_NO_AVG) h = p->cfg.avg_depth - 1;
  return h < first_frame ? h : first_frame;
}

void glfer_gram_required_span(const glfer_gram_plan *p, long long first_frame, long long nframes,
                              long long *lo, long long *hi)
{
  const long long f0 = first_frame - halo_frames(p, first_frame);
  long long l = f0 * p->hop - (p->cfg.n - p->hop);
  if (p->cfg.sub_mean && l > 0) l = (l / p->hop) * p->hop;   /* whole blocks for the block means */
  *lo = l;
  *hi = (first_frame + nframes) * (long long) p->hop;
}

int glfer_gram_window(const glfer_gram_plan *p, float *w)
{
  memcpy(w, p->h_window, sizeof(float) * p->cfg.n);
  return 0;
}

int glfer_gram_tapers(const glfer_gram_plan *p, double *tapers, double *lambda)
{
  if (p->cfg.mode != GLFER_MODE_MTM) return fail(GLFER_EINVAL, "plan is not a multitaper plan");
  memcpy(tapers, p->h_tapers, sizeof(double) * (size_t) p->ntapers * p->cfg.n);
  memcpy(lambda, p->h_lambda, sizeof(double) * p->ntapers);
  return 0;
}

void glfer_gram_plan_destroy(glfer_gram_plan *p)
{
  if (!p) return;
  glb_set_device(p->cfg.device);
  for (int i = 0; i < NSLOT; i++) {
    slot_t *s = &p->slot[i];
    if (s->stream) glb_stream_sync(s->stream);
    glb_free(s->d_samples); glb_free(s->d_pcm); glb_free(s->d_means); glb_free(s->d_psd); glb_free(s->d_avg);
    glb_free(s->d_ret); glb_free(s->d_var); glb_free(s->d_cand); glb_free(s->d_peak); glb_free(s->d_unres);
    glb_event_destroy(s->ev0); glb_event_destroy(s->ev1); glb_event_destroy(s->ev2); glb_event_destroy(s->ev3);
    glb_display_slot_free(&s->disp);
    glb_stream_destroy(s->stream);
  }
  glb_free(p->d_tapers);
  glb_free(p->d_ftapers); glb_free(p->d_u0); glb_free(p->d_fspec); glb_free(p->d_ftest);
  glb_free(p->d_cand_all);
  glb_free(p->d_peak_all);
  glb_display_free(&p->disp);
  glb_tables_destroy(p->tables);
  if (p->h_scal) glb_host_free(p->h_scal);
  free(p->h_window); free(p->h_tapers); free(p->h_lambda);
  free(p);
}

int glfer_gram_plan_create(const glfer_gram_config *cfg, glfer_gram_plan **out)
{
  g_msg[0] = 0;
  if (!cfg || !out) return fail(GLFER_EINVAL, "null argument");
  *out = NULL;
  if (!glb_fft_supported(cfg->n)) return fail(GLFER_EINVAL, "FFT size must be a power of two in 32..32768");
  if (cfg->mode != GLFER_MODE_FFT && cfg->mode != GLFER_MODE_MTM && cfg->mode != GLFER_MODE_LMP)
    return fail(GLFER_EINVAL, "unknown mode");
  if (cfg->mode == GLFER_MODE_LMP) {
    if (cfg->lmp_av < 2) return fail(GLFER_EINVAL, "lmp_av must be >= 2 (lmp.c:145 divides by lmp_av - 1)");
    if (cfg->avg_mode != GLFER_NO_AVG) return fail(GLFER_EINVAL, "frame averaging is not available in LMP mode");
  }
  const int hop = glb_hop(cfg->n, cfg->overlap);
  if (hop < 1 || hop > cfg->n) return fail(GLFER_EINVAL, "overlap leaves no new samples per block");
  if (cfg->mode == GLFER_MODE_MTM && (cfg->mtm_kmax < 0 || cfg->mtm_kmax > 31))
    return fail(GLFER_EINVAL, "mtm_kmax must be in 0..31 (32 eigenvectors exist)");
  if (cfg->avg_mode != GLFER_NO_AVG) {
    if (cfg->avg_mode < 1 || cfg->avg_mode > 3) return fail(GLFER_EINVAL, "unknown avg_mode");
    if (cfg->avg_depth < 1) return fail(GLFER_EINVAL, "avg_depth < 1");
    if (cfg->avg_minbin < 0 || cfg->avg_maxbin < cfg->avg_minbin || cfg->avg_maxbin > cfg->n / 2 + 1)
      return fail(GLFER_EINVAL, "averaging band outside [0, n/2+1]");
  }
  int ndev = 0;
  if (glb_device_count(&ndev) != GLB_OK || ndev < 1)
    return fail(GLFER_ENODEV, "no CUDA device (libglfer_b200 has no CPU fallback)");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(GLFER_EINVAL, "device ordinal out of range");
  TRY(glb_set_device(cfg->device));

  glfer_gram_plan *p = calloc(1, sizeof *p);
  if (!p) return fail(GLFER_ENOMEM, "out of memory");
  p->cfg = *cfg;
  p->hop = hop;
  p->bins = cfg->n / 2 + 1;
  p->avg_cols = (cfg->avg_mode != GLFER_NO_AVG && cfg->avg_band_only) ? cfg->avg_maxbin - cfg->avg_minbin : p->bins;
  if (p->avg_cols < 1) p->avg_cols = 1;
  const int n = cfg->n;
  p->taper_scale = (float) (1.0 / (2.0 * sqrt((double) n)));
  p->h_window = malloc(sizeof(float) * n);
  float *scaled = NULL;
  int rc = 0;
  if (cfg->mode == GLFER_MODE_LMP) p->cfg.window_type = RECTANGULAR_WINDOW;     /* source.c:395 */
  if (cfg->mode == GLFER_MODE_FFT || cfg->mode == GLFER_MODE_LMP) {
    p->ntapers = 1;
    glb_window_table(n, p->cfg.window_type, p->h_window);
    scaled = malloc(sizeof(float) * n);
    for (int i = 0; i < n; i++) {
      /* a rectangular window is NOT applied by the reference (fft.c:146-148): weight 1 */
      const double w = (p->cfg.window_type == RECTANGULAR_WINDOW) ? 1.0 : (double) p->h_window[i];
      scaled[i] = (float) (w * (double) p->taper_scale);
    }
  } else {
    p->ntapers = cfg->mtm_kmax + 1;
    glb_window_table(n, RECTANGULAR_WINDOW, p->h_window);
    p->h_tapers = malloc(sizeof(double) * (size_t) p->ntapers * n);
    p->h_lambda = malloc(sizeof(double) * p->ntapers);
    /* mtm_params_t.w is a float (mtm.h:42) promoted to double (mtm.c:68) */
    if (glb_dpss(n, (double) cfg->mtm_w, cfg->mtm_kmax, p->h_tapers, p->h_lambda) != 0) {
      glfer_gram_plan_destroy(p);
      return fail(GLFER_EINVAL, "DPSS computation failed");
    }
    if (cfg->mtm_ftest) {
      /* mtm_init, mtm.c:78-84,123-136: U0 in double, sum_U0_sqr and hn through float accumulators */
      const int K = p->ntapers;
      double *u0 = malloc(sizeof(double) * K);
      float *ft = malloc(sizeof(float) * (size_t) (K + 1) * n);
      float s2 = 0.0f;
      glb_mtm_ftest_weights(n, K, p->h_tapers, u0, ft, &s2);
      for (int i = 0; i < n; i++) {
        ft[i] = (float) ((double) ft[i] * (double) p->taper_scale);
        for (int k = 0; k < K; k++) ft[(size_t) (k + 1) * n + i] = (float) (p->h_tapers[(size_t) k * n + i] * (double) p->taper_scale);
      }
      p->sum_u0_sqr = (double) s2;
      rc = shim(glb_malloc((void **) &p->d_ftapers, sizeof(float) * (size_t) (K + 1) * n));
      if (rc == 0) rc = shim(glb_memcpy_h2d(p->d_ftapers, ft, sizeof(float) * (size_t) (K + 1) * n, NULL));
      if (rc == 0) rc = shim(glb_malloc((void **) &p->d_u0, sizeof(double) * K));
      if (rc == 0) rc = shim(glb_memcpy_h2d(p->d_u0, u0, sizeof(double) * K, NULL));
      free(u0); free(ft);
      if (rc != 0) { glfer_gram_plan_destroy(p); return rc; }
    }
    scaled = malloc(sizeof(float) * (size_t) p->ntapers * n);
    for (int k = 0; k < p->ntapers; k++) {
      if (!(p->h_lambda[k] > 0.0)) {
        free(scaled);
        glfer_gram_plan_destroy(p);
        return fail(GLFER_EINVAL, "DPSS eigenvalue not positive: reduce mtm_kmax or raise mtm_w");
      }
      const double g = (double) p->taper_scale / sqrt(p->h_lambda[k]);
      for (int i = 0; i < n; i++) scaled[(size_t) k * n + i] = (float) (p->h_tapers[(size_t) k * n + i] * g);
    }
  }
  p->taper_sym = 0;
  if (p->ntapers == 1) {
    /* every window of fft.c:37-82 comes out mirror-symmetric bit for bit; checked, not assumed */
    p->taper_sym = 1;
    for (int i = 0; i < n / 2; i++)
      if (memcmp(&scaled[i], &scaled[n - 1 - i], sizeof(float)) != 0) { p->taper_sym = 0; break; }
  }
  rc = shim(glb_malloc((void **) &p->d_tapers, sizeof(float) * (size_t) p->ntapers * n));
  if (rc == 0) rc = shim(glb_memcpy_h2d(p->d_tapers, scaled, sizeof(float) * (size_t) p->ntapers * n, NULL));
  free(scaled);
  if (rc == 0) rc = shim(glb_tables_create(n, &p->tables));
  for (int i = 0; i < NSLOT && rc == 0; i++) {
    rc = shim(glb_stream_create(&p->slot[i].stream));
    if (rc == 0) rc = shim(glb_event_create(&p->slot[i].ev0));
    if (rc == 0) rc = shim(glb_event_create(&p->slot[i].ev1));
    if (rc == 0) rc = shim(glb_event_create(&p->slot[i].ev2));
    if (rc == 0) rc = shim(glb_event_create(&p->slot[i].ev3));
    if (rc == 0) rc = shim(glb_event_create(&p->slot[i].disp.ev_agc));
    if (rc == 0) rc = shim(glb_malloc((void **) &p->slot[i].d_unres, sizeof(int)));
  }
  if (rc != 0) {
    char keep[512];
    snprintf(keep, sizeof keep, "%s", g_msg);
    glfer_gram_plan_destroy(p);
    snprintf(g_msg, sizeof g_msg, "%s", keep);
    return rc;
  }
  *out = p;
  return GLFER_OK;
}

int glb_ensure(void **ptr, size_t *cap, size_t want, size_t elem)
{
  if (want <= *cap) return 0;
  if (*ptr) TRY(glb_free(*ptr));
  *ptr = NULL;
  *cap = 0;
  TRY(glb_malloc(ptr, want * elem));
  *cap = want;
  return 0;
}

static int stage_slot(glfer_gram_plan *p, slot_t *s, const float *samples, const short *pcm, long long origin,
                      long long count)
{
  if (count < 0) return fail(GLFER_EINVAL, "negative sample count");
  TRY(glb_ensure((void **) &s->d_samples, &s->samples_cap, (size_t) count + 2, sizeof(float)));
  if (pcm) {
    TRY(glb_ensure((void **) &s->d_pcm, &s->pcm_cap, (size_t) count, sizeof(short)));
    TRY(glb_memcpy_h2d(s->d_pcm, pcm, sizeof(short) * (size_t) count, s->stream));
    TRY(glb_launch_pcm16_to_float(s->d_pcm, s->d_samples, count, s->stream));
  } else {
    TRY(glb_memcpy_h2d(s->d_samples, samples, sizeof(float) * (size_t) count, s->stream));
  }
  s->s_origin = origin;
  s->s_count = count;
  (void) p;
  return 0;
}

/* queue the kernels of frames [first, first + nframes) on a slot */
static int exec_slot(glfer_gram_plan *p, slot_t *s, long long first, long long nframes, int *cand_out,
                     const fused_levels *fl)
{
  const glfer_gram_config *c = &p->cfg;
  /* frame averaging inside the spectrogram kernel: band-only rows, ring-kernel geometry, small band history.
     The kernel pre-rolls the depth - 1 frames before every group itself, so the launch covers exactly the
     requested frames (the staged samples still include the pre-roll of the first group). */
  const int fuse_avg = g_fused_avg && !fl && c->avg_mode != GLFER_NO_AVG && c->avg_band_only && c->mode == GLFER_MODE_FFT &&
                       c->a <= 0.0f && !c->limiter && !c->zero_history && (s->s_origin % 4) == 0 &&
                       glb_gram_fused_avg_ok(c->n, p->hop, c->avg_depth, c->avg_maxbin - c->avg_minbin);
  const long long halo = fuse_avg ? 0 : halo_frames(p, first);
  const long long f0 = first - halo, nf = nframes + halo;
  long long lo, hi;
  glfer_gram_required_span(p, first, nframes, &lo, &hi);
  if (lo < 0) lo = 0;
  if (lo < s->s_origin || hi > s->s_origin + s->s_count)
    return fail(GLFER_EINVAL, "staged samples do not cover the requested frames (see glfer_gram_required_span)");
  if (!fl) TRY(glb_ensure((void **) &s->d_psd, &s->psd_cap, (size_t) nf * p->bins, sizeof(float)));

  const float *d_means = NULL;
  long long means_first = 0;
  const int fused_mean = c->sub_mean && glb_gram_fused_mean_ok(c->n, p->hop);
  if (c->sub_mean && !fused_mean) {
    /* irregular hop: block means from a pre-pass over the staged samples */
    const long long b_lo = lo / p->hop, b_hi = first + nframes;      /* blocks [b_lo, b_hi) */
    TRY(glb_ensure((void **) &s->d_means, &s->means_cap, (size_t) (b_hi - b_lo), sizeof(float)));
    TRY(glb_launch_block_means(s->d_samples, s->s_origin, s->s_count, p->hop, b_lo, b_hi - b_lo, s->d_means, s->stream));
    d_means = s->d_means;
    means_first = b_lo;
  }
  glb_gram_args g;
  memset(&g, 0, sizeof g);
  g.n = c->n;
  g.hop = p->hop;
  g.samples = s->d_samples;
  g.origin = s->s_origin;
  g.count = s->s_count;
  g.tapers = p->d_tapers;
  g.ntapers = p->ntapers;
  g.taper_symmetric = p->taper_sym;
  g.block_means = d_means;
  g.means_first_block = means_first;
  g.fused_mean = fused_mean;
  /* RA9MB and the limiter never reach the spectrum in multitaper mode: mtm_do rebuilds
     inbuf_fft from inbuf_audio (mtm.c:190-192) */
  g.ra9mb_a = (c->mode == GLFER_MODE_FFT) ? c->a : 0.0f;
  g.limiter = (c->mode == GLFER_MODE_FFT) ? c->limiter : 0;
  g.zero_history = c->zero_history;
  g.taper_scale = p->taper_scale;
  g.first_frame = f0;
  g.nframes = nf;
  g.rows = fl ? NULL : s->d_psd;
  g.row_stride = p->bins;
  if (fl) {                           /* levels straight from the kernel's registers: no float rows at all */
    g.levels = s->disp.d_levels;
    g.levels_stride = p->bins;
    g.level_tables = p->disp.level_tables;
    g.levels_log = fl->log_scale;
    g.level_lut = p->disp.d_level_lut;
    g.level_min = fl->dmin;
    g.level_max = fl->dmax;
    g.level_thr = fl->thr;
  }
  g.rows_db = (c->avg_mode == GLFER_NO_AVG && c->mode != GLFER_MODE_LMP) ? c->scale_db : 0;   /* averaging / LMP need linear PSD */
  g.spectrum = NULL;
  g.tables = p->tables;
  glb_avg_args a;
  memset(&a, 0, sizeof a);
  if (c->avg_mode != GLFER_NO_AVG) {
    TRY(glb_ensure((void **) &s->d_avg, &s->avg_cap, (size_t) nframes * p->avg_cols, sizeof(float)));
    if ((size_t) nframes > s->scal_cap) {
      glb_free(s->d_ret); glb_free(s->d_var); glb_free(s->d_cand); glb_free(s->d_peak);
      s->d_ret = s->d_var = NULL; s->d_cand = s->d_peak = NULL; s->scal_cap = 0;
      TRY(glb_malloc((void **) &s->d_ret, sizeof(double) * (size_t) nframes));
      TRY(glb_malloc((void **) &s->d_var, sizeof(double) * (size_t) nframes));
      TRY(glb_malloc((void **) &s->d_cand, sizeof(int) * (size_t) nframes));
      TRY(glb_malloc((void **) &s->d_peak, sizeof(int) * (size_t) nframes));
      s->scal_cap = (size_t) nframes;
    }
    a.mode = c->avg_mode;
    a.depth = c->avg_depth;
    a.minbin = c->avg_minbin;
    a.maxbin = c->avg_maxbin;
    a.max0 = c->avg_max0;
    a.nbins = p->bins;
    a.psd = s->d_psd;
    a.psd_first_frame = f0;
    a.psd_stride = p->bins;
    a.first_frame = first;
    a.nframes = nframes;
    a.out_double = 0;
    a.avg_rows = s->d_avg;
    a.out_stride = p->avg_cols;
    a.band_only = c->avg_band_only;
    a.rows_db = c->scale_db;
    a.ret = s->d_ret;
    a.peak_cand = cand_out ? cand_out : s->d_cand;
    a.variance = s->d_var;
    a.peakbin_init = c->avg_peakbin_init;
    a.unresolved = s->d_unres;
    a.sequential = 0;
    if (fuse_avg || c->avg_mode == GLFER_AVG_SUMAVG) TRY(glb_memset(s->d_unres, 0, sizeof(int), s->stream));
  }
  if (fuse_avg) g.fused_avg = &a;
  if (s->time_gram) TRY(glb_event_record(s->ev2, s->stream));
  TRY(glb_launch_gram(&g, s->stream));
  if (s->time_gram) TRY(glb_event_record(s->ev3, s->stream));

  if (c->avg_mode != GLFER_NO_AVG) {
    if (fuse_avg) {
      if (c->avg_mode == GLFER_AVG_SUMAVG) {
        /* a frame without a *peakbin write needs the carried value for its variance (avg.c:279): rare; the
           chunk is then redone in two passes, in order */
        int unres = 0;
        TRY(glb_memcpy_d2h(&unres, s->d_unres, sizeof(int), s->stream));
        TRY(glb_stream_sync(s->stream));
        if (unres > 0) {
          const int keep = g_fused_avg;
          g_fused_avg = 0;
          const int rc2 = exec_slot(p, s, first, nframes, cand_out, NULL);
          g_fused_avg = keep;
          return rc2;
        }
      }
    } else if (c->avg_mode == GLFER_AVG_SUMAVG) {
      TRY(glb_launch_avg(&a, s->stream));
      int unres = 0;
      TRY(glb_memcpy_d2h(&unres, s->d_unres, sizeof(int), s->stream));
      TRY(glb_stream_sync(s->stream));
      if (unres > 0) {             /* a chunk began before any *peakbin write: walk in order */
        a.sequential = 1;
        TRY(glb_launch_avg(&a, s->stream));
      }
    } else {
      TRY(glb_launch_avg(&a, s->stream));
    }
    /* with cand_out the caller resolves the carried *peakbin once over the whole run */
    if (!cand_out) TRY(glb_launch_peak_carry(s->d_cand, s->d_peak, nframes, c->avg_peakbin_init, s->stream));
  }
  if (c->mode == GLFER_MODE_LMP) {
    /* the rows handed out are the detector statistic over the ring of the last lmp_av PSD rows */
    TRY(glb_ensure((void **) &s->d_avg, &s->avg_cap, (size_t) nframes * p->bins, sizeof(float)));
    TRY(glb_launch_lmp(s->d_psd, f0, p->bins, 0, p->bins, first, nframes, c->lmp_av, c->scale_db, s->d_avg, p->bins, s->stream));
  }
  s->out_first = first;
  s->out_nframes = nframes;
  s->out_halo = halo;
  return 0;
}

static int fetch_slot(glfer_gram_plan *p, slot_t *s, float *psd_rows, float *avg_rows, double *avg_ret,
                      int *avg_peakbin, double *avg_variance)
{
  const size_t nf = (size_t) s->out_nframes;
  if (psd_rows) {
    const float *src = (p->cfg.mode == GLFER_MODE_LMP) ? s->d_avg : s->d_psd + (size_t) s->out_halo * p->bins;
    TRY(glb_memcpy_d2h(psd_rows, src, sizeof(float) * nf * p->bins, s->stream));
  }
  if (p->cfg.avg_mode != GLFER_NO_AVG) {
    if (avg_rows) TRY(glb_memcpy_d2h(avg_rows, s->d_avg, sizeof(float) * nf * p->avg_cols, s->stream));
    if (avg_ret) TRY(glb_memcpy_d2h(avg_ret, s->d_ret, sizeof(double) * nf, s->stream));
    if (avg_peakbin) TRY(glb_memcpy_d2h(avg_peakbin, s->d_peak, sizeof(int) * nf, s->stream));
    if (avg_variance) TRY(glb_memcpy_d2h(avg_variance, s->d_var, sizeof(double) * nf, s->stream));
  }
  return 0;
}

/* ---------------------------------------------------------------- device-resident API */
int glfer_gram_stage(glfer_gram_plan *p, const float *samples, long long origin, long long count)
{
  g_msg[0] = 0;
  TRY(glb_set_device(p->cfg.device));
  return stage_slot(p, &p->slot[0], samples, NULL, origin, count);
}

int glfer_gram_stage_pcm16(glfer_gram_plan *p, const short *pcm, long long origin, long long count)
{
  g_msg[0] = 0;
  TRY(glb_set_device(p->cfg.device));
  return stage_slot(p, &p->slot[0], NULL, pcm, origin, count);
}

int glfer_gram_exec(glfer_gram_plan *p, long long first_frame, long long nframes, float *kernel_ms)
{
  g_msg[0] = 0;
  if (nframes < 0 || first_frame < 0) return fail(GLFER_EINVAL, "negative frame range");
  TRY(glb_set_device(p->cfg.device));
  slot_t *s = &p->slot[0];
  s->time_gram = kernel_ms != NULL;
  if (kernel_ms) TRY(glb_event_record(s->ev0, s->stream));
  int rc = exec_slot(p, s, first_frame, nframes, NULL, NULL);
  s->time_gram = 0;
  if (rc != 0) return rc;
  if (kernel_ms) {
    TRY(glb_event_record(s->ev1, s->stream));
    TRY(glb_event_sync(s->ev1));
    TRY(glb_event_elapsed_ms(s->ev0, s->ev1, kernel_ms));
  }
  return 0;
}

int glfer_gram_last_gram_ms(glfer_gram_plan *p, float *ms)
{
  TRY(glb_set_device(p->cfg.device));
  return shim(glb_event_elapsed_ms(p->slot[0].ev2, p->slot[0].ev3, ms));
}

int glfer_gram_sync(glfer_gram_plan *p)
{
  TRY(glb_set_device(p->cfg.device));
  for (int i = 0; i < NSLOT; i++) TRY(glb_stream_sync(p->slot[i].stream));
  return 0;
}

int glfer_gram_fetch(glfer_gram_plan *p, float *psd_rows, float *avg_rows, double *avg_ret, int *avg_peakbin,
                     double *avg_variance)
{
  g_msg[0] = 0;
  TRY(glb_set_device(p->cfg.device));
  int rc = fetch_slot(p, &p->slot[0], psd_rows, avg_rows, avg_ret, avg_peakbin, avg_variance);
  if (rc != 0) return rc;
  return shim(glb_stream_sync(p->slot[0].stream));
}

/* ---------------------------------------------------------------- harmonic F-test
 * One chunk: the complex spectrum of every frame under hn and under each taper (ntapers + 1 launches of the
 * general kernel with its spectrum output), then mtm.c:204-233 per bin.  Not a throughput path: the
 * reference itself computes the statistic only to discard it. */
static int ftest_slot(glfer_gram_plan *p, slot_t *s, long long first, long long nframes)
{
  const glfer_gram_config *c = &p->cfg;
  const size_t plane = (size_t) nframes * p->bins;
  TRY(glb_ensure((void **) &p->d_fspec, &p->fspec_cap, plane * 2 * (size_t) (p->ntapers + 1), sizeof(float)));
  TRY(glb_ensure((void **) &p->d_ftest, &p->ftest_cap, plane, sizeof(float)));
  long long lo, hi;
  glfer_gram_required_span(p, first, nframes, &lo, &hi);
  if (lo < 0) lo = 0;
  const float *d_means = NULL;
  long long means_first = 0;
  const int fused_mean = c->sub_mean && glb_gram_fused_mean_ok(c->n, p->hop);
  if (c->sub_mean && !fused_mean) {
    const long long b_lo = lo / p->hop, b_hi = first + nframes;
    TRY(glb_ensure((void **) &s->d_means, &s->means_cap, (size_t) (b_hi - b_lo), sizeof(float)));
    TRY(glb_launch_block_means(s->d_samples, s->s_origin, s->s_count, p->hop, b_lo, b_hi - b_lo, s->d_means, s->stream));
    d_means = s->d_means;
    means_first = b_lo;
  }
  for (int j = 0; j <= p->ntapers; j++) {
    glb_gram_args g;
    memset(&g, 0, sizeof g);
    g.n = c->n;
    g.hop = p->hop;
    g.samples = s->d_samples;
    g.origin = s->s_origin;
    g.count = s->s_count;
    g.tapers = p->d_ftapers + (size_t) j * c->n;
    g.ntapers = 1;
    g.block_means = d_means;
    g.means_first_block = means_first;
    g.fused_mean = fused_mean;
    g.zero_history = c->zero_history;
    g.taper_scale = p->taper_scale;
    g.first_frame = first;
    g.nframes = nframes;
    g.spectrum = p->d_fspec + (size_t) j * plane * 2;
    g.tables = p->tables;
    TRY(glb_launch_gram(&g, s->stream));
  }
  return shim(glb_launch_ftest(p->d_fspec, nframes, p->bins, c->n, p->ntapers, p->d_u0, p->sum_u0_sqr, p->d_ftest, p->bins, s->stream));
}

int glfer_gram_run_mtm_ftest(glfer_gram_plan *p, const float *samples, long long origin, long long count,
                             long long first_frame, long long nframes, float *psd_rows, float *ftest_rows)
{
  g_msg[0] = 0;
  if (!p || !samples) return fail(GLFER_EINVAL, "null argument");
  if (p->cfg.mode != GLFER_MODE_MTM || !p->d_ftapers) return fail(GLFER_EINVAL, "plan was not created as a multitaper plan with mtm_ftest = 1");
  if (nframes < 0 || first_frame < 0) return fail(GLFER_EINVAL, "negative frame range");
  if (nframes == 0) return 0;
  TRY(glb_set_device(p->cfg.device));
  long long lo, hi;
  glfer_gram_required_span(p, first_frame, nframes, &lo, &hi);
  if (lo < 0) lo = 0;
  if (lo < origin || hi > origin + count)
    return fail(GLFER_EINVAL, "samples do not cover the requested frames (see glfer_gram_required_span)");
  /* chunks bounded by the spectra they need: (ntapers + 1) complex rows per frame */
  long long cf = (256LL << 20) / ((long long) (p->ntapers + 1) * p->bins * 8);
  if (cf < 16) cf = 16;
  slot_t *s = &p->slot[0];
  long long done = 0;
  while (done < nframes) {
    const long long c0 = first_frame + done;
    const long long cn = (nframes - done < cf) ? nframes - done : cf;
    long long clo, chi;
    glfer_gram_required_span(p, c0, cn, &clo, &chi);
    if (clo < 0) clo = 0;
    TRY(stage_slot(p, s, samples + (clo - origin), NULL, clo, chi - clo));
    if (psd_rows) {
      TRY(exec_slot(p, s, c0, cn, NULL, NULL));
      TRY(fetch_slot(p, s, psd_rows + (size_t) done * p->bins, NULL, NULL, NULL, NULL));
    }
    if (ftest_rows) {
      TRY(ftest_slot(p, s, c0, cn));
      TRY(glb_memcpy_d2h(ftest_rows + (size_t) done * p->bins, p->d_ftest, sizeof(float) * (size_t) cn * p->bins, s->stream));
    }
    TRY(glb_stream_sync(s->stream));
    done += cn;
  }
  return 0;
}

/* ---------------------------------------------------------------- host-buffer API */
/* The small per-frame outputs (ret, variance, peakbin) are downloaded chunk by chunk.  Into the
   caller's arrays directly, each of those copies would block the host thread whenever the array is pageable
   -- and with it the chunk pipeline (measured: C2 end to end 48 ms instead of 28 ms per hour of signal) -- so
   they land in pinned staging owned by the plan and are handed over once at the end of the run. */
static int scal_staging(glfer_gram_plan *p, size_t bytes, void **out)
{
  if (bytes > p->h_scal_cap) {
    if (p->h_scal) glb_host_free(p->h_scal);
    p->h_scal = NULL; p->h_scal_cap = 0;
    const size_t cap = bytes + bytes / 2 + 4096;
    TRY(glb_host_alloc(&p->h_scal, cap));
    p->h_scal_cap = cap;
  }
  *out = p->h_scal;
  return 0;
}

static long long chunk_frames(const glfer_gram_plan *p)
{
  /* ~32 MiB of new samples per chunk: large enough to run the copy engines and the
     kernel at full rate, small enough that the slots overlap well */
  long long mib = 32;
  const char *e = getenv("GLFER_B200_CHUNK_MIB");            /* experiments */
  if (e && atoi(e) > 0) mib = atoi(e);
  long long f = (mib << 20) / ((long long) p->hop * 4);
  if (f < 64) f = 64;
  const long long min_avg = 16LL * p->cfg.avg_depth;
  if (p->cfg.avg_mode != GLFER_NO_AVG && f < min_avg) f = min_avg;
  return f;
}

/* (A ramp of chunk sizes at both ends of a run was tried and dropped: the download stream trails the upload
   stream by one full-size chunk whatever the sizes at the ends, so fill + drain stay one chunk = 0.7 of the
   15 ms an hour of signal takes; 32 MiB is where that balances the ~28 us each further chunk costs.) */
static int run_impl(glfer_gram_plan *p, const float *samples, const short *pcm, long long origin, long long count,
                    long long first_frame, long long nframes, float *psd_rows, float *avg_rows, double *avg_ret,
                    int *avg_peakbin, double *avg_variance)
{
  g_msg[0] = 0;
  if (nframes < 0 || first_frame < 0) return fail(GLFER_EINVAL, "negative frame range");
  if (nframes == 0) return 0;
  TRY(glb_set_device(p->cfg.device));
  long long lo, hi;
  glfer_gram_required_span(p, first_frame, nframes, &lo, &hi);
  if (lo < 0) lo = 0;
  if (lo < origin || hi > origin + count)
    return fail(GLFER_EINVAL, "samples do not cover the requested frames (see glfer_gram_required_span)");
  const long long cf = chunk_frames(p);
  const int avg_on = p->cfg.avg_mode != GLFER_NO_AVG;
  /* *peakbin is carried from frame to frame (avg.c:129-133).  SUMAVG needs the carried
     value inside the kernel (variance excludes it, avg.c:279), so its chunks hand the
     value over serially; the other modes collect per-frame candidates for the whole run
     and resolve the carry once at the end, keeping the slots fully overlapped. */
  const int serial_carry = avg_on && p->cfg.avg_mode == GLFER_AVG_SUMAVG;
  const int defer_carry = avg_on && !serial_carry;
  if (defer_carry) {
    if ((size_t) nframes > p->cand_all_cap) {
      glb_free(p->d_cand_all); glb_free(p->d_peak_all);
      p->d_cand_all = p->d_peak_all = NULL; p->cand_all_cap = 0;
      TRY(glb_malloc((void **) &p->d_cand_all, sizeof(int) * (size_t) nframes));
      TRY(glb_malloc((void **) &p->d_peak_all, sizeof(int) * (size_t) nframes));
      p->cand_all_cap = (size_t) nframes;
    }
  }
  int carried_peak = p->cfg.avg_peakbin_init;
  const int saved_init = p->cfg.avg_peakbin_init;
  int rc = 0;
  double *st_ret = NULL, *st_var = NULL;
  int *st_pk = NULL;
  if (avg_on && (avg_ret || avg_variance || avg_peakbin)) {
    void *base = NULL;
    TRY(scal_staging(p, (size_t) nframes * (2 * sizeof(double) + sizeof(int)), &base));
    st_ret = (double *) base;
    st_var = st_ret + nframes;
    st_pk = (int *) (st_var + nframes);
  }
  long long done = 0;
  int ci = 0;
  /* chunk c runs on slot c % 2; before reusing a slot wait for its previous chunk */
  while (done < nframes && rc == 0) {
    slot_t *s = &p->slot[ci % NSLOT];
    const long long c0 = first_frame + done;
    const long long cn = (nframes - done < cf) ? nframes - done : cf;
    rc = shim(glb_stream_sync(s->stream));
    if (rc) break;
    if (serial_carry && ci > 0) {
      slot_t *prev = &p->slot[(ci - 1) % NSLOT];
      int last = 0;
      rc = shim(glb_memcpy_d2h(&last, prev->d_peak + (prev->out_nframes - 1), sizeof(int), prev->stream));
      if (rc == 0) rc = shim(glb_stream_sync(prev->stream));
      if (rc) break;
      carried_peak = last;
    }
    p->cfg.avg_peakbin_init = carried_peak;
    long long clo, chi;
    glfer_gram_required_span(p, c0, cn, &clo, &chi);
    if (clo < 0) clo = 0;
    rc = stage_slot(p, s, samples ? samples + (clo - origin) : NULL, pcm ? pcm + (clo - origin) : NULL, clo, chi - clo);
    if (rc) break;
    rc = exec_slot(p, s, c0, cn, defer_carry ? p->d_cand_all + done : NULL, NULL);
    if (rc) break;
    rc = fetch_slot(p, s, psd_rows ? psd_rows + (size_t) done * p->bins : NULL,
                    avg_rows ? avg_rows + (size_t) done * p->avg_cols : NULL, avg_ret ? st_ret + done : NULL,
                    (avg_peakbin && !defer_carry) ? st_pk + done : NULL,
                    avg_variance ? st_var + done : NULL);
    done += cn;
    ci++;
  }
  for (int i = 0; i < NSLOT; i++) {
    int r2 = shim(glb_stream_sync(p->slot[i].stream));
    if (rc == 0) rc = r2;
  }
  p->cfg.avg_peakbin_init = saved_init;
  if (rc == 0 && defer_carry && avg_peakbin) {
    void *st = p->slot[0].stream;
    rc = shim(glb_launch_peak_carry(p->d_cand_all, p->d_peak_all, nframes, saved_init, st));
    if (rc == 0) rc = shim(glb_memcpy_d2h(st_pk, p->d_peak_all, sizeof(int) * (size_t) nframes, st));
    if (rc == 0) rc = shim(glb_stream_sync(st));
  }
  if (rc == 0 && avg_on) {
    if (avg_ret) memcpy(avg_ret, st_ret, sizeof(double) * (size_t) nframes);
    if (avg_variance) memcpy(avg_variance, st_var, sizeof(double) * (size_t) nframes);
    if (avg_peakbin) memcpy(avg_peakbin, st_pk, sizeof(int) * (size_t) nframes);
  }
  return rc;
}

int glfer_gram_run(glfer_gram_plan *p, const float *samples, long long origin, long long count,
                   long long first_frame, long long nframes, float *psd_rows, float *avg_rows, double *avg_ret,
                   int *avg_peakbin, double *avg_variance)
{
  if (!p || !samples) return fail(GLFER_EINVAL, "null argument");
  return run_impl(p, samples, NULL, origin, count, first_frame, nframes, psd_rows, avg_rows, avg_ret, avg_peakbin,
                  avg_variance);
}

int glfer_gram_run_pcm16(glfer_gram_plan *p, const short *pcm, long long origin, long long count,
                         long long first_frame, long long nframes, float *psd_rows, float *avg_rows,
                         double *avg_ret, int *avg_peakbin, double *avg_variance)
{
  if (!p || !pcm) return fail(GLFER_EINVAL, "null argument");
  return run_impl(p, NULL, pcm, origin, count, first_frame, nframes, psd_rows, avg_rows, avg_ret, avg_peakbin,
                  avg_variance);
}

/* ---------------------------------------------------------------- display mapping
 * The tail of main_window_draw (g_main.c:1109-1229) for a whole run: the estimator's rows of each chunk go
 * through the display chain of host/display.c (floor statistics, AGC, levels / RGB), or, with a fixed range
 * and the estimator's own rows shown, the spectrogram kernel writes the levels itself.  Only 1 (levels) or
 * 3 (RGB) bytes per bin go back to the host. */
static int run_display_impl(glfer_gram_plan *p, const float *samples, const short *pcm, long long origin,
                            long long count, long long first_frame, long long nframes,
                            const glfer_display_config *dc, float *agc_state, unsigned char *levels,
                            unsigned char *rgb, float *range_out)
{
  g_msg[0] = 0;
  if (!dc) return fail(GLFER_EINVAL, "null display config");
  if (nframes < 0 || first_frame < 0) return fail(GLFER_EINVAL, "negative frame range");
  if (p->cfg.scale_db) return fail(GLFER_EINVAL, "display mapping needs linear rows (scale_db = 0)");
  if (rgb && !dc->colortab) return fail(GLFER_EINVAL, "RGB output needs a 256-entry palette");
  if (p->cfg.avg_mode != GLFER_NO_AVG && p->cfg.avg_band_only)
    return fail(GLFER_EINVAL, "the display shows whole averaged rows: plan must not be avg_band_only");
  if (dc->autoscale && first_frame > 0 && !agc_state)
    return fail(GLFER_EINVAL, "autoscale from frame > 0 needs the carried AGC state");
  if (nframes == 0) return 0;
  TRY(glb_set_device(p->cfg.device));
  long long lo, hi;
  glfer_gram_required_span(p, first_frame, nframes, &lo, &hi);
  if (lo < 0) lo = 0;
  if (lo < origin || hi > origin + count)
    return fail(GLFER_EINVAL, "samples do not cover the requested frames (see glfer_gram_required_span)");
  glb_display_run dr;
  TRY(glb_display_begin(&p->disp, &dr, dc, agc_state, nframes, 1, range_out != NULL, p->slot[0].stream));
  const long long cf = chunk_frames(p);
  const int avg_on = p->cfg.avg_mode != GLFER_NO_AVG;
  /* fixed display range, rows shown = the estimator's own rows: the spectrogram kernel writes the 8-bit
     levels itself and no float row ever reaches HBM (1 byte per bin instead of 4 + 4 + 1) */
  const int plain = p->cfg.mode != GLFER_MODE_FFT || (p->cfg.a <= 0.0f && !p->cfg.limiter);   /* RA9MB / limiter: two passes */
  const int fuse = g_fused_levels && !dc->autoscale && !avg_on && p->cfg.mode != GLFER_MODE_LMP && !rgb && plain;
  const fused_levels fl = { dc->log_scale, dr.fixed[1], dr.fixed[0], dr.thr };
  int rc = 0, ci = 0;
  long long done = 0;
  while (done < nframes && rc == 0) {
    slot_t *s = &p->slot[ci % NSLOT];
    const long long c0 = first_frame + done;
    const long long cn = (nframes - done < cf) ? nframes - done : cf;
    rc = shim(glb_stream_sync(s->stream));
    if (rc) break;
    long long clo, chi;
    glfer_gram_required_span(p, c0, cn, &clo, &chi);
    if (clo < 0) clo = 0;
    rc = stage_slot(p, s, samples ? samples + (clo - origin) : NULL, pcm ? pcm + (clo - origin) : NULL, clo, chi - clo);
    if (rc) break;
    rc = glb_display_reserve(&s->disp, cn, p->bins, rgb != NULL);
    if (rc) break;
    rc = exec_slot(p, s, c0, cn, NULL, fuse ? &fl : NULL);
    if (rc) break;
    if (!fuse) {
      /* psdbuf of the GUI: the estimator's output row, which in LMP mode is the statistic */
      const float *d_psd = (p->cfg.mode == GLFER_MODE_LMP) ? s->d_avg : s->d_psd + (size_t) s->out_halo * p->bins;
      const float *d_shown = avg_on ? s->d_avg : d_psd;               /* g_main.c:1192-1201 */
      rc = glb_display_map(&p->disp, &dr, &s->disp, ci > 0 ? &p->slot[(ci - 1) % NSLOT].disp : NULL, d_psd, d_shown,
                           p->bins, c0, cn, cn, done, p->cfg.overlap, rgb != NULL, s->stream);
      if (rc) break;
    }
    rc = glb_display_fetch(&dr, &s->disp, cn, cn, p->bins, done, levels, rgb, s->stream);
    done += cn;
    ci++;
  }
  for (int i = 0; i < NSLOT; i++) {
    int r2 = shim(glb_stream_sync(p->slot[i].stream));
    if (rc == 0) rc = r2;
  }
  if (rc == 0) rc = glb_display_end(&p->disp, &dr, nframes, agc_state, range_out);
  return rc;
}

int glfer_gram_run_display(glfer_gram_plan *p, const float *samples, long long origin, long long count,
                           long long first_frame, long long nframes, const glfer_display_config *dc,
                           float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range)
{
  if (!p || !samples) return fail(GLFER_EINVAL, "null argument");
  return run_display_impl(p, samples, NULL, origin, count, first_frame, nframes, dc, agc_state, levels, rgb, display_range);
}

int glfer_gram_run_display_pcm16(glfer_gram_plan *p, const short *pcm, long long origin, long long count,
                                 long long first_frame, long long nframes, const glfer_display_config *dc,
                                 float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range)
{
  if (!p || !pcm) return fail(GLFER_EINVAL, "null argument");
  return run_display_impl(p, NULL, pcm, origin, count, first_frame, nframes, dc, agc_state, levels, rgb, display_range);
}

int glfer_b200_map_levels(const float *rows, long long nrows, int nbins, const glfer_display_config *dc,
                          const float *range, unsigned char *levels, int device)
{
  g_msg[0] = 0;
  if (!rows || !dc || !levels || nrows < 0 || nbins < 1) return fail(GLFER_EINVAL, "bad arguments");
  if (nrows == 0) return 0;
  int ndev = 0;
  if (glb_device_count(&ndev) != GLB_OK || ndev < 1) return fail(GLFER_ENODEV, "no CUDA device (libglfer_b200 has no CPU fallback)");
  TRY(glb_set_device(device));
  void *tables = NULL, *d_rows = NULL, *d_lev = NULL, *d_range = NULL, *d_lut = NULL;
  const size_t cells = (size_t) nrows * nbins;
  const float thr = dc->thr_level / 100.0;
  float fixed[2] = { 0.0f, 0.0f };
  int rc = glb_make_level_tables(&tables);
  if (rc == 0) rc = shim(glb_malloc(&d_rows, sizeof(float) * cells));
  if (rc == 0) rc = shim(glb_malloc(&d_lev, cells));
  if (rc == 0) rc = shim(glb_memcpy_h2d(d_rows, rows, sizeof(float) * cells, NULL));
  if (rc == 0 && range) {
    rc = shim(glb_malloc(&d_range, sizeof(float) * 2 * (size_t) nrows));
    if (rc == 0) rc = shim(glb_memcpy_h2d(d_range, range, sizeof(float) * 2 * (size_t) nrows, NULL));
  } else if (rc == 0) {
    unsigned char lut[GLB_DB_NTHR];
    glb_fixed_display_range(dc->max_level_db, dc->min_level_db, dc->log_scale, &fixed[0], &fixed[1]);
    glb_level_lut(fixed[1], fixed[0], thr, lut);
    rc = shim(glb_malloc(&d_lut, sizeof lut));
    if (rc == 0) rc = shim(glb_memcpy_h2d(d_lut, lut, sizeof lut, NULL));
  }
  if (rc == 0) rc = shim(glb_launch_levels(d_rows, nbins, nbins, nrows, d_range, range ? NULL : fixed, dc->log_scale, thr,
                                           tables, d_lut, NULL, d_lev, NULL, NULL));
  if (rc == 0) rc = shim(glb_memcpy_d2h(levels, d_lev, cells, NULL));
  glb_free(d_rows); glb_free(d_lev); glb_free(d_range); glb_free(d_lut);
  glb_level_tables_destroy(tables);
  return rc;
}

/* ---------------------------------------------------------------- time sharding */
void glfer_gram_shard_range(long long nframes, int ndev, int g, long long *first, long long *count)
{
  /* contiguous, as even as possible: the first (nframes % ndev) shards get one extra frame */
  const long long base = nframes / ndev, extra = nframes % ndev;
  *first = g * base + (g < extra ? g : extra);
  *count = base + (g < extra ? 1 : 0);
}

typedef struct {
  glfer_gram_config cfg;
  const float *samples;
  long long nsamples, first, count;
  float *psd_rows, *avg_rows;
  double *avg_ret, *avg_variance;
  int *avg_peakbin;
  int bins;
  int rc;
  char msg[512];
} shard_job;

static void *shard_main(void *arg)
{
  shard_job *j = arg;
  glfer_gram_plan *p = NULL;
  j->rc = glfer_gram_plan_create(&j->cfg, &p);
  if (j->rc == 0) {
    const size_t off = (size_t) j->first * j->bins, aoff = (size_t) j->first * p->avg_cols;
    j->rc = glfer_gram_run(p, j->samples, 0, j->nsamples, j->first, j->count, j->psd_rows ? j->psd_rows + off : NULL,
                           j->avg_rows ? j->avg_rows + aoff : NULL, j->avg_ret ? j->avg_ret + j->first : NULL,
                           j->avg_peakbin ? j->avg_peakbin + j->first : NULL,
                           j->avg_variance ? j->avg_variance + j->first : NULL);
  }
  if (j->rc != 0) snprintf(j->msg, sizeof j->msg, "%s", glfer_b200_last_error());
  glfer_gram_plan_destroy(p);
  return NULL;
}

int glfer_gram_run_sharded(const glfer_gram_config *cfg, int ndev, const int *devices, const float *samples,
                           long long nsamples, float *psd_rows, float *avg_rows, double *avg_ret, int *avg_peakbin,
                           double *avg_variance)
{
  g_msg[0] = 0;
  if (!cfg || !samples || ndev < 1 || ndev > 64) return fail(GLFER_EINVAL, "bad arguments");
  const int hop = glb_hop(cfg->n, cfg->overlap);
  if (hop < 1) return fail(GLFER_EINVAL, "overlap leaves no new samples per block");
  const long long nframes = nsamples / hop;
  shard_job jobs[64];
  pthread_t th[64];
  int started[64];
  for (int g = 0; g < ndev; g++) {
    shard_job *j = &jobs[g];
    memset(j, 0, sizeof *j);
    j->cfg = *cfg;
    j->cfg.device = devices ? devices[g] : g;
    if (g > 0) j->cfg.avg_peakbin_init = -1;
    j->samples = samples;
    j->nsamples = nsamples;
    glfer_gram_shard_range(nframes, ndev, g, &j->first, &j->count);
    j->psd_rows = psd_rows; j->avg_rows = avg_rows; j->avg_ret = avg_ret;
    j->avg_peakbin = avg_peakbin; j->avg_variance = avg_variance;
    j->bins = cfg->n / 2 + 1;
    started[g] = pthread_create(&th[g], NULL, shard_main, j) == 0;
    if (!started[g]) {
      j->rc = GLFER_ENOMEM;
      snprintf(j->msg, sizeof j->msg, "pthread_create failed");
    }
  }
  int rc = 0;
  for (int g = 0; g < ndev; g++) {
    if (started[g]) pthread_join(th[g], NULL);
    if (jobs[g].rc != 0 && rc == 0) {
      rc = jobs[g].rc;
      snprintf(g_msg, sizeof g_msg, "shard %d: %s", g, jobs[g].msg);
    }
  }
  /* the carried *peakbin (avg.c:129-133) is the one sequential dependency between shards:
     shards g > 0 ran with the sentinel -1 as their initial value, so leading frames that
     never wrote *peakbin are recognisable and inherit the previous shard's last value */
  if (rc == 0 && avg_peakbin && cfg->avg_mode != GLFER_NO_AVG) {
    for (int g = 1; g < ndev && rc == 0; g++) {
      const long long f0 = jobs[g].first, f1 = f0 + jobs[g].count;
      long long k = 0;
      while (f0 + k < f1 && avg_peakbin[f0 + k] < 0) k++;
      if (k == 0) continue;
      const int carried = (f0 > 0) ? avg_peakbin[f0 - 1] : cfg->avg_peakbin_init;
      for (long long f = f0; f < f0 + k; f++) avg_peakbin[f] = carried;
      /* SUMAVG: the variance of those frames excluded the sentinel instead of the carried bin
         (avg.c:279): recompute them with the true value */
      if (cfg->avg_mode == GLFER_AVG_SUMAVG && avg_variance) {
        glfer_gram_config c2 = *cfg;
        c2.device = devices ? devices[g] : g;
        c2.avg_peakbin_init = carried;
        glfer_gram_plan *p2 = NULL;
        rc = glfer_gram_plan_create(&c2, &p2);
        if (rc == 0) rc = glfer_gram_run(p2, samples, 0, nsamples, f0, k, NULL, NULL, NULL, NULL, avg_variance + f0);
        glfer_gram_plan_destroy(p2);
      }
    }
  }
  return rc;
}
