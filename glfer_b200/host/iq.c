/* iq.c -- I/Q spectrogram plans: two-sided rows of complex (SDR baseband) recordings (include/glfer_b200.h).
 *
 * The frames of an interleaved (I, Q) stream are complex FFT frames of n samples; one shim entry,
 * glb_launch_iq_gram (csrc/iq.cu), computes their rows on whichever path serves the geometry (the fused ring
 * kernel, or the general kernel followed by the zoom's split).  This file only moves data: a run walks the frames
 * in chunks of ~32 MiB of input on ISLOT streams, each chunk uploads its complex samples (the n - hop samples it
 * shares with the previous chunk again), converts int16 input to float on the device, computes its rows and copies
 * them back while the next chunk uploads.  Device memory is bounded by the chunk, not by the recording.
 *
 * The display entries (glfer_iq_run_display*) bring back 8-bit levels instead of rows.  With a fixed range and no
 * RGB the spectrogram kernel maps its own powers (glb_iq_gram_args.levels) and no float row is ever stored;
 * otherwise each chunk's rows stay on the device and go through the display chain of host/display.c.
 *
 * Multitaper plans (glfer_iq_plan_create_mtm, and the zoom's) upload K' DPSS tapers, [K'][2n] floats, each scaled as
 * the real multitaper plan scales its own (host/gram.c); the row sums the K' eigen-spectra.  They always bring float
 * rows to the device: their waterfall goes through the display chain, for a fixed range too.  They also upload the
 * harmonic F-test's hn taper and U0 values (glb_iq_ftest_table), n + K' values: every multitaper plan serves
 * glfer_iq_run_mtm_ftest, whose chunks bring back F rows beside or instead of the rows.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include "glb_host.h"

#define ISLOT 3

#define ITRY(x) do { int rc_ = glb_host_shim(x); if (rc_ != 0) return rc_; } while (0)

typedef struct {
  void *stream;
  short *d_pcm;               /* int16 input of the chunk */
  size_t pcm_cap;             /* shorts */
  float *d_in;                /* interleaved (I, Q) floats of the chunk */
  size_t in_cap;              /* floats */
  float *d_rows;
  size_t rows_cap;            /* floats */
  float *d_ftest;             /* F rows (glfer_iq_run_mtm_ftest) */
  size_t ftest_cap;           /* floats */
  void *d_scratch;
  size_t scratch_cap;         /* bytes */
  glb_display_slot disp;      /* display mapping */
} islot;

struct glfer_iq_plan {
  glfer_iq_config cfg;
  int hop;
  float *d_taper;             /* [ntapers][2n]: w[i] (or v_k[i] / sqrt(lambda_k)) on both halves of complex sample i,
                                 times taper_scale */
  int taper_sym;              /* bit k: taper k is mirror-symmetric bit for bit */
  float taper_scale;
  int ntapers;                /* 1: periodogram, K' = mtm_kmax + 1: multitaper */
  double *h_tapers, *h_lambda;  /* multitaper: the unscaled DPSS [K'][n] and eigenvalues (glfer_iq_tapers) */
  float *d_ftab;              /* multitaper: the F-test's table (glb_iq_ftest_table): hn [2n], then (U0_k, sqrt(lambda_k)) */
  float ftest_s;              /* S = sum_k U0_k^2 */
  void *tables;               /* FFT tables of the 2n-float frames */
  islot slot[ISLOT];
  glb_display disp;
};

void glfer_iq_config_default(glfer_iq_config *c)
{
  memset(c, 0, sizeof *c);
  c->n = 4096;
  c->window_type = HANNING_WINDOW;
  c->overlap = 0.5f;
  c->device = 0;
}

int glfer_iq_hop(const glfer_iq_plan *p) { return p->hop; }
int glfer_iq_bins(const glfer_iq_plan *p) { return p->cfg.n; }

long long glfer_iq_num_frames(const glfer_iq_plan *p, long long nsamples)
{
  return nsamples <= 0 ? 0 : nsamples / p->hop;
}

void glfer_iq_required_span(const glfer_iq_plan *p, long long first_frame, long long nframes, long long *lo,
                            long long *hi)
{
  *lo = first_frame * p->hop - (p->cfg.n - p->hop);
  *hi = (first_frame + nframes) * p->hop;
}

void glfer_iq_plan_destroy(glfer_iq_plan *p)
{
  if (!p) return;
  glb_set_device(p->cfg.device);
  for (int i = 0; i < ISLOT; i++) {
    islot *s = &p->slot[i];
    if (s->stream) glb_stream_sync(s->stream);
    glb_free(s->d_pcm); glb_free(s->d_in); glb_free(s->d_rows); glb_free(s->d_ftest); glb_free(s->d_scratch);
    glb_display_slot_free(&s->disp);
    glb_stream_destroy(s->stream);
  }
  glb_display_free(&p->disp);
  glb_free(p->d_taper);
  glb_free(p->d_ftab);
  glb_tables_destroy(p->tables);
  free(p->h_tapers); free(p->h_lambda);
  free(p);
}

/* The DPSS of a complex multitaper plan (I/Q or zoom) and its taper table, built as host/gram.c builds the real
 * plan's: h_tapers [K'][n] and h_lambda [K'] from glb_dpss, table [K'][2n] floats with
 * v_k[i] taper_scale / sqrt(lambda_k) on both floats of complex sample i, sym: bit k when taper k reads the same
 * backwards bit for bit.  Validation as glfer_gram_plan_create; needs no device. */
int glb_iq_mtm_tapers(int n, float mtm_w, int mtm_kmax, float taper_scale, double **h_tapers, double **h_lambda,
                      float **table, int *sym)
{
  *h_tapers = NULL; *h_lambda = NULL; *table = NULL; *sym = 0;
  if (mtm_kmax < 0 || mtm_kmax > 31) return glb_host_fail(GLFER_EINVAL, "mtm_kmax must be in 0..31 (32 eigenvectors exist)");
  if (!(mtm_w > 0.0f)) return glb_host_fail(GLFER_EINVAL, "mtm_w must be > 0");
  const int K = mtm_kmax + 1;
  double *tap = malloc(sizeof(double) * (size_t) K * n);
  double *lam = malloc(sizeof(double) * K);
  float *tab = malloc(sizeof(float) * (size_t) K * 2 * n);
  if (!tap || !lam || !tab) { free(tap); free(lam); free(tab); return glb_host_fail(GLFER_ENOMEM, "out of memory"); }
  /* the real plan's call: mtm_params_t.w is a float promoted to double */
  if (glb_dpss(n, (double) mtm_w, mtm_kmax, tap, lam) != 0) {
    free(tap); free(lam); free(tab);
    return glb_host_fail(GLFER_EINVAL, "DPSS computation failed");
  }
  for (int k = 0; k < K; k++) {
    if (!(lam[k] > 0.0)) {
      free(tap); free(lam); free(tab);
      return glb_host_fail(GLFER_EINVAL, "DPSS eigenvalue not positive: reduce mtm_kmax or raise mtm_w");
    }
    const double g = (double) taper_scale / sqrt(lam[k]);
    float *t = tab + (size_t) k * 2 * n;
    for (int i = 0; i < n; i++) t[2 * i] = t[2 * i + 1] = (float) (tap[(size_t) k * n + i] * g);
    int s = 1;
    for (int i = 0; i < n && s; i++)
      if (memcmp(&t[i], &t[2 * n - 1 - i], sizeof(float)) != 0) s = 0;
    *sym |= s << k;
  }
  *h_tapers = tap; *h_lambda = lam; *table = tab;
  return 0;
}

/* The harmonic F-test's table of a complex multitaper plan, uploaded to *d_ftab: hn (glb_mtm_ftest_weights, as the real
 * plan builds it) times taper_scale on both floats of complex sample i, [2n] floats, then the K' pairs
 * (U0_k, sqrt(lambda_k)) that undo the per-taper weight of the taper table in the residual (glb_iq_gram_args). */
int glb_iq_ftest_table(int n, int K, const double *h_tapers, const double *h_lambda, float taper_scale, float **d_ftab,
                       float *s)
{
  double *u0 = malloc(sizeof(double) * K);
  float *hn = malloc(sizeof(float) * n);
  float *tab = malloc(sizeof(float) * (2 * (size_t) n + 2 * (size_t) K));
  int rc = 0;
  if (!u0 || !hn || !tab) rc = glb_host_fail(GLFER_ENOMEM, "out of memory");
  if (rc == 0) {
    glb_mtm_ftest_weights(n, K, h_tapers, u0, hn, s);
    for (int i = 0; i < n; i++) tab[2 * i] = tab[2 * i + 1] = (float) ((double) hn[i] * (double) taper_scale);
    for (int k = 0; k < K; k++) {
      tab[2 * n + 2 * k] = (float) u0[k];
      tab[2 * n + 2 * k + 1] = (float) sqrt(h_lambda[k]);
    }
    const size_t bytes = sizeof(float) * (2 * (size_t) n + 2 * (size_t) K);
    rc = glb_host_shim(glb_malloc((void **) d_ftab, bytes));
    if (rc == 0) rc = glb_host_shim(glb_memcpy_h2d(*d_ftab, tab, bytes, NULL));
  }
  free(u0); free(hn); free(tab);
  return rc;
}

/* tab: NULL (periodogram: the window), or the multitaper table of glb_iq_mtm_tapers */
static int build_taper(glfer_iq_plan *p, const float *tab)
{
  const int n = p->cfg.n;
  float *w = malloc(sizeof(float) * n);
  float *taper = malloc(sizeof(float) * 2 * n);
  int rc = 0;
  if (!w || !taper) rc = glb_host_fail(GLFER_ENOMEM, "out of memory");
  if (rc == 0 && !tab) {
    /* as the zoom (host/zoom.c): the window on both floats of a complex sample, times 1 / (2 sqrt(2n)) */
    glb_window_table(n, p->cfg.window_type, w);
    for (int i = 0; i < n; i++) {
      const double wi = p->cfg.window_type == RECTANGULAR_WINDOW ? 1.0 : (double) w[i];
      taper[2 * i] = taper[2 * i + 1] = (float) (wi * (double) p->taper_scale);
    }
    p->taper_sym = 1;
    for (int i = 0; i < n; i++)
      if (memcmp(&taper[i], &taper[2 * n - 1 - i], sizeof(float)) != 0) { p->taper_sym = 0; break; }
    tab = taper;
  }
  const size_t bytes = sizeof(float) * 2 * (size_t) n * p->ntapers;
  if (rc == 0) rc = glb_host_shim(glb_malloc((void **) &p->d_taper, bytes));
  if (rc == 0) rc = glb_host_shim(glb_memcpy_h2d(p->d_taper, tab, bytes, NULL));
  if (rc == 0) rc = glb_host_shim(glb_tables_create(2 * n, &p->tables));
  free(w); free(taper);
  return rc;
}

static int iq_plan_create(const glfer_iq_config *cfg, int mtm, float mtm_w, int mtm_kmax, glfer_iq_plan **out)
{
  glb_host_clear_error();
  if (!cfg || !out) return glb_host_fail(GLFER_EINVAL, "null argument");
  *out = NULL;
  if (cfg->n < 32 || cfg->n > 16384 || (cfg->n & (cfg->n - 1)) != 0)
    return glb_host_fail(GLFER_EINVAL, "I/Q FFT size must be a power of two in 32..16384");
  if (cfg->window_type < 0 || cfg->window_type > 7) return glb_host_fail(GLFER_EINVAL, "unknown window type");
  const int hop = glb_hop(cfg->n, cfg->overlap);
  if (hop < 1 || hop > cfg->n) return glb_host_fail(GLFER_EINVAL, "overlap leaves no new samples per block");
  const float taper_scale = (float) (1.0 / (2.0 * sqrt(2.0 * cfg->n)));
  double *h_tapers = NULL, *h_lambda = NULL;
  float *tab = NULL;
  int sym = 0;
  if (mtm) {
    const int rc = glb_iq_mtm_tapers(cfg->n, mtm_w, mtm_kmax, taper_scale, &h_tapers, &h_lambda, &tab, &sym);
    if (rc != 0) return rc;
  }
  int ndev = 0;
  int rc = 0;
  if (glb_device_count(&ndev) != GLB_OK || ndev < 1)
    rc = glb_host_fail(GLFER_ENODEV, "no CUDA device (libglfer_b200 has no CPU fallback)");
  else if (cfg->device < 0 || cfg->device >= ndev)
    rc = glb_host_fail(GLFER_EINVAL, "device ordinal out of range");
  else
    rc = glb_host_shim(glb_set_device(cfg->device));
  glfer_iq_plan *p = rc == 0 ? calloc(1, sizeof *p) : NULL;
  if (rc == 0 && !p) rc = glb_host_fail(GLFER_ENOMEM, "out of memory");
  if (rc != 0) {
    free(h_tapers); free(h_lambda); free(tab);
    return rc;
  }
  p->cfg = *cfg;
  p->hop = hop;
  p->taper_scale = taper_scale;
  p->ntapers = mtm ? mtm_kmax + 1 : 1;
  p->h_tapers = h_tapers;
  p->h_lambda = h_lambda;
  p->taper_sym = sym;
  rc = build_taper(p, tab);
  free(tab);
  if (rc == 0 && mtm)
    rc = glb_iq_ftest_table(cfg->n, p->ntapers, h_tapers, h_lambda, taper_scale, &p->d_ftab, &p->ftest_s);
  for (int i = 0; i < ISLOT && rc == 0; i++) {
    rc = glb_host_shim(glb_stream_create(&p->slot[i].stream));
    if (rc == 0) rc = glb_host_shim(glb_event_create(&p->slot[i].disp.ev_agc));
  }
  if (rc != 0) {
    char keep[512];
    strncpy(keep, glfer_b200_last_error(), sizeof keep - 1);
    keep[sizeof keep - 1] = 0;
    glfer_iq_plan_destroy(p);
    glb_host_fail(rc, keep);
    return rc;
  }
  *out = p;
  return GLFER_OK;
}

int glfer_iq_plan_create(const glfer_iq_config *cfg, glfer_iq_plan **out)
{
  return iq_plan_create(cfg, 0, 0.0f, 0, out);
}

int glfer_iq_plan_create_mtm(const glfer_iq_config *cfg, float mtm_w, int mtm_kmax, glfer_iq_plan **out)
{
  return iq_plan_create(cfg, 1, mtm_w, mtm_kmax, out);
}

int glfer_iq_tapers(const glfer_iq_plan *p, double *tapers, double *lambda)
{
  if (!p || !tapers || !lambda) return glb_host_fail(GLFER_EINVAL, "null argument");
  if (!p->h_tapers) return glb_host_fail(GLFER_EINVAL, "plan is not a multitaper plan");
  memcpy(tapers, p->h_tapers, sizeof(double) * (size_t) p->ntapers * p->cfg.n);
  memcpy(lambda, p->h_lambda, sizeof(double) * p->ntapers);
  return 0;
}

/* grow-only device buffers */
static int iensure(void **ptr, size_t *cap, size_t want, size_t elem)
{
  if (want <= *cap) return 0;
  if (*ptr) ITRY(glb_free(*ptr));
  *ptr = NULL;
  *cap = 0;
  ITRY(glb_malloc(ptr, want * elem));
  *cap = want;
  return 0;
}

static long long iq_chunk_frames(const glfer_iq_plan *p)
{
  /* ~32 MiB of new float input per chunk, as the spectrogram's and the zoom's pipelines; at least one frame */
  const long long f = (32LL << 20) / ((long long) p->hop * 8);
  return f < 1 ? 1 : f;
}

/* frames [c0, c0 + cn) on slot s: with fl the fixed-range levels into s->disp.d_levels, otherwise rows into s->d_rows
 * (rows_on) and F rows into s->d_ftest (ftest_on) */
static int iq_chunk(glfer_iq_plan *p, islot *s, const void *src, int pcm16, long long origin, long long c0,
                    long long cn, const glb_display_run *fl, int rows_on, int ftest_on)
{
  const long long n = p->cfg.n, hop = p->hop;
  long long lo = c0 * hop - (n - hop);
  const long long hi = (c0 + cn) * hop;
  if (lo < 0) lo = 0;
  /* the fused kernel reads whole hop blocks with 16-byte bulk copies: stage from an even complex index when the
     caller's samples reach that far back (the regular hops are even, so lo already is) */
  if ((lo & 1) && lo - 1 >= origin) lo--;
  const long long cnt = hi - lo;
  ITRY(iensure((void **) &s->d_in, &s->in_cap, (size_t) (2 * cnt), sizeof(float)));
  if (pcm16) {
    ITRY(iensure((void **) &s->d_pcm, &s->pcm_cap, (size_t) (2 * cnt), sizeof(short)));
    ITRY(glb_memcpy_h2d(s->d_pcm, (const short *) src + 2 * (lo - origin), sizeof(short) * 2 * (size_t) cnt, s->stream));
    ITRY(glb_launch_pcm16_to_float(s->d_pcm, s->d_in, 2 * cnt, s->stream));
  } else {
    ITRY(glb_memcpy_h2d(s->d_in, (const float *) src + 2 * (lo - origin), sizeof(float) * 2 * (size_t) cnt, s->stream));
  }
  if (!fl && rows_on) ITRY(iensure((void **) &s->d_rows, &s->rows_cap, (size_t) (cn * n), sizeof(float)));
  if (ftest_on) ITRY(iensure((void **) &s->d_ftest, &s->ftest_cap, (size_t) (cn * n), sizeof(float)));
  const long long sb = glb_iq_gram_scratch_bytes((int) n, (int) hop, cn, fl != NULL, p->ntapers, ftest_on);
  if (sb > 0) ITRY(iensure(&s->d_scratch, &s->scratch_cap, (size_t) sb, 1));
  glb_iq_gram_args g;
  memset(&g, 0, sizeof g);
  g.n = (int) n;
  g.hop = (int) hop;
  g.samples = s->d_in;
  g.origin = lo;
  g.count = cnt;
  g.taper = p->d_taper;
  g.taper_symmetric = p->taper_sym;
  g.taper_scale = p->taper_scale;
  g.ntapers = p->ntapers;
  g.first_frame = c0;
  g.nframes = cn;
  g.rows = (fl || !rows_on) ? NULL : s->d_rows;
  g.tables = p->tables;
  g.scratch = sb > 0 ? s->d_scratch : NULL;
  if (fl) {
    g.levels = s->disp.d_levels;
    g.levels_stride = n;
    g.level_tables = p->disp.level_tables;
    g.levels_log = fl->dc->log_scale;
    g.level_lut = p->disp.d_level_lut;
    g.level_min = fl->fixed[1];
    g.level_max = fl->fixed[0];
    g.level_thr = fl->thr;
  }
  if (ftest_on) {
    g.ftest = s->d_ftest;
    g.ftest_taper = p->d_ftab;
    g.ftest_u0 = p->d_ftab + 2 * n;
    g.ftest_s = p->ftest_s;
  }
  ITRY(glb_launch_iq_gram(&g, s->stream));
  return 0;
}

/* rows and/or F rows (ftest_on: glfer_iq_run_mtm_ftest; rows or ftest may then be NULL) */
static int iq_run_impl(glfer_iq_plan *p, const void *src, int pcm16, long long origin, long long count,
                       long long first_frame, long long nframes, float *rows, int ftest_on, float *ftest)
{
  glb_host_clear_error();
  if (!p || !src || (!ftest_on && !rows)) return glb_host_fail(GLFER_EINVAL, "null argument");
  if (ftest_on) {
    if (!p->h_tapers) return glb_host_fail(GLFER_EINVAL, "the F-test needs a multitaper plan (glfer_iq_plan_create_mtm)");
    if (p->ntapers < 2) return glb_host_fail(GLFER_EINVAL, "the F-test needs mtm_kmax >= 1 (K' - 1 degrees of freedom)");
    if (!rows && !ftest) return glb_host_fail(GLFER_EINVAL, "null argument: rows and ftest are both NULL");
  }
  if (nframes < 0 || first_frame < 0) return glb_host_fail(GLFER_EINVAL, "negative frame range");
  if (origin < 0 || count < 0) return glb_host_fail(GLFER_EINVAL, "negative origin or sample count");
  if (nframes == 0) return 0;
  ITRY(glb_set_device(p->cfg.device));
  long long lo, hi;
  glfer_iq_required_span(p, first_frame, nframes, &lo, &hi);
  if (lo < 0) lo = 0;
  if (lo < origin || hi > origin + count)
    return glb_host_fail(GLFER_EINVAL, "samples do not cover the requested frames (see glfer_iq_required_span)");
  const long long cf = iq_chunk_frames(p);
  int rc = 0, ci = 0;
  long long done = 0;
  while (done < nframes && rc == 0) {
    islot *s = &p->slot[ci % ISLOT];
    const long long cn = (nframes - done < cf) ? nframes - done : cf;
    rc = glb_host_shim(glb_stream_sync(s->stream));
    if (rc) break;
    rc = iq_chunk(p, s, src, pcm16, origin, first_frame + done, cn, NULL, rows != NULL, ftest != NULL);
    if (rc == 0 && rows)
      rc = glb_host_shim(glb_memcpy_d2h(rows + (size_t) done * p->cfg.n, s->d_rows, sizeof(float) * (size_t) (cn * p->cfg.n),
                                        s->stream));
    if (rc == 0 && ftest)
      rc = glb_host_shim(glb_memcpy_d2h(ftest + (size_t) done * p->cfg.n, s->d_ftest,
                                        sizeof(float) * (size_t) (cn * p->cfg.n), s->stream));
    done += cn;
    ci++;
  }
  for (int i = 0; i < ISLOT; i++) {
    const int r2 = glb_host_shim(glb_stream_sync(p->slot[i].stream));
    if (rc == 0) rc = r2;
  }
  return rc;
}

int glfer_iq_run(glfer_iq_plan *p, const float *iq, long long origin, long long count, long long first_frame,
                 long long nframes, float *rows)
{
  return iq_run_impl(p, iq, 0, origin, count, first_frame, nframes, rows, 0, NULL);
}

int glfer_iq_run_pcm16(glfer_iq_plan *p, const short *iq, long long origin, long long count, long long first_frame,
                       long long nframes, float *rows)
{
  return iq_run_impl(p, iq, 1, origin, count, first_frame, nframes, rows, 0, NULL);
}

int glfer_iq_run_mtm_ftest(glfer_iq_plan *p, const float *iq, long long origin, long long count, long long first_frame,
                           long long nframes, float *rows, float *ftest)
{
  return iq_run_impl(p, iq, 0, origin, count, first_frame, nframes, rows, 1, ftest);
}

int glfer_iq_run_mtm_ftest_pcm16(glfer_iq_plan *p, const short *iq, long long origin, long long count,
                                 long long first_frame, long long nframes, float *rows, float *ftest)
{
  return iq_run_impl(p, iq, 1, origin, count, first_frame, nframes, rows, 1, ftest);
}

/* main_window_draw's mapping of the plan's own rows (include/glfer_b200.h, glfer_iq_run_display) */
static int iq_run_display_impl(glfer_iq_plan *p, const void *src, int pcm16, long long origin, long long count,
                               long long first_frame, long long nframes, const glfer_display_config *dc,
                               float *agc_state, unsigned char *levels, unsigned char *rgb, float *range_out)
{
  glb_host_clear_error();
  if (!p || !src || !dc) return glb_host_fail(GLFER_EINVAL, "null argument");
  if (nframes < 0 || first_frame < 0) return glb_host_fail(GLFER_EINVAL, "negative frame range");
  if (origin < 0 || count < 0) return glb_host_fail(GLFER_EINVAL, "negative origin or sample count");
  if (rgb && !dc->colortab) return glb_host_fail(GLFER_EINVAL, "RGB output needs a 256-entry palette");
  if (dc->autoscale && first_frame > 0 && !agc_state)
    return glb_host_fail(GLFER_EINVAL, "autoscale from frame > 0 needs the carried AGC state");
  if (nframes == 0) return 0;
  ITRY(glb_set_device(p->cfg.device));
  long long lo, hi;
  glfer_iq_required_span(p, first_frame, nframes, &lo, &hi);
  if (lo < 0) lo = 0;
  if (lo < origin || hi > origin + count)
    return glb_host_fail(GLFER_EINVAL, "samples do not cover the requested frames (see glfer_iq_required_span)");
  const int n = p->cfg.n;
  glb_display_run dr;
  ITRY(glb_display_begin(&p->disp, &dr, dc, agc_state, nframes, range_out != NULL, p->slot[0].stream));
  /* fixed range without RGB: the spectrogram kernel writes the levels itself (periodogram plans only) */
  const int fuse = glb_host_fused_levels() && !dc->autoscale && !rgb && p->ntapers == 1;
  const long long cf = iq_chunk_frames(p);
  int rc = 0, ci = 0;
  long long done = 0;
  while (done < nframes && rc == 0) {
    islot *s = &p->slot[ci % ISLOT];
    const long long c0 = first_frame + done;
    const long long cn = (nframes - done < cf) ? nframes - done : cf;
    rc = glb_host_shim(glb_stream_sync(s->stream));
    if (rc == 0) rc = glb_display_reserve(&s->disp, cn, n, rgb != NULL);
    if (rc == 0) rc = iq_chunk(p, s, src, pcm16, origin, c0, cn, fuse ? &dr : NULL, !fuse, 0);
    if (rc == 0 && !fuse)
      rc = glb_display_map(&p->disp, &dr, &s->disp, ci > 0 ? &p->slot[(ci - 1) % ISLOT].disp : NULL, s->d_rows, s->d_rows,
                           n, c0, cn, done, p->cfg.overlap, rgb != NULL, s->stream);
    if (rc == 0) rc = glb_display_fetch(&s->disp, cn, n, done, levels, rgb, s->stream);
    done += cn;
    ci++;
  }
  for (int i = 0; i < ISLOT; i++) {
    const int r2 = glb_host_shim(glb_stream_sync(p->slot[i].stream));
    if (rc == 0) rc = r2;
  }
  if (rc == 0) rc = glb_display_end(&p->disp, &dr, nframes, agc_state, range_out);
  return rc;
}

int glfer_iq_run_display(glfer_iq_plan *p, const float *iq, long long origin, long long count, long long first_frame,
                         long long nframes, const glfer_display_config *dc, float *agc_state, unsigned char *levels,
                         unsigned char *rgb, float *display_range)
{
  return iq_run_display_impl(p, iq, 0, origin, count, first_frame, nframes, dc, agc_state, levels, rgb, display_range);
}

int glfer_iq_run_display_pcm16(glfer_iq_plan *p, const short *iq, long long origin, long long count,
                               long long first_frame, long long nframes, const glfer_display_config *dc,
                               float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range)
{
  return iq_run_display_impl(p, iq, 1, origin, count, first_frame, nframes, dc, agc_state, levels, rgb, display_range);
}
