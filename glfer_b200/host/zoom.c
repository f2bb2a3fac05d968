/* zoom.c -- zoom spectrogram plans: sub-hertz bins around a chosen frequency (include/glfer_b200.h).
 *
 * Mix to DC, low-pass and decimate by D on the device (zoom_decim_kernel, csrc/zoom.cu), then complex FFT
 * frames of the decimated stream.  The frame stage reuses the general spectrogram kernel: the decimated
 * stream seen as interleaved floats is a real stream of 2n points per frame at hop 2 hop, its taper is the
 * window duplicated over (re, im) of each complex sample, and its `spectrum` output X[k], k = 0..n, is
 * turned into the complex FFT rows by zoom_split_kernel.
 *
 * A run walks the frames in chunks of ~32 MiB of input on ZSLOT streams.  Each chunk uploads only the input
 * of its new decimated samples (plus the 2K-sample filter halo) and takes the n - hop decimated samples its
 * first frame shares with the previous chunk from that chunk's buffer, device to device: every input sample
 * crosses PCIe once, and device memory is bounded by the chunk, not by the recording.
 *
 * I/Q plans (glfer_zoom_plan_create_iq) take complex input, interleaved (I, Q), through the complex decimator
 * (glb_launch_zoom_decim_iq) and accept a signed centre; everything after the decimator is the same.
 *
 * The display entries (glfer_zoom_run_display*) keep each chunk's rows on the device and map them through the
 * display chain of host/display.c: only the 8-bit levels (or RGB) come back.
 *
 * Multitaper plans (glfer_zoom_plan_create_mtm / _create_iq_mtm) replace the window by K' DPSS tapers
 * (glb_iq_mtm_tapers, host/iq.c); the frame stage then runs one spectrum per taper into the same scratch plane.
 * They also hold the harmonic F-test's table (glb_iq_ftest_table): glfer_zoom_run[_iq]_mtm_ftest add the hn spectrum
 * and the mu and den planes to that scratch and bring back F rows beside or instead of the rows.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include "glb_host.h"

#define ZSLOT 3

#define ZTRY(x) do { int rc_ = glb_host_shim(x); if (rc_ != 0) return rc_; } while (0)

typedef struct {
  void *stream, *ev_dec;      /* ev_dec: this chunk's decimated samples are written */
  void *d_in;                 /* input span of the chunk (float or int16) */
  size_t in_cap;              /* bytes */
  float *d_y;                 /* y[m], m in [y_base, y_end), as (re, im) pairs */
  size_t y_cap;               /* complex samples */
  long long y_base, y_end;
  float *d_spec;              /* [frames][n + 1] (re, im) pairs */
  size_t spec_cap;            /* floats */
  float *d_rows;
  size_t rows_cap;            /* floats */
  float *d_ftest;             /* F rows (glfer_zoom_run[_iq]_mtm_ftest) */
  size_t ftest_cap;           /* floats */
  glb_display_slot disp;      /* display mapping */
} zslot;

struct glfer_zoom_plan {
  glfer_zoom_config cfg;
  int hop, K;
  unsigned step;
  float *d_taps;              /* [33 D] (re, im) pairs: g[j] = h[K - j] e^{+2 pi i phi(K - j)}, zero past 2K */
  float *d_taper;             /* [ntapers][2n]: w[i] (or v_k[i] / sqrt(lambda_k)) on both halves of complex sample i,
                                 times taper_scale */
  int taper_sym;              /* bit k: taper k is mirror-symmetric bit for bit */
  float taper_scale;
  int ntapers;                /* 1: periodogram, K' = mtm_kmax + 1: multitaper */
  double *h_tapers, *h_lambda;  /* multitaper: the unscaled DPSS [K'][n] and eigenvalues (glfer_zoom_tapers) */
  float *d_ftab;              /* multitaper: the F-test's table (glb_iq_ftest_table): hn [2n], then (U0_k, sqrt(lambda_k)) */
  float ftest_s;              /* S = sum_k U0_k^2 */
  int iq;                     /* 1: complex (I, Q) input (glfer_zoom_plan_create_iq), signed centre */
  void *tables;               /* FFT tables of the 2n-point real transform */
  zslot slot[ZSLOT];
  glb_display disp;
};

/* I0 by its power series, in double (converges quickly for the beta of the design) */
static double bessel_i0_series(double x)
{
  const double q = 0.25 * x * x;
  double s = 1.0, t = 1.0;
  for (int k = 1; k < 500; k++) {
    t *= q / ((double) k * (double) k);
    s += t;
    if (t < 1e-18 * s) break;
  }
  return s;
}

int glfer_zoom_taps(int decim, float *taps)
{
  if (decim < 2 || decim > 1024) return glb_host_fail(GLFER_EINVAL, "zoom decimation must be in 2..1024");
  if (!taps) return glb_host_fail(GLFER_EINVAL, "null argument");
  const int K = 16 * decim, L = 2 * K + 1;
  const double fc = 0.5 / decim, beta = 0.1102 * (100.0 - 8.7);
  double *h = malloc(sizeof(double) * L);
  if (!h) return glb_host_fail(GLFER_ENOMEM, "out of memory");
  const double i0b = bessel_i0_series(beta);
  for (int l = 0; l <= K; l++) {
    const double a = 2.0 * fc * l;
    const double sinc = l == 0 ? 1.0 : sin(M_PI * a) / (M_PI * a);
    const double r = (double) l / K;
    const double v = 2.0 * fc * sinc * bessel_i0_series(beta * sqrt(1.0 - r * r)) / i0b;
    h[K + l] = v;
    h[K - l] = v;
  }
  double sum = 0.0;
  for (int j = 0; j < L; j++) sum += h[j];
  for (int j = 0; j < L; j++) taps[j] = (float) (h[j] / sum);
  free(h);
  return 0;
}

void glfer_zoom_config_default(glfer_zoom_config *c)
{
  memset(c, 0, sizeof *c);
  c->n = 4096;
  c->decim = 256;
  c->window_type = HANNING_WINDOW;
  c->overlap = 0.0f;
  c->center_hz = 800.0;
  c->sample_rate = 48000.0;
  c->device = 0;
}

int glfer_zoom_hop(const glfer_zoom_plan *p) { return p->hop; }
int glfer_zoom_bins(const glfer_zoom_plan *p) { return p->cfg.n; }
double glfer_zoom_center_hz(const glfer_zoom_plan *p)
{
  /* an I/Q plan's step is a signed 32-bit fraction of a turn: centres below the dial are negative */
  const double s = p->iq ? (double) (int) p->step : (double) p->step;
  return s * p->cfg.sample_rate / 4294967296.0;
}

long long glfer_zoom_num_frames(const glfer_zoom_plan *p, long long nsamples)
{
  const long long last = nsamples - 1 - p->K;           /* m D <= last */
  const long long md = last < 0 ? 0 : last / p->cfg.decim + 1;
  return md / p->hop;
}

void glfer_zoom_required_span(const glfer_zoom_plan *p, long long first_frame, long long nframes, long long *lo,
                              long long *hi)
{
  const long long D = p->cfg.decim;
  const long long m_lo = first_frame * p->hop - (p->cfg.n - p->hop);
  const long long m_hi = (first_frame + nframes) * p->hop;        /* y[m_lo .. m_hi) */
  *lo = m_lo * D - p->K;
  *hi = (m_hi - 1) * D + p->K + 1;
}

void glfer_zoom_plan_destroy(glfer_zoom_plan *p)
{
  if (!p) return;
  glb_set_device(p->cfg.device);
  for (int i = 0; i < ZSLOT; i++) {
    zslot *s = &p->slot[i];
    if (s->stream) glb_stream_sync(s->stream);
    glb_free(s->d_in); glb_free(s->d_y); glb_free(s->d_spec); glb_free(s->d_rows); glb_free(s->d_ftest);
    glb_event_destroy(s->ev_dec);
    glb_display_slot_free(&s->disp);
    glb_stream_destroy(s->stream);
  }
  glb_display_free(&p->disp);
  glb_free(p->d_taps);
  glb_free(p->d_taper);
  glb_free(p->d_ftab);
  glb_tables_destroy(p->tables);
  free(p->h_tapers); free(p->h_lambda);
  free(p);
}

/* mtab: NULL (periodogram: the window), or the multitaper table of glb_iq_mtm_tapers */
static int build_tables(glfer_zoom_plan *p, const float *mtab)
{
  const glfer_zoom_config *c = &p->cfg;
  const int D = c->decim, K = p->K, n = c->n;
  float *h = malloc(sizeof(float) * (2 * K + 1));
  float *g = calloc((size_t) 66 * D, sizeof(float));
  float *w = malloc(sizeof(float) * n);
  float *taper = malloc(sizeof(float) * 2 * n);
  int rc = 0;
  if (!h || !g || !w || !taper) rc = glb_host_fail(GLFER_ENOMEM, "out of memory");
  if (rc == 0) rc = glfer_zoom_taps(D, h);
  if (rc == 0) {
    /* g[j] = h[K - j] e^{+2 pi i phi(K - j)}: h is symmetric, so h[K - j] is taps[j] */
    for (int j = 0; j <= 2 * K; j++) {
      const unsigned ph = (unsigned) ((long long) (K - j) * (long long) p->step);
      const double a = 2.0 * M_PI * (double) ph / 4294967296.0;
      g[2 * j] = (float) ((double) h[j] * cos(a));
      g[2 * j + 1] = (float) ((double) h[j] * sin(a));
    }
    if (!mtab) {
      glb_window_table(n, c->window_type, w);
      for (int i = 0; i < n; i++) {
        /* as the spectrogram: a rectangular window is not applied (weight 1) */
        const double wi = c->window_type == RECTANGULAR_WINDOW ? 1.0 : (double) w[i];
        taper[2 * i] = taper[2 * i + 1] = (float) (wi * (double) p->taper_scale);
      }
      p->taper_sym = 1;
      for (int i = 0; i < n; i++)
        if (memcmp(&taper[i], &taper[2 * n - 1 - i], sizeof(float)) != 0) { p->taper_sym = 0; break; }
      mtab = taper;
    }
    const size_t tbytes = sizeof(float) * 2 * (size_t) n * p->ntapers;
    rc = glb_host_shim(glb_malloc((void **) &p->d_taps, sizeof(float) * 66 * (size_t) D));
    if (rc == 0) rc = glb_host_shim(glb_memcpy_h2d(p->d_taps, g, sizeof(float) * 66 * (size_t) D, NULL));
    if (rc == 0) rc = glb_host_shim(glb_malloc((void **) &p->d_taper, tbytes));
    if (rc == 0) rc = glb_host_shim(glb_memcpy_h2d(p->d_taper, mtab, tbytes, NULL));
    if (rc == 0) rc = glb_host_shim(glb_tables_create(2 * n, &p->tables));
  }
  free(h); free(g); free(w); free(taper);
  return rc;
}

static int zoom_plan_create(const glfer_zoom_config *cfg, int iq, int mtm, float mtm_w, int mtm_kmax,
                            glfer_zoom_plan **out)
{
  glb_host_clear_error();
  if (!cfg || !out) return glb_host_fail(GLFER_EINVAL, "null argument");
  *out = NULL;
  if (cfg->n < 32 || cfg->n > 16384 || (cfg->n & (cfg->n - 1)) != 0)
    return glb_host_fail(GLFER_EINVAL, "zoom FFT size must be a power of two in 32..16384");
  if (cfg->decim < 2 || cfg->decim > 1024) return glb_host_fail(GLFER_EINVAL, "zoom decimation must be in 2..1024");
  if (cfg->window_type < 0 || cfg->window_type > 7) return glb_host_fail(GLFER_EINVAL, "unknown window type");
  const int hop = glb_hop(cfg->n, cfg->overlap);
  if (hop < 1 || hop > cfg->n) return glb_host_fail(GLFER_EINVAL, "overlap leaves no new samples per block");
  if (!(cfg->sample_rate > 0.0) || !isfinite(cfg->sample_rate)) return glb_host_fail(GLFER_EINVAL, "sample rate must be positive");
  if (!iq && !(cfg->center_hz >= 0.0 && cfg->center_hz <= 0.5 * cfg->sample_rate))
    return glb_host_fail(GLFER_EINVAL, "centre frequency must be in [0, sample_rate / 2]");
  if (iq && !(cfg->center_hz >= -0.5 * cfg->sample_rate && cfg->center_hz <= 0.5 * cfg->sample_rate))
    return glb_host_fail(GLFER_EINVAL, "I/Q centre frequency must be in [-sample_rate / 2, sample_rate / 2]");
  const float taper_scale = (float) (1.0 / (2.0 * sqrt(2.0 * cfg->n)));
  double *h_tapers = NULL, *h_lambda = NULL;
  float *mtab = NULL;
  int sym = 0;
  if (mtm) {
    const int rc = glb_iq_mtm_tapers(cfg->n, mtm_w, mtm_kmax, taper_scale, &h_tapers, &h_lambda, &mtab, &sym);
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
  glfer_zoom_plan *p = rc == 0 ? calloc(1, sizeof *p) : NULL;
  if (rc == 0 && !p) rc = glb_host_fail(GLFER_ENOMEM, "out of memory");
  if (rc != 0) {
    free(h_tapers); free(h_lambda); free(mtab);
    return rc;
  }
  p->cfg = *cfg;
  p->hop = hop;
  p->K = 16 * cfg->decim;
  p->iq = iq;
  /* modulo 2^32: a negative I/Q centre is a step above 2^31 */
  p->step = (unsigned) (unsigned long long) llround(cfg->center_hz / cfg->sample_rate * 4294967296.0);
  p->taper_scale = taper_scale;
  p->ntapers = mtm ? mtm_kmax + 1 : 1;
  p->h_tapers = h_tapers;
  p->h_lambda = h_lambda;
  p->taper_sym = sym;
  rc = build_tables(p, mtab);
  free(mtab);
  if (rc == 0 && mtm)
    rc = glb_iq_ftest_table(cfg->n, p->ntapers, h_tapers, h_lambda, taper_scale, &p->d_ftab, &p->ftest_s);
  for (int i = 0; i < ZSLOT && rc == 0; i++) {
    rc = glb_host_shim(glb_stream_create(&p->slot[i].stream));
    if (rc == 0) rc = glb_host_shim(glb_event_create(&p->slot[i].ev_dec));
    if (rc == 0) rc = glb_host_shim(glb_event_create(&p->slot[i].disp.ev_agc));
  }
  if (rc != 0) {
    char keep[512];
    strncpy(keep, glfer_b200_last_error(), sizeof keep - 1);
    keep[sizeof keep - 1] = 0;
    glfer_zoom_plan_destroy(p);
    glb_host_fail(rc, keep);
    return rc;
  }
  *out = p;
  return GLFER_OK;
}

int glfer_zoom_plan_create(const glfer_zoom_config *cfg, glfer_zoom_plan **out)
{
  return zoom_plan_create(cfg, 0, 0, 0.0f, 0, out);
}

int glfer_zoom_plan_create_iq(const glfer_zoom_config *cfg, glfer_zoom_plan **out)
{
  return zoom_plan_create(cfg, 1, 0, 0.0f, 0, out);
}

int glfer_zoom_plan_create_mtm(const glfer_zoom_config *cfg, float mtm_w, int mtm_kmax, glfer_zoom_plan **out)
{
  return zoom_plan_create(cfg, 0, 1, mtm_w, mtm_kmax, out);
}

int glfer_zoom_plan_create_iq_mtm(const glfer_zoom_config *cfg, float mtm_w, int mtm_kmax, glfer_zoom_plan **out)
{
  return zoom_plan_create(cfg, 1, 1, mtm_w, mtm_kmax, out);
}

int glfer_zoom_tapers(const glfer_zoom_plan *p, double *tapers, double *lambda)
{
  if (!p || !tapers || !lambda) return glb_host_fail(GLFER_EINVAL, "null argument");
  if (!p->h_tapers) return glb_host_fail(GLFER_EINVAL, "plan is not a multitaper plan");
  memcpy(tapers, p->h_tapers, sizeof(double) * (size_t) p->ntapers * p->cfg.n);
  memcpy(lambda, p->h_lambda, sizeof(double) * p->ntapers);
  return 0;
}

/* grow-only device buffers */
static int zensure(void **ptr, size_t *cap, size_t want, size_t elem)
{
  if (want <= *cap) return 0;
  if (*ptr) ZTRY(glb_free(*ptr));
  *ptr = NULL;
  *cap = 0;
  ZTRY(glb_malloc(ptr, want * elem));
  *cap = want;
  return 0;
}

static long long zoom_chunk_frames(const glfer_zoom_plan *p)
{
  /* ~32 MiB of new float input per chunk, as the spectrogram's pipeline; at least one frame */
  const long long per_frame = (long long) p->hop * p->cfg.decim * (p->iq ? 8 : 4);
  const long long f = (32LL << 20) / per_frame;
  return f < 1 ? 1 : f;
}

/* rows of frames [c0, c0 + cn) into s->d_rows (rows_on) and F rows into s->d_ftest (ftest_on); prev: the slot of the
 * previous chunk of this run, or NULL */
static int zoom_chunk(glfer_zoom_plan *p, zslot *s, const zslot *prev, const void *src, int pcm16,
                      long long origin, long long c0, long long cn, int rows_on, int ftest_on)
{
  const glfer_zoom_config *c = &p->cfg;
  const long long D = c->decim, n = c->n, hop = p->hop;
  const long long m_lo = c0 * hop - (n - hop), m_hi = (c0 + cn) * hop;
  long long base, from;                   /* y held from `base`; decimated here from `from` */
  if (prev) {
    base = m_lo > prev->y_base ? m_lo : prev->y_base;
    from = prev->y_end;
  } else {
    base = m_lo > 0 ? m_lo : 0;
    from = base;
  }
  ZTRY(zensure((void **) &s->d_y, &s->y_cap, (size_t) (m_hi - base), 2 * sizeof(float)));
  long long x_lo = from * D - p->K;
  const long long x_hi = (m_hi - 1) * D + p->K + 1;
  if (x_lo < 0) x_lo = 0;
  const size_t esz = (pcm16 ? sizeof(short) : sizeof(float)) * (p->iq ? 2 : 1);
  ZTRY(zensure(&s->d_in, &s->in_cap, (size_t) (x_hi - x_lo) * esz, 1));
  ZTRY(glb_memcpy_h2d(s->d_in, (const char *) src + (size_t) (x_lo - origin) * esz, (size_t) (x_hi - x_lo) * esz,
                      s->stream));
  if (from > base) {
    /* the history this chunk's first frame shares with the previous chunk */
    ZTRY(glb_stream_wait_event(s->stream, prev->ev_dec));
    ZTRY(glb_memcpy_d2d(s->d_y, prev->d_y + 2 * (base - prev->y_base), (size_t) (from - base) * 2 * sizeof(float),
                        s->stream));
  }
  if (p->iq)
    ZTRY(glb_launch_zoom_decim_iq(s->d_in, pcm16, x_lo, x_hi - x_lo, (int) D, p->d_taps,
                                  (unsigned) ((unsigned long long) D * p->step), from, m_hi - from,
                                  s->d_y + 2 * (from - base), s->stream));
  else
    ZTRY(glb_launch_zoom_decim(s->d_in, pcm16, x_lo, x_hi - x_lo, (int) D, p->d_taps,
                               (unsigned) ((unsigned long long) D * p->step), from, m_hi - from,
                               s->d_y + 2 * (from - base), s->stream));
  ZTRY(glb_event_record(s->ev_dec, s->stream));
  s->y_base = base;
  s->y_end = m_hi;

  /* the general path's scratch (glb_launch_iq_gram_general): the spectrum, and for the F-test the mu and den planes */
  ZTRY(zensure((void **) &s->d_spec, &s->spec_cap, (size_t) cn * ((n + 1) * 2 + (ftest_on ? 3 * n : 0)), sizeof(float)));
  if (rows_on) ZTRY(zensure((void **) &s->d_rows, &s->rows_cap, (size_t) cn * n, sizeof(float)));
  if (ftest_on) ZTRY(zensure((void **) &s->d_ftest, &s->ftest_cap, (size_t) cn * n, sizeof(float)));
  glb_iq_gram_args g;
  memset(&g, 0, sizeof g);
  g.n = (int) n;
  g.hop = (int) hop;
  g.samples = s->d_y;
  g.origin = base;
  g.count = m_hi - base;
  g.taper = p->d_taper;
  g.taper_symmetric = p->taper_sym;
  g.taper_scale = p->taper_scale;
  g.ntapers = p->ntapers;
  g.first_frame = c0;
  g.nframes = cn;
  g.rows = rows_on ? s->d_rows : NULL;
  g.tables = p->tables;
  g.scratch = s->d_spec;
  if (ftest_on) {
    g.ftest = s->d_ftest;
    g.ftest_taper = p->d_ftab;
    g.ftest_u0 = p->d_ftab + 2 * n;
    g.ftest_s = p->ftest_s;
  }
  ZTRY(glb_launch_iq_gram_general(&g, s->stream));
  return 0;
}

/* rows and/or F rows (ftest_on: glfer_zoom_run[_iq]_mtm_ftest; rows or ftest may then be NULL) */
static int zoom_run_impl(glfer_zoom_plan *p, int iq, const void *src, int pcm16, long long origin, long long count,
                         long long first_frame, long long nframes, float *rows, int ftest_on, float *ftest)
{
  glb_host_clear_error();
  if (!p || !src || (!ftest_on && !rows)) return glb_host_fail(GLFER_EINVAL, "null argument");
  if (iq != p->iq)
    return glb_host_fail(GLFER_EINVAL, iq ? "glfer_zoom_run_iq needs a plan from glfer_zoom_plan_create_iq"
                                          : "an I/Q zoom plan runs through glfer_zoom_run_iq / glfer_zoom_run_iq_pcm16");
  if (ftest_on) {
    if (!p->h_tapers) return glb_host_fail(GLFER_EINVAL, "the F-test needs a multitaper zoom plan");
    if (p->ntapers < 2) return glb_host_fail(GLFER_EINVAL, "the F-test needs mtm_kmax >= 1 (K' - 1 degrees of freedom)");
    if (!rows && !ftest) return glb_host_fail(GLFER_EINVAL, "null argument: rows and ftest are both NULL");
  }
  if (nframes < 0 || first_frame < 0) return glb_host_fail(GLFER_EINVAL, "negative frame range");
  if (origin < 0 || count < 0) return glb_host_fail(GLFER_EINVAL, "negative origin or sample count");
  if (nframes == 0) return 0;
  ZTRY(glb_set_device(p->cfg.device));
  long long lo, hi;
  glfer_zoom_required_span(p, first_frame, nframes, &lo, &hi);
  if (lo < 0) lo = 0;
  if (lo < origin || hi > origin + count)
    return glb_host_fail(GLFER_EINVAL, "samples do not cover the requested frames (see glfer_zoom_required_span)");
  const long long cf = zoom_chunk_frames(p);
  int rc = 0, ci = 0;
  long long done = 0;
  const zslot *prev = NULL;
  while (done < nframes && rc == 0) {
    zslot *s = &p->slot[ci % ZSLOT];
    const long long cn = (nframes - done < cf) ? nframes - done : cf;
    rc = glb_host_shim(glb_stream_sync(s->stream));
    if (rc) break;
    rc = zoom_chunk(p, s, prev, src, pcm16, origin, first_frame + done, cn, rows != NULL, ftest != NULL);
    if (rc == 0 && rows)
      rc = glb_host_shim(glb_memcpy_d2h(rows + (size_t) done * p->cfg.n, s->d_rows, sizeof(float) * (size_t) cn * p->cfg.n,
                                        s->stream));
    if (rc == 0 && ftest)
      rc = glb_host_shim(glb_memcpy_d2h(ftest + (size_t) done * p->cfg.n, s->d_ftest,
                                        sizeof(float) * (size_t) cn * p->cfg.n, s->stream));
    prev = s;
    done += cn;
    ci++;
  }
  for (int i = 0; i < ZSLOT; i++) {
    const int r2 = glb_host_shim(glb_stream_sync(p->slot[i].stream));
    if (rc == 0) rc = r2;
  }
  return rc;
}

int glfer_zoom_run(glfer_zoom_plan *p, const float *samples, long long origin, long long count,
                   long long first_frame, long long nframes, float *rows)
{
  return zoom_run_impl(p, 0, samples, 0, origin, count, first_frame, nframes, rows, 0, NULL);
}

int glfer_zoom_run_pcm16(glfer_zoom_plan *p, const short *pcm, long long origin, long long count,
                         long long first_frame, long long nframes, float *rows)
{
  return zoom_run_impl(p, 0, pcm, 1, origin, count, first_frame, nframes, rows, 0, NULL);
}

int glfer_zoom_run_iq(glfer_zoom_plan *p, const float *iq, long long origin, long long count,
                      long long first_frame, long long nframes, float *rows)
{
  return zoom_run_impl(p, 1, iq, 0, origin, count, first_frame, nframes, rows, 0, NULL);
}

int glfer_zoom_run_iq_pcm16(glfer_zoom_plan *p, const short *iq, long long origin, long long count,
                            long long first_frame, long long nframes, float *rows)
{
  return zoom_run_impl(p, 1, iq, 1, origin, count, first_frame, nframes, rows, 0, NULL);
}

int glfer_zoom_run_mtm_ftest(glfer_zoom_plan *p, const float *samples, long long origin, long long count,
                             long long first_frame, long long nframes, float *rows, float *ftest)
{
  return zoom_run_impl(p, 0, samples, 0, origin, count, first_frame, nframes, rows, 1, ftest);
}

int glfer_zoom_run_mtm_ftest_pcm16(glfer_zoom_plan *p, const short *pcm, long long origin, long long count,
                                   long long first_frame, long long nframes, float *rows, float *ftest)
{
  return zoom_run_impl(p, 0, pcm, 1, origin, count, first_frame, nframes, rows, 1, ftest);
}

int glfer_zoom_run_iq_mtm_ftest(glfer_zoom_plan *p, const float *iq, long long origin, long long count,
                                long long first_frame, long long nframes, float *rows, float *ftest)
{
  return zoom_run_impl(p, 1, iq, 0, origin, count, first_frame, nframes, rows, 1, ftest);
}

int glfer_zoom_run_iq_mtm_ftest_pcm16(glfer_zoom_plan *p, const short *iq, long long origin, long long count,
                                      long long first_frame, long long nframes, float *rows, float *ftest)
{
  return zoom_run_impl(p, 1, iq, 1, origin, count, first_frame, nframes, rows, 1, ftest);
}

/* main_window_draw's mapping of the plan's own rows (include/glfer_b200.h, glfer_zoom_run_display) */
static int zoom_run_display_impl(glfer_zoom_plan *p, int iq, const void *src, int pcm16, long long origin,
                                 long long count, long long first_frame, long long nframes,
                                 const glfer_display_config *dc, float *agc_state, unsigned char *levels,
                                 unsigned char *rgb, float *range_out)
{
  glb_host_clear_error();
  if (!p || !src || !dc) return glb_host_fail(GLFER_EINVAL, "null argument");
  if (iq != p->iq)
    return glb_host_fail(GLFER_EINVAL, iq ? "glfer_zoom_run_display_iq needs a plan from glfer_zoom_plan_create_iq"
                                          : "an I/Q zoom plan runs through glfer_zoom_run_display_iq / _iq_pcm16");
  if (nframes < 0 || first_frame < 0) return glb_host_fail(GLFER_EINVAL, "negative frame range");
  if (origin < 0 || count < 0) return glb_host_fail(GLFER_EINVAL, "negative origin or sample count");
  if (rgb && !dc->colortab) return glb_host_fail(GLFER_EINVAL, "RGB output needs a 256-entry palette");
  if (dc->autoscale && first_frame > 0 && !agc_state)
    return glb_host_fail(GLFER_EINVAL, "autoscale from frame > 0 needs the carried AGC state");
  if (nframes == 0) return 0;
  ZTRY(glb_set_device(p->cfg.device));
  long long lo, hi;
  glfer_zoom_required_span(p, first_frame, nframes, &lo, &hi);
  if (lo < 0) lo = 0;
  if (lo < origin || hi > origin + count)
    return glb_host_fail(GLFER_EINVAL, "samples do not cover the requested frames (see glfer_zoom_required_span)");
  const int n = p->cfg.n;
  glb_display_run dr;
  ZTRY(glb_display_begin(&p->disp, &dr, dc, agc_state, nframes, range_out != NULL, p->slot[0].stream));
  const long long cf = zoom_chunk_frames(p);
  int rc = 0, ci = 0;
  long long done = 0;
  const zslot *prev = NULL;
  while (done < nframes && rc == 0) {
    zslot *s = &p->slot[ci % ZSLOT];
    const long long c0 = first_frame + done;
    const long long cn = (nframes - done < cf) ? nframes - done : cf;
    rc = glb_host_shim(glb_stream_sync(s->stream));
    if (rc == 0) rc = glb_display_reserve(&s->disp, cn, n, rgb != NULL);
    if (rc == 0) rc = zoom_chunk(p, s, prev, src, pcm16, origin, c0, cn, 1, 0);
    if (rc == 0)
      rc = glb_display_map(&p->disp, &dr, &s->disp, prev ? &prev->disp : NULL, s->d_rows, s->d_rows, n, c0, cn, done,
                           p->cfg.overlap, rgb != NULL, s->stream);
    if (rc == 0) rc = glb_display_fetch(&s->disp, cn, n, done, levels, rgb, s->stream);
    prev = s;
    done += cn;
    ci++;
  }
  for (int i = 0; i < ZSLOT; i++) {
    const int r2 = glb_host_shim(glb_stream_sync(p->slot[i].stream));
    if (rc == 0) rc = r2;
  }
  if (rc == 0) rc = glb_display_end(&p->disp, &dr, nframes, agc_state, range_out);
  return rc;
}

int glfer_zoom_run_display(glfer_zoom_plan *p, const float *samples, long long origin, long long count,
                           long long first_frame, long long nframes, const glfer_display_config *dc,
                           float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range)
{
  return zoom_run_display_impl(p, 0, samples, 0, origin, count, first_frame, nframes, dc, agc_state, levels, rgb,
                               display_range);
}

int glfer_zoom_run_display_pcm16(glfer_zoom_plan *p, const short *pcm, long long origin, long long count,
                                 long long first_frame, long long nframes, const glfer_display_config *dc,
                                 float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range)
{
  return zoom_run_display_impl(p, 0, pcm, 1, origin, count, first_frame, nframes, dc, agc_state, levels, rgb,
                               display_range);
}

int glfer_zoom_run_display_iq(glfer_zoom_plan *p, const float *iq, long long origin, long long count,
                              long long first_frame, long long nframes, const glfer_display_config *dc,
                              float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range)
{
  return zoom_run_display_impl(p, 1, iq, 0, origin, count, first_frame, nframes, dc, agc_state, levels, rgb,
                               display_range);
}

int glfer_zoom_run_display_iq_pcm16(glfer_zoom_plan *p, const short *iq, long long origin, long long count,
                                    long long first_frame, long long nframes, const glfer_display_config *dc,
                                    float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range)
{
  return zoom_run_display_impl(p, 1, iq, 1, origin, count, first_frame, nframes, dc, agc_state, levels, rgb,
                               display_range);
}
