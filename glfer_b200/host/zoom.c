/* zoom.c -- zoom spectrogram plans: sub-hertz bins around a chosen frequency (include/glfer_b200.h).
 *
 * Mix to DC, low-pass and decimate by D on the device (zoom_decim_kernel, csrc/zoom.cu), then complex FFT
 * frames of the decimated stream.  The frame stage is the I/Q plans' (host/cframe.c) on its general path
 * (glb_launch_iq_gram_general): the decimated stream seen as interleaved floats is a real stream of 2n points per
 * frame at hop 2 hop, its taper is the window duplicated over (re, im) of each complex sample, and the general
 * spectrogram kernel's `spectrum` output X[k], k = 0..n, is turned into the complex FFT rows by zoom_split_kernel.
 *
 * A run walks the frames in chunks of ~32 MiB of input on the frame stage's slots.  Each chunk uploads only the input
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
 * Multitaper plans (glfer_zoom_plan_create_mtm / _create_iq_mtm) replace the window by K' DPSS tapers; the frame stage
 * then runs one spectrum per taper into the same scratch plane.  glfer_zoom_run[_iq]_mtm_ftest add the hn spectrum and
 * the mu and den planes to that scratch and bring back F rows beside or instead of the rows.
 *
 * Banks (glfer_zoom_plan_create_bank[_mtm]) hold C centres of one config.  Each chunk's input is uploaded once and the
 * bank decimator (glb_launch_zoom_bank_decim) writes every channel's decimated samples at the channel stride the frame
 * stage asks for; one frame stage launch then covers all channels.  A single-centre plan keeps zoom_decim_kernel.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include "glb_host.h"

typedef struct {
  glb_cslot cs;               /* stream, rows, F rows, scratch (the spectrum), display */
  void *ev_dec;               /* this chunk's decimated samples are written */
  void *d_in;                 /* input span of the chunk (float or int16) */
  size_t in_cap;              /* bytes */
  float *d_y;                 /* y[m], m in [y_base, y_end), as (re, im) pairs */
  size_t y_cap;               /* complex samples */
  long long y_base, y_end;
  long long y_stride;         /* complex samples between two channels' y[y_base] (banks) */
} zslot;

struct glfer_zoom_plan {
  glfer_zoom_config cfg;
  int K;
  int nchan;                  /* channels (centres): 1 for the single-centre constructors */
  unsigned step[GLB_ZOOM_MAX_CHANNELS];
  float *d_taps;              /* [nchan][33 D] (re, im) pairs: g[j] = h[K - j] e^{+2 pi i phi(K - j)}, zero past 2K */
  int iq;                     /* 1: complex (I, Q) input (glfer_zoom_plan_create_iq), signed centre */
  glb_cframe fs;
  zslot slot[GLB_CSLOTS];
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

int glfer_zoom_hop(const glfer_zoom_plan *p) { return p->fs.hop; }
int glfer_zoom_bins(const glfer_zoom_plan *p) { return p->cfg.n; }
int glfer_zoom_channels(const glfer_zoom_plan *p) { return p->nchan; }
double glfer_zoom_channel_center_hz(const glfer_zoom_plan *p, int c)
{
  if (c < 0 || c >= p->nchan) return NAN;
  /* an I/Q plan's step is a signed 32-bit fraction of a turn: centres below the dial are negative */
  const double s = p->iq ? (double) (int) p->step[c] : (double) p->step[c];
  return s * p->cfg.sample_rate / 4294967296.0;
}
double glfer_zoom_center_hz(const glfer_zoom_plan *p) { return glfer_zoom_channel_center_hz(p, 0); }

long long glfer_zoom_num_frames(const glfer_zoom_plan *p, long long nsamples)
{
  const long long last = nsamples - 1 - p->K;           /* m D <= last */
  const long long md = last < 0 ? 0 : last / p->cfg.decim + 1;
  return md / p->fs.hop;
}

void glfer_zoom_required_span(const glfer_zoom_plan *p, long long first_frame, long long nframes, long long *lo,
                              long long *hi)
{
  const long long D = p->cfg.decim;
  const long long m_lo = first_frame * p->fs.hop - (p->cfg.n - p->fs.hop);
  const long long m_hi = (first_frame + nframes) * p->fs.hop;        /* y[m_lo .. m_hi) */
  *lo = m_lo * D - p->K;
  *hi = (m_hi - 1) * D + p->K + 1;
}

void glfer_zoom_plan_destroy(glfer_zoom_plan *p)
{
  if (!p) return;
  glb_cframe_destroy(&p->fs);
  for (int i = 0; i < GLB_CSLOTS; i++) {
    zslot *s = &p->slot[i];
    glb_free(s->d_in); glb_free(s->d_y);
    glb_event_destroy(s->ev_dec);
  }
  glb_free(p->d_taps);
  free(p);
}

/* the decimator's complex taps of every channel on the device */
static int upload_taps(glfer_zoom_plan *p)
{
  const int D = p->cfg.decim, K = p->K;
  const size_t per = (size_t) 66 * D, bytes = sizeof(float) * per * p->nchan;
  float *h = malloc(sizeof(float) * (2 * K + 1));
  float *g = calloc(per * p->nchan, sizeof(float));
  int rc = 0;
  if (!h || !g) rc = glb_host_fail(GLFER_ENOMEM, "out of memory");
  if (rc == 0) rc = glfer_zoom_taps(D, h);
  for (int c = 0; c < p->nchan && rc == 0; c++) {
    /* g[j] = h[K - j] e^{+2 pi i phi(K - j)}: h is symmetric, so h[K - j] is taps[j] */
    float *gc = g + per * c;
    for (int j = 0; j <= 2 * K; j++) {
      const unsigned ph = (unsigned) ((long long) (K - j) * (long long) p->step[c]);
      const double a = 2.0 * M_PI * (double) ph / 4294967296.0;
      gc[2 * j] = (float) ((double) h[j] * cos(a));
      gc[2 * j + 1] = (float) ((double) h[j] * sin(a));
    }
  }
  if (rc == 0) {
    rc = glb_host_shim(glb_malloc((void **) &p->d_taps, bytes));
    if (rc == 0) rc = glb_host_shim(glb_memcpy_h2d(p->d_taps, g, bytes, NULL));
  }
  free(h); free(g);
  return rc;
}

/* centers[c], c = 0..nchan-1: the channels' centres (cfg->center_hz is not read); validated before any device call */
static int zoom_plan_create(const glfer_zoom_config *cfg, const double *centers, int nchan, int iq, int mtm,
                            float mtm_w, int mtm_kmax, glfer_zoom_plan **out)
{
  glb_host_clear_error();
  if (!cfg || !out || !centers) return glb_host_fail(GLFER_EINVAL, "null argument");
  *out = NULL;
  if (nchan < 1 || nchan > GLB_ZOOM_MAX_CHANNELS) return glb_host_fail(GLFER_EINVAL, "zoom channels must be in 1..32");
  if (cfg->decim < 2 || cfg->decim > 1024) return glb_host_fail(GLFER_EINVAL, "zoom decimation must be in 2..1024");
  if (!(cfg->sample_rate > 0.0) || !isfinite(cfg->sample_rate)) return glb_host_fail(GLFER_EINVAL, "sample rate must be positive");
  for (int c = 0; c < nchan; c++) {
    if (!iq && !(centers[c] >= 0.0 && centers[c] <= 0.5 * cfg->sample_rate))
      return glb_host_fail(GLFER_EINVAL, "centre frequency must be in [0, sample_rate / 2]");
    if (iq && !(centers[c] >= -0.5 * cfg->sample_rate && centers[c] <= 0.5 * cfg->sample_rate))
      return glb_host_fail(GLFER_EINVAL, "I/Q centre frequency must be in [-sample_rate / 2, sample_rate / 2]");
  }
  glfer_zoom_plan *p = calloc(1, sizeof *p);
  if (!p) return glb_host_fail(GLFER_ENOMEM, "out of memory");
  p->cfg = *cfg;
  p->K = 16 * cfg->decim;
  p->iq = iq;
  p->nchan = nchan;
  /* modulo 2^32: a negative I/Q centre is a step above 2^31 */
  for (int c = 0; c < nchan; c++)
    p->step[c] = (unsigned) (unsigned long long) llround(centers[c] / cfg->sample_rate * 4294967296.0);
  glb_cslot *const slot[GLB_CSLOTS] = { &p->slot[0].cs, &p->slot[1].cs, &p->slot[2].cs };
  int rc = glb_cframe_create(&p->fs, slot, cfg->n, cfg->window_type, cfg->overlap, cfg->device, mtm, mtm_w, mtm_kmax,
                             "zoom FFT size must be a power of two in 32..16384");
  if (rc != 0) {
    free(p);
    return rc;
  }
  rc = upload_taps(p);
  for (int i = 0; i < GLB_CSLOTS && rc == 0; i++) rc = glb_host_shim(glb_event_create(&p->slot[i].ev_dec));
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
  return zoom_plan_create(cfg, cfg ? &cfg->center_hz : NULL, 1, 0, 0, 0.0f, 0, out);
}

int glfer_zoom_plan_create_iq(const glfer_zoom_config *cfg, glfer_zoom_plan **out)
{
  return zoom_plan_create(cfg, cfg ? &cfg->center_hz : NULL, 1, 1, 0, 0.0f, 0, out);
}

int glfer_zoom_plan_create_mtm(const glfer_zoom_config *cfg, float mtm_w, int mtm_kmax, glfer_zoom_plan **out)
{
  return zoom_plan_create(cfg, cfg ? &cfg->center_hz : NULL, 1, 0, 1, mtm_w, mtm_kmax, out);
}

int glfer_zoom_plan_create_iq_mtm(const glfer_zoom_config *cfg, float mtm_w, int mtm_kmax, glfer_zoom_plan **out)
{
  return zoom_plan_create(cfg, cfg ? &cfg->center_hz : NULL, 1, 1, 1, mtm_w, mtm_kmax, out);
}

int glfer_zoom_plan_create_bank(const glfer_zoom_config *cfg, const double *centers_hz, int nchan, int iq,
                                glfer_zoom_plan **out)
{
  return zoom_plan_create(cfg, centers_hz, nchan, iq != 0, 0, 0.0f, 0, out);
}

int glfer_zoom_plan_create_bank_mtm(const glfer_zoom_config *cfg, const double *centers_hz, int nchan, int iq,
                                    float mtm_w, int mtm_kmax, glfer_zoom_plan **out)
{
  return zoom_plan_create(cfg, centers_hz, nchan, iq != 0, 1, mtm_w, mtm_kmax, out);
}

int glfer_zoom_tapers(const glfer_zoom_plan *p, double *tapers, double *lambda)
{
  return glb_cframe_tapers(p ? &p->fs : NULL, tapers, lambda);
}

/* the decimated samples of frames [c0, c0 + cn) into slot i's d_y, those its first frame shares with the previous
 * chunk (slot prev) copied device to device (glb_cframe_stage); a bank's channel c at d_y + c z_stride */
static int zoom_stage(void *plan, const glb_cframe_call *c, int i, int prev, long long c0, long long cn,
                      long long z_stride, const float **z, long long *z_origin, long long *z_count)
{
  glfer_zoom_plan *p = plan;
  zslot *s = &p->slot[i];
  const zslot *ps = prev >= 0 ? &p->slot[prev] : NULL;
  const long long D = p->cfg.decim, n = p->fs.n, hop = p->fs.hop;
  const long long m_lo = c0 * hop - (n - hop), m_hi = (c0 + cn) * hop;
  long long base, from;                   /* y held from `base`; decimated here from `from` */
  if (ps) {
    base = m_lo > ps->y_base ? m_lo : ps->y_base;
    from = ps->y_end;
  } else {
    base = m_lo > 0 ? m_lo : 0;
    from = base;
  }
  const int C = p->nchan;
  const long long ys = C > 1 ? z_stride : 0;
  TRY(glb_ensure((void **) &s->d_y, &s->y_cap, (size_t) ((C - 1) * ys + m_hi - base), 2 * sizeof(float)));
  long long x_lo = from * D - p->K;
  const long long x_hi = (m_hi - 1) * D + p->K + 1;
  if (x_lo < 0) x_lo = 0;
  const size_t esz = (c->pcm16 ? sizeof(short) : sizeof(float)) * (p->iq ? 2 : 1);
  TRY(glb_ensure(&s->d_in, &s->in_cap, (size_t) (x_hi - x_lo) * esz, 1));
  TRY(glb_memcpy_h2d(s->d_in, (const char *) c->src + (size_t) (x_lo - c->origin) * esz, (size_t) (x_hi - x_lo) * esz,
                     s->cs.stream));
  if (from > base) {
    /* the history this chunk's first frame shares with the previous chunk */
    TRY(glb_stream_wait_event(s->cs.stream, ps->ev_dec));
    for (int ch = 0; ch < C; ch++)
      TRY(glb_memcpy_d2d(s->d_y + 2 * ch * ys, ps->d_y + 2 * (ch * ps->y_stride + base - ps->y_base),
                         (size_t) (from - base) * 2 * sizeof(float), s->cs.stream));
  }
  /* a channel c >= 1 frame that starts before y[base] reads the samples just below channel c's: zeros, as y[m < 0] */
  for (int ch = 1; ch < C && m_lo < base; ch++)
    TRY(glb_memset(s->d_y + 2 * (ch * ys - (base - m_lo)), 0, (size_t) (base - m_lo) * 2 * sizeof(float),
                   s->cs.stream));
  if (C > 1) {
    unsigned dstep[GLB_ZOOM_MAX_CHANNELS];
    for (int ch = 0; ch < C; ch++) dstep[ch] = (unsigned) ((unsigned long long) D * p->step[ch]);
    TRY(glb_launch_zoom_bank_decim(s->d_in, c->pcm16, p->iq, x_lo, x_hi - x_lo, (int) D, C, p->d_taps, dstep, from,
                                   m_hi - from, s->d_y + 2 * (from - base), ys, s->cs.stream));
  } else if (p->iq)
    TRY(glb_launch_zoom_decim_iq(s->d_in, c->pcm16, x_lo, x_hi - x_lo, (int) D, p->d_taps,
                                 (unsigned) ((unsigned long long) D * p->step[0]), from, m_hi - from,
                                 s->d_y + 2 * (from - base), s->cs.stream));
  else
    TRY(glb_launch_zoom_decim(s->d_in, c->pcm16, x_lo, x_hi - x_lo, (int) D, p->d_taps,
                              (unsigned) ((unsigned long long) D * p->step[0]), from, m_hi - from,
                              s->d_y + 2 * (from - base), s->cs.stream));
  TRY(glb_event_record(s->ev_dec, s->cs.stream));
  s->y_base = base;
  s->y_end = m_hi;
  s->y_stride = ys;
  *z = s->d_y;
  *z_origin = base;
  *z_count = (C - 1) * ys + m_hi - base;
  return 0;
}

/* rows and/or F rows, or display levels: the frame stage's run on the general path with this plan's decimator; iq: the
 * entry takes complex input */
static int zoom_run(glfer_zoom_plan *p, int iq, glb_cframe_call *c)
{
  glb_host_clear_error();
  if (!p) return glb_host_fail(GLFER_EINVAL, "null argument");
  if (iq != p->iq && c->display)
    c->wrong_kind = iq ? "glfer_zoom_run_display_iq needs a plan from glfer_zoom_plan_create_iq"
                       : "an I/Q zoom plan runs through glfer_zoom_run_display_iq / _iq_pcm16";
  else if (iq != p->iq)
    c->wrong_kind = iq ? "glfer_zoom_run_iq needs a plan from glfer_zoom_plan_create_iq"
                       : "an I/Q zoom plan runs through glfer_zoom_run_iq / glfer_zoom_run_iq_pcm16";
  c->plan = p;
  c->stage = zoom_stage;
  c->nchan = p->nchan;
  /* ~32 MiB of new float input per chunk, as the spectrogram's pipeline; at least one frame */
  c->chunk_frames = (32LL << 20) / ((long long) p->fs.hop * p->cfg.decim * (p->iq ? 8 : 4));
  if (c->chunk_frames < 1) c->chunk_frames = 1;
  glfer_zoom_required_span(p, c->first_frame, c->nframes, &c->lo, &c->hi);
  c->general = 1;
  c->no_mtm = "the F-test needs a multitaper zoom plan";
  c->short_span = "samples do not cover the requested frames (see glfer_zoom_required_span)";
  return glb_cframe_run(&p->fs, c);
}

int glfer_zoom_run(glfer_zoom_plan *p, const float *samples, long long origin, long long count,
                   long long first_frame, long long nframes, float *rows)
{
  return zoom_run(p, 0, &(glb_cframe_call) { .src = samples, .origin = origin, .count = count,
                                             .first_frame = first_frame, .nframes = nframes, .rows = rows });
}

int glfer_zoom_run_pcm16(glfer_zoom_plan *p, const short *pcm, long long origin, long long count,
                         long long first_frame, long long nframes, float *rows)
{
  return zoom_run(p, 0, &(glb_cframe_call) { .src = pcm, .pcm16 = 1, .origin = origin, .count = count,
                                             .first_frame = first_frame, .nframes = nframes, .rows = rows });
}

int glfer_zoom_run_iq(glfer_zoom_plan *p, const float *iq, long long origin, long long count,
                      long long first_frame, long long nframes, float *rows)
{
  return zoom_run(p, 1, &(glb_cframe_call) { .src = iq, .origin = origin, .count = count, .first_frame = first_frame,
                                             .nframes = nframes, .rows = rows });
}

int glfer_zoom_run_iq_pcm16(glfer_zoom_plan *p, const short *iq, long long origin, long long count,
                            long long first_frame, long long nframes, float *rows)
{
  return zoom_run(p, 1, &(glb_cframe_call) { .src = iq, .pcm16 = 1, .origin = origin, .count = count,
                                             .first_frame = first_frame, .nframes = nframes, .rows = rows });
}

int glfer_zoom_run_mtm_ftest(glfer_zoom_plan *p, const float *samples, long long origin, long long count,
                             long long first_frame, long long nframes, float *rows, float *ftest)
{
  return zoom_run(p, 0, &(glb_cframe_call) { .src = samples, .origin = origin, .count = count,
                                             .first_frame = first_frame, .nframes = nframes, .ftest_on = 1,
                                             .rows = rows, .ftest = ftest });
}

int glfer_zoom_run_mtm_ftest_pcm16(glfer_zoom_plan *p, const short *pcm, long long origin, long long count,
                                   long long first_frame, long long nframes, float *rows, float *ftest)
{
  return zoom_run(p, 0, &(glb_cframe_call) { .src = pcm, .pcm16 = 1, .origin = origin, .count = count,
                                             .first_frame = first_frame, .nframes = nframes, .ftest_on = 1,
                                             .rows = rows, .ftest = ftest });
}

int glfer_zoom_run_iq_mtm_ftest(glfer_zoom_plan *p, const float *iq, long long origin, long long count,
                                long long first_frame, long long nframes, float *rows, float *ftest)
{
  return zoom_run(p, 1, &(glb_cframe_call) { .src = iq, .origin = origin, .count = count, .first_frame = first_frame,
                                             .nframes = nframes, .ftest_on = 1, .rows = rows, .ftest = ftest });
}

int glfer_zoom_run_iq_mtm_ftest_pcm16(glfer_zoom_plan *p, const short *iq, long long origin, long long count,
                                      long long first_frame, long long nframes, float *rows, float *ftest)
{
  return zoom_run(p, 1, &(glb_cframe_call) { .src = iq, .pcm16 = 1, .origin = origin, .count = count,
                                             .first_frame = first_frame, .nframes = nframes, .ftest_on = 1,
                                             .rows = rows, .ftest = ftest });
}

int glfer_zoom_run_mtm_lines(glfer_zoom_plan *p, const float *samples, long long origin, long long count,
                         long long first_frame, long long nframes, const glfer_lines_config *lc, int *line_count,
                         int *line_bin, float *line_ftest, float *line_psd)
{
  return zoom_run(p, 0, &(glb_cframe_call) { .src = samples, .origin = origin, .count = count,
                                             .first_frame = first_frame, .nframes = nframes, .lines = 1, .lc = lc,
                                             .line_count = line_count, .line_bin = line_bin,
                                             .line_ftest = line_ftest, .line_psd = line_psd });
}

int glfer_zoom_run_mtm_lines_pcm16(glfer_zoom_plan *p, const short *pcm, long long origin, long long count,
                               long long first_frame, long long nframes, const glfer_lines_config *lc, int *line_count,
                               int *line_bin, float *line_ftest, float *line_psd)
{
  return zoom_run(p, 0, &(glb_cframe_call) { .src = pcm, .pcm16 = 1, .origin = origin, .count = count,
                                             .first_frame = first_frame, .nframes = nframes, .lines = 1, .lc = lc,
                                             .line_count = line_count, .line_bin = line_bin,
                                             .line_ftest = line_ftest, .line_psd = line_psd });
}

int glfer_zoom_run_iq_mtm_lines(glfer_zoom_plan *p, const float *iq, long long origin, long long count,
                            long long first_frame, long long nframes, const glfer_lines_config *lc, int *line_count,
                            int *line_bin, float *line_ftest, float *line_psd)
{
  return zoom_run(p, 1, &(glb_cframe_call) { .src = iq, .origin = origin, .count = count,
                                             .first_frame = first_frame, .nframes = nframes, .lines = 1, .lc = lc,
                                             .line_count = line_count, .line_bin = line_bin,
                                             .line_ftest = line_ftest, .line_psd = line_psd });
}

int glfer_zoom_run_iq_mtm_lines_pcm16(glfer_zoom_plan *p, const short *iq, long long origin, long long count,
                                  long long first_frame, long long nframes, const glfer_lines_config *lc, int *line_count,
                                  int *line_bin, float *line_ftest, float *line_psd)
{
  return zoom_run(p, 1, &(glb_cframe_call) { .src = iq, .pcm16 = 1, .origin = origin, .count = count,
                                             .first_frame = first_frame, .nframes = nframes, .lines = 1, .lc = lc,
                                             .line_count = line_count, .line_bin = line_bin,
                                             .line_ftest = line_ftest, .line_psd = line_psd });
}

/* main_window_draw's mapping of the plan's own rows (include/glfer_b200.h, glfer_zoom_run_display) */
int glfer_zoom_run_display(glfer_zoom_plan *p, const float *samples, long long origin, long long count,
                           long long first_frame, long long nframes, const glfer_display_config *dc,
                           float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range)
{
  return zoom_run(p, 0, &(glb_cframe_call) { .src = samples, .origin = origin, .count = count,
                                             .first_frame = first_frame, .nframes = nframes, .display = 1, .dc = dc,
                                             .agc_state = agc_state, .range_out = display_range, .levels = levels,
                                             .rgb = rgb });
}

int glfer_zoom_run_display_pcm16(glfer_zoom_plan *p, const short *pcm, long long origin, long long count,
                                 long long first_frame, long long nframes, const glfer_display_config *dc,
                                 float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range)
{
  return zoom_run(p, 0, &(glb_cframe_call) { .src = pcm, .pcm16 = 1, .origin = origin, .count = count,
                                             .first_frame = first_frame, .nframes = nframes, .display = 1, .dc = dc,
                                             .agc_state = agc_state, .range_out = display_range, .levels = levels,
                                             .rgb = rgb });
}

int glfer_zoom_run_display_iq(glfer_zoom_plan *p, const float *iq, long long origin, long long count,
                              long long first_frame, long long nframes, const glfer_display_config *dc,
                              float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range)
{
  return zoom_run(p, 1, &(glb_cframe_call) { .src = iq, .origin = origin, .count = count, .first_frame = first_frame,
                                             .nframes = nframes, .display = 1, .dc = dc, .agc_state = agc_state,
                                             .range_out = display_range, .levels = levels, .rgb = rgb });
}

int glfer_zoom_run_display_iq_pcm16(glfer_zoom_plan *p, const short *iq, long long origin, long long count,
                                    long long first_frame, long long nframes, const glfer_display_config *dc,
                                    float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range)
{
  return zoom_run(p, 1, &(glb_cframe_call) { .src = iq, .pcm16 = 1, .origin = origin, .count = count,
                                             .first_frame = first_frame, .nframes = nframes, .display = 1, .dc = dc,
                                             .agc_state = agc_state, .range_out = display_range, .levels = levels,
                                             .rgb = rgb });
}
