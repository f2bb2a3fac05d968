/* iq.c -- I/Q spectrogram plans: two-sided rows of complex (SDR baseband) recordings (include/glfer_b200.h).
 *
 * The frames of an interleaved (I, Q) stream are complex FFT frames of n samples; one shim entry,
 * glb_launch_iq_gram (csrc/iq.cu), computes their rows on whichever path serves the geometry (the fused ring
 * kernel, or the general kernel followed by the zoom's split).  Everything after a chunk's samples reach the device --
 * the taper tables, the launch, the downloads, the display chain and the chunk loop -- is the complex frame stage of
 * host/cframe.c, shared with the zoom.  This file only stages the samples: each chunk of ~32 MiB of input uploads its
 * complex samples (the n - hop samples it shares with the previous chunk again) and converts int16 input to float on
 * the device.
 *
 * The display entries (glfer_iq_run_display*) bring back 8-bit levels instead of rows.  With a fixed range and no
 * RGB the spectrogram kernel maps its own powers (glb_iq_gram_args.levels) and no float row is ever stored;
 * otherwise each chunk's rows stay on the device and go through the display chain of host/display.c.
 *
 * Multitaper plans (glfer_iq_plan_create_mtm) always bring float rows to the device: their waterfall goes through the
 * display chain, for a fixed range too.  Every multitaper plan serves glfer_iq_run_mtm_ftest, whose chunks bring back
 * F rows beside or instead of the rows, and glfer_iq_run_mtm_lines, whose chunks keep the F rows on the device and
 * bring back only the lines selected from them.
 */
#include <stdlib.h>
#include <string.h>
#include "glb_host.h"

typedef struct {
  glb_cslot cs;               /* stream, rows, F rows, scratch, display */
  short *d_pcm;               /* int16 input of the chunk */
  size_t pcm_cap;             /* shorts */
  float *d_in;                /* interleaved (I, Q) floats of the chunk */
  size_t in_cap;              /* floats */
} islot;

struct glfer_iq_plan {
  glfer_iq_config cfg;
  glb_cframe fs;
  islot slot[GLB_CSLOTS];
};

void glfer_iq_config_default(glfer_iq_config *c)
{
  memset(c, 0, sizeof *c);
  c->n = 4096;
  c->window_type = HANNING_WINDOW;
  c->overlap = 0.5f;
  c->device = 0;
}

int glfer_iq_hop(const glfer_iq_plan *p) { return p->fs.hop; }
int glfer_iq_bins(const glfer_iq_plan *p) { return p->cfg.n; }

long long glfer_iq_num_frames(const glfer_iq_plan *p, long long nsamples)
{
  return nsamples <= 0 ? 0 : nsamples / p->fs.hop;
}

void glfer_iq_required_span(const glfer_iq_plan *p, long long first_frame, long long nframes, long long *lo,
                            long long *hi)
{
  *lo = first_frame * p->fs.hop - (p->cfg.n - p->fs.hop);
  *hi = (first_frame + nframes) * p->fs.hop;
}

void glfer_iq_plan_destroy(glfer_iq_plan *p)
{
  if (!p) return;
  glb_cframe_destroy(&p->fs);
  for (int i = 0; i < GLB_CSLOTS; i++) { glb_free(p->slot[i].d_pcm); glb_free(p->slot[i].d_in); }
  free(p);
}

static int iq_plan_create(const glfer_iq_config *cfg, int mtm, float mtm_w, int mtm_kmax, glfer_iq_plan **out)
{
  glb_host_clear_error();
  if (!cfg || !out) return glb_host_fail(GLFER_EINVAL, "null argument");
  *out = NULL;
  glfer_iq_plan *p = calloc(1, sizeof *p);
  if (!p) return glb_host_fail(GLFER_ENOMEM, "out of memory");
  p->cfg = *cfg;
  glb_cslot *const slot[GLB_CSLOTS] = { &p->slot[0].cs, &p->slot[1].cs, &p->slot[2].cs };
  const int rc = glb_cframe_create(&p->fs, slot, cfg->n, cfg->window_type, cfg->overlap, cfg->device, mtm, mtm_w,
                                   mtm_kmax, "I/Q FFT size must be a power of two in 32..16384");
  if (rc != 0) {
    free(p);
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
  return glb_cframe_tapers(p ? &p->fs : NULL, tapers, lambda);
}

/* the complex samples of frames [c0, c0 + cn) into slot i's d_in (glb_cframe_stage) */
static int iq_stage(void *plan, const glb_cframe_call *c, int i, int prev, long long c0, long long cn,
                    long long z_stride, const float **z, long long *z_origin, long long *z_count)
{
  glfer_iq_plan *p = plan;
  islot *s = &p->slot[i];
  const long long n = p->fs.n, hop = p->fs.hop;
  long long lo = c0 * hop - (n - hop);
  const long long hi = (c0 + cn) * hop;
  if (lo < 0) lo = 0;
  /* the fused kernel reads whole hop blocks with 16-byte bulk copies: stage from an even complex index when the
     caller's samples reach that far back (the regular hops are even, so lo already is) */
  if ((lo & 1) && lo - 1 >= c->origin) lo--;
  const long long cnt = hi - lo;
  TRY(glb_ensure((void **) &s->d_in, &s->in_cap, (size_t) (2 * cnt), sizeof(float)));
  if (c->pcm16) {
    TRY(glb_ensure((void **) &s->d_pcm, &s->pcm_cap, (size_t) (2 * cnt), sizeof(short)));
    TRY(glb_memcpy_h2d(s->d_pcm, (const short *) c->src + 2 * (lo - c->origin), sizeof(short) * 2 * (size_t) cnt,
                       s->cs.stream));
    TRY(glb_launch_pcm16_to_float(s->d_pcm, s->d_in, 2 * cnt, s->cs.stream));
  } else {
    TRY(glb_memcpy_h2d(s->d_in, (const float *) c->src + 2 * (lo - c->origin), sizeof(float) * 2 * (size_t) cnt,
                       s->cs.stream));
  }
  *z = s->d_in;
  *z_origin = lo;
  *z_count = cnt;
  return 0;
}

/* rows and/or F rows, or display levels: the frame stage's run with this plan's stage */
static int iq_run(glfer_iq_plan *p, glb_cframe_call *c)
{
  glb_host_clear_error();
  if (!p) return glb_host_fail(GLFER_EINVAL, "null argument");
  c->plan = p;
  c->stage = iq_stage;
  /* ~32 MiB of new float input per chunk, as the spectrogram's and the zoom's pipelines; at least one frame */
  c->chunk_frames = (32LL << 20) / ((long long) p->fs.hop * 8);
  if (c->chunk_frames < 1) c->chunk_frames = 1;
  glfer_iq_required_span(p, c->first_frame, c->nframes, &c->lo, &c->hi);
  /* fixed range without RGB: the spectrogram kernel writes the levels itself (periodogram plans only) */
  c->fuse = c->display && c->dc && glb_host_fused_levels() && !c->dc->autoscale && !c->rgb && p->fs.ntapers == 1;
  c->no_mtm = "the F-test needs a multitaper plan (glfer_iq_plan_create_mtm)";
  c->short_span = "samples do not cover the requested frames (see glfer_iq_required_span)";
  return glb_cframe_run(&p->fs, c);
}

int glfer_iq_run(glfer_iq_plan *p, const float *iq, long long origin, long long count, long long first_frame,
                 long long nframes, float *rows)
{
  return iq_run(p, &(glb_cframe_call) { .src = iq, .origin = origin, .count = count, .first_frame = first_frame,
                                        .nframes = nframes, .rows = rows });
}

int glfer_iq_run_pcm16(glfer_iq_plan *p, const short *iq, long long origin, long long count, long long first_frame,
                       long long nframes, float *rows)
{
  return iq_run(p, &(glb_cframe_call) { .src = iq, .pcm16 = 1, .origin = origin, .count = count,
                                        .first_frame = first_frame, .nframes = nframes, .rows = rows });
}

int glfer_iq_run_mtm_ftest(glfer_iq_plan *p, const float *iq, long long origin, long long count, long long first_frame,
                           long long nframes, float *rows, float *ftest)
{
  return iq_run(p, &(glb_cframe_call) { .src = iq, .origin = origin, .count = count, .first_frame = first_frame,
                                        .nframes = nframes, .ftest_on = 1, .rows = rows, .ftest = ftest });
}

int glfer_iq_run_mtm_ftest_pcm16(glfer_iq_plan *p, const short *iq, long long origin, long long count,
                                 long long first_frame, long long nframes, float *rows, float *ftest)
{
  return iq_run(p, &(glb_cframe_call) { .src = iq, .pcm16 = 1, .origin = origin, .count = count,
                                        .first_frame = first_frame, .nframes = nframes, .ftest_on = 1, .rows = rows,
                                        .ftest = ftest });
}

int glfer_iq_run_mtm_lines(glfer_iq_plan *p, const float *iq, long long origin, long long count, long long first_frame,
                           long long nframes, const glfer_lines_config *lc, int *line_count, int *line_bin,
                           float *line_ftest, float *line_psd)
{
  return iq_run(p, &(glb_cframe_call) { .src = iq, .origin = origin, .count = count, .first_frame = first_frame,
                                        .nframes = nframes, .lines = 1, .lc = lc, .line_count = line_count,
                                        .line_bin = line_bin, .line_ftest = line_ftest, .line_psd = line_psd });
}

int glfer_iq_run_mtm_lines_pcm16(glfer_iq_plan *p, const short *iq, long long origin, long long count,
                                 long long first_frame, long long nframes, const glfer_lines_config *lc,
                                 int *line_count, int *line_bin, float *line_ftest, float *line_psd)
{
  return iq_run(p, &(glb_cframe_call) { .src = iq, .pcm16 = 1, .origin = origin, .count = count,
                                        .first_frame = first_frame, .nframes = nframes, .lines = 1, .lc = lc,
                                        .line_count = line_count, .line_bin = line_bin, .line_ftest = line_ftest,
                                        .line_psd = line_psd });
}

/* main_window_draw's mapping of the plan's own rows (include/glfer_b200.h, glfer_iq_run_display) */
int glfer_iq_run_display(glfer_iq_plan *p, const float *iq, long long origin, long long count, long long first_frame,
                         long long nframes, const glfer_display_config *dc, float *agc_state, unsigned char *levels,
                         unsigned char *rgb, float *display_range)
{
  return iq_run(p, &(glb_cframe_call) { .src = iq, .origin = origin, .count = count, .first_frame = first_frame,
                                        .nframes = nframes, .display = 1, .dc = dc, .agc_state = agc_state,
                                        .range_out = display_range, .levels = levels, .rgb = rgb });
}

int glfer_iq_run_display_pcm16(glfer_iq_plan *p, const short *iq, long long origin, long long count,
                               long long first_frame, long long nframes, const glfer_display_config *dc,
                               float *agc_state, unsigned char *levels, unsigned char *rgb, float *display_range)
{
  return iq_run(p, &(glb_cframe_call) { .src = iq, .pcm16 = 1, .origin = origin, .count = count,
                                        .first_frame = first_frame, .nframes = nframes, .display = 1, .dc = dc,
                                        .agc_state = agc_state, .range_out = display_range, .levels = levels,
                                        .rgb = rgb });
}
