/* cframe.c -- the complex frame stage shared by the I/Q (host/iq.c) and zoom (host/zoom.c) plans.
 *
 * Both plans turn a chunk of their input into complex samples on the device -- the I/Q plan uploads them, the zoom
 * mixes, filters and decimates them -- and from there do the same work: complex FFT frames of n samples through one
 * shim entry (glb_launch_iq_gram, or glb_launch_iq_gram_general for the zoom), rows and/or the harmonic F-test's F rows
 * back to the host, 8-bit levels through the display chain of host/display.c, or the harmonic lines selected from the
 * F rows on the device (glb_launch_ftest_lines).  This unit owns that work: the taper
 * table (the window, or K' DPSS tapers, each scaled as the real multitaper plan scales its own in host/gram.c) with the
 * F-test's table and the FFT tables, the GLB_CSLOTS streams with their rows, F rows and scratch, the argument checks of
 * the run entries and the chunk loop.  The plan supplies its per-chunk stage as a callback.
 *
 * A run walks the frames in chunks on the slots in turn: a slot's stream is synchronised before the slot is reused, so
 * a chunk's kernels and downloads overlap the next chunk's upload, and device memory is bounded by the chunk, not by
 * the recording.
 *
 * A zoom bank's call has C channels: the stage lays the channels' samples at a fixed stride, and one frame stage
 * launch covers every channel (glb_cframe_stage), so the launches per chunk do not grow with C.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include "glb_host.h"

/* 1 when the [2n]-float taper t reads the same backwards bit for bit */
static int mirrored(const float *t, int n)
{
  for (int i = 0; i < n; i++)
    if (memcmp(&t[i], &t[2 * n - 1 - i], sizeof(float)) != 0) return 0;
  return 1;
}

/* The DPSS of a complex multitaper plan and its taper table, built as host/gram.c builds the real plan's: h_tapers
 * [K'][n] and h_lambda [K'] from glb_dpss, table [K'][2n] floats with v_k[i] taper_scale / sqrt(lambda_k) on both
 * floats of complex sample i, sym: bit k when taper k reads the same backwards bit for bit.  Validation as
 * glfer_gram_plan_create; needs no device. */
static int glb_iq_mtm_tapers(int n, float mtm_w, int mtm_kmax, float taper_scale, double **h_tapers, double **h_lambda,
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
    *sym |= mirrored(t, n) << k;
  }
  *h_tapers = tap; *h_lambda = lam; *table = tab;
  return 0;
}

/* The harmonic F-test's table of a complex multitaper plan, uploaded to *d_ftab: hn (glb_mtm_ftest_weights, as the real
 * plan builds it) times taper_scale on both floats of complex sample i, [2n] floats, then the K' pairs
 * (U0_k, sqrt(lambda_k)) that undo the per-taper weight of the taper table in the residual (glb_iq_gram_args). */
static int glb_iq_ftest_table(int n, int K, const double *h_tapers, const double *h_lambda, float taper_scale,
                              float **d_ftab, float *s)
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

/* the taper table on the device -- tab: the multitaper table of glb_iq_mtm_tapers, or NULL for the window on both
 * floats of a complex sample, times taper_scale -- and the FFT tables of the 2n-float frames */
static int upload_taper(glb_cframe *f, int window_type, const float *tab)
{
  const int n = f->n;
  float *w = malloc(sizeof(float) * n);
  float *taper = malloc(sizeof(float) * 2 * n);
  int rc = 0;
  if (!w || !taper) rc = glb_host_fail(GLFER_ENOMEM, "out of memory");
  if (rc == 0 && !tab) {
    glb_window_table(n, window_type, w);
    for (int i = 0; i < n; i++) {
      /* as the spectrogram: a rectangular window is not applied (weight 1) */
      const double wi = window_type == RECTANGULAR_WINDOW ? 1.0 : (double) w[i];
      taper[2 * i] = taper[2 * i + 1] = (float) (wi * (double) f->taper_scale);
    }
    f->taper_sym = mirrored(taper, n);
    tab = taper;
  }
  const size_t bytes = sizeof(float) * 2 * (size_t) n * f->ntapers;
  if (rc == 0) rc = glb_host_shim(glb_malloc((void **) &f->d_taper, bytes));
  if (rc == 0) rc = glb_host_shim(glb_memcpy_h2d(f->d_taper, tab, bytes, NULL));
  if (rc == 0) rc = glb_host_shim(glb_tables_create(2 * n, &f->tables));
  free(w); free(taper);
  return rc;
}

int glb_cframe_create(glb_cframe *f, glb_cslot *const slot[GLB_CSLOTS], int n, int window_type, float overlap,
                      int device, int mtm, float mtm_w, int mtm_kmax, const char *size_msg)
{
  memset(f, 0, sizeof *f);
  for (int i = 0; i < GLB_CSLOTS; i++) f->slot[i] = slot[i];
  if (n < 32 || n > 16384 || (n & (n - 1)) != 0) return glb_host_fail(GLFER_EINVAL, size_msg);
  if (window_type < 0 || window_type > 7) return glb_host_fail(GLFER_EINVAL, "unknown window type");
  const int hop = glb_hop(n, overlap);
  if (hop < 1 || hop > n) return glb_host_fail(GLFER_EINVAL, "overlap leaves no new samples per block");
  f->n = n;
  f->hop = hop;
  f->overlap = overlap;
  f->device = device;
  f->taper_scale = (float) (1.0 / (2.0 * sqrt(2.0 * n)));
  f->ntapers = mtm ? mtm_kmax + 1 : 1;
  float *tab = NULL;
  if (mtm) {
    const int rc = glb_iq_mtm_tapers(n, mtm_w, mtm_kmax, f->taper_scale, &f->h_tapers, &f->h_lambda, &tab,
                                     &f->taper_sym);
    if (rc != 0) return rc;
  }
  int ndev = 0;
  int rc = 0;
  if (glb_device_count(&ndev) != GLB_OK || ndev < 1)
    rc = glb_host_fail(GLFER_ENODEV, "no CUDA device (libglfer_b200 has no CPU fallback)");
  else if (device < 0 || device >= ndev)
    rc = glb_host_fail(GLFER_EINVAL, "device ordinal out of range");
  else
    rc = glb_host_shim(glb_set_device(device));
  if (rc != 0) {
    free(f->h_tapers); free(f->h_lambda); free(tab);
    return rc;
  }
  rc = upload_taper(f, window_type, tab);
  free(tab);
  if (rc == 0 && mtm)
    rc = glb_iq_ftest_table(n, f->ntapers, f->h_tapers, f->h_lambda, f->taper_scale, &f->d_ftab, &f->ftest_s);
  for (int i = 0; i < GLB_CSLOTS && rc == 0; i++) {
    rc = glb_host_shim(glb_stream_create(&slot[i]->stream));
    if (rc == 0) rc = glb_host_shim(glb_event_create(&slot[i]->disp.ev_agc));
  }
  if (rc != 0) {
    char keep[512];
    strncpy(keep, glfer_b200_last_error(), sizeof keep - 1);
    keep[sizeof keep - 1] = 0;
    glb_cframe_destroy(f);
    glb_host_fail(rc, keep);
  }
  return rc;
}

void glb_cframe_destroy(glb_cframe *f)
{
  glb_set_device(f->device);
  for (int i = 0; i < GLB_CSLOTS; i++) {
    glb_cslot *s = f->slot[i];
    if (s->stream) glb_stream_sync(s->stream);
    glb_free(s->d_rows); glb_free(s->d_ftest); glb_free(s->d_scratch); glb_free(s->d_lines);
    if (s->h_lines) glb_host_free(s->h_lines);
    glb_display_slot_free(&s->disp);
    glb_stream_destroy(s->stream);
  }
  glb_display_free(&f->disp);
  glb_free(f->d_taper);
  glb_free(f->d_ftab);
  glb_tables_destroy(f->tables);
  free(f->h_tapers); free(f->h_lambda);
}

int glb_cframe_tapers(const glb_cframe *f, double *tapers, double *lambda)
{
  if (!f || !tapers || !lambda) return glb_host_fail(GLFER_EINVAL, "null argument");
  if (!f->h_tapers) return glb_host_fail(GLFER_EINVAL, "plan is not a multitaper plan");
  memcpy(tapers, f->h_tapers, sizeof(double) * (size_t) f->ntapers * f->n);
  memcpy(lambda, f->h_lambda, sizeof(double) * f->ntapers);
  return 0;
}

/* frames [c0, cn) of the staged samples z ([z_origin, z_origin + z_count)) on slot s: with c->fuse the fixed-range
 * levels into s->disp.d_levels, otherwise rows into s->d_rows (when the run wants them) and F rows into s->d_ftest
 * (always for a lines run, whose rows are wanted only for line_psd) */
static int cframe_launch(glb_cframe *f, glb_cslot *s, const glb_cframe_call *c, const glb_display_run *dr,
                         const float *z, long long z_origin, long long z_count, long long c0, long long cn)
{
  const long long n = f->n;
  const int rows_on = c->display ? !c->fuse : c->lines ? c->line_psd != NULL : c->rows != NULL;
  const int ftest_on = c->ftest != NULL || c->lines;
  if (rows_on) TRY(glb_ensure((void **) &s->d_rows, &s->rows_cap, (size_t) (cn * n), sizeof(float)));
  if (ftest_on) TRY(glb_ensure((void **) &s->d_ftest, &s->ftest_cap, (size_t) (cn * n), sizeof(float)));
  const long long sb = c->general ? glb_iq_gram_general_scratch_bytes((int) n, cn, c->fuse, ftest_on)
                                  : glb_iq_gram_scratch_bytes((int) n, f->hop, cn, c->fuse, f->ntapers, ftest_on);
  if (sb > 0) TRY(glb_ensure(&s->d_scratch, &s->scratch_cap, (size_t) sb, 1));
  glb_iq_gram_args g;
  memset(&g, 0, sizeof g);
  g.n = (int) n;
  g.hop = f->hop;
  g.samples = z;
  g.origin = z_origin;
  g.count = z_count;
  g.taper = f->d_taper;
  g.taper_symmetric = f->taper_sym;
  g.taper_scale = f->taper_scale;
  g.ntapers = f->ntapers;
  g.first_frame = c0;
  g.nframes = cn;
  g.rows = rows_on ? s->d_rows : NULL;
  g.tables = f->tables;
  g.scratch = sb > 0 ? s->d_scratch : NULL;
  if (c->fuse) {
    g.levels = s->disp.d_levels;
    g.levels_stride = n;
    g.level_tables = f->disp.level_tables;
    g.levels_log = c->dc->log_scale;
    g.level_lut = f->disp.d_level_lut;
    g.level_min = dr->fixed[1];
    g.level_max = dr->fixed[0];
    g.level_thr = dr->thr;
  }
  if (ftest_on) {
    g.ftest = s->d_ftest;
    g.ftest_taper = f->d_ftab;
    g.ftest_u0 = f->d_ftab + 2 * n;
    g.ftest_s = f->ftest_s;
  }
  TRY(c->general ? glb_launch_iq_gram_general(&g, s->stream) : glb_launch_iq_gram(&g, s->stream));
  return 0;
}

/* bytes of one chunk's line arrays for nf output frames: count [nf] ints, then bin [nf][max_lines] ints, F and psd
 * [nf][max_lines] floats when wanted; the device buffer and its pinned staging share the layout */
static size_t lines_bytes(const glb_cframe_call *c, long long nf)
{
  const size_t slots = (size_t) nf * c->lc->max_lines;
  return sizeof(int) * ((size_t) nf + slots) + sizeof(float) * slots * ((c->line_ftest != NULL) + (c->line_psd != NULL));
}

/* the lines of the chunk's F rows on slot s (nchan channels at a stride of crows rows), downloaded in one copy to the
 * slot's pinned staging, which glb_cframe_run hands over once the slot's stream is synchronised */
static int lines_chunk(glb_cframe *f, glb_cslot *s, const glb_cframe_call *c, float thr, int nchan, long long cn,
                       long long crows, long long done)
{
  const long long nf = nchan * cn;
  const size_t slots = (size_t) nf * c->lc->max_lines, bytes = lines_bytes(c, nf);
  TRY(glb_ensure(&s->d_lines, &s->dlines_cap, bytes, 1));
  if (bytes > s->hlines_cap) {
    /* into the caller's arrays directly, each chunk's copy would block the host thread whenever they are pageable,
       and with it the chunk pipeline (as the display range, host/display.c) */
    if (s->h_lines) glb_host_free(s->h_lines);
    s->h_lines = NULL; s->hlines_cap = 0;
    const size_t cap = bytes + bytes / 2 + 4096;
    TRY(glb_host_alloc(&s->h_lines, cap));
    s->hlines_cap = cap;
  }
  int *d_count = s->d_lines, *d_bin = d_count + nf;
  float *d_f = (float *) (d_bin + slots);
  float *d_p = d_f + (c->line_ftest ? slots : 0);
  TRY(glb_launch_ftest_lines(s->d_ftest, c->line_psd ? s->d_rows : NULL, f->n, f->n, cn, nchan, crows, thr,
                             c->lc->max_lines, c->lc->bin_lo, c->lc->bin_hi, d_count, d_bin,
                             c->line_ftest ? d_f : NULL, c->line_psd ? d_p : NULL, s->stream));
  TRY(glb_memcpy_d2h(s->h_lines, s->d_lines, bytes, s->stream));
  s->lines_done = done;
  s->lines_cn = cn;
  return 0;
}

/* the staged lines of slot s (its stream synchronised) into the caller's arrays */
static void lines_handover(const glb_cframe_call *c, glb_cslot *s, int nchan)
{
  const long long cn = s->lines_cn, nf = nchan * cn, M = c->lc->max_lines;
  const size_t slots = (size_t) nf * M;
  const int *h_count = s->h_lines, *h_bin = h_count + nf;
  const float *h_f = (const float *) (h_bin + slots);
  const float *h_p = h_f + (c->line_ftest ? slots : 0);
  for (int ch = 0; ch < nchan; ch++) {
    const size_t to = (size_t) (ch * c->nframes + s->lines_done), from = (size_t) (ch * cn);
    const size_t m = sizeof(float) * (size_t) (cn * M);
    memcpy(c->line_count + to, h_count + from, sizeof(int) * (size_t) cn);
    memcpy(c->line_bin + to * M, h_bin + from * M, m);
    if (c->line_ftest) memcpy(c->line_ftest + to * M, h_f + from * M, m);
    if (c->line_psd) memcpy(c->line_psd + to * M, h_p + from * M, m);
  }
  s->lines_cn = 0;
}

int glb_cframe_run(glb_cframe *f, const glb_cframe_call *c)
{
  if (!c->src || (c->display ? !c->dc : c->lines ? (!c->lc || !c->line_count || !c->line_bin)
                                                  : (!c->ftest_on && !c->rows)))
    return glb_host_fail(GLFER_EINVAL, "null argument");
  if (c->wrong_kind) return glb_host_fail(GLFER_EINVAL, c->wrong_kind);
  if (c->ftest_on || c->lines) {
    if (!f->h_tapers) return glb_host_fail(GLFER_EINVAL, c->no_mtm);
    if (f->ntapers < 2) return glb_host_fail(GLFER_EINVAL, "the F-test needs mtm_kmax >= 1 (K' - 1 degrees of freedom)");
    if (c->ftest_on && !c->rows && !c->ftest) return glb_host_fail(GLFER_EINVAL, "null argument: rows and ftest are both NULL");
  }
  float thr = 0.0f;
  if (c->lines) {
    const int rt = glfer_ftest_threshold(f->ntapers, c->lc->pfa, &thr);
    if (rt != 0) return rt;
    if (c->lc->max_lines < 1 || c->lc->max_lines > 1024) return glb_host_fail(GLFER_EINVAL, "max_lines must be in 1..1024");
    if (c->lc->bin_lo < 0 || c->lc->bin_lo >= c->lc->bin_hi || c->lc->bin_hi > f->n)
      return glb_host_fail(GLFER_EINVAL, "bin range must satisfy 0 <= bin_lo < bin_hi <= n");
  }
  if (c->nframes < 0 || c->first_frame < 0) return glb_host_fail(GLFER_EINVAL, "negative frame range");
  if (c->origin < 0 || c->count < 0) return glb_host_fail(GLFER_EINVAL, "negative origin or sample count");
  if (c->display) {
    if (c->rgb && !c->dc->colortab) return glb_host_fail(GLFER_EINVAL, "RGB output needs a 256-entry palette");
    if (c->dc->autoscale && c->first_frame > 0 && !c->agc_state)
      return glb_host_fail(GLFER_EINVAL, "autoscale from frame > 0 needs the carried AGC state");
  }
  if (c->nframes == 0) return 0;
  TRY(glb_set_device(f->device));
  if ((c->lo < 0 ? 0 : c->lo) < c->origin || c->hi > c->origin + c->count)
    return glb_host_fail(GLFER_EINVAL, c->short_span);
  const int n = f->n;
  const int nchan = c->nchan > 1 ? c->nchan : 1;
  glb_display_run dr;
  if (c->display)
    TRY(glb_display_begin(&f->disp, &dr, c->dc, c->agc_state, c->nframes, nchan, c->range_out != NULL,
                          f->slot[0]->stream));
  int rc = 0, ci = 0;
  long long done = 0;
  for (int i = 0; i < GLB_CSLOTS; i++) f->slot[i]->lines_cn = 0;
  while (done < c->nframes && rc == 0) {
    const int i = ci % GLB_CSLOTS, prev = ci > 0 ? (ci - 1) % GLB_CSLOTS : -1;
    glb_cslot *s = f->slot[i];
    const long long c0 = c->first_frame + done;
    const long long cn = (c->nframes - done < c->chunk_frames) ? c->nframes - done : c->chunk_frames;
    /* channels at a stride of crows frames, so that one launch of nl frames covers them all: frame c0 + c crows + j is
       channel c's frame c0 + j, and the crows - cn frames between two channels are computed and never fetched */
    const long long crows = nchan > 1 ? cn + (n - f->hop + f->hop - 1) / f->hop : cn;
    const long long nl = (nchan - 1) * crows + cn;
    const float *z = NULL;
    long long z_origin = 0, z_count = 0;
    rc = glb_host_shim(glb_stream_sync(s->stream));
    if (rc == 0 && s->lines_cn) lines_handover(c, s, nchan);
    if (rc == 0 && c->display) rc = glb_display_reserve(&s->disp, nl, n, c->rgb != NULL);
    if (rc == 0) rc = c->stage(c->plan, c, i, prev, c0, cn, crows * f->hop, &z, &z_origin, &z_count);
    if (rc == 0) rc = cframe_launch(f, s, c, &dr, z, z_origin, z_count, c0, nl);
    if (rc == 0 && c->display && !c->fuse)
      rc = glb_display_map(&f->disp, &dr, &s->disp, prev >= 0 ? &f->slot[prev]->disp : NULL, s->d_rows, s->d_rows, n,
                           c0, cn, crows, done, f->overlap, c->rgb != NULL, s->stream);
    if (rc == 0 && c->display)
      rc = glb_display_fetch(&dr, &s->disp, cn, crows, n, done, c->levels, c->rgb, s->stream);
    if (rc == 0 && c->lines) rc = lines_chunk(f, s, c, thr, nchan, cn, crows, done);
    for (int ch = 0; ch < nchan && rc == 0; ch++) {
      const size_t to = (size_t) (ch * c->nframes + done) * n, from = (size_t) (ch * crows) * n;
      if (c->rows)
        rc = glb_host_shim(glb_memcpy_d2h(c->rows + to, s->d_rows + from, sizeof(float) * (size_t) (cn * n),
                                          s->stream));
      if (rc == 0 && c->ftest)
        rc = glb_host_shim(glb_memcpy_d2h(c->ftest + to, s->d_ftest + from, sizeof(float) * (size_t) (cn * n),
                                          s->stream));
    }
    done += cn;
    ci++;
  }
  for (int i = 0; i < GLB_CSLOTS; i++) {
    const int r2 = glb_host_shim(glb_stream_sync(f->slot[i]->stream));
    if (rc == 0) rc = r2;
    if (rc == 0 && f->slot[i]->lines_cn) lines_handover(c, f->slot[i], nchan);
    f->slot[i]->lines_cn = 0;
  }
  if (rc == 0 && c->display) rc = glb_display_end(&f->disp, &dr, c->nframes, c->agc_state, c->range_out);
  return rc;
}
