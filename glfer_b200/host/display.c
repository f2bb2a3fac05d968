/* display.c -- the display chain of main_window_draw (g_main.c:1109-1229) over device rows, shared by every plan
 * type that offers a *_run_display entry (gram.c, iq.c, zoom.c).
 *
 * Per run: the plan's device state (carried AGC levels, palette, the fixed range's level look-up table, the dB
 * thresholds) is uploaded once.  Per chunk of rows on a slot: per-row floor statistics (compute_floor), the AGC
 * of the display range -- a recurrence over frames, walked in order on the device and carried from chunk to
 * chunk through an event chain between the slots -- then 8-bit levels / RGB.  Only 1 (levels) or 3 (RGB) bytes
 * per bin go back to the host, plus the per-frame range through pinned staging.
 */
#include <stdlib.h>
#include <string.h>
#include "glb_host.h"

/* dB thresholds from the host's libm (host/levels.c) on the current device */
int glb_make_level_tables(void **tables)
{
  float *tf = malloc(sizeof(float) * GLB_DB_NTHR);
  double *td = malloc(sizeof(double) * GLB_DB_NTHR);
  if (!tf || !td) { free(tf); free(td); return glb_host_fail(GLFER_ENOMEM, "out of memory"); }
  glb_db_thresholds_f(tf);
  glb_db_thresholds_d(td);
  const int rc = glb_host_shim(glb_level_tables_create(tf, td, GLB_DB_NTHR, tables));
  free(tf); free(td);
  return rc;
}

void glb_display_free(glb_display *d)
{
  glb_free(d->d_agc_state); glb_free(d->d_colortab); glb_free(d->d_level_lut);
  glb_level_tables_destroy(d->level_tables);
  if (d->h_range) glb_host_free(d->h_range);
  memset(d, 0, sizeof *d);
}

void glb_display_slot_free(glb_display_slot *s)
{
  glb_event_destroy(s->ev_agc);
  glb_free(s->d_stats); glb_free(s->d_range); glb_free(s->d_levels); glb_free(s->d_rgb);
  memset(s, 0, sizeof *s);
}

int glb_display_begin(glb_display *d, glb_display_run *r, const glfer_display_config *dc, const float *agc_state,
                      long long nframes, int nchan, int want_range, void *stream)
{
  memset(r, 0, sizeof *r);
  r->dc = dc;
  r->nchan = nchan;
  r->nframes = nframes;
  if (!d->d_agc_state) {
    TRY(glb_malloc((void **) &d->d_agc_state, 2 * GLB_ZOOM_MAX_CHANNELS * sizeof(float)));
    TRY(glb_malloc((void **) &d->d_colortab, 768));
    TRY(glb_malloc((void **) &d->d_level_lut, GLB_DB_NTHR));
    /* the device never evaluates 10 log10 itself */
    const int rt = glb_make_level_tables(&d->level_tables);
    if (rt != 0) return rt;
  }
  if (want_range && dc->autoscale) {
    /* into the caller's array directly, each chunk's copy would block the host thread whenever that array is
       pageable, and with it the chunk pipeline: pinned staging owned by the plan, handed over at the end */
    const size_t bytes = sizeof(float) * 2 * (size_t) nframes * nchan;
    if (bytes > d->h_range_cap) {
      if (d->h_range) glb_host_free(d->h_range);
      d->h_range = NULL; d->h_range_cap = 0;
      const size_t cap = bytes + bytes / 2 + 4096;
      TRY(glb_host_alloc((void **) &d->h_range, cap));
      d->h_range_cap = cap;
    }
    r->st_range = d->h_range;
  }
  float state[2 * GLB_ZOOM_MAX_CHANNELS];
  for (int i = 0; i < 2 * nchan; i++) state[i] = agc_state ? agc_state[i] : 0.0f;
  TRY(glb_memcpy_h2d(d->d_agc_state, state, sizeof(float) * 2 * nchan, stream));
  r->thr = dc->thr_level / 100.0;                            /* g_main.c:1098 */
  if (!dc->autoscale) {
    /* fixed levels, g_main.c:1126-1138; in the log scales the level of every integer dB value is
       tabulated once on the host with the reference's own arithmetic */
    unsigned char lut[GLB_DB_NTHR];
    glb_fixed_display_range(dc->max_level_db, dc->min_level_db, dc->log_scale, &r->fixed[0], &r->fixed[1]);
    glb_level_lut(r->fixed[1], r->fixed[0], r->thr, lut);
    TRY(glb_memcpy_h2d(d->d_level_lut, lut, sizeof lut, stream));
  }
  if (dc->colortab) TRY(glb_memcpy_h2d(d->d_colortab, dc->colortab, 768, stream));
  TRY(glb_stream_sync(stream));
  return 0;
}

int glb_display_reserve(glb_display_slot *s, long long nframes, int nbins, int rgb)
{
  const int rc = glb_ensure((void **) &s->d_levels, &s->levels_cap, (size_t) nframes * nbins, 1);
  if (rc != 0 || !rgb) return rc;
  return glb_ensure((void **) &s->d_rgb, &s->rgb_cap, (size_t) nframes * nbins * 3, 1);
}

int glb_display_map(const glb_display *d, const glb_display_run *r, glb_display_slot *s, const glb_display_slot *prev,
                    const float *d_psd, const float *d_shown, int nbins, long long c0, long long cn, long long crows,
                    long long done, float overlap, int rgb, void *stream)
{
  const glfer_display_config *dc = r->dc;
  const float *d_range = NULL;
  const long long nrows = (r->nchan - 1) * crows + cn;
  if (dc->autoscale) {
    if ((size_t) nrows > s->stats_cap) {
      glb_free(s->d_stats); glb_free(s->d_range);
      s->d_stats = s->d_range = NULL; s->stats_cap = 0;
      TRY(glb_malloc((void **) &s->d_stats, sizeof(float) * 4 * (size_t) nrows));
      TRY(glb_malloc((void **) &s->d_range, sizeof(float) * 2 * (size_t) nrows));
      s->stats_cap = (size_t) nrows;
    }
    /* compute_floor always looks at the raw PSD row (g_main.c:1109) */
    TRY(glb_launch_floor_stats(d_psd, nbins, nbins, nrows, s->d_stats, stream));
    /* the recurrence continues where the previous chunk (other slot) stopped; one chain per channel */
    if (prev) TRY(glb_stream_wait_event(stream, prev->ev_agc));
    for (int c = 0; c < r->nchan; c++)
      TRY(glb_launch_agc(s->d_stats + 4 * c * crows, cn, c0, overlap, dc->log_scale, d->d_agc_state + 2 * c,
                         s->d_range + 2 * c * crows, stream));
    TRY(glb_event_record(s->ev_agc, stream));
    d_range = s->d_range;
    for (int c = 0; r->st_range && c < r->nchan; c++)
      TRY(glb_memcpy_d2h(r->st_range + 2 * (c * r->nframes + done), s->d_range + 2 * c * crows,
                         sizeof(float) * 2 * (size_t) cn, stream));
  }
  /* rows between the channels' rows (crows > cn) are mapped too and never fetched */
  TRY(glb_launch_levels(d_shown, nbins, nbins, nrows, d_range, dc->autoscale ? NULL : r->fixed, dc->log_scale, r->thr,
                        d->level_tables, d->d_level_lut, dc->colortab ? d->d_colortab : NULL, s->d_levels,
                        rgb ? s->d_rgb : NULL, stream));
  return 0;
}

int glb_display_fetch(const glb_display_run *r, const glb_display_slot *s, long long cn, long long crows, int nbins,
                      long long done, unsigned char *levels, unsigned char *rgb, void *stream)
{
  for (int c = 0; c < r->nchan; c++) {
    const size_t to = (size_t) (c * r->nframes + done) * nbins, from = (size_t) (c * crows) * nbins;
    if (levels) TRY(glb_memcpy_d2h(levels + to, s->d_levels + from, (size_t) cn * nbins, stream));
    if (rgb) TRY(glb_memcpy_d2h(rgb + to * 3, s->d_rgb + from * 3, (size_t) cn * nbins * 3, stream));
  }
  return 0;
}

int glb_display_end(const glb_display *d, const glb_display_run *r, long long nframes, float *agc_state,
                    float *range_out)
{
  if (agc_state && r->dc->autoscale)
    TRY(glb_memcpy_d2h(agc_state, d->d_agc_state, 2 * sizeof(float) * r->nchan, NULL));
  if (r->st_range) memcpy(range_out, r->st_range, sizeof(float) * 2 * (size_t) nframes * r->nchan);
  return 0;
}
