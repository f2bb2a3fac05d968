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

#define DTRY(x) do { int rc_ = glb_host_shim(x); if (rc_ != 0) return rc_; } while (0)

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

static int dgrow(void **ptr, size_t *cap, size_t want)
{
  if (want <= *cap) return 0;
  if (*ptr) DTRY(glb_free(*ptr));
  *ptr = NULL;
  *cap = 0;
  DTRY(glb_malloc(ptr, want));
  *cap = want;
  return 0;
}

int glb_display_begin(glb_display *d, glb_display_run *r, const glfer_display_config *dc, const float *agc_state,
                      long long nframes, int want_range, void *stream)
{
  memset(r, 0, sizeof *r);
  r->dc = dc;
  if (!d->d_agc_state) {
    DTRY(glb_malloc((void **) &d->d_agc_state, 2 * sizeof(float)));
    DTRY(glb_malloc((void **) &d->d_colortab, 768));
    DTRY(glb_malloc((void **) &d->d_level_lut, GLB_DB_NTHR));
    /* the device never evaluates 10 log10 itself */
    const int rt = glb_make_level_tables(&d->level_tables);
    if (rt != 0) return rt;
  }
  if (want_range && dc->autoscale) {
    /* into the caller's array directly, each chunk's copy would block the host thread whenever that array is
       pageable, and with it the chunk pipeline: pinned staging owned by the plan, handed over at the end */
    const size_t bytes = sizeof(float) * 2 * (size_t) nframes;
    if (bytes > d->h_range_cap) {
      if (d->h_range) glb_host_free(d->h_range);
      d->h_range = NULL; d->h_range_cap = 0;
      const size_t cap = bytes + bytes / 2 + 4096;
      DTRY(glb_host_alloc((void **) &d->h_range, cap));
      d->h_range_cap = cap;
    }
    r->st_range = d->h_range;
  }
  float state[2] = { agc_state ? agc_state[0] : 0.0f, agc_state ? agc_state[1] : 0.0f };
  DTRY(glb_memcpy_h2d(d->d_agc_state, state, sizeof state, stream));
  r->thr = dc->thr_level / 100.0;                            /* g_main.c:1098 */
  if (!dc->autoscale) {
    /* fixed levels, g_main.c:1126-1138; in the log scales the level of every integer dB value is
       tabulated once on the host with the reference's own arithmetic */
    unsigned char lut[GLB_DB_NTHR];
    glb_fixed_display_range(dc->max_level_db, dc->min_level_db, dc->log_scale, &r->fixed[0], &r->fixed[1]);
    glb_level_lut(r->fixed[1], r->fixed[0], r->thr, lut);
    DTRY(glb_memcpy_h2d(d->d_level_lut, lut, sizeof lut, stream));
  }
  if (dc->colortab) DTRY(glb_memcpy_h2d(d->d_colortab, dc->colortab, 768, stream));
  DTRY(glb_stream_sync(stream));
  return 0;
}

int glb_display_reserve(glb_display_slot *s, long long nframes, int nbins, int rgb)
{
  const int rc = dgrow((void **) &s->d_levels, &s->levels_cap, (size_t) nframes * nbins);
  if (rc != 0 || !rgb) return rc;
  return dgrow((void **) &s->d_rgb, &s->rgb_cap, (size_t) nframes * nbins * 3);
}

int glb_display_map(const glb_display *d, const glb_display_run *r, glb_display_slot *s, const glb_display_slot *prev,
                    const float *d_psd, const float *d_shown, int nbins, long long c0, long long cn, long long done,
                    float overlap, int rgb, void *stream)
{
  const glfer_display_config *dc = r->dc;
  const float *d_range = NULL;
  if (dc->autoscale) {
    if ((size_t) cn > s->stats_cap) {
      glb_free(s->d_stats); glb_free(s->d_range);
      s->d_stats = s->d_range = NULL; s->stats_cap = 0;
      DTRY(glb_malloc((void **) &s->d_stats, sizeof(float) * 4 * (size_t) cn));
      DTRY(glb_malloc((void **) &s->d_range, sizeof(float) * 2 * (size_t) cn));
      s->stats_cap = (size_t) cn;
    }
    /* compute_floor always looks at the raw PSD row (g_main.c:1109) */
    DTRY(glb_launch_floor_stats(d_psd, nbins, nbins, cn, s->d_stats, stream));
    /* the recurrence continues where the previous chunk (other slot) stopped */
    if (prev) DTRY(glb_stream_wait_event(stream, prev->ev_agc));
    DTRY(glb_launch_agc(s->d_stats, cn, c0, overlap, dc->log_scale, d->d_agc_state, s->d_range, stream));
    DTRY(glb_event_record(s->ev_agc, stream));
    d_range = s->d_range;
    if (r->st_range) DTRY(glb_memcpy_d2h(r->st_range + 2 * done, s->d_range, sizeof(float) * 2 * (size_t) cn, stream));
  }
  DTRY(glb_launch_levels(d_shown, nbins, nbins, cn, d_range, dc->autoscale ? NULL : r->fixed, dc->log_scale, r->thr,
                         d->level_tables, d->d_level_lut, dc->colortab ? d->d_colortab : NULL, s->d_levels,
                         rgb ? s->d_rgb : NULL, stream));
  return 0;
}

int glb_display_fetch(const glb_display_slot *s, long long cn, int nbins, long long done, unsigned char *levels,
                      unsigned char *rgb, void *stream)
{
  if (levels) DTRY(glb_memcpy_d2h(levels + (size_t) done * nbins, s->d_levels, (size_t) cn * nbins, stream));
  if (rgb) DTRY(glb_memcpy_d2h(rgb + (size_t) done * nbins * 3, s->d_rgb, (size_t) cn * nbins * 3, stream));
  return 0;
}

int glb_display_end(const glb_display *d, const glb_display_run *r, long long nframes, float *agc_state,
                    float *range_out)
{
  if (agc_state && r->dc->autoscale) DTRY(glb_memcpy_d2h(agc_state, d->d_agc_state, 2 * sizeof(float), NULL));
  if (r->st_range) memcpy(range_out, r->st_range, sizeof(float) * 2 * (size_t) nframes);
  return 0;
}
