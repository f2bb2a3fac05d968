/* glb_host.h -- internals shared by the C host layer (not installed). */
#ifndef GLB_HOST_H
#define GLB_HOST_H

#include "../../include/fft.h"
#include "../../include/mtm.h"
#include "../../include/avg.h"
#include "../../include/lmp.h"
#include "../../include/glfer_b200.h"
#include "../../include/glb_shim.h"

double glb_bessel_i0(double x);
void glb_window_table(int n, int window_type, float *w);
int glb_dpss(int n, double nw, int kmax, double *tapers, double *lambda);
/* host/dpss.c: U0 (double), S and hn (float) of the harmonic F-test from K unit-energy tapers [K][n] */
void glb_mtm_ftest_weights(int n, int K, const double *tapers, double *u0, float *hn, float *s);
/* host/iq.c: DPSS and [K'][2n] taper table of a complex multitaper plan (I/Q or zoom); sym: bit k = taper k mirror-symmetric */
int glb_iq_mtm_tapers(int n, float mtm_w, int mtm_kmax, float taper_scale, double **h_tapers, double **h_lambda,
                      float **table, int *sym);
/* host/iq.c: the F-test's device table of a complex multitaper plan, hn [2n] then (U0_k, sqrt(lambda_k)) [K'], and S */
int glb_iq_ftest_table(int n, int K, const double *h_tapers, const double *h_lambda, float taper_scale, float **d_ftab,
                       float *s);
int glb_hop(int n, float overlap);
/* the message slot of glfer_b200_last_error() (gram.c), for the other host units */
int glb_host_fail(int code, const char *msg);
int glb_host_shim(int rc);
void glb_host_clear_error(void);

/* display mapping tables (host/levels.c) */
#define GLB_DB_JMIN (-450)
#define GLB_DB_JMAX 390
#define GLB_DB_NTHR (GLB_DB_JMAX - GLB_DB_JMIN + 1)
int glb_short_db_f(float x);
int glb_short_db_d(double x);
void glb_db_thresholds_f(float *thr);
void glb_db_thresholds_d(double *thr);
unsigned char glb_level_u8(float sig_level, float dmin, float dmax, float thr);
void glb_level_lut(float dmin, float dmax, float thr, unsigned char *lut);
void glb_fixed_display_range(float max_level_db, float min_level_db, int log_scale, float *dmax, float *dmin);

/* the display chain over device rows (host/display.c), shared by the plans' *_run_display entries */
typedef struct {                /* per plan */
  float *d_agc_state;           /* carried AGC levels (display_max_lvl, display_min_lvl) */
  unsigned char *d_colortab, *d_level_lut;
  void *level_tables;           /* dB thresholds on the device (host/levels.c) */
  float *h_range;               /* pinned staging of the per-frame display range */
  size_t h_range_cap;           /* bytes */
} glb_display;
typedef struct {                /* per slot (stream) of a plan */
  void *ev_agc;                 /* this slot's AGC step is queued: the next chunk's recurrence waits for it */
  float *d_stats, *d_range;
  unsigned char *d_levels, *d_rgb;
  size_t stats_cap, levels_cap, rgb_cap;
} glb_display_slot;
typedef struct {                /* one run */
  const glfer_display_config *dc;
  float thr;                    /* thr_level / 100 */
  float fixed[2];               /* fixed display range (display_max, display_min), dB in the log scales */
  float *st_range;              /* staging of the caller's display_range, or NULL */
} glb_display_run;
int glb_make_level_tables(void **tables);
void glb_display_free(glb_display *d);
void glb_display_slot_free(glb_display_slot *s);
/* device state for a run (synchronises `stream`); want_range: the caller asked for display_range */
int glb_display_begin(glb_display *d, glb_display_run *r, const glfer_display_config *dc, const float *agc_state,
                      long long nframes, int want_range, void *stream);
/* the slot's level (and RGB) buffers for nframes rows of nbins */
int glb_display_reserve(glb_display_slot *s, long long nframes, int nbins, int rgb);
/* levels (and RGB) of the cn device rows d_shown (floor statistics of d_psd when autoscaling) of frames [c0, c0 + cn),
 * frames [done, done + cn) of the run; prev: the slot of the run's previous chunk, or NULL for the first */
int glb_display_map(const glb_display *d, const glb_display_run *r, glb_display_slot *s, const glb_display_slot *prev,
                    const float *d_psd, const float *d_shown, int nbins, long long c0, long long cn, long long done,
                    float overlap, int rgb, void *stream);
/* download the slot's levels / RGB (either may be NULL) to rows [done, done + cn) */
int glb_display_fetch(const glb_display_slot *s, long long cn, int nbins, long long done, unsigned char *levels,
                      unsigned char *rgb, void *stream);
/* after the run's streams are synchronised: the carried AGC state and the staged display range */
int glb_display_end(const glb_display *d, const glb_display_run *r, long long nframes, float *agc_state,
                    float *range_out);
/* testing aid glfer_b200_set_fused_levels (gram.c): 0 = levels always in a second pass over float rows */
int glb_host_fused_levels(void);

/* values of the hidden globals (weak `opt` / `glfer` when the host program has them) */
int glb_autoscale(void);
int glb_first_buffer(void);

/* abort the way the reference does on allocation failure (fft.c:249-252) */
void glb_fatal(const char *where);

#endif
