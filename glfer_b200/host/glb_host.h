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
int glb_hop(int n, float overlap);
/* the message slot of glfer_b200_last_error() (gram.c), for the other host units */
int glb_host_fail(int code, const char *msg);
int glb_host_shim(int rc);
void glb_host_clear_error(void);
#define TRY(x) do { int rc_ = glb_host_shim(x); if (rc_ != 0) return rc_; } while (0)
/* grow-only device buffer (gram.c): *ptr holds at least want elements of elem bytes, *cap counts elements */
int glb_ensure(void **ptr, size_t *cap, size_t want, size_t elem);

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
  int nchan;                    /* channels: the caller's arrays are [nchan][nframes]..., one AGC chain each */
  long long nframes;
} glb_display_run;
int glb_make_level_tables(void **tables);
void glb_display_free(glb_display *d);
void glb_display_slot_free(glb_display_slot *s);
/* device state for a run (synchronises `stream`); nchan: channels of a zoom bank (1..GLB_ZOOM_MAX_CHANNELS, 1
 * elsewhere), agc_state [nchan][2]; want_range: the caller asked for display_range */
int glb_display_begin(glb_display *d, glb_display_run *r, const glfer_display_config *dc, const float *agc_state,
                      long long nframes, int nchan, int want_range, void *stream);
/* the slot's level (and RGB) buffers for nframes rows of nbins */
int glb_display_reserve(glb_display_slot *s, long long nframes, int nbins, int rgb);
/* levels (and RGB) of the cn device rows d_shown (floor statistics of d_psd when autoscaling) of frames [c0, c0 + cn),
 * frames [done, done + cn) of the run; channel c's rows start at row c crows (crows >= cn; the slot is reserved for
 * (nchan - 1) crows + cn rows); prev: the slot of the run's previous chunk, or NULL for the first */
int glb_display_map(const glb_display *d, const glb_display_run *r, glb_display_slot *s, const glb_display_slot *prev,
                    const float *d_psd, const float *d_shown, int nbins, long long c0, long long cn, long long crows,
                    long long done, float overlap, int rgb, void *stream);
/* download the slot's levels / RGB (either may be NULL) of each channel to its rows [done, done + cn) */
int glb_display_fetch(const glb_display_run *r, const glb_display_slot *s, long long cn, long long crows, int nbins,
                      long long done, unsigned char *levels, unsigned char *rgb, void *stream);
/* after the run's streams are synchronised: the carried AGC state and the staged display range */
int glb_display_end(const glb_display *d, const glb_display_run *r, long long nframes, float *agc_state,
                    float *range_out);
/* testing aid glfer_b200_set_fused_levels (gram.c): 0 = levels always in a second pass over float rows */
int glb_host_fused_levels(void);

/* the complex frame stage of the I/Q and zoom plans (host/cframe.c): everything after a chunk's complex samples are
 * on the device.  Chunks in flight: three, as the real plan's (gram.c). */
#define GLB_CSLOTS 3
typedef struct {                /* per slot (stream); embedded in the plan's own slot */
  void *stream;
  float *d_rows;
  size_t rows_cap;              /* floats */
  float *d_ftest;               /* F rows (*_mtm_ftest) */
  size_t ftest_cap;             /* floats */
  void *d_scratch;              /* the general path's (glb_iq_gram_scratch_bytes) */
  size_t scratch_cap;           /* bytes */
  glb_display_slot disp;        /* display mapping */
  void *d_lines, *h_lines;      /* *_run_mtm_lines: the chunk's line arrays on the device and their pinned staging */
  size_t dlines_cap, hlines_cap;     /* bytes */
  long long lines_done, lines_cn;    /* h_lines holds frames [lines_done, lines_done + lines_cn) of the run (0: none) */
} glb_cslot;
typedef struct {                /* per plan */
  int n, hop, device;
  float overlap;
  float *d_taper;               /* [ntapers][2n]: w[i] (or v_k[i] / sqrt(lambda_k)) on both halves of complex sample i,
                                   times taper_scale */
  int taper_sym;                /* bit k: taper k is mirror-symmetric bit for bit */
  float taper_scale;            /* 1 / (2 sqrt(2n)) */
  int ntapers;                  /* 1: periodogram, K' = mtm_kmax + 1: multitaper */
  double *h_tapers, *h_lambda;  /* multitaper: the unscaled DPSS [K'][n] and eigenvalues */
  float *d_ftab;                /* multitaper: the F-test's table: hn [2n], then (U0_k, sqrt(lambda_k)) [K'] */
  float ftest_s;                /* S = sum_k U0_k^2 */
  void *tables;                 /* FFT tables of the 2n-float frames */
  glb_display disp;
  glb_cslot *slot[GLB_CSLOTS];  /* in the plan's slots */
} glb_cframe;
/* Validates n (size_msg: the plan's message), window_type, overlap and, for mtm, the DPSS parameters before any device
 * call; then selects the device, uploads the taper table (the window, or the K' DPSS tapers) and the F-test's table,
 * builds the FFT tables and creates the slots' streams.  On failure f owns nothing and the message is kept. */
int glb_cframe_create(glb_cframe *f, glb_cslot *const slot[GLB_CSLOTS], int n, int window_type, float overlap,
                      int device, int mtm, float mtm_w, int mtm_kmax, const char *size_msg);
/* synchronises and frees the slots' buffers and streams and the plan's tables (not f itself) */
void glb_cframe_destroy(glb_cframe *f);
/* glfer_iq_tapers / glfer_zoom_tapers (f: NULL for a NULL plan) */
int glb_cframe_tapers(const glb_cframe *f, double *tapers, double *lambda);
typedef struct glb_cframe_call glb_cframe_call;
/* the plan's stage of a chunk: the complex samples that frames [c0, c0 + cn) read, on the device of slot i (prev: the
 * slot of the run's previous chunk, or -1), on that slot's stream; *z holds samples [*z_origin, *z_origin + *z_count).
 * A call with nchan > 1 channels lays channel c's samples at z + c z_stride (complex samples, z_stride = crows hop),
 * so that frame c0 + c crows + j of one launch is frame c0 + j of channel c; the stage zeroes what a channel c >= 1
 * frame reads before its channel's samples (stream indices < 0), and *z_count covers the last channel. */
typedef int (*glb_cframe_stage)(void *plan, const glb_cframe_call *c, int i, int prev, long long c0, long long cn,
                                long long z_stride, const float **z, long long *z_origin, long long *z_count);
struct glb_cframe_call {        /* one run entry's call */
  const void *src;              /* the caller's samples [origin, origin + count), float or int16 (pcm16) */
  int pcm16;
  long long origin, count, first_frame, nframes;
  int ftest_on;                 /* a *_mtm_ftest entry: rows or ftest may be NULL */
  float *rows, *ftest;
  int display;                  /* a *_run_display entry: levels / RGB of dc's mapping */
  const glfer_display_config *dc;
  float *agc_state, *range_out;
  unsigned char *levels, *rgb;
  int lines;                    /* a *_run_mtm_lines entry: the F rows stay on the device, only the lines come back */
  const glfer_lines_config *lc;
  int *line_count, *line_bin;
  float *line_ftest, *line_psd;
  /* from the plan */
  int nchan;                    /* channels (zoom bank): the caller's outputs are [nchan][nframes]...; 0 or 1: one */
  void *plan;
  glb_cframe_stage stage;
  long long chunk_frames;
  long long lo, hi;             /* the plan's required span of the frames */
  int general;                  /* 1: glb_launch_iq_gram_general (the zoom), 0: glb_launch_iq_gram */
  int fuse;                     /* display: the spectrogram kernel writes fixed-range levels itself, no float rows */
  const char *wrong_kind;       /* non-NULL: the entry does not serve this plan (checked after the null arguments) */
  const char *no_mtm, *short_span;   /* the plan's messages: F-test without a multitaper plan, samples short */
};
/* checks the call, then walks its frames in chunks of chunk_frames on the slots in turn: the plan's stage, the launch,
 * and the rows / F rows downloads, the display chain or the line selection */
int glb_cframe_run(glb_cframe *f, const glb_cframe_call *c);

/* values of the hidden globals (weak `opt` / `glfer` when the host program has them) */
int glb_autoscale(void);
int glb_first_buffer(void);

/* abort the way the reference does on allocation failure (fft.c:249-252) */
void glb_fatal(const char *where);

#endif
