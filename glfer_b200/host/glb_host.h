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

/* values of the hidden globals (weak `opt` / `glfer` when the host program has them) */
int glb_autoscale(void);
int glb_first_buffer(void);

/* abort the way the reference does on allocation failure (fft.c:249-252) */
void glb_fatal(const char *where);

#endif
