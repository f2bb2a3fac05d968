/* dpss.c -- discrete prolate spheroidal (Slepian) tapers, host, double precision.
 *
 * A fresh implementation of the method the reference uses (g-l_dpss.c:288-347, after
 * Thomson 1982 appendix A): the sinc kernel sin(c(x-y)) / (pi(x-y)), c = pi * NW, is
 * discretised on the 32 Gauss-Legendre nodes of [-1,1] and symmetrised with the square
 * roots of the weights; the eigenvectors of that 32x32 matrix, ordered by |eigenvalue|
 * descending, are interpolated through the same kernel to n points centred at
 * 2(i + 1/2)/n - 1 and normalised to unit energy.  sig[k] = lambda_k - 1.
 * Eigenvectors are determined up to sign (and up to rotation inside numerically
 * degenerate eigenvalue clusters); the multitaper PSD is invariant to both.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include "glb_host.h"

#define GLQ 32

/* nodes and weights of the GLQ-point Gauss-Legendre rule by Newton iteration on P_n */
static void gauss_legendre(double *x, double *w)
{
  for (int i = 0; i < (GLQ + 1) / 2; i++) {
    double z = cos(M_PI * (i + 0.75) / (GLQ + 0.5));
    double pp = 1.0;
    for (int it = 0; it < 100; it++) {
      double p0 = 1.0, p1 = z;
      for (int k = 2; k <= GLQ; k++) {
        const double p2 = ((2.0 * k - 1.0) * z * p1 - (k - 1.0) * p0) / k;
        p0 = p1;
        p1 = p2;
      }
      pp = GLQ * (z * p1 - p0) / (z * z - 1.0);
      const double dz = p1 / pp;
      z -= dz;
      if (fabs(dz) < 1e-16) break;
    }
    x[i] = -z;
    x[GLQ - 1 - i] = z;
    w[i] = w[GLQ - 1 - i] = 2.0 / ((1.0 - z * z) * pp * pp);
  }
}

/* cyclic Jacobi eigen-solver for a dense symmetric matrix (row-major, n x n).
 * On return d[] holds the eigenvalues and the columns of e the eigenvectors. */
static int jacobi_eigen(double *a, int n, double *d, double *e, int max_sweeps)
{
  for (int i = 0; i < n; i++)
    for (int j = 0; j < n; j++) e[i * n + j] = (i == j) ? 1.0 : 0.0;
  for (int sweep = 0; sweep < max_sweeps; sweep++) {
    double off = 0.0;
    for (int p = 0; p < n; p++)
      for (int q = p + 1; q < n; q++) off += a[p * n + q] * a[p * n + q];
    if (off == 0.0) break;
    for (int p = 0; p < n - 1; p++) {
      for (int q = p + 1; q < n; q++) {
        const double apq = a[p * n + q];
        if (apq == 0.0) continue;
        const double app = a[p * n + p], aqq = a[q * n + q];
        if (fabs(apq) < 1e-300 || (fabs(app) + 100.0 * fabs(apq) == fabs(app) && fabs(aqq) + 100.0 * fabs(apq) == fabs(aqq))) {
          a[p * n + q] = a[q * n + p] = 0.0;
          continue;
        }
        const double theta = (aqq - app) / (2.0 * apq);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < n; k++) {              /* columns p, q */
          const double akp = a[k * n + p], akq = a[k * n + q];
          a[k * n + p] = c * akp - s * akq;
          a[k * n + q] = s * akp + c * akq;
        }
        for (int k = 0; k < n; k++) {              /* rows p, q */
          const double apk = a[p * n + k], aqk = a[q * n + k];
          a[p * n + k] = c * apk - s * aqk;
          a[q * n + k] = s * apk + c * aqk;
        }
        a[p * n + q] = a[q * n + p] = 0.0;
        for (int k = 0; k < n; k++) {
          const double ekp = e[k * n + p], ekq = e[k * n + q];
          e[k * n + p] = c * ekp - s * ekq;
          e[k * n + q] = s * ekp + c * ekq;
        }
      }
    }
  }
  for (int i = 0; i < n; i++) d[i] = a[i * n + i];
  return 0;
}

/* tapers: [kmax+1][n] row-major doubles; lambda: [kmax+1] */
int glb_dpss(int n, double nw, int kmax, double *tapers, double *lambda)
{
  if (n < 1 || kmax < 0 || kmax >= GLQ) return -1;
  double gx[GLQ], gw[GLQ], ker[GLQ * GLQ], ev[GLQ], evec[GLQ * GLQ];
  const double c = M_PI * nw;
  gauss_legendre(gx, gw);
  for (int i = 0; i < GLQ; i++)
    for (int j = 0; j < GLQ; j++) {
      const double d = gx[i] - gx[j];
      const double k = (i == j) ? c / M_PI : sin(c * d) / (M_PI * d);
      ker[i * GLQ + j] = k * sqrt(gw[i] * gw[j]);
    }
  jacobi_eigen(ker, GLQ, ev, evec, 100);
  /* order by |eigenvalue| descending (stable selection) */
  int order[GLQ];
  for (int i = 0; i < GLQ; i++) order[i] = i;
  for (int i = 0; i < GLQ - 1; i++) {
    int best = i;
    for (int j = i + 1; j < GLQ; j++)
      if (fabs(ev[order[j]]) > fabs(ev[order[best]])) best = j;
    const int tmp = order[i];
    order[i] = order[best];
    order[best] = tmp;
  }
  /* interpolate: v_k[i] = sum_j sqrt(w_j) E[j][k] sin(c a) / (pi a), a = 2(i+.5)/n - 1 - x_j */
  double sw[GLQ];
  for (int j = 0; j < GLQ; j++) sw[j] = sqrt(gw[j]);
  for (int k = 0; k <= kmax; k++) memset(tapers + (size_t) k * n, 0, sizeof(double) * n);
  for (int i = 0; i < n; i++) {
    double sinc[GLQ];
    for (int j = 0; j < GLQ; j++) {
      const double a = (2.0 * (i + 0.5) / n) - 1.0 - gx[j];
      sinc[j] = sw[j] * sin(c * a) / (M_PI * a);
    }
    for (int k = 0; k <= kmax; k++) {
      const int col = order[k];
      double acc = 0.0;
      for (int j = 0; j < GLQ; j++) acc += sinc[j] * evec[j * GLQ + col];
      tapers[(size_t) k * n + i] = acc;
    }
  }
  for (int k = 0; k <= kmax; k++) {
    double *v = tapers + (size_t) k * n;
    double e = 0.0;
    for (int i = 0; i < n; i++) e += v[i] * v[i];
    const double r = sqrt(e);
    for (int i = 0; i < n; i++) v[i] /= r;
    lambda[k] = ev[order[k]];
  }
  return 0;
}

/* reference-compatible entry point (g-l_dpss.h:23): v is an NR-style 1-offset matrix */
int gl_dpss(int nmax, int kmax, int n, double w, double **v, double *sig, int *totit)
{
  (void) nmax;
  double *tap = malloc(sizeof(double) * (size_t) (kmax + 1) * n);
  double *lam = malloc(sizeof(double) * (kmax + 1));
  if (!tap || !lam) { free(tap); free(lam); return -1; }
  const int rc = glb_dpss(n, w, kmax, tap, lam);
  if (rc == 0) {
    for (int k = 0; k <= kmax; k++) {
      sig[k] = lam[k] - 1.0;
      for (int i = 0; i < n; i++) v[i + 1][k] = tap[(size_t) k * n + i];
    }
  }
  if (totit) *totit = 0;
  free(tap);
  free(lam);
  return rc;
}

/* The harmonic F-test's weights of K unit-energy tapers [K][n] (mtm_init, mtm.c:78-84,123-136): u0[k] = sum_i v_k[i] in
 * double, s = sum_k u0[k]^2 and hn[i] = sum_k u0[k] v_k[i] / s through float accumulators, as the reference rounds them.
 * Shared by the real multitaper plan (host/gram.c) and the complex ones (host/iq.c, host/zoom.c). */
void glb_mtm_ftest_weights(int n, int K, const double *tapers, double *u0, float *hn, float *s)
{
  float s2 = 0.0f;
  for (int k = 0; k < K; k++) {
    double acc = 0.0;
    for (int i = 0; i < n; i++) acc += tapers[(size_t) k * n + i];
    u0[k] = acc;
    s2 += u0[k] * u0[k];
  }
  for (int i = 0; i < n; i++) {
    float h = 0.0f;
    for (int k = 0; k < K; k++) h += u0[k] * tapers[(size_t) k * n + i];
    hn[i] = h / s2;
  }
  *s = s2;
}

/* include/glfer_b200.h: the F(2, 2K' - 2) threshold of a per-bin false-alarm probability, in double, rounded to float */
int glfer_ftest_threshold(int ntapers, double pfa, float *thr)
{
  if (!thr) return glb_host_fail(GLFER_EINVAL, "null argument");
  if (ntapers < 2) return glb_host_fail(GLFER_EINVAL, "the F-test needs K' >= 2 tapers (K' - 1 degrees of freedom)");
  if (!(pfa > 0.0 && pfa < 1.0)) return glb_host_fail(GLFER_EINVAL, "pfa must be in (0, 1)");
  const double m = ntapers - 1;
  *thr = (float) (m * expm1(-log(pfa) / m));
  return 0;
}
