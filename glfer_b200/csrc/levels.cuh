// levels.cuh -- device side of the display mapping (main_window_draw, g_main.c:1186-1229), shared by the
// spectrogram kernels (fused 8-bit output) and levels_kernel (rows already in HBM).
//
// Log scales: the level is (short) (10.0 * log10(x)) evaluated by the host's libm (see host/levels.c).
// The device never evaluates that expression; it locates x between the host-computed thresholds
// thr[j - JMIN] = smallest float with level >= j.  lg2.approx gives 10 log10 x to ~1.2e-4 dB, so
// unless the estimate lies within 5e-4 dB of an integer its truncation is the exact level; the rare
// remaining inputs (and zero / negative / non-finite ones) take a binary search over the table.
#pragma once
#include <cuda_runtime.h>

namespace glb {

constexpr int kDbJmin = -450, kDbJmax = 390, kDbN = kDbJmax - kDbJmin + 1;   // host/glb_host.h GLB_DB_*

// largest j with thr[j - JMIN] <= x; JMIN when x is below every threshold
__device__ __forceinline__ int db_search(float x, const float *__restrict__ thr) {
  int lo = 0, hi = kDbN - 1;            // invariant: thr[lo] <= x (thr[0] is the smallest subnormal)
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (__ldg(thr + mid) <= x) lo = mid; else hi = mid - 1;
  }
  return lo + kDbJmin;
}

// (short) (10.0 * log10((double) x)) as the x86-64 host computes it
__device__ __forceinline__ int trunc_db(float x, const float *__restrict__ thr) {
  if (!(x > 0.f) || x > 3.4028234e38f) return 0;         // 0, negative, NaN, +inf: cvttsd2si overflow -> (short) 0
  const float d = 3.0102999566398120f * __log2f(x);       // 10 log10 x, |error| < 1.2e-4 over the float range
  const float r = (d + 12582912.f) - 12582912.f;          // nearest integer (|d| < 2^22)
  if (fabsf(d - r) < 5e-4f || x < 1.1754944e-38f) return db_search(x, thr);
  return (int) d;                                          // truncation towards zero, as the C conversion
}

// the same for a double input (averaged rows are doubles in the reference, g_main.c:1193)
__device__ __forceinline__ int trunc_db(double x, const double *__restrict__ thr) {
  if (!(x > 0.0) || x > 1.7976931348623157e308) return 0;
  const float xf = (float) x;
  if (xf >= 1.1754944e-38f && xf <= 3.4028234e38f) {
    const float d = 3.0102999566398120f * __log2f(xf);    // rounding x to float moves d by < 3e-6 dB
    const float r = (d + 12582912.f) - 12582912.f;
    if (fabsf(d - r) >= 5e-4f) return (int) d;
  }
  int lo = 0, hi = kDbN - 1;
  if (x < thr[0]) return kDbJmin;                          // below 1e-45: level < JMIN cannot reach the palette
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (thr[mid] <= x) lo = mid; else hi = mid - 1;
  }
  return lo + kDbJmin;
}

// g_main.c:1206,1221-1229
__device__ __forceinline__ unsigned char level_u8(float sig_level, float dmin, float dmax, float thr) {
  const float f = 255 * ((sig_level - dmin) / (dmax - dmin));
  if ((double) f < 255.0 * (double) thr) return 0;
  if (f > 255) return 255;
  if (thr == 0.f) return (unsigned char) f;                // (f - 0) / 1 in double is f itself
  return (unsigned char) (((double) f - 255.0 * (double) thr) / (1.0 - (double) thr));
}

// the device tables behind glb_level_tables_create's handle
struct LevelTables {
  float *thr_f;
  double *thr_d;
};

// what the fused epilogue and levels_kernel need to map a value
struct LevelMap {
  const float *thr;            // [kDbN] float thresholds (log scales)
  const unsigned char *lut;    // [kDbN] level of integer dB j for a FIXED display range, or nullptr
  int log_scale;
  float dmin, dmax, thr_level; // display range (dB in the log scales) and threshold fraction when lut == nullptr
};

__device__ __forceinline__ unsigned char map_level(float x, const LevelMap &m) {
  if (m.log_scale) {
    const int s = trunc_db(x, m.thr);
    if (m.lut) return __ldg(m.lut + (s - kDbJmin));
    return level_u8((float) s, m.dmin, m.dmax, m.thr_level);
  }
  return level_u8(x, m.dmin, m.dmax, m.thr_level);
}

}  // namespace glb
