// iq_core.cuh -- epilogue of the fused I/Q spectrogram kernel (gram_iq_kernel, iq.cu).
//
// The ring kernel transforms a frame of N = 2M floats as the M complex points z[m] = x[2m] + i x[2m+1] and
// then splits the result into the real FFT of the N floats.  For an interleaved (I, Q) stream those points
// are the complex samples themselves, so the complex FFT of a frame of n = M samples is the ring kernel's
// transform without the split: after the last pass thread t holds (Z[k], Z[M - k]) in (v[rp], v[15 - rp]),
// k = slot_bin<M>(t, 2 rp), and thread 0 also holds Z[M/2] (thread0_fixup, fft_core.cuh).  Power of Z[k]
// goes to row position (k + M/2) mod M, the fft-shifted order of the I/Q contract.
//
// __host__ __device__ like fft_core.cuh, so tests/emu/emu_iq.cpp runs the same functions on the CPU.
#pragma once
#include "fft_core.cuh"

namespace glb {

// |Z|^2 of the thread's bins, by slot (slot 2 rp: bin k, slot 2 rp + 1: bin M - k, slot 16: bin M/2 on thread
// 0).  Thread 0's slot 1 is bin M, i.e. Z[0] again: it is computed but never stored (iq_slot_stored).
// T0 = false: the caller knows that t != 0 (as emit_bins_rt).
template <int M, bool T0 = true>
GLB_HD void iq_emit_power(float2 *v, int t, float scale, float (&yv)[17]) {
  if (T0 && t == 0) {
    const float2 z = thread0_fixup(v);
    yv[16] = scale * norm2(z);
  }
#pragma unroll
  for (int rp = 0; rp < 8; rp++) {
    yv[2 * rp] = scale * norm2(v[rp]);
    yv[2 * rp + 1] = scale * norm2(v[15 - rp]);
  }
}

// The same powers added to a multitaper row's per-slot sums (acc[slot] += scale |Z|^2, the order of iq_emit_power)
template <int M, bool T0 = true>
GLB_HD void iq_add_power(float2 *v, int t, float scale, float (&acc)[17]) {
  if (T0 && t == 0) {
    const float2 z = thread0_fixup(v);
    acc[16] += scale * norm2(z);
  }
#pragma unroll
  for (int rp = 0; rp < 8; rp++) {
    acc[2 * rp] += scale * norm2(v[rp]);
    acc[2 * rp + 1] += scale * norm2(v[15 - rp]);
  }
}

// Harmonic F-test (gram_iq_ftest_kernel, iq.cu; the general path's split kernels, zoom.cu).  The hn transform leaves
// mu by slot (the slots of iq_emit_power) at mu[slot * stride]: stride 1 for an array in registers, the thread count
// for a per-thread column of shared memory.  Each taper's transform then adds its power to acc exactly as
// iq_add_power does, and its residual to den.  The uploaded taper carries taper_scale / sqrt(lambda_k): sl = sqrt(lambda_k)
// undoes the per-taper factor, the common taper_scale cancels in F.  The residual is formed directly: the expanded
// sum |y_k|^2 - |sum U0_k y_k|^2 / S needs no mu but cancels in FP32 on exactly the bins where F is large.
GLB_HD float iq_ftest_resid(float2 z, float2 mu, float u0, float sl) {
  const float rr = z.x * sl - mu.x * u0, ri = z.y * sl - mu.y * u0;
  return rr * rr + ri * ri;
}
// fnum = (K' - 1) S; IEEE division (0 / 0 is NaN, as on an all-zero frame)
GLB_HD float iq_ftest_value(float2 mu, float den, float fnum) { return fnum * norm2(mu) / den; }

template <int M, bool T0 = true>
GLB_HD void iq_emit_mu(float2 *v, int t, float2 *mu, int stride) {
  if (T0 && t == 0) mu[16 * stride] = thread0_fixup(v);
#pragma unroll
  for (int rp = 0; rp < 8; rp++) {
    mu[2 * rp * stride] = v[rp];
    mu[(2 * rp + 1) * stride] = v[15 - rp];
  }
}

template <int M, bool T0 = true>
GLB_HD void iq_add_ftest(float2 *v, int t, float scale, float u0, float sl, const float2 *mu, int stride,
                         float (&acc)[17], float (&den)[17]) {
  if (T0 && t == 0) {
    const float2 z = thread0_fixup(v);
    acc[16] += scale * norm2(z);
    den[16] += iq_ftest_resid(z, mu[16 * stride], u0, sl);
  }
#pragma unroll
  for (int rp = 0; rp < 8; rp++) {
    acc[2 * rp] += scale * norm2(v[rp]);
    acc[2 * rp + 1] += scale * norm2(v[15 - rp]);
    den[2 * rp] += iq_ftest_resid(v[rp], mu[2 * rp * stride], u0, sl);
    den[2 * rp + 1] += iq_ftest_resid(v[15 - rp], mu[(2 * rp + 1) * stride], u0, sl);
  }
}

template <int M> GLB_HD bool iq_slot_stored(int t, int slot) { return slot == 16 ? t == 0 : !(t == 0 && slot == 1); }

// Row positions as four per-thread bases plus compile-time offsets (the stores of a warp cover 32
// consecutive floats, ascending for slots 2 rp and descending for slots 2 rp + 1, as the real kernel's):
//   rp < 4 : k = t + 2 rp T      -> t + 8T + 2 rp T,             M - k -> 8T - t - 2 rp T
//   rp >= 4: k = khi + 2(rp-4) T -> (t ? t - 8T : T) + 2 rp T,   M - k -> (t ? 24T - t : 15T) - 2 rp T
// slot 16 (Z[M/2]) lands at position 0.
template <int M> GLB_HD void iq_row_bases(int t, int (&b)[4]) {
  constexpr int T = M / kPoints;
  b[0] = t + 8 * T;
  b[1] = 8 * T - t;
  b[2] = t != 0 ? t - 8 * T : T;
  b[3] = t != 0 ? 24 * T - t : 15 * T;
}
template <int M> GLB_HD int iq_slot_offset(const int (&b)[4], int slot) {
  constexpr int T = M / kPoints;
  if (slot == 16) return 0;
  const int rp = slot >> 1, hi = rp >= 4 ? 2 : 0;
  return (slot & 1) ? b[1 + hi] - 2 * rp * T : b[hi] + 2 * rp * T;
}

// Display pixels of the LEV epilogue: pixel i shows row position M - 1 - i (highest frequency first, as
// main_window_draw draws a row), so the bases are the row bases mirrored and the offsets change sign.  A run of
// 32 consecutive row positions stays 32 consecutive bytes, now descending for slots 2 rp and ascending for
// slots 2 rp + 1; slot 16 (row position 0) lands on pixel M - 1.
template <int M> GLB_HD void iq_pixel_bases(int t, int (&b)[4]) {
  iq_row_bases<M>(t, b);
#pragma unroll
  for (int i = 0; i < 4; i++) b[i] = M - 1 - b[i];
}
template <int M> GLB_HD int iq_pixel_offset(const int (&b)[4], int slot) {
  constexpr int T = M / kPoints;
  if (slot == 16) return M - 1;
  const int rp = slot >> 1, hi = rp >= 4 ? 2 : 0;
  return (slot & 1) ? b[1 + hi] + 2 * rp * T : b[hi] - 2 * rp * T;
}

}  // namespace glb
