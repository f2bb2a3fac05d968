// zoom.cu -- kernels of the zoom spectrogram (host/zoom.c): mix a centre frequency to DC, low-pass and
// decimate by D, then turn the general spectrogram kernel's real-FFT output of the decimated stream into
// complex-FFT rows.
//
//   zoom_decim_kernel<T>  the hot path.  y[m] = e^{-2 pi i phi(mD)} sum_j g[j] x[mD - K + j], j = 0..2K,
//                         with the complex taps g[j] = h[K - j] e^{+2 pi i phi(K - j)} built on the host.
//                         Polyphase form: phase p = j mod D owns the 33 taps g[p + tD] (zero-padded past
//                         2K), and its contribution to output m is a 33-tap FIR over the stream
//                         u_p[q] = x[qD - K + p].  A lane holds the taps of one phase in registers and
//                         streams u_p once for kZR consecutive outputs: each loaded sample feeds up to
//                         2 kZR FMAs, so the loop runs on the FP32 pipe, not on loads.  Lanes take
//                         consecutive phases (coalesced loads of x and of the taps, no shared-memory
//                         stride-D access); a lane walks the phases p = sl, sl + 32, ... of its group in
//                         order, and the lane partials are summed in a fixed order through shared memory.
//                         The sum order of an output therefore depends on D only, never on where the
//                         output falls in a launch or chunk.  int16 input is converted in registers.
//                         T = float2 / short2: complex (I, Q) input, four FMAs per tap in an order that
//                         rounds exactly as the real kernel's when Q = 0.
//   zoom_split_kernel     X[k], k = 0..Nz, of the interleaved (re, im) stream seen as 2 Nz real points ->
//                         Z[k] = E + iO of the complex frame -> |Z|^2 / Nz in fft-shifted bin order.
//   iq_mtm_split_kernel   the same split for one taper of a multitaper row: taper 0 stores |Z_0|^2 / Nz, taper
//                         k > 0 adds |Z_k|^2 / Nz to the row, so the tapers are summed in the order k = 0..K'-1.
//   iq_ftest_*_kernel     the harmonic F-test on the general path: the hn spectrum split into the mu plane, each
//                         taper's split adding its power to the row and its residual to the den plane, the quotient.
#include <cuda_runtime.h>
#include <atomic>
#include <cstdio>
#include <cstring>
#include "../../include/glb_shim.h"
#include "iq_core.cuh"

extern std::atomic<unsigned long long> g_launches;   // gram_kernels.cu

#define ZCU(call)                                                                             \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess) {                                                                  \
      char m_[512];                                                                           \
      snprintf(m_, sizeof m_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),         \
               __FILE__, __LINE__);                                                           \
      glb_set_error(m_);                                                                      \
      return GLB_ECUDA;                                                                       \
    }                                                                                         \
  } while (0)

constexpr int kZR = 16;        // outputs per lane group
constexpr int kZT = 33;        // taps per phase: 32 D + 1 taps, zero-padded to 33 D
constexpr int kZWarps = 8;

static __device__ __forceinline__ float zload(const float *x, long long i, long long count) {
  return (i >= 0 && i < count) ? __ldg(x + i) : 0.f;
}
// wav_fmt.c:113: (float) s / 32768 (a power-of-two scale: exact, so equal to the float path's input)
static __device__ __forceinline__ float zload(const short *x, long long i, long long count) {
  return (i >= 0 && i < count) ? (float) __ldg(x + i) * (1.f / 32768.f) : 0.f;
}
// complex input: interleaved (I, Q) floats or int16 pairs, converted as above
static __device__ __forceinline__ float2 zload(const float2 *x, long long i, long long count) {
  return (i >= 0 && i < count) ? __ldg(x + i) : make_float2(0.f, 0.f);
}
static __device__ __forceinline__ float2 zload(const short2 *x, long long i, long long count) {
  if (i < 0 || i >= count) return make_float2(0.f, 0.f);
  const short2 s = __ldg(x + i);
  return make_float2((float) s.x * (1.f / 32768.f), (float) s.y * (1.f / 32768.f));
}
template <typename T> struct ZComplex { static constexpr bool value = false; };
template <> struct ZComplex<float2> { static constexpr bool value = true; };
template <> struct ZComplex<short2> { static constexpr bool value = true; };

template <typename T>
__global__ void __launch_bounds__(kZWarps * 32, ZComplex<T>::value ? 1 : 0)
zoom_decim_kernel(const T *__restrict__ x, long long origin, long long count, int D, int LG, int G,
                  const float2 *__restrict__ taps, unsigned dstep, long long m_first, long long m_count,
                  float2 *__restrict__ y) {
  __shared__ float part[kZWarps][32][2 * kZR + 1];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int per_blk = G * kZR;
  const long long nblk = (m_count + per_blk - 1) / per_blk;
  const int gi = lane / LG, sl = lane - gi * LG;
  const bool active = gi < G;
  const long long K = 16LL * D;
  for (long long b = (long long) blockIdx.x * kZWarps + w; b < nblk; b += (long long) gridDim.x * kZWarps) {
    const long long mb = m_first + b * per_blk;
    float ar[kZR], ai[kZR];
#pragma unroll
    for (int r = 0; r < kZR; r++) ar[r] = ai[r] = 0.f;
    if (active) {
      const long long i0 = (mb + (long long) gi * kZR) * D - K - origin;
      for (int p = sl; p < D; p += LG) {
        float tr[kZT], ti[kZT];
#pragma unroll
        for (int t = 0; t < kZT; t++) {
          const float2 c = __ldg(taps + t * D + p);
          tr[t] = c.x;
          ti[t] = c.y;
        }
        const long long ip = i0 + p;
#pragma unroll
        for (int q = 0; q < kZR + kZT - 1; q++) {
          const auto u = zload(x, ip + (long long) q * D, count);
#pragma unroll
          for (int r = 0; r < kZR; r++) {
            const int t = q - r;
            if (t >= 0 && t < kZT) {
              if constexpr (ZComplex<T>::value) {
                ar[r] = fmaf(tr[t], u.x, ar[r]);
                ar[r] = fmaf(-ti[t], u.y, ar[r]);
                ai[r] = fmaf(ti[t], u.x, ai[r]);
                ai[r] = fmaf(tr[t], u.y, ai[r]);
              } else {
                ar[r] = fmaf(tr[t], u, ar[r]);
                ai[r] = fmaf(ti[t], u, ai[r]);
              }
            }
          }
        }
      }
    }
#pragma unroll
    for (int r = 0; r < kZR; r++) {
      part[w][lane][2 * r] = ar[r];
      part[w][lane][2 * r + 1] = ai[r];
    }
    __syncwarp();
    for (int o = lane; o < per_blk; o += 32) {
      const int g = o / kZR, r = o - g * kZR;
      const long long m = mb + o;
      float sr = 0.f, si = 0.f;
      for (int s = 0; s < LG; s++) {
        sr += part[w][g * LG + s][2 * r];
        si += part[w][g * LG + s][2 * r + 1];
      }
      if (m < m_first + m_count) {
        // phi(mD) 2^32 exactly in 32-bit arithmetic; as a signed value / 2^31 it is the angle in half-turns
        const unsigned ph = (unsigned) (unsigned long long) m * dstep;
        float sn, cs;
        sincospif((float) (int) ph * 4.656612873077393e-10f, &sn, &cs);
        y[m - m_first] = make_float2(fmaf(sr, cs, si * sn), fmaf(si, cs, -(sr * sn)));
      }
    }
    __syncwarp();
  }
}

__global__ void zoom_split_kernel(const float2 *__restrict__ spec, int nz, long long nframes, float inv_nz,
                                  float *__restrict__ rows) {
  const long long total = nframes * nz;
  const long long stride = (long long) gridDim.x * blockDim.x;
  for (long long idx = (long long) blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += stride) {
    const long long f = idx / nz;
    const int j = (int) (idx - f * nz);
    const int k = (j + nz / 2) & (nz - 1);
    const float2 *X = spec + f * (nz + 1);
    const float2 a = X[k], c = X[nz - k];
    // E = (X[k] + conj X[Nz-k]) / 2,  O = (X[k] - conj X[Nz-k]) / (2 W^k),  W = e^{-i pi / Nz}
    const float er = 0.5f * (a.x + c.x), ei = 0.5f * (a.y - c.y);
    const float dr = 0.5f * (a.x - c.x), di = 0.5f * (a.y + c.y);
    float sn, cs;
    sincospif((float) k / (float) nz, &sn, &cs);
    const float orr = dr * cs - di * sn, oi = dr * sn + di * cs;
    const float zr = er - oi, zi = ei + orr;          // Z = E + i O
    rows[idx] = (zr * zr + zi * zi) * inv_nz;
  }
}

// zoom_split_kernel's arithmetic, kept apart so that the periodogram's kernel keeps its exact instructions
__global__ void iq_mtm_split_kernel(const float2 *__restrict__ spec, int nz, long long nframes, float inv_nz, int add,
                                    float *__restrict__ rows) {
  const long long total = nframes * nz;
  const long long stride = (long long) gridDim.x * blockDim.x;
  for (long long idx = (long long) blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += stride) {
    const long long f = idx / nz;
    const int j = (int) (idx - f * nz);
    const int k = (j + nz / 2) & (nz - 1);
    const float2 *X = spec + f * (nz + 1);
    const float2 a = X[k], c = X[nz - k];
    const float er = 0.5f * (a.x + c.x), ei = 0.5f * (a.y - c.y);
    const float dr = 0.5f * (a.x - c.x), di = 0.5f * (a.y + c.y);
    float sn, cs;
    sincospif((float) k / (float) nz, &sn, &cs);
    const float orr = dr * cs - di * sn, oi = dr * sn + di * cs;
    const float zr = er - oi, zi = ei + orr;
    const float pw = (zr * zr + zi * zi) * inv_nz;
    rows[idx] = add ? rows[idx] + pw : pw;
  }
}

// The harmonic F-test on the general path (glb_launch_iq_gram_general with ftest).  Z[k] of a frame as the splits above
// form it; the kernels below are the complex-output split of the hn spectrum (the mu plane), the split of one taper's
// spectrum that adds its power to the rows as iq_mtm_split_kernel does and its residual to the den plane, and the
// quotient.  The residual and F are the fused kernel's (iq_core.cuh).
static __device__ __forceinline__ float2 iq_split_z(const float2 *X, int nz, int k) {
  const float2 a = X[k], c = X[nz - k];
  const float er = 0.5f * (a.x + c.x), ei = 0.5f * (a.y - c.y);
  const float dr = 0.5f * (a.x - c.x), di = 0.5f * (a.y + c.y);
  float sn, cs;
  sincospif((float) k / (float) nz, &sn, &cs);
  const float orr = dr * cs - di * sn, oi = dr * sn + di * cs;
  return make_float2(er - oi, ei + orr);
}

__global__ void iq_ftest_mu_kernel(const float2 *__restrict__ spec, int nz, long long nframes, float2 *__restrict__ mu) {
  const long long total = nframes * nz;
  const long long stride = (long long) gridDim.x * blockDim.x;
  for (long long idx = (long long) blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += stride) {
    const long long f = idx / nz;
    const int j = (int) (idx - f * nz);
    mu[idx] = iq_split_z(spec + f * (nz + 1), nz, (j + nz / 2) & (nz - 1));
  }
}

// taper k: u0k = (U0_k, sqrt(lambda_k)); add = 0 stores (taper 0), 1 adds; rows may be nullptr
__global__ void iq_ftest_split_kernel(const float2 *__restrict__ spec, int nz, long long nframes, float inv_nz, int add,
                                      const float2 *__restrict__ u0, int k, const float2 *__restrict__ mu,
                                      float *__restrict__ rows, float *__restrict__ den) {
  const long long total = nframes * nz;
  const long long stride = (long long) gridDim.x * blockDim.x;
  const float2 w = u0[k];
  for (long long idx = (long long) blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += stride) {
    const long long f = idx / nz;
    const int j = (int) (idx - f * nz);
    const float2 z = iq_split_z(spec + f * (nz + 1), nz, (j + nz / 2) & (nz - 1));
    if (rows) {
      const float pw = (z.x * z.x + z.y * z.y) * inv_nz;
      rows[idx] = add ? rows[idx] + pw : pw;
    }
    const float r = glb::iq_ftest_resid(z, mu[idx], w.x, w.y);
    den[idx] = add ? den[idx] + r : r;
  }
}

__global__ void iq_ftest_f_kernel(const float2 *__restrict__ mu, const float *__restrict__ den, long long total, float fnum,
                                  float *__restrict__ ftest) {
  const long long stride = (long long) gridDim.x * blockDim.x;
  for (long long idx = (long long) blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += stride)
    ftest[idx] = glb::iq_ftest_value(mu[idx], den[idx], fnum);
}

static int sm_count() {
  int dev = 0, sms = 148;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return sms;
}

template <typename T>
static int launch_decim(const T *x, long long origin, long long count, int decim, const void *taps, unsigned dstep,
                        long long m_first, long long m_count, void *y, void *stream) {
  const int lg = decim < 32 ? decim : 32;
  const int g = 32 / lg;
  const long long nblk = (m_count + (long long) g * kZR - 1) / ((long long) g * kZR);
  long long ctas = (nblk + kZWarps - 1) / kZWarps;
  const long long cap = (long long) sm_count() * 8;
  if (ctas > cap) ctas = cap;
  zoom_decim_kernel<T><<<(int) ctas, kZWarps * 32, 0, (cudaStream_t) stream>>>(
      x, origin, count, decim, lg, g, (const float2 *) taps, dstep, m_first, m_count, (float2 *) y);
  ZCU(cudaGetLastError());
  g_launches++;
  return GLB_OK;
}

extern "C" int glb_launch_zoom_decim(const void *x, int pcm16, long long origin, long long count, int decim,
                                     const void *taps, unsigned dstep, long long m_first, long long m_count,
                                     void *y, void *stream) {
  if (decim < 2 || decim > 1024 || !taps || !y || origin < 0 || count < 0 || m_first < 0) {
    glb_set_error("glb_launch_zoom_decim: invalid arguments");
    return GLB_EINVAL;
  }
  if (m_count <= 0) return GLB_OK;
  if (pcm16) return launch_decim((const short *) x, origin, count, decim, taps, dstep, m_first, m_count, y, stream);
  return launch_decim((const float *) x, origin, count, decim, taps, dstep, m_first, m_count, y, stream);
}

extern "C" int glb_launch_zoom_decim_iq(const void *x, int pcm16, long long origin, long long count, int decim,
                                        const void *taps, unsigned dstep, long long m_first, long long m_count,
                                        void *y, void *stream) {
  if (decim < 2 || decim > 1024 || !taps || !y || origin < 0 || count < 0 || m_first < 0) {
    glb_set_error("glb_launch_zoom_decim_iq: invalid arguments");
    return GLB_EINVAL;
  }
  if (m_count <= 0) return GLB_OK;
  if (pcm16) return launch_decim((const short2 *) x, origin, count, decim, taps, dstep, m_first, m_count, y, stream);
  return launch_decim((const float2 *) x, origin, count, decim, taps, dstep, m_first, m_count, y, stream);
}

extern "C" int glb_launch_zoom_split(const void *spec, int nz, long long nframes, float *rows, void *stream) {
  if (nz < 2 || (nz & (nz - 1)) != 0 || !spec || !rows) {
    glb_set_error("glb_launch_zoom_split: invalid arguments");
    return GLB_EINVAL;
  }
  if (nframes <= 0) return GLB_OK;
  const long long total = nframes * nz;
  long long ctas = (total + 255) / 256;
  const long long cap = (long long) sm_count() * 16;
  if (ctas > cap) ctas = cap;
  zoom_split_kernel<<<(int) ctas, 256, 0, (cudaStream_t) stream>>>((const float2 *) spec, nz, nframes,
                                                                  (float) (1.0 / nz), rows);
  ZCU(cudaGetLastError());
  g_launches++;
  return GLB_OK;
}

// The general path of complex frames: the interleaved stream seen as a real stream of 2n floats per frame at hop
// 2 hop, the general spectrogram kernel's spectrum output X[k], k = 0..n, then zoom_split_kernel.  The zoom's frame
// stage (host/zoom.c) and the I/Q spectrogram's non-fused launches (iq.cu).  Multitaper (ntapers > 1): one spectrum
// per taper into the same scratch plane, each followed by iq_mtm_split_kernel, which sums the tapers into the rows.
extern "C" int glb_launch_iq_gram_general(const glb_iq_gram_args *a, void *stream) {
  if (!a || (!a->rows && !a->ftest) || a->nframes < 0 || a->ntapers < 0 || a->ntapers > 32 ||
      (a->ftest && (a->ntapers < 2 || !a->ftest_taper || !a->ftest_u0))) {
    glb_set_error("glb_launch_iq_gram_general: invalid arguments");
    return GLB_EINVAL;
  }
  if (a->nframes == 0) return GLB_OK;
  if (!a->scratch) {
    glb_set_error("glb_launch_iq_gram_general: needs scratch for the spectrum (glb_iq_gram_scratch_bytes)");
    return GLB_EINVAL;
  }
  glb_gram_args g;
  memset(&g, 0, sizeof g);
  g.n = 2 * a->n;
  g.hop = 2 * a->hop;
  g.samples = a->samples;
  g.origin = 2 * a->origin;
  g.count = 2 * a->count;
  g.tapers = a->taper;
  g.ntapers = 1;
  g.taper_symmetric = a->taper_symmetric;
  g.taper_scale = a->taper_scale;
  g.first_frame = a->first_frame;
  g.nframes = a->nframes;
  g.spectrum = (float *) a->scratch;
  g.tables = a->tables;
  g.general_only = 1;
  if (a->ntapers <= 1) {
    int rc = glb_launch_gram(&g, stream);
    if (rc != GLB_OK) return rc;
    return glb_launch_zoom_split(a->scratch, a->n, a->nframes, a->rows, stream);
  }
  const int nz = a->n;
  const long long total = a->nframes * nz;
  long long ctas = (total + 255) / 256;
  const long long cap = (long long) sm_count() * 16;
  if (ctas > cap) ctas = cap;
  if (a->ftest) {
    float2 *mu = reinterpret_cast<float2 *>((float *) a->scratch + a->nframes * (long long) (nz + 1) * 2);
    float *den = reinterpret_cast<float *>(mu + total);
    g.tapers = a->ftest_taper;
    g.taper_symmetric = 0;
    int rc = glb_launch_gram(&g, stream);
    if (rc != GLB_OK) return rc;
    iq_ftest_mu_kernel<<<(int) ctas, 256, 0, (cudaStream_t) stream>>>((const float2 *) a->scratch, nz, a->nframes, mu);
    ZCU(cudaGetLastError());
    g_launches++;
    for (int k = 0; k < a->ntapers; k++) {
      g.tapers = a->taper + (size_t) k * 2 * nz;
      g.taper_symmetric = (int) (((unsigned) a->taper_symmetric >> k) & 1u);
      rc = glb_launch_gram(&g, stream);
      if (rc != GLB_OK) return rc;
      iq_ftest_split_kernel<<<(int) ctas, 256, 0, (cudaStream_t) stream>>>(
          (const float2 *) a->scratch, nz, a->nframes, (float) (1.0 / nz), k > 0, (const float2 *) a->ftest_u0, k, mu,
          a->rows, den);
      ZCU(cudaGetLastError());
      g_launches++;
    }
    const float fnum = (float) ((double) (a->ntapers - 1) * (double) a->ftest_s);
    iq_ftest_f_kernel<<<(int) ctas, 256, 0, (cudaStream_t) stream>>>(mu, den, total, fnum, a->ftest);
    ZCU(cudaGetLastError());
    g_launches++;
    return GLB_OK;
  }
  for (int k = 0; k < a->ntapers; k++) {
    g.tapers = a->taper + (size_t) k * 2 * nz;
    g.taper_symmetric = (int) (((unsigned) a->taper_symmetric >> k) & 1u);
    int rc = glb_launch_gram(&g, stream);
    if (rc != GLB_OK) return rc;
    iq_mtm_split_kernel<<<(int) ctas, 256, 0, (cudaStream_t) stream>>>((const float2 *) a->scratch, nz, a->nframes,
                                                                         (float) (1.0 / nz), k > 0, a->rows);
    ZCU(cudaGetLastError());
    g_launches++;
  }
  return GLB_OK;
}
