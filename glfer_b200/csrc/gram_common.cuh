// gram_common.cuh -- the spectrogram kernels proper (general, TMA ring, warp-per-frame) and their
// launch logic, shared by the translation units that instantiate them for a subset of FFT sizes
// (gram_part.cu, compiled once per subset so the sizes build in parallel) and by gram_kernels.cu
// (C-ABI shim, tables, the small kernels).
#pragma once
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cstdint>
#include <atomic>
#include <vector>
#include <algorithm>

#include "fft_core.cuh"
#include "fft_wpf.cuh"
#include "levels.cuh"
#include "avg_frame.cuh"
#include "tables.hpp"
#include "../../include/glb_shim.h"

using namespace glb;

// shared state of the library (defined in gram_kernels.cu)
extern std::atomic<unsigned long long> g_launches;
extern int g_big_pair;
extern int g_kernel_pref;            // 0 auto, 1 general, 2 ring, 3 warp-per-frame, 4 two frames per thread
extern int g_last_family;            // family of the last spectrogram kernel launched (same numbering)
extern "C" void glb_set_error(const char *msg);

#define CU(call)                                                                              \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess) {                                                                  \
      char m_[512];                                                                           \
      snprintf(m_, sizeof m_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_),         \
               __FILE__, __LINE__);                                                           \
      glb_set_error(m_);                                                                      \
      return (e_ == cudaErrorNoDevice || e_ == cudaErrorInsufficientDriver) ? GLB_ENODEV      \
             : (e_ == cudaErrorMemoryAllocation ? GLB_ENOMEM : GLB_ECUDA);                    \
    }                                                                                         \
  } while (0)

// ------------------------------------------------------------------------- gram kernel
struct KParams {
  const float *samples;
  long long origin, count;
  const float *tapers;
  int ntapers;
  int taper_sym;              // 1: periodogram taper with w[i] == w[N - 1 - i] bit for bit
  const float *means;         // pre-computed block means (general geometry), or nullptr
  long long means_first_block;
  int fused_mean;             // 1: block means are computed inside the kernel (regular geometry)
  int qs;                     // regular geometry: hop = 2T << qs
  float inv_hop_mean;         // 1 / hop
  int hop, n_ov, cblk;        // cblk = ceil(n_ov / hop)
  float inv_hop;
  float ra9mb_a;
  int limiter;
  int zero_hist;              // 1: the n_ov history samples of every frame are zero (general kernel only)
  float lim_scale;            // taper_scale^0.9
  float spec_scale;           // 1 / (2 taper_scale)
  long long first_frame, nframes;
  int frames_per_group;
  float *rows;
  long long row_stride;
  int rows_db;
  float2 *spectrum;
  const float2 *tw, *vtab, *roots;
  // fused display mapping (g_main.c:1186-1229): 8-bit palette indices, pixel i = bin M - i, beside or
  // instead of the float rows
  unsigned char *levels;
  long long lev_stride;
  LevelMap lm;
  // fused frame averaging (ring kernel, AVG instantiations): the launch's frames are averaged by the kernel
  // that computes them; av.first_frame / av.nframes are the launch's own, av.psd is unused
  int av_on;
  glb_avg_args av;
};

#ifndef GLB_REG_TARGET
#define GLB_REG_TARGET 80
#endif
#ifndef GLB_STREAM_STORE
#define GLB_STREAM_STORE 1
#endif

template <int M> struct Geo {
  static constexpr int N = 2 * M;
  static constexpr int T = M / kPoints;
  static constexpr int G = (T >= 128) ? 1 : 128 / T;   // frame groups per CTA
  static constexpr int THREADS = G * T;
  static constexpr int NW = (T + 31) / 32;             // warps per group
  // frames are staged in shared memory by TMA bulk copies, one frame ahead, when the
  // staging buffer still leaves room for >= 2 CTAs per SM
  static constexpr bool STAGE = (M <= 4096);           // (used by the multitaper variant only)
  // twiddles kept in registers across frames instead of per-frame table loads
  static constexpr bool RT = (M <= 2048);
  static constexpr size_t BUF_BYTES = (size_t) BufSize<M>::value * sizeof(float2);      // multiple of 16
  static constexpr size_t RED_BYTES = 16 * NW * sizeof(float) + 16 * sizeof(float);     // partial sums + means
  // per frame group: FFT buffer | [staging buffer] | reduction scratch | mbarrier
  static __host__ __device__ constexpr size_t stage_bytes(bool multi) { return (STAGE && multi) ? (size_t) N * sizeof(float) : 0; }
  static __host__ __device__ constexpr size_t group_bytes(bool multi) { return ((BUF_BYTES + stage_bytes(multi) + RED_BYTES + 16 + 15) / 16) * 16; }
  // table-twiddle plans (N >= 8192) keep the twiddles of their mid passes in shared memory (one
  // copy per CTA, a few KB: they depend on k = j mod Ns only)
  static constexpr size_t TWS_BYTES = RT ? 0 : (size_t) TwOffset<M, (Plan<M>::NP > 1 ? Plan<M>::NP - 1 : 0)>::value * sizeof(float2);
  static __host__ __device__ constexpr size_t smem_bytes(bool multi) { return (size_t) G * group_bytes(multi) + TWS_BYTES; }
  // CTAs per SM the register allocation is tuned for (~GLB_REG_TARGET registers per thread)
  static constexpr int MINB_ = 65536 / (THREADS * (THREADS >= 512 ? 64 : GLB_REG_TARGET));
  static constexpr int MINB = MINB_ < 1 ? 1 : (MINB_ > 16 ? 16 : MINB_);
};

// Barrier of one frame group (T threads; a CTA of 128 threads holds 128 / T groups): nothing a
// group touches in shared memory is shared with another group, so groups that fit a warp
// (N <= 1024) synchronise with a warp-level sync (+3 % at N = 1024); larger groups use the
// CTA-wide barrier.
#ifndef GLB_CTA_BARRIER
#define GLB_CTA_BARRIER 0             // 1 (experiments): every group barrier is a CTA-wide bar.sync
#endif
template <int M> __device__ __forceinline__ void group_sync(int g) {
  constexpr int T = M / kPoints;
  if constexpr (GLB_CTA_BARRIER) {
    (void) g;
    __syncthreads();
  } else if constexpr (T <= 32) {
    __syncwarp();                       // a frame group is (part of) one warp: its buffers never leave the warp
  } else {
    // (a named barrier per 2-warp group at N = 2048 measured 6 % slower than the CTA-wide one)
    (void) g;
    __syncthreads();
  }
}

// ---- mbarrier / TMA bulk-copy helpers (1-D cp.async.bulk global -> shared) ----
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned) __cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// checked build: a bulk copy must read inside the staged samples [lo, hi)
#define GLB_CHECK_SRC(p, src, floats) GLB_CHECK((src) >= (p).samples && (src) + (floats) <= (p).samples + (p).count)
// ... and a row store must land inside the launch's rows
#define GLB_CHECK_ROW(p, ptr) GLB_CHECK((ptr) >= (p).rows && (ptr) < (p).rows + (p).nframes * (p).row_stride)
__device__ __forceinline__ void tma_load_1d(void *dst, const void *src, unsigned bytes, unsigned long long *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ float2 ldg2(const float2 *p) { return __ldg(p); }
// The taper table is the one global array every frame re-reads; with ~28 KB of L1 left beside the
// shared-memory carve-out it stays resident only if its lines are the last to go and the row
// stores do not allocate.
#ifndef GLB_L1_POLICY
#define GLB_L1_POLICY 1
#endif
__device__ __forceinline__ float2 ld_taper(const float2 *p) {
#if GLB_L1_POLICY
  float2 r;
  asm("ld.global.nc.L1::evict_last.v2.f32 {%0, %1}, [%2];" : "=f"(r.x), "=f"(r.y) : "l"(p));
  return r;
#else
  return __ldg(p);
#endif
}

// frame f can be fetched by one bulk copy: entirely inside the staged samples, no zero
// history, 16-byte aligned
__device__ __forceinline__ bool frame_bulk_ok(const KParams &p, long long f, int n) {
  const long long s0 = f * (long long) p.hop - p.n_ov;
  const long long rel = s0 - p.origin;
  return (s0 >= 0) && (rel >= 0) && (rel + n <= p.count) && ((rel & 3) == 0) && !p.zero_hist;
}

// Raw samples of one frame: x[q] = (y[2m], y[2m+1]), m = t + T q; zeros before the stream.
template <int M>
__device__ __forceinline__ void load_raw(float2 (&x)[kPoints], int t, const KParams &p, long long f, const float *stage,
                                         bool staged) {
  constexpr int T = M / kPoints, N = 2 * M;
  if (staged) {
    const float2 *s2 = reinterpret_cast<const float2 *>(stage);
#pragma unroll
    for (int q = 0; q < kPoints; q++) x[q] = s2[t + T * q];
    return;
  }
  const long long s0 = f * (long long) p.hop - p.n_ov;
  const long long rel = s0 - p.origin;
  if ((s0 >= 0) && (rel >= 0) && (rel + N <= p.count) && !p.zero_hist) {
    if ((rel & 1) == 0) {
      const float2 *src = reinterpret_cast<const float2 *>(p.samples + rel);
#pragma unroll
      for (int q = 0; q < kPoints; q++) x[q] = ldg2(src + t + T * q);
    } else {
      // interior frame at an odd offset (odd hops): pairs straddle the 8-byte alignment
      const float *src = p.samples + rel + 2 * t;
#pragma unroll
      for (int q = 0; q < kPoints; q++) x[q] = make_float2(__ldg(src + 2 * T * q), __ldg(src + 2 * T * q + 1));
    }
    return;
  }
#pragma unroll
  for (int q = 0; q < kPoints; q++) {
    float y[2];
#pragma unroll
    for (int e = 0; e < 2; e++) {
      const int i = 2 * (t + T * q) + e;
      const long long s = s0 + i;
      const long long r = s - p.origin;
      y[e] = (s >= 0 && r >= 0 && r < p.count && !(p.zero_hist && i < p.n_ov)) ? __ldg(p.samples + r) : 0.f;
    }
    x[q] = make_float2(y[0], y[1]);
  }
}

// Block-mean removal inside the kernel (prepare_audio, fft.c:86-96) for the regular
// geometry hop = 2T << QS, n_ov a multiple of hop: the frame is NB = 16 >> QS whole hop
// blocks, block b = registers q with (q >> QS) == b.  Every thread sums its share of each
// block, warps reduce by shuffle, the group combines through shared memory.  A block gets
// the same summation tree in every frame it appears in, so its mean is bit-identical
// across frames (and across time shards).  Zero history sums to a zero mean.
// `reuse` (groups of more than one warp): the warp partial sums of this frame are still in `red`
// from an earlier taper of the same frame: no summation, no shuffles, no barrier.
template <int M, int QS>
__device__ __forceinline__ void remove_block_means(float2 (&x)[kPoints], int t, float *red, float inv_hop, int g, bool reuse) {
  constexpr int T = M / kPoints, NW = (T + 31) / 32, NB = kPoints >> QS;
  constexpr int W = T < 32 ? T : 32;      // lanes of a warp that belong to this group
  float bs[NB];
  if (NW == 1 || !reuse) {
#pragma unroll
    for (int b = 0; b < NB; b++) {
      float s = 0.f;
#pragma unroll
      for (int q = b << QS; q < (b + 1) << QS; q++) s += x[q].x + x[q].y;
#pragma unroll
      for (int o = W / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      bs[b] = s;
    }
  }
  if (NW > 1) {
    if (!reuse) {
      const int w = t >> 5;
      if ((t & 31) == 0) {
#pragma unroll
        for (int b = 0; b < NB; b++) red[b * NW + w] = bs[b];
      }
      group_sync<M>(g);
    }
#pragma unroll
    for (int b = 0; b < NB; b++) {
      float s = 0.f;
#pragma unroll
      for (int w2 = 0; w2 < NW; w2++) s += red[b * NW + w2];
      bs[b] = s;
    }
  }
#pragma unroll
  for (int q = 0; q < kPoints; q++) {
    const float m = bs[q >> QS] * inv_hop;
    x[q].x -= m;
    x[q].y -= m;
  }
}

template <int M>
__device__ __forceinline__ void remove_block_means_qs(float2 (&x)[kPoints], int t, float *red, const KParams &p, int g, bool reuse) {
  switch (p.qs) {
    case 4: remove_block_means<M, 4>(x, t, red, p.inv_hop_mean, g, reuse); break;
    case 3: remove_block_means<M, 3>(x, t, red, p.inv_hop_mean, g, reuse); break;
    case 2: remove_block_means<M, 2>(x, t, red, p.inv_hop_mean, g, reuse); break;
    case 1: remove_block_means<M, 1>(x, t, red, p.inv_hop_mean, g, reuse); break;
    default: remove_block_means<M, 0>(x, t, red, p.inv_hop_mean, g, reuse); break;
  }
}

// pre-computed block means, any geometry: block of frame sample i is
// f - cblk + floor((i + cblk*hop - n_ov) / hop); samples before the stream keep 0
template <int M>
__device__ __forceinline__ void remove_table_means(float2 (&x)[kPoints], int t, const KParams &p, long long f) {
  constexpr int T = M / kPoints;
  const long long s0 = f * (long long) p.hop - p.n_ov;
  const float *mu = p.means + (f - p.cblk - p.means_first_block);
  const float off = (float) (p.cblk * p.hop - p.n_ov) + 0.5f;
#pragma unroll
  for (int q = 0; q < kPoints; q++) {
    const int i = 2 * (t + T * q);
    const int h0 = p.zero_hist ? p.n_ov : 0;          // zeroed history keeps its zeros
    if (s0 + i >= 0 && i >= h0) x[q].x -= __ldg(mu + (int) (((float) i + off) * p.inv_hop));
    if (s0 + i + 1 >= 0 && i + 1 >= h0) x[q].y -= __ldg(mu + (int) (((float) (i + 1) + off) * p.inv_hop));
  }
}

// RA9MB -> taper -> limiter (fft.c:127-156); the common case is the bare multiply
template <int M, bool PLAIN>
__device__ __forceinline__ void apply_taper(float2 (&v)[kPoints], const float2 (&x)[kPoints], int t, const KParams &p,
                                            const float *tap) {
  constexpr int T = M / kPoints;
  const float2 *w2 = reinterpret_cast<const float2 *>(tap);
  if (PLAIN || (p.ra9mb_a <= 0.f && p.limiter == 0)) {
#pragma unroll
    for (int q = 0; q < kPoints; q++) {
      const float2 w = ld_taper(w2 + t + T * q);
      v[q] = mul2(x[q], w);
    }
    return;
  }
#pragma unroll
  for (int q = 0; q < kPoints; q++) {
    const float2 w = ldg2(w2 + t + T * q);
    float y[2] = {x[q].x, x[q].y};
    const float ww[2] = {w.x, w.y};
#pragma unroll
    for (int e = 0; e < 2; e++) {
      if (p.ra9mb_a > 0.f) y[e] = y[e] / (p.ra9mb_a + y[e] * y[e]);
      y[e] *= ww[e];
      if (p.limiter == 1) {
        const float m = p.lim_scale * powf(fabsf(y[e]), 0.1f);
        y[e] = (y[e] > 0.f) ? m : -m;
      }
    }
    v[q] = make_float2(y[0], y[1]);
  }
}

template <int M, int P, bool RT> struct MidPasses {
  static __device__ __forceinline__ void run(float2 (&v)[kPoints], int t, float2 *buf, const float2 *tw, const TwRegs &tr, int g) {
    if constexpr (P < Plan<M>::NP - 1) {
      pass_load<M>(v, t, buf);
      if constexpr (RT) {
        pass_compute_rt<M, P>(v, tr);
        group_sync<M>(g);               // every thread has read before anyone overwrites
        pass_scatter<M, P>(v, t, buf);
      } else {
        group_sync<M>(g);
        pass_store<M, P>(v, t, buf, tw);
      }
      group_sync<M>(g);
      MidPasses<M, P + 1, RT>::run(v, t, buf, tw, tr, g);
    }
  }
};

// MULTI: multitaper (K' tapers per frame, frame staged in shared memory by TMA one frame
// ahead and re-read per taper).  PLAIN: no RA9MB / limiter code in the kernel.
// LEV: 8-bit display levels beside / instead of the float rows (separate instantiations: as a run-time
// branch the display epilogue cost the float path registers, +14 % on the odd-hop workload).
template <int M, bool MULTI, bool PLAIN, bool LEV = false>
__global__ void __launch_bounds__(Geo<M>::THREADS, Geo<M>::MINB) gram_kernel(const KParams p) {
  using GeoM = Geo<M>;
  constexpr int T = GeoM::T, G = GeoM::G, N = GeoM::N;
  constexpr bool STAGE = GeoM::STAGE && MULTI;
  constexpr bool RT = GeoM::RT;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int g = threadIdx.x / T;
  const int t = threadIdx.x % T;
  unsigned char *gbase = smem_raw + (size_t) g * GeoM::group_bytes(MULTI);
  float2 *buf = reinterpret_cast<float2 *>(gbase);
  float *stage = reinterpret_cast<float *>(gbase + GeoM::BUF_BYTES);
  float *red = reinterpret_cast<float *>(gbase + GeoM::BUF_BYTES + GeoM::stage_bytes(MULTI));
  unsigned long long *mbar = reinterpret_cast<unsigned long long *>(gbase + GeoM::BUF_BYTES + GeoM::stage_bytes(MULTI) + GeoM::RED_BYTES);
  const long long gid = (long long) blockIdx.x * G + g;
  const long long fb = gid * p.frames_per_group;
  unsigned phase = 0;

  TwRegs tr;
  if constexpr (RT) load_tw_regs<M>(tr, t, p.tw, p.vtab);
  // table-twiddle plans: mid-pass twiddles from shared memory (global loads of 29 twiddles per
  // thread and transform kept the L1TEX pipe busy and the warps waiting on L2)
  const float2 *tw_mid = p.tw;
  if constexpr (!RT) {
    float2 *tws = reinterpret_cast<float2 *>(smem_raw + (size_t) G * GeoM::group_bytes(MULTI));
    constexpr int kMid = TwOffset<M, Plan<M>::NP - 1>::value;
    for (int i = threadIdx.x; i < kMid; i += GeoM::THREADS) tws[i] = p.tw[i];
    __syncthreads();
    tw_mid = tws;
  }

  if (STAGE) {
    if (t == 0) {
      mbar_init(mbar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (t == 0 && fb < p.nframes && frame_bulk_ok(p, p.first_frame + fb, N)) {
      const long long f0 = p.first_frame + fb;
      mbar_expect_tx(mbar, N * 4);
      tma_load_1d(stage, p.samples + (f0 * (long long) p.hop - p.n_ov - p.origin), N * 4, mbar);
    }
  }

  for (int it = 0; it < p.frames_per_group; ++it) {
    const long long fl = fb + it;
    const bool active = fl < p.nframes;
    const long long f = p.first_frame + fl;
    const bool staged = STAGE && active && frame_bulk_ok(p, f, N);
    const bool next_there = (it + 1 < p.frames_per_group) && (fl + 1 < p.nframes);
    const bool next_staged = STAGE && next_there && frame_bulk_ok(p, f + 1, N);
    if (staged) {
      mbar_wait(mbar, phase);
      phase ^= 1;
    }
    if (!STAGE && next_there) {
      // pull the next frame's new hop block towards L2 while this frame is computed
      const long long nb = (f + 1) * (long long) p.hop - p.origin;       // first new sample, buffer index
      for (int i = t * 32; i < p.hop; i += T * 32)
        if (nb + i >= 0 && nb + i < p.count) asm volatile("prefetch.global.L2 [%0];" ::"l"(p.samples + nb + i));
    }
    float acc[17];
    if (MULTI) {
#pragma unroll
      for (int i = 0; i < 17; i++) acc[i] = 0.f;
    }
    const int ntap = MULTI ? p.ntapers : 1;
    for (int j = 0; j < ntap; ++j) {
      float2 v[kPoints];
      {
        float2 x[kPoints];
        // Control flow around the warp shuffles / barriers of the mean removal depends only
        // on j (uniform over the CTA), never on a group's own frame: groups of one warp or
        // CTA can sit on different kinds of frames.
        if (MULTI && STAGE && j > 0) {
          // multitaper: tapers after the first read the cleaned copy kept in the staging buffer
          const float2 *s2 = reinterpret_cast<const float2 *>(stage);
#pragma unroll
          for (int q = 0; q < kPoints; q++) x[q] = s2[t + T * q];
        } else {
          if (active) {
            load_raw<M>(x, t, p, f, stage, staged);
          } else {
#pragma unroll
            for (int q = 0; q < kPoints; q++) x[q] = make_float2(0.f, 0.f);
          }
          if (p.fused_mean) remove_block_means_qs<M>(x, t, red, p, g, MULTI && j > 0);
          else if (p.means != nullptr && active) remove_table_means<M>(x, t, p, f);
          if (MULTI && STAGE && ntap > 1) {
            float2 *s2 = reinterpret_cast<float2 *>(stage);
#pragma unroll
            for (int q = 0; q < kPoints; q++) s2[t + T * q] = x[q];     // own elements only: no hazard
          }
        }
        apply_taper<M, PLAIN>(v, x, t, p, p.tapers + (size_t) j * N);
      }
      if constexpr (RT) {
        pass_compute_rt<M, 0>(v, tr);
        group_sync<M>(g);              // (A) the previous transform's last pass has been read by all
        pass_scatter<M, 0>(v, t, buf);
      } else {
        group_sync<M>(g);
        pass_store<M, 0>(v, t, buf, p.tw);
      }
      if (STAGE && next_staged && j == ntap - 1 && t == 0) {
        // past barrier (A) everyone is done reading the staging buffer: fetch the next frame
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_expect_tx(mbar, N * 4);
        tma_load_1d(stage, p.samples + ((f + 1) * (long long) p.hop - p.n_ov - p.origin), N * 4, mbar);
      }
      group_sync<M>(g);
      MidPasses<M, 1, RT>::run(v, t, buf, tw_mid, tr, g);
      auto sink_multi = [&](int slot, float2 a, bool) { acc[slot] += norm2(a); };
      float *row = (!MULTI && active && p.rows) ? p.rows + fl * p.row_stride : nullptr;
      unsigned char *lrow = (LEV && !MULTI && active) ? p.levels + fl * p.lev_stride : nullptr;
      float2 *sp = (!MULTI && active && p.spectrum) ? p.spectrum + fl * (long long) (M + 1) : nullptr;
      const bool db = p.rows_db != 0;
      const float ss = p.spec_scale;
      auto sink_single = [&](int slot, float2 a, bool cj) {
        const int bin = slot_bin<M>(t, slot);
        if constexpr (LEV) {
          if (lrow) lrow[M - bin] = map_level(norm2(a), p.lm);
        }
        if (row) {
          float y = norm2(a);
          if (db) y = 10.f * log10f(y);
          row[bin] = y;
        }
        if (sp) sp[bin] = make_float2(a.x * ss, cj ? -a.y * ss : a.y * ss);
      };
      if constexpr (RT) {
        last_pass_rt<M>(v, t, buf, p.tw, tr);
        if (MULTI) emit_bins_rt<M>(v, t, tr, sink_multi);
        else emit_bins_rt<M>(v, t, tr, sink_single);
      } else {
        // last pass and split from 6 loaded bases, the register-twiddle code path
        TwRegs tl;
        load_last_regs<M>(tl, t, p.tw, p.vtab);
        last_pass_load<M>(v, t, buf);
        last_pass_compute_rt<M>(v, t, tl);
        if (MULTI) emit_bins_rt<M>(v, t, tl, sink_multi);
        else emit_bins_rt<M>(v, t, tl, sink_single);
      }
      // no barrier here: (A) of the next transform orders these reads before its stores
    }
    if (LEV && MULTI && active) {
      unsigned char *lrow = p.levels + fl * p.lev_stride;
#pragma unroll
      for (int slot = 0; slot < 17; slot++)
        if (slot < 16 || t == 0) lrow[M - slot_bin<M>(t, slot)] = map_level(acc[slot], p.lm);
    }
    if (MULTI && active && p.rows) {
      float *row = p.rows + fl * p.row_stride;
      const bool db = p.rows_db != 0;
#pragma unroll
      for (int slot = 0; slot < 17; slot++) {
        if (slot < 16 || t == 0) {
          float y = acc[slot];
          if (db) y = 10.f * log10f(y);
          row[slot_bin<M>(t, slot)] = y;
        }
      }
    }
  }
}

// ------------------------------------------------------------------------- ring kernel
// The fast path for the regular geometry (hop = 2T << QS, N - hop a multiple of hop: 0, 50,
// 75, 87.5, 93.75 % overlap; no RA9MB / limiter).  A frame is NB = 16 >> QS whole hop blocks.
// Each frame group keeps the last NB blocks of its run in a shared-memory ring that is
// filled by TMA bulk copies (cp.async.bulk + mbarrier), always one block ahead of the FFT
// (the oldest slot is handed to the next copy as soon as the frame is in registers), so every
// sample crosses HBM -> SM exactly once, whatever the overlap, and the DRAM latency hides
// behind the current frame's transform.  The mean of a block (sub_mean) is formed once, from the
// registers of the frame in which it is the newest block (ring_fetch), and kept beside the ring
// for the NB - 1 frames that use the block again.
#ifndef GLB_RING_EXTRA
#define GLB_RING_EXTRA 0  // 1: one spare slot, the next block is requested at the top of a frame;
#endif                    // 0: NB slots, requested after barrier (A) into the oldest block's slot
struct RingLayout {
  int slots;            // NB + GLB_RING_EXTRA
  size_t ring_off, red_off, mu_off, mbar_off, hist_off, group_bytes;
};

// hist_floats: fused averaging keeps the last `depth` PSD rows of the averaging band ([depth][band] floats)
template <int M>
__host__ __device__ inline RingLayout ring_layout(int hop, int nb, int hist_floats = 0) {
  RingLayout L;
  L.slots = nb + GLB_RING_EXTRA;
  L.ring_off = Geo<M>::BUF_BYTES;
  L.red_off = L.ring_off + (size_t) L.slots * hop * sizeof(float);
  L.mu_off = L.red_off + (size_t) 18 * Geo<M>::NW * sizeof(float);
  L.mbar_off = ((L.mu_off + 18 * sizeof(float) + 7) / 8) * 8;
  L.hist_off = ((L.mbar_off + 18 * sizeof(unsigned long long) + 15) / 16) * 16;
  L.group_bytes = ((L.hist_off + (size_t) hist_floats * sizeof(float) + 15) / 16) * 16;
  return L;
}

// mean of one ring block: every thread sums its (1 << qs) float2 entries, warps reduce by
// shuffle, the group combines through `red` (one barrier).  The summation tree of a block is
// the same wherever the block sits in a frame: its mean is bit-identical in every frame, group
// and time shard.  Must be called by all threads of the CTA (contains a block barrier).
template <int M>
__device__ __forceinline__ float ring_block_partial(const float *blk, int qs, int t, float *red) {
  constexpr int T = M / kPoints, NW = (T + 31) / 32, W = T < 32 ? T : 32;
  const float2 *b2 = reinterpret_cast<const float2 *>(blk);
  float s = 0.f;
  for (int i = 0; i < (1 << qs); i++) {
    const float2 a = b2[t + T * i];
    s += a.x + a.y;
  }
#pragma unroll
  for (int o = W / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (NW > 1 && (t & 31) == 0) red[t >> 5] = s;
  return s;
}
// after a block barrier that follows ring_block_partial()
template <int M>
__device__ __forceinline__ float ring_block_total(float s_warp, const float *red, float inv_hop) {
  constexpr int T = M / kPoints, NW = (T + 31) / 32;
  float s = s_warp;
  if (NW > 1) {
    s = 0.f;
#pragma unroll
    for (int w = 0; w < NW; w++) s += red[w];
  }
  return s * inv_hop;
}
template <int M>
__device__ __forceinline__ float ring_block_mean(const float *blk, int qs, int t, float *red, float inv_hop, int g) {
  constexpr int T = M / kPoints, NW = (T + 31) / 32;
  const float s = ring_block_partial<M>(blk, qs, t, red);
  if (NW > 1) group_sync<M>(g);
  return ring_block_total<M>(s, red, inv_hop);
}

// Top of a frame: the NB blocks of the frame from the ring into registers, block means removed.
// `new_mean`: the newest block has just landed and its mean is not known yet; it is summed from
// the registers just loaded (same order as ring_block_partial, so the mean of a block is the
// same bits wherever it is formed), combined across the warps of the group through `red` with
// one block barrier, and left in mu_new / mu[slot_newest].  The loads of the other blocks are
// in flight across that barrier.
template <int M, int QS>
__device__ __forceinline__ void ring_fetch(float2 (&x)[kPoints], int t, const float *ring, int hop, int slot_oldest,
                                           int slots, float *mu, float &mu_new, bool sub, bool new_mean, float *red,
                                           float inv_hop, int g) {
  constexpr int T = M / kPoints, NB = kPoints >> QS, NW = (T + 31) / 32, W = T < 32 ? T : 32;
  int sidx = slot_oldest;
  int slot_of[NB];
#pragma unroll
  for (int b = 0; b < NB; b++) {
    const float2 *bp = reinterpret_cast<const float2 *>(ring + (size_t) sidx * hop);
    slot_of[b] = sidx;
#pragma unroll
    for (int i = 0; i < (1 << QS); i++) x[(b << QS) + i] = bp[t + T * i];
    sidx = (sidx + 1 == slots) ? 0 : sidx + 1;
  }
  if (!sub) return;
  if (new_mean) {
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < (1 << QS); i++) {
      const float2 a = x[((NB - 1) << QS) + i];
      s += a.x + a.y;
    }
#pragma unroll
    for (int o = W / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (NW > 1) {
      if ((t & 31) == 0) red[t >> 5] = s;
      group_sync<M>(g);
    }
    mu_new = ring_block_total<M>(s, red, inv_hop);
    if (t == 0) mu[slot_of[NB - 1]] = mu_new;
  }
#pragma unroll
  for (int b = 0; b < NB; b++) {
    const float m = (b == NB - 1) ? mu_new : mu[slot_of[b]];
#pragma unroll
    for (int i = 0; i < (1 << QS); i++) x[(b << QS) + i] = sub2(x[(b << QS) + i], bc(m));
  }
}

// One PSD row out of the registers (slot numbering of fft_core.cuh): slot 2 rp is bin k, slot
// 2 rp + 1 is bin M - k, k = t + rp 2T except for the upper four pairs of thread 0; base pointers
// plus immediates.  Thread 0 also owns bin M/2.
__device__ __forceinline__ void st_row(float *p, float y) {
#if GLB_L1_POLICY
  asm volatile("st.global.L1::no_allocate.f32 [%0], %1;" ::"l"(p), "f"(y) : "memory");
#elif GLB_STREAM_STORE
  __stcs(p, y);
#else
  *p = y;
#endif
}
template <int M>
__device__ __forceinline__ void store_row(float *row, int t, const float (&yv)[17]) {
  constexpr int T = M / kPoints;
  const int kh = khi<M>(t) - 8 * T;
  float *ra = row + t, *rb = row + (M - t), *rah = row + kh, *rbh = row + (M - kh);
  GLB_CHECK(t >= 0 && t <= M && kh + 14 * T <= M && M - kh - 14 * T >= 0);
#pragma unroll
  for (int rp = 0; rp < 8; rp++) {
    st_row((rp < 4 ? ra : rah) + rp * 2 * T, yv[2 * rp]);
    st_row((rp < 4 ? rb : rbh) - rp * 2 * T, yv[2 * rp + 1]);
  }
  if (t == 0) st_row(row + M / 2, yv[16]);
}

// The same row as 8-bit display levels: pixel i shows bin M - i (g_main.c:1193-1201), so the bins a warp
// stores together are still 32 consecutive bytes.  Only compiled into the LEV = true instantiations of the
// ring kernel: as a run-time branch of the one kernel it cost the float-row path registers (spills at
// N = 1024, +4 % at N = 16384).
template <int M>
__device__ __forceinline__ void store_levels(unsigned char *lrow, int t, const float (&yv)[17], const LevelMap &lm) {
  constexpr int T = M / kPoints;
  const int kh = khi<M>(t) - 8 * T;
  unsigned char *pa = lrow + (M - t), *pb = lrow + t, *pah = lrow + (M - kh), *pbh = lrow + kh;
#pragma unroll
  for (int rp = 0; rp < 8; rp++) {
    *((rp < 4 ? pa : pah) - rp * 2 * T) = map_level(yv[2 * rp], lm);
    *((rp < 4 ? pb : pbh) + rp * 2 * T) = map_level(yv[2 * rp + 1], lm);
  }
  if (t == 0) lrow[M - M / 2] = map_level(yv[16], lm);
}

// mid passes of the ring kernel
template <int M, int P, bool RT> struct RingMidPasses {
  static __device__ __forceinline__ void run(float2 (&v)[kPoints], int t, float2 *buf, const float2 *tw, const TwRegs &tr, int g) {
    if constexpr (P < Plan<M>::NP - 1) {
      pass_load<M>(v, t, buf);
      if constexpr (RT) {
        pass_compute_rt<M, P>(v, tr);
        group_sync<M>(g);                // every thread has read before anyone overwrites
        pass_scatter<M, P>(v, t, buf);
      } else {
        group_sync<M>(g);
        pass_store<M, P>(v, t, buf, tw);
      }
      group_sync<M>(g);
      RingMidPasses<M, P + 1, RT>::run(v, t, buf, tw, tr, g);
    }
  }
};

// N = 16384 (512 threads, one CTA per SM because of its 138 KB of shared memory): the periodogram
// variant may use 128 registers, enough to keep the twiddles of its two mid passes in registers
template <int M, bool MULTI> struct RingGeo {
  static constexpr bool BIG = (M == 8192) && !MULTI;
  static constexpr bool RT = Geo<M>::RT || BIG;
#ifndef GLB_MULTI_MINB
#define GLB_MULTI_MINB 4          // CTAs per SM the 128-thread multitaper ring kernel is compiled for: 115 registers, no
                                  // spills (6 / 5 / 4 / 3 CTAs: 3.34 / 3.17 / 3.03 / 3.02 ms on C3); 0 = as the periodogram
#endif
  static constexpr int MINB = BIG ? 1 : ((MULTI && GLB_MULTI_MINB > 0 && Geo<M>::THREADS == 128) ? GLB_MULTI_MINB : Geo<M>::MINB);
};
// AVG: the sliding frame averaging (update_avg_*, avg.c:108-298) fused in.  A group pre-rolls the depth - 1
// frames before its run (their rows belong to the previous group and are not stored), every frame leaves
// the PSD of the averaging band in a [depth][band] history in shared memory, and one warp -- a different
// one each frame -- forms the averaged band row, the return value, the *peakbin candidate and the variance
// of the frame before, right after barrier (A) has made that frame's history entries visible.  The
// arithmetic is avg_frame_warp() of the stand-alone kernel: identical bits.  Band-only output rows.
template <int M, bool MULTI, int QSC, bool LEV, bool AVG = false>
__global__ void __launch_bounds__(Geo<M>::THREADS, (RingGeo<M, MULTI>::MINB)) gram_ring_kernel(const KParams p) {
  using GeoM = Geo<M>;
  constexpr int T = GeoM::T, G = GeoM::G, N = GeoM::N;
  constexpr bool RT = RingGeo<M, MULTI>::RT;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int g = threadIdx.x / T;
  const int t = threadIdx.x % T;
  const int qs = QSC >= 0 ? QSC : p.qs;
  const int hop = QSC >= 0 ? ((2 * T) << (QSC >= 0 ? QSC : 0)) : p.hop;
  const int nb = kPoints >> qs;                                  // nb blocks per frame
  const int av_band = AVG ? p.av.maxbin - p.av.minbin : 0, av_depth = AVG ? p.av.depth : 1;
  const RingLayout L = ring_layout<M>(hop, nb, AVG ? av_band * av_depth : 0);
  const int slots = L.slots;
  unsigned char *gbase = smem_raw + (size_t) g * L.group_bytes;
  float2 *buf = reinterpret_cast<float2 *>(gbase);
  float *ring = reinterpret_cast<float *>(gbase + L.ring_off);
  float *red = reinterpret_cast<float *>(gbase + L.red_off);
  float *mu = reinterpret_cast<float *>(gbase + L.mu_off);
  unsigned long long *mbar = reinterpret_cast<unsigned long long *>(gbase + L.mbar_off);
  float *hist = reinterpret_cast<float *>(gbase + L.hist_off);
  const long long gid = (long long) blockIdx.x * G + g;
  const long long fb = gid * p.frames_per_group;
  const bool group_active = fb < p.nframes;
  // fused averaging: pre-roll of depth - 1 frames (fewer at the very start of the recording)
  const int pre = (AVG && group_active) ? (int) ((p.first_frame + fb < av_depth - 1) ? p.first_frame + fb : av_depth - 1) : 0;
  const long long f_first = p.first_frame + fb - pre;
  const long long b0 = f_first - (nb - 1);                       // oldest block of the first frame
  const bool sub = p.fused_mean != 0;
  const unsigned blk_bytes = (unsigned) hop * 4u;
  unsigned phase_bits = 0;                                       // one parity bit per ring slot

  TwRegs tr;
  if constexpr (RT) load_tw_regs<M>(tr, t, p.tw, p.vtab);

  if (t == 0) {
    for (int sl = 0; sl < slots; sl++) mbar_init(&mbar[sl], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // table-twiddle plans (one group per CTA): mid-pass twiddles in shared memory, behind the group
  const float2 *tw_mid = p.tw;
  if constexpr (!RT) {
    float2 *tws = reinterpret_cast<float2 *>(smem_raw + (size_t) G * L.group_bytes);
    constexpr int kMid = TwOffset<M, Plan<M>::NP - 1>::value;
    for (int i = threadIdx.x; i < kMid; i += GeoM::THREADS) tws[i] = p.tw[i];
    tw_mid = tws;
  }
  group_sync<M>(g);

  // prologue: the nb blocks of the first frame (zeros before the stream start, fft.c:103-108)
  for (int lb = 0; lb < nb; lb++) {
    const long long blk = b0 + lb;
    if (group_active) {
      if (blk < 0) {
        float2 *z = reinterpret_cast<float2 *>(ring + (size_t) lb * hop);
        for (int i = 0; i < (1 << qs); i++) z[t + T * i] = make_float2(0.f, 0.f);
      } else if (t == 0) {
        GLB_CHECK_SRC(p, p.samples + (blk * hop - p.origin), hop);
        mbar_expect_tx(&mbar[lb], blk_bytes);
        tma_load_1d(ring + (size_t) lb * hop, p.samples + (blk * hop - p.origin), blk_bytes, &mbar[lb]);
      }
    }
  }
  float mu_new = 0.f;
  for (int lb = 0; lb < nb; lb++) {
    const long long blk = b0 + lb;
    if (group_active && blk >= 0) {
      mbar_wait(&mbar[lb], 0);
      phase_bits ^= 1u << lb;
    }
    if (sub) {
      group_sync<M>(g);                                           // zero fill visible to all (uniform: groups differ in blk)
      const float m = ring_block_mean<M>(ring + (size_t) lb * hop, qs, t, red + lb * GeoM::NW, p.inv_hop_mean, g);
      mu_new = (blk < 0) ? 0.f : m;
      if (t == 0) mu[lb] = mu_new;
    }
  }
  group_sync<M>(g);                                               // zero fill and mu[] visible

  // (CTAs that share an SM start together; a start offset per arrival rank on the SM -- rank x 400 ... 4 371 cycles,
  // or two / three clusters half / a third of a frame apart -- changed nothing here: 0.424 ... 0.430 ms.)
  int slot_new = nb - 1;                                         // slot of the newest block of frame `it`
  // loop state carried incrementally (no 64-bit multiplies per frame): frames of this group that
  // exist, the row to write and the block the next bulk copy reads
  const int nact = (group_active ? (int) ((p.nframes - fb < p.frames_per_group) ? p.nframes - fb : p.frames_per_group) : 0) + pre;
  float *row_ptr = p.rows + (fb - pre) * p.row_stride;           // (never dereferenced when p.rows is null / in the pre-roll)
  unsigned char *lev_ptr = p.levels + fb * p.lev_stride;
  const float *next_src = p.samples + ((f_first + 1) * (long long) hop - p.origin);
  // fused averaging: which of this thread's 17 bins lie in the band (bit per slot)
  unsigned av_mask = 0;
  if constexpr (AVG) {
#pragma unroll
    for (int slot = 0; slot < 17; slot++) {
      const unsigned rel = (unsigned) (slot_bin<M>(t, slot) - p.av.minbin);
      if (rel < (unsigned) av_band && (slot < 16 || t == 0)) av_mask |= 1u << slot;
    }
  }
  auto av_frame = [&](int itf) {
    // averaged row of the frame computed in iteration itf (an output frame), by the calling warp.  History
    // row of frame gg: (gg mod depth), found from the frame's own row by a 32-bit step back (no 64-bit
    // modulo per access: the first version spent 60 % of the kernel in them)
    const int lane = t & 31;
    const long long gf = f_first + itf;                          // global index of the frame
    const int sf = (int) ((unsigned long long) gf % (unsigned) av_depth);
    auto psd_at = [&](long long gg, int b) -> float {
      int s = sf - (int) (gf - gg);                              // 0 <= gf - gg < depth
      if (s < 0) s += av_depth;
      return hist[s * av_band + (b - p.av.minbin)];
    };
    avg_frame_warp<float>(p.av, fb + (itf - pre), lane, psd_at);
  };
  int hslot = (AVG && group_active) ? (int) ((unsigned long long) f_first % (unsigned) av_depth) : 0;   // history row of frame `it`
  // (fused averaging: the pre-roll, plus one idle iteration in which the last frame of a full run is averaged)
  const int n_iter = p.frames_per_group + (AVG ? av_depth : 0);
  for (int it = 0; it < n_iter; ++it, row_ptr += p.row_stride, lev_ptr += p.lev_stride, next_src += hop) {
    const bool active = it < nact;
    const bool storing = !AVG || it >= pre;                      // pre-roll frames only feed the history
    const bool next_there = it + 1 < nact;
    const int slot_next = (slot_new + 1 == slots) ? 0 : slot_new + 1;
    if (it > 0 && active) {
      // block f was requested one frame ago
      mbar_wait(&mbar[slot_new], (phase_bits >> slot_new) & 1u);
      phase_bits ^= 1u << slot_new;
    }
    auto request_next = [&]() {
      GLB_CHECK_SRC(p, next_src, hop);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_expect_tx(&mbar[slot_next], blk_bytes);
      tma_load_1d(ring + (size_t) slot_next * hop, next_src, blk_bytes, &mbar[slot_next]);
    };
    // spare slot: slot_next held block f - nb, whose last readers passed a block barrier in frame f - 1
    if (GLB_RING_EXTRA && next_there && t == 0) request_next();
    // slot of block f - nb + 1: next to the spare slot, or (tight ring) the slot block f + 1 will take
    const int slot_oldest = GLB_RING_EXTRA ? ((slot_next + 1 == slots) ? 0 : slot_next + 1) : slot_next;
    float acc[17];
    if (MULTI) {
#pragma unroll
      for (int i = 0; i < 17; i++) acc[i] = 0.f;
    }
    const int ntap = MULTI ? p.ntapers : 1;
    // the frame's samples, block means removed: fetched once, kept in registers across the tapers
    // (the multitaper variant is compiled for 4 CTAs per SM and has the registers for it)
    float2 x[kPoints];
    const bool nm = it > 0;            // the newest block has just landed: its mean is formed in ring_fetch
    float *redn = red + slot_new * GeoM::NW;
    if constexpr (QSC >= 0) {
      ring_fetch<M, (QSC >= 0 ? QSC : 0)>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, sub, nm, redn, p.inv_hop_mean, g);
    } else {
      switch (qs) {
        case 4: ring_fetch<M, 4>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, sub, nm, redn, p.inv_hop_mean, g); break;
        case 3: ring_fetch<M, 3>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, sub, nm, redn, p.inv_hop_mean, g); break;
        case 2: ring_fetch<M, 2>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, sub, nm, redn, p.inv_hop_mean, g); break;
        case 1: ring_fetch<M, 1>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, sub, nm, redn, p.inv_hop_mean, g); break;
        default: ring_fetch<M, 0>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, sub, nm, redn, p.inv_hop_mean, g); break;
      }
    }
    // (requesting the next taper's 16 pairs right after the multiply, to take their L2 latency off
    // the next transform, measured slower: 32 more live registers -> 3 CTAs/SM or spills)
    for (int j = 0; j < ntap; ++j) {
      float2 v[kPoints];
      apply_taper<M, true>(v, x, t, p, p.tapers + (size_t) j * N);
      if constexpr (RT) {
        pass_compute_rt<M, 0>(v, tr);
        group_sync<M>(g);              // (A) the previous transform's last pass has been read by all
        pass_scatter<M, 0>(v, t, buf);
      } else {
        group_sync<M>(g);
        pass_store<M, 0>(v, t, buf, p.tw);
      }
      // tight ring: the frame is in registers, so past the first (A) nobody reads the ring any more
      if (!GLB_RING_EXTRA && next_there && j == 0 && t == 0) request_next();
      if constexpr (AVG) {
        // the frame before is complete in the history (its stores precede barrier (A)); its reader is done
        // before the next barrier, i.e. before this frame's epilogue overwrites the oldest history row
        if (it > pre && it - 1 < nact && (t >> 5) == ((it - 1) & (Geo<M>::NW - 1))) av_frame(it - 1);
      }
      group_sync<M>(g);
      RingMidPasses<M, 1, RT>::run(v, t, buf, tw_mid, tr, g);
      float *row = row_ptr;
      const bool db = p.rows_db != 0;
      float yv[17];
      yv[16] = 1.f;                     // only thread 0 has a 17th bin
      auto sink_multi = [&](int slot, float2 a, bool) { acc[slot] += norm2(a); };
      auto sink_single = [&](int slot, float2 a, bool) { yv[slot] = norm2(a); };
      const bool w0 = t < 32;           // warp-uniform: only the warp that holds thread 0 pays for its re-ordering
      if constexpr (RT) {
        last_pass_rt<M>(v, t, buf, p.tw, tr);
        if (MULTI) {
          if (w0) emit_bins_rt<M, true>(v, t, tr, sink_multi);
          else emit_bins_rt<M, false>(v, t, tr, sink_multi);
        } else {
          if (w0) emit_bins_rt<M, true>(v, t, tr, sink_single);
          else emit_bins_rt<M, false>(v, t, tr, sink_single);
        }
      } else {
        // table-twiddle plans: last pass and split from 6 loaded bases, the register-twiddle code path
        TwRegs tl;
        load_last_regs<M>(tl, t, p.tw, p.vtab);
        last_pass_load<M>(v, t, buf);
        last_pass_compute_rt<M>(v, t, tl);
        if (MULTI) {
          if (w0) emit_bins_rt<M, true>(v, t, tl, sink_multi);
          else emit_bins_rt<M, false>(v, t, tl, sink_multi);
        } else {
          if (w0) emit_bins_rt<M, true>(v, t, tl, sink_single);
          else emit_bins_rt<M, false>(v, t, tl, sink_single);
        }
      }
      if (!MULTI) {
        // the row leaves the registers here: one store per bin, streaming (written once, never
        // re-read by this kernel); the display levels and the dB conversion are uniform branches
        if constexpr (LEV) {
          if (active) store_levels<M>(lev_ptr, t, yv, p.lm);
        }
        if (!LEV || p.rows != nullptr) {
          if (db) {
#pragma unroll
            for (int slot = 0; slot < 17; slot++) yv[slot] = 10.f * log10f(yv[slot]);
          }
          if constexpr (AVG) {
            if (active && av_mask != 0) {
              float *hrow = hist + hslot * av_band - p.av.minbin;
#pragma unroll
              for (int slot = 0; slot < 17; slot++)
                if (av_mask & (1u << slot)) hrow[slot_bin<M>(t, slot)] = yv[slot];
            }
          }
          if (active && storing) {
            GLB_CHECK_ROW(p, row);
            GLB_CHECK_ROW(p, row + M);
            store_row<M>(row, t, yv);
          }
        }
      }
    }
    if (MULTI && active) {
      float *row = row_ptr;
      const bool db = p.rows_db != 0;
      if constexpr (LEV) store_levels<M>(lev_ptr, t, acc, p.lm);
      if (!LEV || p.rows != nullptr) {
#pragma unroll
        for (int slot = 0; slot < 17; slot++) {
          if (slot < 16 || t == 0) {
            float y = acc[slot];
            if (db) y = 10.f * log10f(y);
            row[slot_bin<M>(t, slot)] = y;
          }
        }
      }
    }
    slot_new = slot_next;
    if constexpr (AVG) hslot = (hslot + 1 == av_depth) ? 0 : hslot + 1;
  }
}

// (Tried and removed: the periodogram's taper values in TENSOR MEMORY -- 32 words per thread written once with
// tcgen05.st and read back every frame with tcgen05.ld, to take 16 of a frame's 96 L1 / shared-memory accesses per
// thread off the busiest pipe.  0.5435 against 0.4229 ms on the metric workload, 0.489 against 0.387 ms at N = 1024:
// 16 KB per frame through tcgen05.ld cost ~400 cycles per frame and SM, i.e. tensor memory delivers ~40 bytes per
// clock to the register file in the 32x32b shape, a third of shared memory.  It pays where the volume is small and
// the shared memory it frees is worth more: the multitaper row of gram_big.cu.)
// (Tried in round 2 and removed again, commit 5cac14a: a ring kernel that forms the sums of the NEXT frame's newest
// block at the end of a frame, behind the row stores, so that one barrier at the end of the frame both publishes
// them and frees the exchange buffer -- four block barriers per frame instead of five and no sum / shuffle chain
// in front of the transform.  Bit-identical rows, and exactly as fast: 0.4240 against 0.4237 ms on the metric
// workload, 0.829 against 0.824 ms at 75 % overlap.  With six CTAs per SM the other groups fill those stalls
// already; the kernel is bound by pipe throughput (FP32 lanes, shared-memory wavefronts, issue), not by latency.)

// (Also tried and removed, commit e1c816e: the same kernel as TWO frame groups of 128 threads per CTA, each on its own named
// barrier, held half a frame apart by the handshake that gave the 32-point kernel 14 % at N = 16384 (gram_big.cu).
// Bit-identical rows; 0.479 ms with the handshake, 0.488 ms free-running, against 0.423 ms for six independent
// 128-thread CTAs per SM: six groups drift apart on their own, and named 128-thread barriers cost more than they win.)

// mid passes of the pair kernel (both frames through each pass, float4 exchange)
template <int M, int P> struct PairMidPasses {
  static __device__ __forceinline__ void run(float2 (&va)[kPoints], float2 (&vb)[kPoints], int t, float4 *buf, const TwRegs &tr) {
    if constexpr (P < Plan<M>::NP - 1) {
      pass_load2<M>(va, vb, t, buf);
      pass_compute_rt<M, P>(va, tr);
      pass_compute_rt<M, P>(vb, tr);
      __syncthreads();                  // every thread has read before anyone overwrites
      pass_scatter2<M, P>(va, vb, t, buf);
      __syncthreads();
      PairMidPasses<M, P + 1>::run(va, vb, t, buf, tr);
    }
  }
};

// ------------------------------------------------------------------------- pair kernel
// Periodogram fast path for 50 % and 75 % overlap (register-twiddle plans): every thread carries
// the same 16 points of TWO consecutive frames f, f + 1 through the transform.  The two frames
// share the taper loads and all but one of their ring blocks, the exchange buffer holds float4
// entries (frame A's value, frame B's value) so every shared-memory access is 128 bits, and the
// five block barriers, the loop bookkeeping and the address arithmetic are paid once per pair.
// The two independent butterfly streams also give the scheduler twice the ILP per warp.
// Ring: the NB + 1 blocks of the pair; after barrier (A) the two oldest slots are handed to one
// bulk-copy transaction (two copies, one mbarrier) for the blocks of the next pair.
template <int M, int QS> struct PairGeo {
  static constexpr int T = M / kPoints, NB = kPoints >> QS, SLOTS = NB + 1, NW = (T + 31) / 32;
  static constexpr int HOP = (2 * T) << QS;                          // samples per block
  static constexpr int G = Geo<M>::G, THREADS = Geo<M>::THREADS;
  static constexpr size_t BUF_BYTES = (size_t) BufSize<M>::value * sizeof(float4);
  static constexpr size_t RING_OFF = BUF_BYTES;
  static constexpr size_t RED_OFF = RING_OFF + (size_t) SLOTS * HOP * sizeof(float);
  static constexpr size_t MU_OFF = RED_OFF + (((size_t) (NB + 1) * NW * sizeof(float) + 15) / 16) * 16;
  static constexpr size_t MBAR_OFF = MU_OFF + (((size_t) SLOTS * sizeof(float) + 15) / 16) * 16;
  static constexpr size_t GROUP_BYTES = MBAR_OFF + 16;
  static constexpr size_t SMEM = (size_t) G * GROUP_BYTES;
  static constexpr int MINB_ = 65536 / (THREADS * 168);
  static constexpr int MINB = MINB_ < 1 ? 1 : MINB_;
};

template <int M, int QS>
__global__ void __launch_bounds__(Geo<M>::THREADS, (PairGeo<M, QS>::MINB)) gram_pair_kernel(const KParams p) {
  using PG = PairGeo<M, QS>;
  constexpr int T = PG::T, G = PG::G, N = 2 * M, NB = PG::NB, SLOTS = PG::SLOTS, NW = PG::NW, HOP = PG::HOP;
  constexpr int BQ = 1 << QS;                                        // float2 entries per thread and block
  constexpr int W = T < 32 ? T : 32;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int g = threadIdx.x / T;
  const int t = threadIdx.x % T;
  unsigned char *gbase = smem_raw + (size_t) g * PG::GROUP_BYTES;
  float4 *buf = reinterpret_cast<float4 *>(gbase);
  float *ring = reinterpret_cast<float *>(gbase + PG::RING_OFF);
  float *red = reinterpret_cast<float *>(gbase + PG::RED_OFF);
  float *mu = reinterpret_cast<float *>(gbase + PG::MU_OFF);
  unsigned long long *mbar = reinterpret_cast<unsigned long long *>(gbase + PG::MBAR_OFF);
  const long long gid = (long long) blockIdx.x * G + g;
  const long long fb = gid * p.frames_per_group;                    // frames_per_group is even
  const bool group_active = fb < p.nframes;
  const long long f_first = p.first_frame + fb;
  const bool sub = p.fused_mean != 0;
  constexpr unsigned blk_bytes = (unsigned) HOP * 4u;
  unsigned phase = 0;

  TwRegs tr;
  load_tw_regs<M>(tr, t, p.tw, p.vtab);

  if (t == 0) {
    mbar_init(mbar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  // prologue: blocks f_first - NB + 1 .. f_first + 1 into slots 0..NB (zeros before the stream
  // start, fft.c:103-108, and for a block past the last frame of the launch)
  {
    const long long b0 = f_first - (NB - 1);
    const bool b_there = fb + 1 < p.nframes;                         // frame B of the first pair exists
    unsigned bytes = 0;
#pragma unroll
    for (int lb = 0; lb <= NB; lb++) {
      const long long blk = b0 + lb;
      const bool want = group_active && blk >= 0 && (lb < NB || b_there);
      if (!want) {
        float2 *z = reinterpret_cast<float2 *>(ring + (size_t) lb * HOP);
#pragma unroll
        for (int i = 0; i < BQ; i++) z[t + T * i] = make_float2(0.f, 0.f);
      } else {
        bytes += blk_bytes;
      }
    }
    if (bytes != 0) {
      if (t == 0) {
        mbar_expect_tx(mbar, bytes);
#pragma unroll
        for (int lb = 0; lb <= NB; lb++) {
          const long long blk = b0 + lb;
          if (blk >= 0 && (lb < NB || b_there))
            tma_load_1d(ring + (size_t) lb * HOP, p.samples + (blk * HOP - p.origin), blk_bytes, mbar);
        }
      }
      mbar_wait(mbar, phase);
      phase ^= 1;
    }
    __syncthreads();                                                 // zero fill visible
    // means of the NB - 1 oldest blocks; the two newest are summed from registers in the loop
    if (sub) {
#pragma unroll
      for (int lb = 0; lb < NB - 1; lb++) {
        const float m = ring_block_mean<M>(ring + (size_t) lb * HOP, QS, t, red + lb * NW, p.inv_hop_mean, g);
        if (t == 0) mu[lb] = m;
      }
      __syncthreads();
    }
  }

  int s0 = 0;                                                        // slot of the oldest block of the pair
  bool pending = false;                                              // a bulk copy for this pair is in flight
  for (int it = 0; it < p.frames_per_group; it += 2) {
    const long long fl = fb + it;
    const bool active_a = fl < p.nframes, active_b = fl + 1 < p.nframes;
    const long long f = p.first_frame + fl;
    if (pending) {
      mbar_wait(mbar, phase);
      phase ^= 1;
    }
    int slot_of[NB + 1];
#pragma unroll
    for (int lb = 0; lb <= NB; lb++) slot_of[lb] = (s0 + lb) % SLOTS;

    float2 va[kPoints], vb[kPoints];
    {
      // the NB + 1 blocks of the pair: frame A is x[0..15], frame B is x[BQ..BQ+15]
      float2 x[kPoints + BQ];
#pragma unroll
      for (int lb = 0; lb <= NB; lb++) {
        const float2 *bp = reinterpret_cast<const float2 *>(ring + (size_t) slot_of[lb] * HOP);
#pragma unroll
        for (int i = 0; i < BQ; i++) x[lb * BQ + i] = bp[t + T * i];
      }
      float m[NB + 1];
#pragma unroll
      for (int lb = 0; lb <= NB; lb++) m[lb] = 0.f;
      if (sub) {
        // the two newest blocks: sums from the registers just loaded, in the order of
        // ring_block_partial (a block's mean is the same bits wherever it is formed)
        float sn[2];
#pragma unroll
        for (int e = 0; e < 2; e++) {
          float a = 0.f;
#pragma unroll
          for (int i = 0; i < BQ; i++) {
            const float2 c = x[(NB - 1 + e) * BQ + i];
            a += c.x + c.y;
          }
#pragma unroll
          for (int o = W / 2; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
          sn[e] = a;
        }
        if (NW > 1) {
          if ((t & 31) == 0) {
            red[t >> 5] = sn[0];
            red[NW + (t >> 5)] = sn[1];
          }
          __syncthreads();
        }
        m[NB - 1] = ring_block_total<M>(sn[0], red, p.inv_hop_mean);
        m[NB] = ring_block_total<M>(sn[1], red + NW, p.inv_hop_mean);
#pragma unroll
        for (int lb = 0; lb < NB - 1; lb++) m[lb] = mu[slot_of[lb]];
        if (t == 0) {
          mu[slot_of[NB - 1]] = m[NB - 1];
          mu[slot_of[NB]] = m[NB];
        }
      }
      const float2 *w2 = reinterpret_cast<const float2 *>(p.tapers);
#pragma unroll
      for (int q = 0; q < kPoints; q++) {
        const float2 w = ld_taper(w2 + t + T * q);
        va[q] = mul2(sub2(x[q], bc(m[q >> QS])), w);
        vb[q] = mul2(sub2(x[q + BQ], bc(m[(q >> QS) + 1])), w);
      }
    }
    pass_compute_rt<M, 0>(va, tr);
    pass_compute_rt<M, 0>(vb, tr);
    __syncthreads();                   // (A) the previous pair's last pass and this pair's ring reads are done
    pass_scatter2<M, 0>(va, vb, t, buf);
    {
      // the two oldest slots take the newest blocks of the next pair
      const bool next_a = (it + 2 < p.frames_per_group) && (fl + 2 < p.nframes);
      const bool next_b = next_a && (fl + 3 < p.nframes);
      pending = next_a;
      if (next_a && t == 0) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_expect_tx(mbar, next_b ? 2 * blk_bytes : blk_bytes);
        tma_load_1d(ring + (size_t) slot_of[0] * HOP, p.samples + ((f + 2) * (long long) HOP - p.origin), blk_bytes, mbar);
        if (next_b)
          tma_load_1d(ring + (size_t) slot_of[1] * HOP, p.samples + ((f + 3) * (long long) HOP - p.origin), blk_bytes, mbar);
      }
    }
    __syncthreads();
    PairMidPasses<M, 1>::run(va, vb, t, buf, tr);
    last_pass_load2<M>(va, vb, t, buf);
    const bool db = p.rows_db != 0;
    const bool w0 = t < 32;
#pragma unroll
    for (int e = 0; e < 2; e++) {
      float2 *v = e == 0 ? va : vb;
      last_pass_compute_rt<M>(v, t, tr);
      float yv[17];
      yv[16] = 1.f;
      auto sink = [&](int slot, float2 a, bool) { yv[slot] = norm2(a); };
      if (w0) emit_bins_rt<M, true>(v, t, tr, sink);
      else emit_bins_rt<M, false>(v, t, tr, sink);
      if (db) {
#pragma unroll
        for (int slot = 0; slot < 17; slot++) yv[slot] = 10.f * log10f(yv[slot]);
      }
      if (e == 0 ? active_a : active_b) store_row<M>(p.rows + (fl + e) * p.row_stride, t, yv);
    }
    s0 = (s0 + 2) % SLOTS;
  }
}

// ------------------------------------------------------------------------- warp-per-frame kernel
// Periodogram fast path for N = 512..4096: a frame never leaves its warp (fft_wpf.cuh), so the
// kernel has no block barrier at all.  Warps walk contiguous runs of INTERIOR frames (no zero
// history, fully inside the staged samples, 8-byte aligned); the few edge frames of a
// recording are launched through the general kernel by the host code below.
#ifndef GLB_WPF_MINB
#define GLB_WPF_MINB 5
#endif
constexpr int kWpfWarps = 2;          // warps per CTA (independent of each other)

// block-mean removal inside one lane group: hop = 2T << QW; block b = registers q with (q >> QW) == b
template <int M, int QW>
__device__ __forceinline__ void wpf_remove_means(float2 (&x)[kWP], float inv_hop) {
  constexpr int T = Wpf<M>::T, NB = kWP >> QW;
#pragma unroll
  for (int b = 0; b < NB; b++) {
    float s = 0.f;
#pragma unroll
    for (int q = b << QW; q < (b + 1) << QW; q++) s += x[q].x + x[q].y;
#pragma unroll
    for (int o = T / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float m = s * inv_hop;
#pragma unroll
    for (int q = b << QW; q < (b + 1) << QW; q++) {
      x[q].x -= m;
      x[q].y -= m;
    }
  }
}

template <int M>
__global__ void __launch_bounds__(32 * kWpfWarps, GLB_WPF_MINB) gram_wpf_kernel(const KParams p) {
  constexpr int T = Wpf<M>::T, N = 2 * M, FPW = 32 / T;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane / T, t = lane % T;
  float2 *tile = reinterpret_cast<float2 *>(smem_raw) + (size_t) (warp * FPW + g) * (Wpf<M>::TILE + 2);
  const long long gid = ((long long) blockIdx.x * kWpfWarps + warp) * FPW + g;
  const long long fb = gid * p.frames_per_group;

  WpfRegs rg;
  wpf_load_regs<M>(rg, t, p.roots, p.vtab);
  const float2 *w2 = reinterpret_cast<const float2 *>(p.tapers) + t;
  const bool db = p.rows_db != 0;

  for (int it = 0; it < p.frames_per_group; ++it) {
    const long long fl = fb + it;
    const bool active = fl < p.nframes;
    // inactive tail iterations recompute the group's last frame without storing (keeps the
    // warp converged for the shuffles and __syncwarp below)
    const long long fe = active ? fl : (p.nframes - 1);
    const long long f = p.first_frame + fe;
    const float2 *src = reinterpret_cast<const float2 *>(p.samples + (f * (long long) p.hop - p.n_ov - p.origin)) + t;
    float2 v[kWP];
#pragma unroll
    for (int q = 0; q < kWP; q++) v[q] = ldg2(src + T * q);
    if (fl + 1 < p.nframes && it + 1 < p.frames_per_group) {
      // pull the next frame's new hop block towards L2 behind this frame's arithmetic
      const float *nx = p.samples + ((f + 1) * (long long) p.hop - p.origin);
      for (int i = t * 32; i < p.hop; i += T * 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(nx + i));
    }
    if (p.fused_mean) {
      switch (p.qs) {
        case 6: wpf_remove_means<M, 6>(v, p.inv_hop_mean); break;
        case 5: wpf_remove_means<M, 5>(v, p.inv_hop_mean); break;
        case 4: wpf_remove_means<M, 4>(v, p.inv_hop_mean); break;
        case 3: wpf_remove_means<M, 3>(v, p.inv_hop_mean); break;
        default: wpf_remove_means<M, 2>(v, p.inv_hop_mean); break;
      }
    }
#pragma unroll
    for (int q = 0; q < kWP; q++) {
      const float2 w = ldg2(w2 + T * q);
      v[q].x *= w.x;
      v[q].y *= w.y;
    }
    wpf_pass_a<M>(v);
    __syncwarp();                      // the previous frame's gathers are done
    wpf_scatter<M>(v, t, tile);
    __syncwarp();
    wpf_gather<M>(v, t, tile);
    wpf_pass_b<M>(v, t, rg);
    float *row = p.rows + fe * p.row_stride;
    wpf_emit<M>(v, t, rg, [&](int, int bin, float2 a, bool) {
      float y = norm2(a);
      if (db) y = 10.f * log10f(y);
      if (active) row[bin] = y;
    });
  }
}

template <int M>
inline int launch_wpf(const KParams &kp, cudaStream_t st) {
  int dev = 0, sms = 0;
  CU(cudaGetDevice(&dev));
  CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  constexpr int FPW = 32 / Wpf<M>::T;
  const size_t smem = (size_t) kWpfWarps * FPW * (Wpf<M>::TILE + 2) * sizeof(float2);
  static thread_local int occ_cache[64];
  int &occ = occ_cache[dev & 63];
  if (occ == 0) {
    CU(cudaFuncSetAttribute(gram_wpf_kernel<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, gram_wpf_kernel<M>, 32 * kWpfWarps, smem));
    if (occ < 1) occ = 1;
  }
  long long groups = (long long) sms * occ * kWpfWarps * FPW;
  if (groups > kp.nframes) groups = kp.nframes;
  if (groups < 1) groups = 1;
  KParams k = kp;
  k.frames_per_group = (int) ((kp.nframes + groups - 1) / groups);
  const long long used = (kp.nframes + k.frames_per_group - 1) / k.frames_per_group;
  const int ctas = (int) ((used + kWpfWarps * FPW - 1) / (kWpfWarps * FPW));
  gram_wpf_kernel<M><<<ctas, 32 * kWpfWarps, smem, st>>>(k);
  CU(cudaGetLastError());
  g_launches++;
  g_last_family = 3;
  return GLB_OK;
}

// which kernel family serves a launch (tests / experiments can pin one)

template <int M>
inline int launch_gram_m(const KParams &kp, bool multi, int groups_hint, cudaStream_t st, int allow) {
  using GeoM = Geo<M>;
  int dev = 0, sms = 0;
  CU(cudaGetDevice(&dev));
  CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const bool plain = multi || (kp.ra9mb_a <= 0.f && kp.limiter == 0);
  // ---- fastest path (N <= 4096 periodograms): warp-per-frame kernel on the interior frames
  if constexpr (M >= 256 && M <= 2048) {
    constexpr int unitw = 2 * Wpf<M>::T;
    int qw = -1;
    for (int s2 = 2; s2 <= 6; s2++)
      if (kp.hop == (unitw << s2)) qw = s2;
    const bool mean_ok = !kp.fused_mean || (qw >= 0 && (kp.n_ov % kp.hop) == 0);
    const bool pref_ok = (allow & 4) != 0;
    if (pref_ok && !multi && plain && kp.rows != nullptr && kp.levels == nullptr && kp.spectrum == nullptr && kp.means == nullptr && mean_ok &&
        (kp.hop % 2) == 0 && ((kp.n_ov + kp.origin) % 2) == 0 && ((reinterpret_cast<uintptr_t>(kp.samples) & 7) == 0)) {
      // interior frames: f*hop - n_ov >= max(origin, 0) and the frame ends inside the staged samples
      const long long lo_s = kp.origin > 0 ? kp.origin : 0;
      long long f_lo = (lo_s + kp.n_ov + kp.hop - 1) / kp.hop;
      long long f_hi = (kp.origin + kp.count - kp.hop) / kp.hop + 1;       // exclusive: (f+1)*hop <= origin+count
      if (f_lo < kp.first_frame) f_lo = kp.first_frame;
      if (f_hi > kp.first_frame + kp.nframes) f_hi = kp.first_frame + kp.nframes;
      if (f_hi > f_lo) {
        KParams kw = kp;
        kw.qs = qw;
        kw.first_frame = f_lo;
        kw.nframes = f_hi - f_lo;
        kw.rows = kp.rows + (f_lo - kp.first_frame) * kp.row_stride;
        int rc = launch_wpf<M>(kw, st);
        if (rc != GLB_OK) return rc;
        // edge frames before / after the interior run go through the kernels below
        KParams ke = kp;
        if (f_lo > kp.first_frame) {
          ke.nframes = f_lo - kp.first_frame;
          rc = launch_gram_m<M>(ke, multi, groups_hint, st, 1);
          if (rc != GLB_OK) return rc;
        }
        if (f_hi < kp.first_frame + kp.nframes) {
          ke = kp;
          ke.first_frame = f_hi;
          ke.nframes = kp.first_frame + kp.nframes - f_hi;
          ke.rows = kp.rows + (f_hi - kp.first_frame) * kp.row_stride;
          rc = launch_gram_m<M>(ke, multi, groups_hint, st, 1);
          if (rc != GLB_OK) return rc;
        }
        return GLB_OK;
      }
    }
  }
  // ---- fast path: regular geometry, rows only, 16-byte aligned blocks -> TMA ring / pair kernel
  {
    const int unit = 2 * GeoM::T;
    int qs = -1;
    for (int s2 = 0; s2 <= 4; s2++)
      if (kp.hop == (unit << s2)) qs = s2;
    // the fast paths read whole hop blocks without bounds checks: the staged span must cover every
    // block of the launch that lies inside the stream (blocks before sample 0 are the zero history)
    const long long blk_lo = (kp.first_frame - kp.n_ov / kp.hop) * (long long) kp.hop;
    const long long blk_hi = (kp.first_frame + kp.nframes) * (long long) kp.hop;
    const bool covered = kp.origin <= (blk_lo > 0 ? blk_lo : 0) && blk_hi <= kp.origin + kp.count;
    const bool regular = qs >= 0 && (kp.n_ov % kp.hop) == 0 && (kp.hop % 4) == 0 && (kp.origin % 4) == 0 &&
                         ((reinterpret_cast<uintptr_t>(kp.samples) & 15) == 0) && covered;
    if constexpr (GeoM::RT && M >= 256) {
      // 50 % / 75 % overlap periodograms: two frames per thread (selectable family: measured
      // 0.431 ms vs 0.422 ms for the ring kernel on the metric workload, 3 CTAs/SM vs 6)
      if (regular && !multi && plain && kp.rows != nullptr && kp.levels == nullptr && kp.spectrum == nullptr && kp.means == nullptr &&
          (allow & 8) != 0 && (qs == 3 || qs == 2) && kp.nframes >= 2) {
        void (*pk)(const KParams) = qs == 3 ? gram_pair_kernel<M, 3> : gram_pair_kernel<M, 2>;
        const size_t smem = qs == 3 ? PairGeo<M, 3>::SMEM : PairGeo<M, 2>::SMEM;
        static thread_local int occ_pair[2][64];
        int &occ = occ_pair[qs - 2][dev & 63];
        if (occ == 0) {
          CU(cudaFuncSetAttribute(pk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
          CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pk, GeoM::THREADS, smem));
          if (occ < 1) occ = -1;
        }
        if (occ >= 1) {
          long long groups = groups_hint > 0 ? groups_hint : (long long) sms * occ * GeoM::G;
          if (groups > (kp.nframes + 1) / 2) groups = (kp.nframes + 1) / 2;
          if (groups < 1) groups = 1;
          KParams k = kp;
          k.qs = qs;
          long long fpg = (kp.nframes + groups - 1) / groups;
          fpg += fpg & 1;                                            // whole pairs per group
          k.frames_per_group = (int) fpg;
          long long used = (kp.nframes + fpg - 1) / fpg;
          int ctas = (int) ((used + GeoM::G - 1) / GeoM::G);
          pk<<<ctas, GeoM::THREADS, smem, st>>>(k);
          CU(cudaGetLastError());
          g_launches++;
          g_last_family = 4;
          return GLB_OK;
        }
      }
    }
    if (regular && plain && (kp.rows != nullptr || kp.levels != nullptr) && kp.spectrum == nullptr && kp.means == nullptr &&
        (allow & 2) != 0) {
      const int nb = kPoints >> qs;
      const bool avg = kp.av_on != 0;
      const int hist_floats = avg ? kp.av.depth * (kp.av.maxbin - kp.av.minbin) : 0;
      const RingLayout L = ring_layout<M>(kp.hop, nb, hist_floats);
      size_t smem = (size_t) GeoM::G * L.group_bytes + ((multi ? RingGeo<M, true>::RT : RingGeo<M, false>::RT) ? 0 : Geo<M>::TWS_BYTES);
      if (const char *e = getenv("GLB_SMEM_PAD_KB")) smem += (size_t) atoi(e) * 1024;     // experiments: cap the CTAs per SM
      if (smem <= 227 * 1024) {
        // 50 % and 75 % overlap have kernels with the ring geometry folded in
        void (*rk)(const KParams) = nullptr;
        const bool lev = kp.levels != nullptr;       // 8-bit display levels: a second set of instantiations
        if (avg) {
          // fused frame averaging: one frame group per CTA, periodogram, float rows (N = 4096, 8192)
          if constexpr (M == 2048 || M == 4096) {
            if (multi || lev) { glb_set_error("glb_launch_gram: fused averaging is for periodogram float rows"); return GLB_EINVAL; }
            rk = qs == 3 ? gram_ring_kernel<M, false, 3, false, true>
                         : (qs == 2 ? gram_ring_kernel<M, false, 2, false, true> : gram_ring_kernel<M, false, -1, false, true>);
            CU(cudaFuncSetAttribute(rk, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
            int occ_a = 0;
            CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_a, rk, GeoM::THREADS, smem));
            if (occ_a < 1) { glb_set_error("glb_launch_gram: fused averaging does not fit shared memory"); return GLB_EINVAL; }
            long long groups = groups_hint > 0 ? groups_hint : (long long) sms * occ_a;
            if (groups > kp.nframes) groups = kp.nframes;
            if (groups < 1) groups = 1;
            KParams k = kp;
            k.qs = qs;
            k.frames_per_group = (int) ((kp.nframes + groups - 1) / groups);
            const long long used = (kp.nframes + k.frames_per_group - 1) / k.frames_per_group;
            rk<<<(int) used, GeoM::THREADS, smem, st>>>(k);
            CU(cudaGetLastError());
            g_launches++;
            g_last_family = 2;
            return GLB_OK;
          } else {
            glb_set_error("glb_launch_gram: fused averaging is available for N = 4096 and 8192 (see glb_gram_fused_avg_ok)");
            return GLB_EINVAL;
          }
        }
        if (qs == 3) rk = multi ? (lev ? gram_ring_kernel<M, true, 3, true> : gram_ring_kernel<M, true, 3, false>)
                                : (lev ? gram_ring_kernel<M, false, 3, true> : gram_ring_kernel<M, false, 3, false>);
        else if (qs == 2) rk = multi ? (lev ? gram_ring_kernel<M, true, 2, true> : gram_ring_kernel<M, true, 2, false>)
                                     : (lev ? gram_ring_kernel<M, false, 2, true> : gram_ring_kernel<M, false, 2, false>);
        else rk = multi ? (lev ? gram_ring_kernel<M, true, -1, true> : gram_ring_kernel<M, true, -1, false>)
                        : (lev ? gram_ring_kernel<M, false, -1, true> : gram_ring_kernel<M, false, -1, false>);
        static thread_local int occ_ring[2][2][5][64];
        int &occ = occ_ring[lev ? 1 : 0][multi ? 1 : 0][qs][dev & 63];
        if (occ == 0) {
          // opt in to the device maximum once: the ring size (hence the launch's smem) varies with the overlap
          CU(cudaFuncSetAttribute(rk, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
          CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, rk, GeoM::THREADS, smem));
          if (occ < 1) occ = -1;
        }
        // big frames: the ring must not cost more residency than it saves in traffic
        int occ_generic_bound = (int) ((227 * 1024) / GeoM::smem_bytes(false));
        // (N = 16384: one 512-thread CTA per SM with the ring still beats two without, 2.39 vs 2.55 ms)
        const bool worth = occ >= 2 || (occ >= 1 && occ_generic_bound <= 1) || GeoM::THREADS >= 512 || g_kernel_pref == 2;
        if (occ >= 1 && worth) {
          long long groups = groups_hint > 0 ? groups_hint : (long long) sms * occ * GeoM::G;
          // Several waves of shorter frame runs instead of one run per resident group: groups that share an SM
          // do not progress at the same rate, and with a single wave the early finishers leave their slots
          // idle for the rest of the launch; with more CTAs than slots the block scheduler refills them.  A run
          // pays one prologue (the nb - 1 history blocks and their means, other CTAs of the SM hide it), so
          // runs stay >= kRingMinRun frames.  Metric workload (N = 4096, 84 375 frames, B200): 1 / 2 / 3 / 4 / 6
          // waves 0.423 / 0.405 / 0.398 / 0.395 / 0.396-0.401 ms.  Rows do not depend on the split.
          constexpr int kRingWaves = 4, kRingMinRun = 16;
          if (groups_hint <= 0 && occ >= 2) {
            int waves = kRingWaves;
            while (waves > 1 && kp.nframes < groups * waves * kRingMinRun) waves--;
            groups *= waves;
          }
          if (groups > kp.nframes) groups = kp.nframes;
          if (groups < 1) groups = 1;
          KParams k = kp;
          k.qs = qs;
          k.frames_per_group = (int) ((kp.nframes + groups - 1) / groups);
          long long used = (kp.nframes + k.frames_per_group - 1) / k.frames_per_group;
          int ctas = (int) ((used + GeoM::G - 1) / GeoM::G);
          rk<<<ctas, GeoM::THREADS, smem, st>>>(k);
          CU(cudaGetLastError());
          g_launches++;
          g_last_family = 2;
          return GLB_OK;
        }
      }
    }
  }
  if (kp.av_on) {
    glb_set_error("glb_launch_gram: fused averaging needs the regular geometry of the ring kernel (see glb_gram_fused_avg_ok)");
    return GLB_EINVAL;
  }
  const int variant = multi ? 2 : (plain ? 1 : 0);
  const bool glev = kp.levels != nullptr;
  if (glev && !plain) {
    glb_set_error("glb_launch_gram: display levels are not available together with RA9MB / limiter");
    return GLB_EINVAL;
  }
  auto kern = glev ? (multi ? gram_kernel<M, true, true, true> : gram_kernel<M, false, true, true>)
                   : (multi ? gram_kernel<M, true, true> : (plain ? gram_kernel<M, false, true> : gram_kernel<M, false, false>));
  // the staging buffer is only carved out for the multitaper variant
  const size_t smem = GeoM::smem_bytes(multi);
  // per (device, variant): opt in to the dynamic shared memory once, cache the occupancy
  static thread_local int occ_cache[6][64];
  int &occ = occ_cache[variant + (glev ? 3 : 0)][dev & 63];
  if (occ == 0) {
    CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, GeoM::THREADS, smem));
    if (occ < 1) occ = 1;
  }
  // resident grid: every CTA slot of the chip holds G frame groups, each walking a
  // contiguous run of frames (keeps the overlapped samples of consecutive frames in L1/L2)
  long long groups = groups_hint > 0 ? groups_hint : (long long) sms * occ * GeoM::G;
  if (groups > kp.nframes) groups = kp.nframes;
  if (groups < 1) groups = 1;
  KParams k = kp;
  k.frames_per_group = (int) ((kp.nframes + groups - 1) / groups);
  long long used = (kp.nframes + k.frames_per_group - 1) / k.frames_per_group;
  int ctas = (int) ((used + GeoM::G - 1) / GeoM::G);
  // regular geometry for the fused block means: hop = 2T << qs, n_ov a multiple of hop
  k.fused_mean = 0;
  k.qs = 0;
  if (kp.fused_mean) {
    const int unit = 2 * GeoM::T;
    int qs = -1;
    for (int s2 = 0; s2 <= 4; s2++)
      if (kp.hop == (unit << s2)) qs = s2;
    if (qs >= 0 && (k.n_ov % kp.hop) == 0) {
      k.fused_mean = 1;
      k.qs = qs;
    } else {
      glb_set_error("glb_launch_gram: fused block means need hop = (N/16) << s, s = 0..4");
      return GLB_EINVAL;
    }
  }
  kern<<<ctas, GeoM::THREADS, smem, st>>>(k);
  CU(cudaGetLastError());
  g_launches++;
  g_last_family = 1;
  return GLB_OK;
}


// one function per translation unit of gram_part.cu: the FFT sizes of that part
#define GLB_DECLARE_PART(K) int glb_gram_part_##K(int m, const KParams &k, bool multi, int groups_hint, cudaStream_t st, int allow)
GLB_DECLARE_PART(0);
GLB_DECLARE_PART(1);
GLB_DECLARE_PART(2);
GLB_DECLARE_PART(3);
// the 32-points-per-thread family for N = 16384 / 32768 (gram_big.cu); -1 = not served
int glb_gram_big(int m, const KParams &k, bool multi, int groups_hint, cudaStream_t st, bool small_too);
