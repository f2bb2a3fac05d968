// lines.cu -- harmonic line selection over device F rows (glb_launch_ftest_lines): the *_run_mtm_lines entries of the
// I/Q and zoom plans (host/cframe.c, include/glfer_b200.h).
//
//   ftest_lines_kernel<V>  one warp per frame (8 per CTA, grid-stride over the launch's frames).  A bin j of
//                          [bin_lo, bin_hi) is a candidate when F[j] > thr, F[j] > F[j - 1] and F[j] >= F[j + 1] (cyclic
//                          neighbours, read from the whole row).  The row is walked in strips of 32 V bins: lane l loads
//                          bins V l .. V l + V - 1 of the strip with one vector load (coalesced), the neighbours inside
//                          the warp come through shuffles and only the two strip edges are re-read.  The first pass
//                          fetches kLnUnroll strips before it examines them, to keep loads in flight.  Candidates are
//                          ranked with ballots and popc, so the first pass stores them in ascending j while it counts
//                          them: a frame with at most max_lines candidates is done in one pass.
//                          A frame with more takes the max_lines largest by (F, -j): a radix select on ln_key (the
//                          order-preserving integer image of the float, as fs_key in gram_kernels.cu), four 8-bit
//                          passes over the row's candidates with a per-warp shared histogram, finds the key T of the
//                          max_lines-th largest; a last pass keeps every candidate above T and the first of those equal
//                          to T in ascending j until the slots are full, again stored in ascending j.
#include <cuda_runtime.h>
#include <atomic>
#include <cstdio>
#include "../../include/glb_shim.h"

extern std::atomic<unsigned long long> g_launches;   // gram_kernels.cu

#define LCU(call)                                                                             \
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

constexpr int kLnWarps = 8;            // frames per CTA
constexpr int kLnCtasPerSm = 4;        // 56 / 62 / 64 registers (V = 1 / 2 / 4), no spills; 5 spills at V = 4
constexpr int kLnUnroll = 4;           // strips in flight per warp in the first pass
constexpr unsigned kFull = 0xffffffffu;

__device__ __forceinline__ unsigned ln_key(float f) {
  const unsigned b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);       // ascending keys <=> ascending floats
}

template <int V>
__device__ __forceinline__ void ln_load(const float *p, float (&v)[V]) {
  if constexpr (V == 4) {
    const float4 t = __ldg(reinterpret_cast<const float4 *>(p));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  } else if constexpr (V == 2) {
    const float2 t = __ldg(reinterpret_cast<const float2 *>(p));
    v[0] = t.x; v[1] = t.y;
  } else {
    v[0] = __ldg(p);
  }
}

// the strip [base, base + 32 V) of the row: its values v and the bin after it (lane 31) or before it (lane 0)
template <int V>
__device__ __forceinline__ void ln_fetch(const float *row, int n, int base, int lane, float (&v)[V], float &edge) {
  // the strip's cyclic edges: lane 0 re-reads the bin before it, lane 31 the bin after it
  const int e = lane == 0 ? (base == 0 ? n - 1 : base - 1) : (base + 32 * V == n ? 0 : base + 32 * V);
  edge = (lane == 0 || lane == 31) ? __ldg(row + e) : 0.f;
  ln_load<V>(row + base + V * lane, v);
}

// the candidate mask of a fetched strip (bit q: bin base + V lane + q)
template <int V>
__device__ __forceinline__ unsigned ln_mask(int base, int lane, float thr, int lo, int hi, const float (&v)[V],
                                            float edge) {
  float left = __shfl_up_sync(kFull, v[V - 1], 1);
  float right = __shfl_down_sync(kFull, v[0], 1);
  if (lane == 0) left = edge;
  if (lane == 31) right = edge;
  unsigned m = 0;
#pragma unroll
  for (int q = 0; q < V; q++) {
    const float l = q == 0 ? left : v[q - 1];
    const float r = q == V - 1 ? right : v[q + 1];
    const int j = base + V * lane + q;
    if (v[q] > thr && v[q] > l && v[q] >= r && j >= lo && j < hi) m |= 1u << q;
  }
  return m;
}

template <int V>
__device__ __forceinline__ unsigned ln_strip(const float *row, int n, int base, int lane, float thr, int lo, int hi,
                                             float (&v)[V]) {
  float edge;
  ln_fetch<V>(row, n, base, lane, v, edge);
  return ln_mask<V>(base, lane, thr, lo, hi, v, edge);
}

// set bits of the strip's masks in ascending j below this lane's bins, and (tot) in the whole strip
template <int V>
__device__ __forceinline__ int ln_below(unsigned m, int lane, int &tot) {
  const unsigned lt = (1u << lane) - 1u;
  int below = 0;
  tot = 0;
#pragma unroll
  for (int q = 0; q < V; q++) {
    const unsigned b = __ballot_sync(kFull, (m >> q) & 1u);
    below += __popc(b & lt);
    tot += __popc(b);
  }
  return below;
}

template <int V>
__global__ void __launch_bounds__(32 * kLnWarps, kLnCtasPerSm)
ftest_lines_kernel(const float *__restrict__ ftest, const float *__restrict__ psd, int n, long long stride, long long cn,
                   int nchan, long long crows, float thr, int max_lines, int lo, int hi, int *__restrict__ count,
                   int *__restrict__ bin, float *__restrict__ out_f, float *__restrict__ out_p) {
  __shared__ int s_hist[kLnWarps][256];
  constexpr int SEG = 32 * V;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int *hist = s_hist[w];
  const int b0 = lo / SEG * SEG;
  const long long nout = cn * nchan;
  for (long long o = (long long) blockIdx.x * kLnWarps + w; o < nout; o += (long long) gridDim.x * kLnWarps) {
    // output frame o = channel ch's frame fr, device row ch crows + fr
    const long long ch = o / cn, fr = o - ch * cn;
    const float *row = ftest + (ch * crows + fr) * stride;
    const float *prow = psd ? psd + (ch * crows + fr) * stride : nullptr;
    int *ob = bin + o * max_lines;
    float *of = out_f ? out_f + o * max_lines : nullptr;
    float *op = out_p ? out_p + o * max_lines : nullptr;
    // ---- one pass: count the candidates, store the first max_lines in ascending j.  kLnUnroll strips are fetched
    // before any is examined: a short launch (a zoom's chunk is a few frames per channel) is bound by load latency
    int total = 0;
    for (int base0 = b0; base0 < hi; base0 += kLnUnroll * SEG) {
      float v[kLnUnroll][V], edge[kLnUnroll];
#pragma unroll
      for (int u = 0; u < kLnUnroll; u++)
        if (base0 + u * SEG < hi) ln_fetch<V>(row, n, base0 + u * SEG, lane, v[u], edge[u]);
#pragma unroll
      for (int u = 0; u < kLnUnroll; u++) {
        const int base = base0 + u * SEG;
        if (base >= hi) break;
        const unsigned m = ln_mask<V>(base, lane, thr, lo, hi, v[u], edge[u]);
        if (__ballot_sync(kFull, m != 0u) == 0u) continue;   // most strips hold no candidate
        int tot;
        int slot = total + ln_below<V>(m, lane, tot);
#pragma unroll
        for (int q = 0; q < V; q++) {
          if ((m >> q) & 1u) {
            if (slot < max_lines) {
              const int j = base + V * lane + q;
              ob[slot] = j;
              if (of) of[slot] = v[u][q];
              if (op) op[slot] = prow[j];
            }
            slot++;
          }
        }
        total += tot;
      }
    }
    if (total <= max_lines) {
      for (int s = total + lane; s < max_lines; s += 32) {
        ob[s] = -1;
        if (of) of[s] = 0.f;
        if (op) op[s] = 0.f;
      }
    } else {
      // ---- overflow: key T of the max_lines-th largest candidate, most significant byte first
      unsigned prefix = 0;
      int want = max_lines;                                 // rank (1-based, descending) still to be located
      for (int pass = 3; pass >= 0; --pass) {
        for (int b = lane; b < 256; b += 32) hist[b] = 0;
        __syncwarp();
        const int sh = 8 * pass;
        const unsigned himask = pass == 3 ? 0u : (0xffffffffu << (sh + 8));
        for (int base = b0; base < hi; base += SEG) {
          float v[V];
          const unsigned m = ln_strip<V>(row, n, base, lane, thr, lo, hi, v);
#pragma unroll
          for (int q = 0; q < V; q++) {
            const unsigned k = ln_key(v[q]);
            if (((m >> q) & 1u) && (k & himask) == prefix) atomicAdd(&hist[(k >> sh) & 255u], 1);
          }
        }
        __syncwarp();
        // lane l owns digits 255 - 8 l .. 248 - 8 l, in descending order
        int loc[8], tot = 0;
#pragma unroll
        for (int d = 0; d < 8; d++) { loc[d] = hist[255 - 8 * lane - d]; tot += loc[d]; }
        int incl = tot;
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
          const int up = __shfl_up_sync(kFull, incl, s);
          if (lane >= s) incl += up;
        }
        int above = incl - tot;                             // candidates in digits above this lane's
        int digit = -1, above_d = 0;
        if (above < want && want <= incl) {
#pragma unroll
          for (int d = 0; d < 8; d++) {
            if (digit < 0 && want <= above + loc[d]) { digit = 255 - 8 * lane - d; above_d = above; }
            if (digit < 0) above += loc[d];
          }
        }
        const int src = __ffs(__ballot_sync(kFull, digit >= 0)) - 1;
        digit = __shfl_sync(kFull, digit, src);
        above_d = __shfl_sync(kFull, above_d, src);
        prefix |= (unsigned) digit << sh;
        want -= above_d;
        __syncwarp();
      }
      // ---- every candidate above T, then `want` of those equal to T in ascending j, stored in ascending j
      int slot0 = 0, ties0 = 0;
      for (int base = b0; base < hi; base += SEG) {
        float v[V];
        const unsigned m = ln_strip<V>(row, n, base, lane, thr, lo, hi, v);
        if (__ballot_sync(kFull, m != 0u) == 0u) continue;
        unsigned sel = 0, tie = 0;
#pragma unroll
        for (int q = 0; q < V; q++) {
          const unsigned k = ln_key(v[q]);
          if ((m >> q) & 1u) {
            if (k > prefix) sel |= 1u << q;
            else if (k == prefix) tie |= 1u << q;
          }
        }
        int ntie;
        int t = ties0 + ln_below<V>(tie, lane, ntie);
#pragma unroll
        for (int q = 0; q < V; q++) {
          if ((tie >> q) & 1u) {
            if (t < want) sel |= 1u << q;
            t++;
          }
        }
        ties0 += ntie;
        int nsel;
        int slot = slot0 + ln_below<V>(sel, lane, nsel);
#pragma unroll
        for (int q = 0; q < V; q++) {
          if ((sel >> q) & 1u) {
            const int j = base + V * lane + q;
            ob[slot] = j;
            if (of) of[slot] = v[q];
            if (op) op[slot] = prow[j];
            slot++;
          }
        }
        slot0 += nsel;
      }
    }
    if (lane == 0) count[o] = total;
  }
}

extern "C" int glb_launch_ftest_lines(const float *ftest, const float *rows, int n, long long stride, long long nframes,
                                      int nchan, long long crows, float thr, int max_lines, int bin_lo, int bin_hi,
                                      int *count, int *bin, float *line_ftest, float *line_psd, void *stream) {
  if (nframes <= 0) return GLB_OK;
  if (n < 32 || n > 16384 || (n & (n - 1)) != 0 || stride < n || stride % 4 != 0 || nchan < 1 ||
      (nchan > 1 && crows < nframes) || max_lines < 1 || max_lines > 1024 || bin_lo < 0 || bin_lo >= bin_hi ||
      bin_hi > n || !ftest || !count || !bin || (line_psd && !rows)) {
    glb_set_error("ftest_lines: invalid arguments");
    return GLB_EINVAL;
  }
  long long ctas = (nframes * nchan + kLnWarps - 1) / kLnWarps;
  if (ctas > 148 * 16) ctas = 148 * 16;
  const float *p = line_psd ? rows : nullptr;
  cudaStream_t st = (cudaStream_t) stream;
  // V bins per lane and strip: the widest vector load whose strip of 32 V bins divides the row
  if (n >= 128)
    ftest_lines_kernel<4><<<(unsigned) ctas, 32 * kLnWarps, 0, st>>>(ftest, p, n, stride, nframes, nchan, crows, thr,
                                                                     max_lines, bin_lo, bin_hi, count, bin, line_ftest,
                                                                     line_psd);
  else if (n == 64)
    ftest_lines_kernel<2><<<(unsigned) ctas, 32 * kLnWarps, 0, st>>>(ftest, p, n, stride, nframes, nchan, crows, thr,
                                                                     max_lines, bin_lo, bin_hi, count, bin, line_ftest,
                                                                     line_psd);
  else
    ftest_lines_kernel<1><<<(unsigned) ctas, 32 * kLnWarps, 0, st>>>(ftest, p, n, stride, nframes, nchan, crows, thr,
                                                                     max_lines, bin_lo, bin_hi, count, bin, line_ftest,
                                                                     line_psd);
  LCU(cudaGetLastError());
  g_launches++;
  return GLB_OK;
}
