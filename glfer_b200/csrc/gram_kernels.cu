// gram_kernels.cu -- the C-ABI CUDA shim: stream/event/memory plumbing, constant tables, the
// launch entry points and the small kernels around the spectrogram kernels proper (which live in
// gram_common.cuh and are instantiated per FFT size by gram_part.cu).
//
// Kernels (all hand-written, no library FFT):
//   gram_kernel<M> / gram_ring_kernel<M> / gram_wpf_kernel<M>   (gram_common.cuh)
//                         overlapped-frame gather -> [block-mean removal] -> [RA9MB] ->
//                         taper multiply -> [limiter] -> real FFT (N = 2M, in registers +
//                         padded shared memory) -> |X|^2 -> [sum over K' tapers with the
//                         1/lambda weights folded into the tapers] -> [10 log10] -> one PSD
//                         row per frame straight to HBM.  Replaces prepare_audio + fft_do +
//                         fft_psd (fft.c:66-226) and the taper loop of mtm_do (mtm.c:189-220).
//   block_means_kernel    mean of every hop block (prepare_audio, fft.c:86-96).
//   avg_kernel            sliding per-bin frame averaging, three normalisations
//                         (update_avg_*, avg.c:108-298).
//   peak_carry_kernel     the carried *peakbin of avg.c:129-133.
//   pcm*_to_float_kernel  WAV sample conversion (wav_fmt.c:105-116).
//
// No tensor cores: the path is an FFT at ~9 flop/B executed, bound by HBM and the
// FP32/shared-memory pipes, not a dense contraction (see DESIGN.md).
#include "gram_common.cuh"

// ------------------------------------------------------------------------- errors
static thread_local char g_err[512] = "";
std::atomic<unsigned long long> g_launches{0};
int g_kernel_pref = 0;               // 0 auto, 1 general, 2 ring, 3 warp-per-frame, 4 two frames per thread
int g_last_family = 0;
int g_force_generic = 0;            // tests: run the general kernel where the ring kernel would be chosen (also iq.cu)

extern "C" const char *glb_last_error(void) { return g_err; }
extern "C" void glb_set_error(const char *msg) { snprintf(g_err, sizeof g_err, "%s", msg ? msg : ""); }
extern "C" unsigned long long glb_kernel_launches(void) { return g_launches.load(); }
extern "C" void glb_force_generic_kernel(int on) { g_force_generic = on; }
extern "C" void glb_set_kernel_preference(int pref) {
  // 6 = automatic choice, but the 32-point kernel never pairs two frame groups in one CTA (A/B measurements)
  g_big_pair = pref != 6;
  g_kernel_pref = pref == 6 ? 0 : pref;
}
extern "C" int glb_last_kernel_family(void) { return g_last_family; }

// ------------------------------------------------------------------------- plumbing
extern "C" int glb_device_count(int *count) {
  int c = 0;
  cudaError_t e = cudaGetDeviceCount(&c);
  if (e != cudaSuccess) {
    snprintf(g_err, sizeof g_err, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    *count = 0;
    return GLB_ENODEV;
  }
  *count = c;
  return GLB_OK;
}
extern "C" int glb_set_device(int dev) { CU(cudaSetDevice(dev)); return GLB_OK; }
extern "C" int glb_sm_count(int dev, int *sms) {
  CU(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev));
  return GLB_OK;
}
extern "C" int glb_malloc(void **p, size_t bytes) { CU(cudaMalloc(p, bytes ? bytes : 1)); return GLB_OK; }
extern "C" int glb_free(void *p) { if (p) CU(cudaFree(p)); return GLB_OK; }
extern "C" int glb_memset(void *p, int v, size_t bytes, void *s) {
  CU(cudaMemsetAsync(p, v, bytes, (cudaStream_t) s));
  return GLB_OK;
}
extern "C" int glb_host_alloc(void **p, size_t bytes) { CU(cudaMallocHost(p, bytes ? bytes : 1)); return GLB_OK; }
extern "C" int glb_host_free(void *p) { if (p) CU(cudaFreeHost(p)); return GLB_OK; }
static int copy_(void *d, const void *s, size_t n, cudaMemcpyKind k, void *stream) {
  if (n == 0) return GLB_OK;
  if (stream) CU(cudaMemcpyAsync(d, s, n, k, (cudaStream_t) stream));
  else CU(cudaMemcpy(d, s, n, k));
  return GLB_OK;
}
extern "C" int glb_memcpy_h2d(void *d, const void *s, size_t n, void *st) { return copy_(d, s, n, cudaMemcpyHostToDevice, st); }
extern "C" int glb_memcpy_d2h(void *d, const void *s, size_t n, void *st) { return copy_(d, s, n, cudaMemcpyDeviceToHost, st); }
extern "C" int glb_memcpy_d2d(void *d, const void *s, size_t n, void *st) { return copy_(d, s, n, cudaMemcpyDeviceToDevice, st); }
extern "C" int glb_stream_create(void **s) {
  cudaStream_t st;
  CU(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  *s = st;
  return GLB_OK;
}
extern "C" int glb_stream_destroy(void *s) { if (s) CU(cudaStreamDestroy((cudaStream_t) s)); return GLB_OK; }
extern "C" int glb_stream_sync(void *s) { CU(cudaStreamSynchronize((cudaStream_t) s)); return GLB_OK; }
extern "C" int glb_stream_wait_event(void *s, void *e) { CU(cudaStreamWaitEvent((cudaStream_t) s, (cudaEvent_t) e, 0)); return GLB_OK; }
extern "C" int glb_device_sync(void) { CU(cudaDeviceSynchronize()); return GLB_OK; }
extern "C" int glb_event_create(void **e) { cudaEvent_t ev; CU(cudaEventCreate(&ev)); *e = ev; return GLB_OK; }
extern "C" int glb_event_destroy(void *e) { if (e) CU(cudaEventDestroy((cudaEvent_t) e)); return GLB_OK; }
extern "C" int glb_event_record(void *e, void *s) { CU(cudaEventRecord((cudaEvent_t) e, (cudaStream_t) s)); return GLB_OK; }
extern "C" int glb_event_sync(void *e) { CU(cudaEventSynchronize((cudaEvent_t) e)); return GLB_OK; }
extern "C" int glb_event_elapsed_ms(void *a, void *b, float *ms) {
  CU(cudaEventElapsedTime(ms, (cudaEvent_t) a, (cudaEvent_t) b));
  return GLB_OK;
}

// ------------------------------------------------------------------------- tables
struct GramTables {
  int n;
  float2 *tw;
  float2 *vtab;
  float2 *roots;     // exp(-2 pi i k / M), k < M (warp-per-frame kernel)
};

template <int M> static std::vector<float2> tw_for() { return build_twiddles<M>(); }

static bool host_twiddles(int m, std::vector<float2> &tw) {
  switch (m) {
    case 16: tw = tw_for<16>(); return true;
    case 32: tw = tw_for<32>(); return true;
    case 64: tw = tw_for<64>(); return true;
    case 128: tw = tw_for<128>(); return true;
    case 256: tw = tw_for<256>(); return true;
    case 512: tw = tw_for<512>(); return true;
    case 1024: tw = tw_for<1024>(); return true;
    case 2048: tw = tw_for<2048>(); return true;
    case 4096: tw = tw_for<4096>(); return true;
    case 8192: tw = tw_for<8192>(); return true;
    case 16384: tw = tw_for<16384>(); return true;
    default: return false;
  }
}

extern "C" int glb_fft_supported(int n) {
  return n >= 32 && n <= 32768 && (n & (n - 1)) == 0;
}

extern "C" int glb_tables_create(int n, void **out) {
  if (!glb_fft_supported(n)) {
    snprintf(g_err, sizeof g_err, "FFT size %d unsupported (power of two, 32..32768)", n);
    return GLB_EINVAL;
  }
  std::vector<float2> tw;
  host_twiddles(n / 2, tw);
  std::vector<float2> vt = build_vtab(n / 2);
  GramTables *t = new GramTables();
  t->n = n;
  t->tw = nullptr;
  t->vtab = nullptr;
  t->roots = nullptr;
  std::vector<float2> rt = build_roots(n / 2);
  CU(cudaMalloc(&t->roots, rt.size() * sizeof(float2)));
  CU(cudaMemcpy(t->roots, rt.data(), rt.size() * sizeof(float2), cudaMemcpyHostToDevice));
  CU(cudaMalloc(&t->tw, tw.size() * sizeof(float2)));
  CU(cudaMalloc(&t->vtab, vt.size() * sizeof(float2)));
  CU(cudaMemcpy(t->tw, tw.data(), tw.size() * sizeof(float2), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(t->vtab, vt.data(), vt.size() * sizeof(float2), cudaMemcpyHostToDevice));
  *out = t;
  return GLB_OK;
}

// the tables of a launch made outside this unit (iq.cu)
int glb_tables_get(const void *tp, int *n, const float2 **tw, const float2 **vtab) {
  const GramTables *t = (const GramTables *) tp;
  if (!t) return GLB_EINVAL;
  *n = t->n;
  *tw = t->tw;
  *vtab = t->vtab;
  return GLB_OK;
}

extern "C" int glb_tables_destroy(void *tp) {
  GramTables *t = (GramTables *) tp;
  if (!t) return GLB_OK;
  cudaFree(t->tw);
  cudaFree(t->vtab);
  cudaFree(t->roots);
  delete t;
  return GLB_OK;
}

// ------------------------------------------------------------------------- display tables
extern "C" int glb_level_tables_create(const float *thr_f, const double *thr_d, int count, void **out) {
  if (!thr_f || !thr_d || count != kDbN) {
    glb_set_error("glb_level_tables_create: expected GLB_DB_NTHR thresholds");
    return GLB_EINVAL;
  }
  LevelTables *t = new LevelTables();
  t->thr_f = nullptr;
  t->thr_d = nullptr;
  CU(cudaMalloc(&t->thr_f, sizeof(float) * count));
  CU(cudaMalloc(&t->thr_d, sizeof(double) * count));
  CU(cudaMemcpy(t->thr_f, thr_f, sizeof(float) * count, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(t->thr_d, thr_d, sizeof(double) * count, cudaMemcpyHostToDevice));
  *out = t;
  return GLB_OK;
}

extern "C" int glb_level_tables_destroy(void *tp) {
  LevelTables *t = (LevelTables *) tp;
  if (!t) return GLB_OK;
  cudaFree(t->thr_f);
  cudaFree(t->thr_d);
  delete t;
  return GLB_OK;
}

extern "C" int glb_gram_fused_mean_ok(int n, int hop) {
  if (!glb_fft_supported(n) || hop < 1 || hop > n) return 0;
  const int unit = n / 16;            // 2T
  if ((n - hop) % hop != 0) return 0;
  for (int s = 0; s <= 4; s++)
    if (hop == (unit << s)) return 1;
  return 0;
}

extern "C" int glb_gram_fused_avg_ok(int n, int hop, int depth, int band) {
  if (n != 4096 && n != 8192) return 0;
  if (!glb_gram_fused_mean_ok(n, hop) || (hop % 4) != 0) return 0;
  if (depth < 1 || band < 2 || (long long) depth * band * 4 > 2048) return 0;
  return g_force_generic == 0 && (g_kernel_pref == 0 || g_kernel_pref == 2);
}

extern "C" int glb_launch_gram(const glb_gram_args *a, void *stream) {
  if (!a || !a->tables || !glb_fft_supported(a->n) || a->hop < 1 || a->hop > a->n || a->ntapers < 1) {
    glb_set_error("glb_launch_gram: invalid arguments");
    return GLB_EINVAL;
  }
  if (a->nframes <= 0) return GLB_OK;
  const GramTables *tb = (const GramTables *) a->tables;
  if (tb->n != a->n) {
    glb_set_error("glb_launch_gram: tables were built for another FFT size");
    return GLB_EINVAL;
  }
  KParams k;
  memset(&k, 0, sizeof k);
  k.samples = a->samples;
  k.origin = a->origin;
  k.count = a->count;
  k.tapers = a->tapers;
  k.ntapers = a->ntapers;
  k.taper_sym = a->ntapers == 1 && a->taper_symmetric;
  k.means = a->block_means;
  k.means_first_block = a->means_first_block;
  k.fused_mean = a->fused_mean;
  k.hop = a->hop;
  k.n_ov = a->n - a->hop;
  k.cblk = (k.n_ov + a->hop - 1) / a->hop;
  k.inv_hop = (float) (1.0 / (double) a->hop);
  k.inv_hop_mean = (float) (1.0 / (double) a->hop);
  k.ra9mb_a = a->ra9mb_a;
  k.limiter = a->limiter;
  k.zero_hist = a->zero_history;
  k.lim_scale = (float) pow((double) a->taper_scale, 0.9);
  k.spec_scale = (float) (1.0 / (2.0 * (double) a->taper_scale));
  k.first_frame = a->first_frame;
  k.nframes = a->nframes;
  k.rows = a->rows;
  k.row_stride = a->row_stride;
  k.rows_db = a->rows_db;
  k.spectrum = (float2 *) a->spectrum;
  k.tw = tb->tw;
  k.vtab = tb->vtab;
  k.roots = tb->roots;
  if (a->levels) {
    if (!a->level_tables) {
      glb_set_error("glb_launch_gram: levels output needs level_tables");
      return GLB_EINVAL;
    }
    if (a->spectrum) {
      glb_set_error("glb_launch_gram: levels and spectrum outputs are exclusive");
      return GLB_EINVAL;
    }
    k.levels = a->levels;
    k.lev_stride = a->levels_stride;
    k.lm.thr = ((const LevelTables *) a->level_tables)->thr_f;
    k.lm.lut = a->levels_log ? a->level_lut : nullptr;
    k.lm.log_scale = a->levels_log;
    k.lm.dmin = a->level_min;
    k.lm.dmax = a->level_max;
    k.lm.thr_level = a->level_thr;
  }
  if (a->fused_avg) {
    const glb_avg_args *av = (const glb_avg_args *) a->fused_avg;
    if (!av->band_only || av->out_double || av->first_frame != a->first_frame || av->nframes != a->nframes || !av->avg_rows ||
        !glb_gram_fused_avg_ok(a->n, a->hop, av->depth, av->maxbin - av->minbin) || a->origin % 4 != 0) {
      glb_set_error("glb_launch_gram: fused averaging not available for this launch");
      return GLB_EINVAL;
    }
    k.av_on = 1;
    k.av = *av;
  }
  if (!a->rows && !a->levels && !a->spectrum) {
    glb_set_error("glb_launch_gram: no output requested");
    return GLB_EINVAL;
  }
  const bool multi = a->ntapers > 1;
  if (multi && a->spectrum) {
    glb_set_error("glb_launch_gram: spectrum output is only defined for one taper");
    return GLB_EINVAL;
  }
  if (a->fused_mean && a->block_means) {
    glb_set_error("glb_launch_gram: fused_mean and block_means are exclusive");
    return GLB_EINVAL;
  }
  cudaStream_t st = (cudaStream_t) stream;
  // kernel families this launch may use: 1 general, 2 TMA ring, 4 warp-per-frame
  // (automatic = ring then general: measured on B200 the ring kernel is the fastest family at
  // N = 4096, 0.726 ms vs 0.746 ms for warp-per-frame, whose 67 KB of straight-line code per
  // frame stalls on instruction fetch; warp-per-frame stays selectable for experiments)
  int allow = 3;                                  // 1 general, 2 ring, 4 warp-per-frame, 8 pair
  if (g_force_generic || g_kernel_pref == 1 || a->zero_history || a->general_only) allow = 1;     // zeroed history: general kernel only
  else if (g_kernel_pref == 3) allow = 7;
  else if (g_kernel_pref == 4) allow = 11;
  const int m = a->n / 2;
  int rc = -1;
  // big frames: the 32-points-per-thread kernel (family 5) unless another family is asked for
  if ((g_kernel_pref == 0 || g_kernel_pref == 5) && !g_force_generic && !a->general_only) rc = glb_gram_big(m, k, multi, a->groups_hint, st, g_kernel_pref == 5);
  if (rc != -1) return rc;
  rc = glb_gram_part_0(m, k, multi, a->groups_hint, st, allow);
  if (rc == -1) rc = glb_gram_part_1(m, k, multi, a->groups_hint, st, allow);
  if (rc == -1) rc = glb_gram_part_2(m, k, multi, a->groups_hint, st, allow);
  if (rc == -1) rc = glb_gram_part_3(m, k, multi, a->groups_hint, st, allow);
  if (rc != -1) return rc;
  return GLB_EINVAL;
}

// ------------------------------------------------------------------------- block means
// One warp per hop block; lanes stride the block, float partial sums, shuffle tree.
__global__ void block_means_kernel(const float *__restrict__ samples, long long origin, long long count,
                                   int hop, long long first_block, long long nblocks, float *__restrict__ means) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long) gridDim.x * blockDim.x) >> 5;
  for (long long b = warp; b < nblocks; b += nwarps) {
    const long long base = (first_block + b) * hop - origin;
    float s = 0.f;
    for (int i = lane; i < hop; i += 32) {
      const long long r = base + i;
      s += (r >= 0 && r < count) ? __ldg(samples + r) : 0.f;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) means[b] = s / (float) hop;
  }
}

extern "C" int glb_launch_block_means(const float *samples, long long origin, long long count, int hop,
                                      long long first_block, long long nblocks, float *means, void *stream) {
  if (nblocks <= 0) return GLB_OK;
  if (hop < 1) { glb_set_error("block_means: hop < 1"); return GLB_EINVAL; }
  const int threads = 256;
  long long ctas = (nblocks * 32 + threads - 1) / threads;
  if (ctas > 148 * 16) ctas = 148 * 16;
  block_means_kernel<<<(int) ctas, threads, 0, (cudaStream_t) stream>>>(samples, origin, count, hop, first_block, nblocks, means);
  CU(cudaGetLastError());
  g_launches++;
  return GLB_OK;
}

// ------------------------------------------------------------------------- PCM ingest
__global__ void pcm16_to_float_kernel(const short *__restrict__ in, float *__restrict__ out, long long n) {
  const long long stride = (long long) gridDim.x * blockDim.x;
  for (long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    out[i] = (float) in[i] / 32768.f;
}
__global__ void pcm8_to_float_kernel(const unsigned char *__restrict__ in, float *__restrict__ out, long long n) {
  const long long stride = (long long) gridDim.x * blockDim.x;
  for (long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
    out[i] = ((float) in[i] - 128.f) / 128.f;
}
extern "C" int glb_launch_pcm16_to_float(const short *pcm, float *out, long long count, void *stream) {
  if (count <= 0) return GLB_OK;
  long long ctas = std::min<long long>((count + 255) / 256, 148 * 32);
  pcm16_to_float_kernel<<<(int) ctas, 256, 0, (cudaStream_t) stream>>>(pcm, out, count);
  CU(cudaGetLastError());
  g_launches++;
  return GLB_OK;
}
extern "C" int glb_launch_pcm8_to_float(const unsigned char *pcm, float *out, long long count, void *stream) {
  if (count <= 0) return GLB_OK;
  long long ctas = std::min<long long>((count + 255) / 256, 148 * 32);
  pcm8_to_float_kernel<<<(int) ctas, 256, 0, (cudaStream_t) stream>>>(pcm, out, count);
  CU(cudaGetLastError());
  g_launches++;
  return GLB_OK;
}

// ------------------------------------------------------------------------- averaging
// One CTA walks a chunk of consecutive frames; threads stride the band
// [minbin, maxbin).  Per bin the window sum cum = sum of the last min(f+1, depth) PSD
// values is held in double in shared memory (the reference keeps double cum[],
// avg.c:119,123) and slid frame to frame; the chunk's first frame sums its window
// directly from the rows, so chunks are independent.
struct AvgRed {
  double mx; int arg; double sum; double mn;
};

template <typename OutT>
__global__ void __launch_bounds__(256) avg_kernel(const glb_avg_args a, int chunk) {
  extern __shared__ double cum[];                    // band doubles
  __shared__ double s_mx[8], s_sum[8], s_mn[8], s_var[8];
  __shared__ int s_arg[8], s_cnt[8];
  __shared__ double b_mx, b_sum, b_mn, b_var;
  __shared__ int b_arg, b_cnt;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int band = a.maxbin - a.minbin;
  const long long c0 = (long long) blockIdx.x * chunk;
  const long long c1 = (c0 + chunk < a.nframes) ? c0 + chunk : a.nframes;
  OutT *out_base = (OutT *) a.avg_rows;
  auto psd_row = [&](long long g2) -> const float * {
    const long long r = a.psd_ring_rows > 0 ? g2 % a.psd_ring_rows : g2 - a.psd_first_frame;
    return a.psd + r * a.psd_stride;
  };
  int carried = a.peakbin_init;
  bool carry_known = (blockIdx.x == 0);

  for (long long fl = c0; fl < c1; ++fl) {
    const long long f = a.first_frame + fl;          // frames since alloc_avg
    const float *row = psd_row(f);
    const long long eff = (f + 1 < a.depth) ? f + 1 : a.depth;   // effdepth after this update
    double mx = -1.0, sum = 0.0, mn = 1.0;
    int arg = -1;
    for (int i = tid; i < band; i += 256) {
      const int b = a.minbin + i;
      double c;
      if (fl == c0) {
        c = 0.0;
        for (long long g2 = f - eff + 1; g2 <= f; ++g2) c += (double) psd_row(g2)[b];
      } else {
        c = cum[i] + (double) row[b];
        if (f - a.depth >= 0) c -= (double) psd_row(f - a.depth)[b];
      }
      cum[i] = c;
      if (arg < 0 || c > mx) { mx = c; arg = b; }     // first maximum within this thread's bins
      sum += c;
      if (c < mn) mn = c;
    }
    // block reduction: max with the lowest bin on ties, sum, min
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double omx = __shfl_xor_sync(0xffffffffu, mx, o);
      const int oarg = __shfl_xor_sync(0xffffffffu, arg, o);
      if (oarg >= 0 && (arg < 0 || omx > mx || (omx == mx && oarg < arg))) { mx = omx; arg = oarg; }
      sum += __shfl_xor_sync(0xffffffffu, sum, o);
      const double omn = __shfl_xor_sync(0xffffffffu, mn, o);
      if (omn < mn) mn = omn;
    }
    if (lane == 0) { s_mx[wid] = mx; s_arg[wid] = arg; s_sum[wid] = sum; s_mn[wid] = mn; }
    __syncthreads();
    if (tid == 0) {
      double m = s_mx[0], sm = s_sum[0], mi = s_mn[0];
      int ar = s_arg[0];
      for (int w = 1; w < 8; w++) {
        if (s_arg[w] >= 0 && (ar < 0 || s_mx[w] > m || (s_mx[w] == m && s_arg[w] < ar))) { m = s_mx[w]; ar = s_arg[w]; }
        sm += s_sum[w];
        if (s_mn[w] < mi) mi = s_mn[w];
      }
      // `double max = psd[minbin]; if (cum > max) { max = cum; *peakbin = index; }` avg.c:111,129-133
      const double m0 = (double) row[a.minbin];
      if (ar >= 0 && m > m0) { b_mx = m; b_arg = ar; } else { b_mx = m0; b_arg = -1; }
      b_sum = sm;
      b_mn = mi;
    }
    __syncthreads();
    const double vmax = b_mx, vsum = b_sum, vmin = b_mn;
    const int cand = b_arg;
    if (cand >= 0) { carried = cand; carry_known = true; }
    const int pk = carried;
    double avgspec = 0.0, retv = 0.0;
    if (a.mode == 2) {
      retv = (vsum - vmax) / ((double) (band - 1) * (double) (eff + 1));
    } else {
      avgspec = (vsum - vmax) / (double) (band - 1);
      retv = vmax / avgspec;
    }
    // output row
    OutT *orow = out_base + fl * a.out_stride;
    double var = 0.0;
    int cnt = 0;
    const int ob0 = a.band_only ? a.minbin : 0, ob1 = a.band_only ? (a.maxbin < a.nbins ? a.maxbin : a.nbins) : a.nbins;
    for (int b = ob0 + tid; b < ob1; b += 256) {
      double y = 1e-15;
      if (b >= a.minbin && b < a.maxbin) {
        const double c = cum[b - a.minbin];
        if (a.mode == 2) {
          y = c / (double) (eff + 1);
        } else if (a.mode == 3) {
          y = a.max0 ? (c - vmin) / (vmax - vmin) : c / avgspec;
        } else {
          if (c - avgspec > 0) {
            y = a.max0 ? (c - avgspec) / (vmax - avgspec) : c / avgspec;
            if (b != pk) { const double r = c / avgspec; var += r * r; cnt++; }
          } else {
            y = 1e-15;
          }
        }
      }
      if (sizeof(OutT) == 4 && a.rows_db) y = 10.0 * log10(y);
      orow[b - ob0] = (OutT) y;
    }
    if (a.mode == 1) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        var += __shfl_xor_sync(0xffffffffu, var, o);
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
      }
      if (lane == 0) { s_var[wid] = var; s_cnt[wid] = cnt; }
      __syncthreads();
      if (tid == 0) {
        double v = 0; int c = 0;
        for (int w = 0; w < 8; w++) { v += s_var[w]; c += s_cnt[w]; }
        b_var = v; b_cnt = c;
      }
      __syncthreads();
    }
    if (tid == 0) {
      if (a.ret) a.ret[fl] = retv;
      if (a.peak_cand) a.peak_cand[fl] = cand;
      if (a.variance) a.variance[fl] = (a.mode == 1) ? b_var / (double) b_cnt : 0.0;
      if (a.mode == 1 && !carry_known && a.unresolved) atomicAdd(a.unresolved, 1);
    }
    __syncthreads();
  }
}

// Direct form for small depths: one warp per frame, no block barrier, no state carried
// between frames.  The window sum of every band bin is re-read from the PSD rows (depth loads
// per bin: consecutive frames share depth-1 of them).  Frames are fully independent, so the grid
// is sized by the frame count.  The per-frame arithmetic lives in avg_frame.cuh, shared with the ring
// kernel's fused averaging.
template <typename OutT>
__global__ void __launch_bounds__(256) avg_direct_kernel(const glb_avg_args a) {
  const int lane = threadIdx.x & 31;
  const long long warp = ((long long) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const long long nwarps = ((long long) gridDim.x * blockDim.x) >> 5;
  auto psd_at = [&](long long g2, int b) -> float {
    const long long r = a.psd_ring_rows > 0 ? g2 % a.psd_ring_rows : g2 - a.psd_first_frame;
    return a.psd[r * a.psd_stride + b];
  };
  // a warp takes a contiguous run of frames: consecutive frames share depth - 1 of their rows
  const long long per = (a.nframes + nwarps - 1) / nwarps;
  const long long fl_end = ((warp + 1) * per < a.nframes) ? (warp + 1) * per : a.nframes;
  for (long long fl = warp * per; fl < fl_end; ++fl) avg_frame_warp<OutT>(a, fl, lane, psd_at);
}

extern "C" int glb_launch_avg(const glb_avg_args *a, void *stream) {
  if (!a || a->mode < 1 || a->mode > 3 || a->depth < 1 || a->minbin < 0 || a->maxbin < a->minbin) {
    glb_set_error("glb_launch_avg: invalid arguments");
    return GLB_EINVAL;
  }
  if (a->nframes <= 0) return GLB_OK;
  const int band = a->maxbin - a->minbin;
  const size_t smem = (size_t) (band > 0 ? band : 1) * sizeof(double);
  if (smem > 200 * 1024) { glb_set_error("glb_launch_avg: band too wide"); return GLB_EINVAL; }
  cudaStream_t st = (cudaStream_t) stream;
  if (!a->sequential && a->depth <= 32) {
    // runs of ~8 frames per warp
    long long ctas = (a->nframes * 4 + 255) / 256;
    if (ctas > 148 * 64) ctas = 148 * 64;
    if (ctas < 1) ctas = 1;
    if (a->out_double) avg_direct_kernel<double><<<(int) ctas, 256, 0, st>>>(*a);
    else avg_direct_kernel<float><<<(int) ctas, 256, 0, st>>>(*a);
    CU(cudaGetLastError());
    g_launches++;
    return GLB_OK;
  }
  int chunk;
  if (a->sequential) {
    chunk = (int) std::min<long long>(a->nframes, 0x7fffffff);
  } else {
    // amortise the direct window sum of a chunk's first frame over >= 8*depth frames
    long long want = std::max<long long>(8LL * a->depth, 16);
    long long by_grid = (a->nframes + 148 * 8 - 1) / (148 * 8);
    chunk = (int) std::max(want, by_grid);
  }
  long long ctas = (a->nframes + chunk - 1) / chunk;
  if (a->out_double) {
    CU(cudaFuncSetAttribute(avg_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
    avg_kernel<double><<<(int) ctas, 256, smem, st>>>(*a, chunk);
  } else {
    CU(cudaFuncSetAttribute(avg_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
    avg_kernel<float><<<(int) ctas, 256, smem, st>>>(*a, chunk);
  }
  CU(cudaGetLastError());
  g_launches++;
  return GLB_OK;
}

// carried peak bin (avg.c:129-133): out[f] = the last written candidate at or before frame f, the
// caller's initial value before the first one.  A "rightmost valid" scan: every CTA owns a chunk
// of frames, finds its carry-in by looking back from the chunk start (coalesced tiles, normally
// one: a candidate is written on almost every frame), then scans its chunk tile by tile with
// warp shuffles.  (The first version walked strided chunks from one CTA: 173 us per 168 750
// frames, 13 % of the C2 step.)
constexpr int kPcThreads = 256;
__device__ __forceinline__ int pc_block_rightmost(int x, int *wtot) {
  // inclusive rightmost-valid scan over the 256 threads of the CTA; returns the scanned value
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int o = __shfl_up_sync(0xffffffffu, x, d);
    if (lane >= d && x < 0) x = o;
  }
  if (lane == 31) wtot[warp] = x;
  __syncthreads();
  int wc = -1;
  for (int k = 0; k < warp; k++)
    if (wtot[k] >= 0) wc = wtot[k];
  if (x < 0) x = wc;
  return x;
}

__global__ void __launch_bounds__(kPcThreads) peak_carry_kernel(const int *__restrict__ cand, int *__restrict__ out,
                                                                long long n, long long per, int init) {
  __shared__ int wtot[kPcThreads / 32];
  __shared__ int s_carry;
  const int tid = threadIdx.x;
  const long long b = (long long) blockIdx.x * per;
  const long long e = (b + per < n) ? b + per : n;
  if (b >= n) return;
  // carry-in: rightmost valid candidate before the chunk
  int carry = init;
  for (long long hi = b; hi > 0; hi -= kPcThreads) {
    // tile [hi - 256, hi) read in ascending order so that the scan's last thread holds the answer
    const long long i = hi - kPcThreads + tid;
    int x = (i >= 0) ? cand[i] : -1;
    x = pc_block_rightmost(x, wtot);
    if (tid == kPcThreads - 1) s_carry = x;
    __syncthreads();
    const int found = s_carry;
    __syncthreads();
    if (found >= 0) {
      carry = found;
      break;
    }
  }
  for (long long tile = b; tile < e; tile += kPcThreads) {
    const long long i = tile + tid;
    int x = (i < e) ? cand[i] : -1;
    x = pc_block_rightmost(x, wtot);
    if (x < 0) x = carry;
    if (i < e) out[i] = x;
    if (tid == kPcThreads - 1) s_carry = x;
    __syncthreads();
    carry = s_carry;
    __syncthreads();
  }
}

extern "C" int glb_launch_peak_carry(const int *cand, int *peakbin, long long nframes, int init, void *stream) {
  if (nframes <= 0) return GLB_OK;
  // chunks of whole tiles, about four CTAs per SM
  long long per = (nframes + 148 * 4 - 1) / (148 * 4);
  per = ((per + kPcThreads - 1) / kPcThreads) * kPcThreads;
  const long long ctas = (nframes + per - 1) / per;
  peak_carry_kernel<<<(unsigned) ctas, kPcThreads, 0, (cudaStream_t) stream>>>(cand, peakbin, nframes, per, init);
  CU(cudaGetLastError());
  g_launches++;
  return GLB_OK;
}

// ------------------------------------------------------------------------- LMP statistic
// lmp_do, lmp.c:131-160: one thread per (frame, bin); the nl rows of the ring are read twice
// (mean, then variance) in slot order and stay in L1/L2.  Double arithmetic throughout, as the
// reference (my, sy, v_hat are doubles); IEEE sqrt and division, so inf / NaN appear exactly
// where the reference produces them (v_hat = 0).
// This general form serves the per-call ring (ring_rows > 0) and ring lengths the run kernel below is not
// instantiated for.
__global__ void __launch_bounds__(256) lmp_kernel(const float *__restrict__ psd, long long psd_first_frame, long long psd_stride,
                                                  int ring_rows, int nbins, long long first_frame, long long nframes, int nl,
                                                  double c0, double c1, int rows_db, float *__restrict__ out, long long out_stride) {
  const int bin = blockIdx.x * blockDim.x + threadIdx.x;
  if (bin >= nbins) return;
  // slot written by frame f = f mod nl, kept incrementally (one 64-bit division per thread)
  int fm = (int) ((first_frame + blockIdx.y) % nl);
  const int fstep = (int) (gridDim.y % (unsigned) nl);
  for (long long fi = blockIdx.y; fi < nframes; fi += gridDim.y) {
    const long long f = first_frame + fi;
    // row of slot j: the latest frame g <= f with g % nl == j, d = (fm - j) mod nl frames back
    const float *cur = psd + (f - psd_first_frame) * psd_stride + bin;
    auto row = [&](int j) -> float {
      if (ring_rows > 0) return psd[(long long) j * psd_stride + bin];
      int d = fm - j;
      if (d < 0) d += nl;
      return (long long) d <= f ? cur[-(long long) d * psd_stride] : 0.f;      // g = f - d < 0: never written
    };
    double my = 0.0, sy = 0.0;
    for (int j = 0; j < nl; j++) my += (double) row(j);
    my /= nl;
    for (int j = 0; j < nl; j++) {
      const double d = (double) row(j) - my;
      sy = __dadd_rn(sy, __dmul_rn(d, d));             // (no FMA contraction: the reference's doubles)
    }
    sy /= (nl - 1);
    double v = __dsub_rn(__dmul_rn(my, my), sy);
    if (v < 0.0) v = 0.0;
    v = 0.5 * (my - sqrt(v));
    float o = (float) (c0 + (nl * my) / (c1 * v));
    if ((double) o <= 1.0e-3) o = 1e-3f;
    if (bin == 0) o = 1e-3f;
    if (rows_db) o = 10.f * log10f(o);
    out[fi * out_stride + bin] = o;
    fm += fstep;
    if (fm >= nl) fm -= nl;
  }
}

// The batch form: one thread walks ONE bin through a run of consecutive frames with the ring in registers, in
// slot order (runs start at multiples of NL, so the slot of every frame of the unrolled body is a compile-time
// index).  A PSD value is loaded once per run instead of 2 nl times per frame, the frame index arithmetic is
// paid once per run, and the divisions by the constants nl and nl - 1 take three operations (Markstein,
// avg_frame.cuh: correctly rounded, the same bits as IEEE division).  Every product and sum is a separate
// IEEE operation (no FMA contraction): the doubles are those of the reference built for baseline x86-64.
// ncu on the general kernel above (profiles/r02_ncu_lmp_*): issue-bound, 416 instructions per (frame, bin) warp,
// 28 % of the samples in the per-thread prologue.
template <int NL>
__global__ void __launch_bounds__(256) lmp_run_kernel(const float *__restrict__ psd, long long psd_first_frame, long long psd_stride,
                                                      int nbins, long long first_frame, long long nframes, long long run0,
                                                      int run_len, long long nruns, double c0, double c1, int rows_db,
                                                      float *__restrict__ out, long long out_stride) {
  const long long w = (long long) blockIdx.x * blockDim.x + threadIdx.x;
  if (w >= nruns * nbins) return;
  const long long run = w / nbins;
  const int bin = (int) (w - run * nbins);
  const long long fa = run0 + run * run_len;                 // a multiple of NL: frame fa + u lives in slot u
  const long long fend = first_frame + nframes;
  const long long fb = (fa + run_len < fend) ? fa + run_len : fend;
  const float *col = psd + bin;
  auto load = [&](long long g) -> double {                   // frames before the stream start were never written: 0
    return (g >= 0 && g >= psd_first_frame) ? (double) __ldg(col + (g - psd_first_frame) * psd_stride) : 0.0;
  };
  constexpr double rn = 1.0 / NL, rn1 = 1.0 / (NL - 1);
  constexpr bool pow2 = (NL & (NL - 1)) == 0, pow2m1 = ((NL - 1) & (NL - 2)) == 0;
  double ring[NL];
  ring[0] = 0.0;
#pragma unroll
  for (int j = 1; j < NL; j++) ring[j] = load(fa - NL + j);
  for (long long base = fa; base < fb; base += NL) {
    double nxt[NL];
#pragma unroll
    for (int u = 0; u < NL; u++) nxt[u] = (base + u < fb) ? load(base + u) : 0.0;
#pragma unroll
    for (int u = 0; u < NL; u++) {
      const long long f = base + u;
      if (f >= fb) break;
      ring[u] = nxt[u];
      if (f < first_frame) continue;
      double my = 0.0;
#pragma unroll
      for (int j = 0; j < NL; j++) my = __dadd_rn(my, ring[j]);
      my = pow2 ? __dmul_rn(my, rn) : avg_div_small(my, (double) NL, rn);
      double sy = 0.0;
#pragma unroll
      for (int j = 0; j < NL; j++) {
        const double d = __dsub_rn(ring[j], my);
        sy = __dadd_rn(sy, __dmul_rn(d, d));
      }
      sy = pow2m1 ? __dmul_rn(sy, rn1) : avg_div_small(sy, (double) (NL - 1), rn1);
      double v = __dsub_rn(__dmul_rn(my, my), sy);
      if (v < 0.0) v = 0.0;
      v = __dmul_rn(0.5, __dsub_rn(my, __dsqrt_rn(v)));
      float o = (float) __dadd_rn(c0, __ddiv_rn(__dmul_rn((double) NL, my), __dmul_rn(c1, v)));
      if ((double) o <= 1.0e-3) o = 1e-3f;
      if (bin == 0) o = 1e-3f;
      if (rows_db) o = 10.f * log10f(o);
      GLB_CHECK(f - first_frame >= 0 && f - first_frame < nframes && bin < nbins);
      out[(f - first_frame) * out_stride + bin] = o;
    }
  }
}

template <int NL>
static void launch_lmp_run(const float *psd, long long psd_first_frame, long long psd_stride, int nbins, long long first_frame,
                           long long nframes, double c0, double c1, int rows_db, float *out, long long out_stride, cudaStream_t st) {
  const int run_len = NL * 8;
  const long long run0 = (first_frame / NL) * NL;
  const long long nruns = (first_frame + nframes - run0 + run_len - 1) / run_len;
  const long long ctas = (nruns * nbins + 255) / 256;
  lmp_run_kernel<NL><<<(unsigned) ctas, 256, 0, st>>>(psd, psd_first_frame, psd_stride, nbins, first_frame, nframes, run0, run_len,
                                                      nruns, c0, c1, rows_db, out, out_stride);
}

extern "C" int glb_launch_lmp(const float *psd, long long psd_first_frame, long long psd_stride, int psd_ring_rows, int nbins,
                              long long first_frame, long long nframes, int nl, int rows_db, float *out, long long out_stride,
                              void *stream) {
  if (nframes <= 0) return GLB_OK;
  if (!psd || !out || nl < 2 || nbins < 1 || first_frame < 0) {
    glb_set_error("glb_launch_lmp: invalid arguments (nl >= 2)");
    return GLB_EINVAL;
  }
  // the two constants of lmp.c:154, in double on the host (IEEE sqrt: the same bits as on the device)
  const double c0 = -sqrt((double) nl / 2.0), c1 = 2.0 * sqrt(2.0 * (double) nl);
  if (psd_ring_rows <= 0 && nl <= 8) {
    cudaStream_t st = (cudaStream_t) stream;
    switch (nl) {
      case 2: launch_lmp_run<2>(psd, psd_first_frame, psd_stride, nbins, first_frame, nframes, c0, c1, rows_db, out, out_stride, st); break;
      case 3: launch_lmp_run<3>(psd, psd_first_frame, psd_stride, nbins, first_frame, nframes, c0, c1, rows_db, out, out_stride, st); break;
      case 4: launch_lmp_run<4>(psd, psd_first_frame, psd_stride, nbins, first_frame, nframes, c0, c1, rows_db, out, out_stride, st); break;
      case 5: launch_lmp_run<5>(psd, psd_first_frame, psd_stride, nbins, first_frame, nframes, c0, c1, rows_db, out, out_stride, st); break;
      case 6: launch_lmp_run<6>(psd, psd_first_frame, psd_stride, nbins, first_frame, nframes, c0, c1, rows_db, out, out_stride, st); break;
      case 7: launch_lmp_run<7>(psd, psd_first_frame, psd_stride, nbins, first_frame, nframes, c0, c1, rows_db, out, out_stride, st); break;
      default: launch_lmp_run<8>(psd, psd_first_frame, psd_stride, nbins, first_frame, nframes, c0, c1, rows_db, out, out_stride, st); break;
    }
    CU(cudaGetLastError());
    g_launches++;
    return GLB_OK;
  }
  const int xb = (nbins + 255) / 256;
  // one frame per CTA row (neighbouring frames run together and share the ring rows in L1/L2;
  // a small persistent grid measured slower: 2.9 vs 2.4 ms per 84 375 rows)
  dim3 grid(xb, (unsigned) std::min<long long>(nframes, 32768));
  lmp_kernel<<<grid, 256, 0, (cudaStream_t) stream>>>(psd, psd_first_frame, psd_stride, psd_ring_rows, nbins, first_frame, nframes, nl,
                                                      c0, c1, rows_db, out, out_stride);
  CU(cudaGetLastError());
  g_launches++;
  return GLB_OK;
}

// ------------------------------------------------------------------------- harmonic F-test
// mtm.c:204-233 per (frame, bin): den accumulates |y_j - mu U0_j|^2 over the tapers in the reference's float
// buffer (`ftest[i] += ...`: double terms, one rounding to float per taper), then
// ftest = kmax |mu|^2 sum_U0_sqr / den in double, stored to float.  DC: real parts only (:205-206,223-224);
// even n: the Nyquist denominator is never accumulated (the loops stop at (n+1)/2) and its numerator is
// mu[n/2]^2 + mu[n - n/2]^2 = twice the (real) Nyquist value squared (:229-233).
__global__ void __launch_bounds__(256) ftest_kernel(const float2 *__restrict__ spec, long long nframes, int nbins, int n,
                                                    int ntapers, const double *__restrict__ u0, double sum_u0_sqr,
                                                    float *__restrict__ out, long long stride) {
  const long long plane = nframes * (long long) nbins;
  const long long total = plane;
  const int half = (n + 1) / 2;
  for (long long idx = (long long) blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long) gridDim.x * blockDim.x) {
    const long long f = idx / nbins;
    const int i = (int) (idx - f * nbins);
    const float2 m = spec[idx];
    const double mr = (double) m.x, mi = (i == 0) ? 0.0 : (double) m.y;
    float den = 0.f;
    double num;
    if (i < half) {
      for (int j = 0; j < ntapers; j++) {
        const float2 y = spec[(long long) (1 + j) * plane + idx];
        const double tr = (double) y.x - mr * u0[j];
        const double ti = (i == 0) ? 0.0 : (double) y.y - mi * u0[j];
        den = (float) ((double) den + (__dmul_rn(tr, tr) + __dmul_rn(ti, ti)));
      }
      num = (double) (ntapers - 1) * (__dmul_rn(mr, mr) + __dmul_rn(mi, mi)) * sum_u0_sqr;
    } else {
      num = (double) (ntapers - 1) * (__dmul_rn(mr, mr) + __dmul_rn(mr, mr)) * sum_u0_sqr;
    }
    out[f * stride + i] = (float) (num / (double) den);
  }
}

extern "C" int glb_launch_ftest(const float *spec, long long nframes, int nbins, int n, int ntapers, const double *u0,
                                double sum_u0_sqr, float *ftest, long long stride, void *stream) {
  if (nframes <= 0) return GLB_OK;
  if (!spec || !u0 || !ftest || ntapers < 1) { glb_set_error("glb_launch_ftest: invalid arguments"); return GLB_EINVAL; }
  long long ctas = (nframes * nbins + 255) / 256;
  if (ctas > 148 * 32) ctas = 148 * 32;
  ftest_kernel<<<(unsigned) ctas, 256, 0, (cudaStream_t) stream>>>((const float2 *) spec, nframes, nbins, n, ntapers, u0,
                                                                  sum_u0_sqr, ftest, stride);
  CU(cudaGetLastError());
  g_launches++;
  return GLB_OK;
}

// ------------------------------------------------------------------------- half-complex PSD
// fft_psd (fft.c:203-226) for a spectrum that did not come from gram_kernel (callers that
// fill outbuf themselves).  phase = atan2(Re, Im), the reference's argument order.
__global__ void halfcomplex_psd_kernel(const float *__restrict__ hc, int n, float *__restrict__ psd,
                                       float *__restrict__ phase) {
  const int half = (n + 1) / 2;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i <= n / 2; i += gridDim.x * blockDim.x) {
    const bool edge = (i == 0) || (n % 2 == 0 && i == n / 2);
    if (!edge && i >= half) continue;
    const float re = hc[i];
    const float im = edge ? 0.f : hc[n - i];
    if (psd) psd[i] = (re * re + im * im) / (float) n;
    if (phase) phase[i] = edge ? 0.f : atan2f(re, im);
  }
}

extern "C" int glb_launch_halfcomplex_psd(const float *hc, int n, float *psd, float *phase, void *stream) {
  if (n < 1) { glb_set_error("halfcomplex_psd: n < 1"); return GLB_EINVAL; }
  const int ctas = (n / 2 + 1 + 255) / 256;
  halfcomplex_psd_kernel<<<ctas, 256, 0, (cudaStream_t) stream>>>(hc, n, psd, phase);
  CU(cudaGetLastError());
  g_launches++;
  return GLB_OK;
}

// ------------------------------------------------------------------------- floor statistics
// compute_floor (fft.c:240-294) per PSD row.  The reference sorts the whole row (qsort, descending) only to
// take its head (sig = largest bin) and to add up its tail: floor = (sum of the entries from index
// (int)(n * 0.95) on, i.e. the K = n - (int)(0.95 n) smallest bins, added in DESCENDING order into a float)
// / 0.05 / n.  One warp per row does exactly that without sorting the row: a four-pass radix select on
// the order-preserving integer image of the floats finds the K-th smallest value, the K smallest bins
// are compacted into shared memory (ties are equal values: which of them are taken does not matter),
// sorted there (bitonic, K <= 1024 entries) and summed by one lane in the reference's order, so the
// float sum rounds identically.  The first maximum (peak value and bin; (0, 0) when no bin is > 0,
// fft.c:284-291) comes from a warp reduction.  (The first version bitonic-sorted all 4096 padded
// entries of every row with a 512-thread CTA: 78 block barriers per row.)
constexpr int kFsWarps = 8;            // rows per CTA
constexpr int kFsMaxK = 1024;          // n <= 20480 bins... n = 16385 gives K = 820

__device__ __forceinline__ unsigned fs_key(float f) {
  const unsigned b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);       // ascending keys <=> ascending floats
}

__global__ void __launch_bounds__(32 * kFsWarps) floor_stats_kernel(const float *__restrict__ rows, long long stride, int nbins,
                                                                  long long nrows, float *__restrict__ stats) {
  __shared__ int s_hist[kFsWarps][256];
  __shared__ float s_cand[kFsWarps][kFsMaxK];
  __shared__ int s_cnt[kFsWarps];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int *hist = s_hist[w];
  float *cand = s_cand[w];
  const int K = nbins - (int) (nbins * 0.95);             // entries of the sorted row from index (int)(n * 0.95) on
  for (long long r = (long long) blockIdx.x * kFsWarps + w; r < nrows; r += (long long) gridDim.x * kFsWarps) {
    const float *row = rows + r * stride;
    // ---- head of the sorted row and the first maximum
    float best = 0.f, top = -INFINITY;
    int best_i = 0x7fffffff;
    for (int i = lane; i < nbins; i += 32) {
      const float v = row[i];
      if (v > best) { best = v; best_i = i; }               // a lane's bins ascend: its first maximum
      top = fmaxf(top, v);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(0xffffffffu, best, o);
      const int oi = __shfl_xor_sync(0xffffffffu, best_i, o);
      if (ob > best || (ob == best && oi < best_i)) { best = ob; best_i = oi; }
      top = fmaxf(top, __shfl_xor_sync(0xffffffffu, top, o));
    }
    // ---- radix select: key of the K-th smallest bin, most significant byte first
    unsigned prefix = 0;
    int want = K;                                           // rank (1-based, ascending) still to be located
    for (int pass = 3; pass >= 0 && K > 0; --pass) {
      for (int b = lane; b < 256; b += 32) hist[b] = 0;
      __syncwarp();
      const int sh = 8 * pass;
      const unsigned himask = (pass == 3) ? 0u : (0xffffffffu << (sh + 8));
      for (int i = lane; i < nbins; i += 32) {
        const unsigned k = fs_key(row[i]);
        if ((k & himask) == (prefix & himask)) atomicAdd(&hist[(k >> sh) & 255u], 1);
      }
      __syncwarp();
      // lane l owns digits 8 l .. 8 l + 7
      int loc[8], tot = 0;
#pragma unroll
      for (int j = 0; j < 8; j++) { loc[j] = hist[8 * lane + j]; tot += loc[j]; }
      int incl = tot;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += up;
      }
      int below = incl - tot;                               // bins in digits before this lane's
      int digit = -1, below_d = 0;
      if (below < want && want <= incl) {
#pragma unroll
        for (int j = 0; j < 8; j++) {
          if (digit < 0 && want <= below + loc[j]) { digit = 8 * lane + j; below_d = below; }
          if (digit < 0) below += loc[j];
        }
      }
      const unsigned who = __ballot_sync(0xffffffffu, digit >= 0);
      const int src = __ffs(who) - 1;
      digit = __shfl_sync(0xffffffffu, digit, src);
      below_d = __shfl_sync(0xffffffffu, below_d, src);
      prefix |= (unsigned) digit << sh;
      want -= below_d;
      __syncwarp();
    }
    // ---- the K smallest bins: every key below the threshold, and `want` of the bins equal to it
    if (lane == 0) s_cnt[w] = 0;
    __syncwarp();
    int np2 = 1;
    while (np2 < K) np2 <<= 1;
    const int n_lt = K - want;
    for (int i = lane; i < nbins && K > 0; i += 32) {
      const float v = row[i];
      if (fs_key(v) < prefix) cand[atomicAdd(&s_cnt[w], 1)] = v;
    }
    __syncwarp();
    float thr_val = 0.f;
    {
      const unsigned b = (prefix & 0x80000000u) ? (prefix & 0x7fffffffu) : ~prefix;
      thr_val = __uint_as_float(b);
    }
    for (int i = n_lt + lane; i < np2; i += 32) cand[i] = (i < K) ? thr_val : -INFINITY;   // ties, then padding
    __syncwarp();
    for (int k2 = 2; k2 <= np2; k2 <<= 1) {
      for (int j = k2 >> 1; j > 0; j >>= 1) {
        for (int i = lane; i < np2; i += 32) {
          const int l = i ^ j;
          if (l > i) {
            const float a = cand[i], b = cand[l];
            const bool desc = ((i & k2) == 0);
            if (desc ? (a < b) : (a > b)) { cand[i] = b; cand[l] = a; }
          }
        }
        __syncwarp();
      }
    }
    if (lane == 0) {
      float fsum = 0.f;
      for (int i = 0; i < K; i++) fsum += cand[i];          // `floor_pwr += tmp_buf[i]`, descending order (fft.c:271-272)
      float fl = (float) ((double) fsum / 0.05);            // `floor_pwr /= 0.05`: double division, stored to float
      fl = fl / (float) nbins;                              // `floor_pwr /= N2`
      float *o = stats + r * 4;
      o[0] = top;
      o[1] = fl;
      o[2] = (best > 0.f) ? best : 0.f;
      o[3] = (best > 0.f) ? (float) best_i : 0.f;
    }
    __syncwarp();
  }
}

// The same statistics with the row held in registers (rows of up to 32 NPL bins, K <= 128): one load per bin, then a
// bit-by-bit descent from the highest bit in which the row's keys differ, counting in registers (no shared-
// memory histogram: the first radix passes of the kernel above put a whole row into two or three counters, 32-way
// conflicts).  The descent stops as soon as at most 128 bins remain at or below the current prefix range -- for
// a noise-like row after some ten bits; those bins are compacted by ballots, sorted as above, and the last K of
// them are summed.  If all 32 bits are spent first, the bins still undecided are equal to the threshold.
// Per 4096 rows of 2049 bins: 65 us -> see profiles/ (the display path's autoscale statistics).
template <int NPL>
__global__ void __launch_bounds__(32 * kFsWarps) floor_stats_reg_kernel(const float *__restrict__ rows, long long stride,
                                                                      int nbins, long long nrows, float *__restrict__ stats) {
  constexpr int CAP = 128;
  __shared__ float s_cand[kFsWarps][CAP];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  float *cand = s_cand[w];
  const int K = nbins - (int) (nbins * 0.95);
  const unsigned full = 0xffffffffu;
  for (long long r = (long long) blockIdx.x * kFsWarps + w; r < nrows; r += (long long) gridDim.x * kFsWarps) {
    const float *row = rows + r * stride;
    unsigned key[NPL];
    float best = 0.f, top = -INFINITY;
    int best_i = 0x7fffffff;
    unsigned kmin = 0xffffffffu, kmax = 0u;
#pragma unroll
    for (int k = 0; k < NPL; k++) {
      const int i = lane + 32 * k;
      if (i < nbins) {
        const float v = __ldg(row + i);
        key[k] = fs_key(v);
        if (v > best) { best = v; best_i = i; }             // a lane's bins ascend: its first maximum
        top = fmaxf(top, v);
        kmin = min(kmin, key[k]);
        kmax = max(kmax, key[k]);
      } else {
        key[k] = 0xffffffffu;                               // padding: above every bin, never gathered
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ob = __shfl_xor_sync(full, best, o);
      const int oi = __shfl_xor_sync(full, best_i, o);
      if (ob > best || (ob == best && oi < best_i)) { best = ob; best_i = oi; }
      top = fmaxf(top, __shfl_xor_sync(full, top, o));
    }
    kmin = __reduce_min_sync(full, kmin);
    kmax = __reduce_max_sync(full, kmax);
    // keys agree above `bit`; P = the common prefix, the range [P, P + 2^(bit+1)) holds every bin
    int bit = 31 - __clz(kmin ^ kmax);                      // -1: all bins equal
    unsigned P = (bit == 31) ? 0u : ((kmin >> (bit + 1)) << (bit + 1));
    int n_lt = 0, n_in = nbins;                             // bins below P / inside the range; n_lt < K <= n_lt + n_in
    while (bit >= 0 && n_lt + n_in > CAP) {
      const unsigned half = 1u << bit;
      int c0 = 0;
#pragma unroll
      for (int k = 0; k < NPL; k++) c0 += (key[k] - P < half) ? 1 : 0;      // (bins below P wrap to huge values)
      c0 = __reduce_add_sync(full, c0);
      if (K <= n_lt + c0) {
        n_in = c0;
      } else {
        n_lt += c0;
        n_in -= c0;
        P += half;
      }
      --bit;
    }
    // candidates: with the range narrowed to <= CAP bins, every bin up to the end of the range; otherwise (all
    // bits spent: the n_in undecided bins equal P) the bins below P, then copies of the threshold up to K
    const bool ties = n_lt + n_in > CAP;
    const unsigned span1 = (bit < 0) ? 0u : (bit == 31) ? 0xffffffffu : ((2u << bit) - 1u);   // range length - 1
    const unsigned last = ties ? P - 1u : P + span1;                         // gather keys <= last (ties: n_lt > 0 => P > 0)
    const bool any = !(ties && n_lt == 0);
    int c = 0;
#pragma unroll
    for (int k = 0; k < NPL; k++) {
      const bool take = any && (lane + 32 * k < nbins) && key[k] <= last;
      const unsigned m = __ballot_sync(full, take);
      if (take) {
        GLB_CHECK(c + __popc(m & ((1u << lane) - 1u)) < CAP);
        const unsigned kk = key[k];
        cand[c + __popc(m & ((1u << lane) - 1u))] = __uint_as_float((kk & 0x80000000u) ? (kk & 0x7fffffffu) : ~kk);
      }
      c += __popc(m);
    }
    if (ties) {
      const float tv = __uint_as_float((P & 0x80000000u) ? (P & 0x7fffffffu) : ~P);
      for (int i = c + lane; i < K; i += 32) cand[i] = tv;
      c = K;
    }
    for (int i = c + lane; i < CAP; i += 32) cand[i] = -INFINITY;            // padding sorts behind the candidates
    __syncwarp();
    for (int k2 = 2; k2 <= CAP; k2 <<= 1) {
      for (int j = k2 >> 1; j > 0; j >>= 1) {
#pragma unroll
        for (int i = lane; i < CAP; i += 32) {
          const int l = i ^ j;
          if (l > i) {
            const float a = cand[i], b = cand[l];
            const bool desc = ((i & k2) == 0);
            if (desc ? (a < b) : (a > b)) { cand[i] = b; cand[l] = a; }
          }
        }
        __syncwarp();
      }
    }
    if (lane == 0) {
      float fsum = 0.f;
      GLB_CHECK(c >= K && c <= CAP);
      for (int i = c - K; i < c; i++) fsum += cand[i];      // the K smallest, descending (fft.c:271-272)
      float fl = (float) ((double) fsum / 0.05);
      fl = fl / (float) nbins;
      float *o = stats + r * 4;
      o[0] = top;
      o[1] = fl;
      o[2] = (best > 0.f) ? best : 0.f;
      o[3] = (best > 0.f) ? (float) best_i : 0.f;
    }
    __syncwarp();
  }
}

extern "C" int glb_launch_floor_stats(const float *rows, long long stride, int nbins, long long nrows, float *stats,
                                      void *stream) {
  if (nrows <= 0) return GLB_OK;
  if (nbins < 1 || nbins - (int) (nbins * 0.95) > kFsMaxK) { glb_set_error("floor_stats: row too wide"); return GLB_EINVAL; }
  long long ctas = (nrows + kFsWarps - 1) / kFsWarps;
  if (ctas > 148 * 16) ctas = 148 * 16;
  const int K = nbins - (int) (nbins * 0.95);
  if (K >= 1 && K <= 128 && nbins <= 32 * 65 && g_kernel_pref != 1) {
    cudaStream_t st = (cudaStream_t) stream;
    if (nbins <= 32 * 17) floor_stats_reg_kernel<17><<<(unsigned) ctas, 32 * kFsWarps, 0, st>>>(rows, stride, nbins, nrows, stats);
    else if (nbins <= 32 * 33) floor_stats_reg_kernel<33><<<(unsigned) ctas, 32 * kFsWarps, 0, st>>>(rows, stride, nbins, nrows, stats);
    else floor_stats_reg_kernel<65><<<(unsigned) ctas, 32 * kFsWarps, 0, st>>>(rows, stride, nbins, nrows, stats);
    CU(cudaGetLastError());
    g_launches++;
    return GLB_OK;
  }
  floor_stats_kernel<<<(unsigned) ctas, 32 * kFsWarps, 0, (cudaStream_t) stream>>>(rows, stride, nbins, nrows, stats);
  CU(cudaGetLastError());
  g_launches++;
  return GLB_OK;
}

// ------------------------------------------------------------------------- display mapping
// main_window_draw, g_main.c:1109-1229, minus the GTK drawing: AGC of the display range from
// the per-row floor statistics, then level -> 8-bit palette index (-> RGB).
//
// agc_kernel: the display range is a recurrence over frames in mixed double/float arithmetic with a
// rounding to float at every step (static float display_max_lvl, g_main.c:1080,1118-1123):
//     lvl = (float) ((1.0 - 0.99) * sig + 0.99 * lvl)
// Rounding makes it non-associative, so the chain itself is walked in order -- but only the chain: the
// maximum and the minimum level are two independent chains on two warps (per step two conversions, one
// multiply and one add on the critical path; the product with the new statistic does not depend on the
// chain and runs ahead), and the dB conversion of the range (two double log10 per frame, most of the cost
// of the first version, where one thread did everything) is done for all frames in parallel afterwards.
// The double products and the sum are kept as separate roundings (__dmul_rn / __dadd_rn: no FMA
// contraction), as the x86-64 reference build computes them.
// state[0..1] = (display_max_lvl, display_min_lvl) carried between calls; stats = floor_stats rows.
constexpr int kAgcTile = 1536;          // frames staged per tile (36 KB of static shared memory)

__global__ void __launch_bounds__(256) agc_kernel(const float *__restrict__ stats, long long nframes, long long first_frame,
                                                  float overlap, int log_scale, float *__restrict__ state,
                                                  float *__restrict__ range /* [nframes][2] */) {
  // per tile: the products (1.0 - 0.99) * stat for both chains, formed by all threads; then the two chains walk
  // the tile out of shared memory (the loads do not depend on the chain and run ahead of it); the level of
  // every frame goes back through shared memory and is written (and converted to dB) by all threads
  __shared__ double s_a[2][kAgcTile];
  __shared__ float s_lvl[2][kAgcTile];
  __shared__ float s_state[2];
  const int tid = threadIdx.x;
  if (tid < 2) s_state[tid] = state[tid];
  __syncthreads();
  for (long long base = 0; base < nframes; base += kAgcTile) {
    const int cnt = (int) ((nframes - base < kAgcTile) ? nframes - base : kAgcTile);
    for (int i = tid; i < 2 * cnt; i += blockDim.x) {
      const int f = i >> 1, chain = i & 1;
      s_a[chain][f] = __dmul_rn(1.0 - 0.99, (double) stats[4 * (base + f) + chain]);
    }
    __syncthreads();
    const int chain = tid >> 5;                        // warp 0: maximum level, warp 1: minimum level
    if (chain < 2 && (tid & 31) == 0) {
      float lvl = s_state[chain];
      int i = 0;
      if (first_frame + base == 0) {                   // glfer.first_buffer == TRUE (g_main.c:1112-1120)
        float s = stats[chain];
        if (overlap > 0.0f) s /= overlap;
        lvl = s;
        s_lvl[chain][0] = lvl;
        i = 1;
      }
#pragma unroll 8
      for (; i < cnt; i++) {                           // g_main.c:1122-1123
        lvl = (float) __dadd_rn(s_a[chain][i], __dmul_rn(0.99, (double) lvl));
        s_lvl[chain][i] = lvl;
      }
      s_state[chain] = lvl;
    }
    __syncthreads();
    for (int i = tid; i < 2 * cnt; i += blockDim.x) {
      const float l = s_lvl[i & 1][i >> 1];
      range[2 * base + i] = log_scale ? (float) (10.0 * log10((double) l)) : l;      // g_main.c:1132-1135
    }
    __syncthreads();
  }
  if (tid < 2) state[tid] = s_state[tid];
}

// levels_kernel: one thread per four consecutive pixels of the [nframes][nbins] level image (one 32-bit
// store; rows are nbins = n/2 + 1 bytes, so a group may straddle two rows).  Pixel i of a row shows bin
// n-1-i (g_main.c:1193-1201); in the log scales the level first passes through the reference's `short`
// level buffer (sig_level = levbuf[..] = 10 log10(x): integer-truncated dB, g_main.c:68,1193-1195), located
// between the host-computed thresholds (levels.cuh) so that it is the host libm's value bit for bit.
// (The first version walked a row per warp, one dependent load per iteration: 59 us per 4096 rows of 2049
// bins, latency-bound at 0.7 TB/s.)
__global__ void __launch_bounds__(256) levels_kernel(const float *__restrict__ rows, long long stride, int nbins,
                                                     long long nframes, const float *__restrict__ range, LevelMap lm,
                                                     const unsigned char *__restrict__ colortab,
                                                     unsigned char *__restrict__ levels, unsigned char *__restrict__ rgb) {
  const long long total = nframes * (long long) nbins;
  const long long p0 = 4 * ((long long) blockIdx.x * blockDim.x + threadIdx.x);
  if (p0 >= total) return;
  long long f = p0 / nbins;
  int i = (int) (p0 - f * nbins);
  const int cnt = (total - p0 < 4) ? (int) (total - p0) : 4;
  float x[4];
  float2 rg[4];
#pragma unroll
  for (int e = 0; e < 4; e++) {
    long long fe = f;
    int ie = i + e;
    while (ie >= nbins) { ie -= nbins; fe++; }
    GLB_CHECK(e >= cnt || (fe < nframes && ie >= 0));
    x[e] = (e < cnt) ? __ldg(rows + fe * stride + (nbins - 1 - ie)) : 0.f;
    rg[e] = (range && e < cnt) ? __ldg(reinterpret_cast<const float2 *>(range) + fe) : make_float2(lm.dmax, lm.dmin);
  }
  unsigned char v[4];
#pragma unroll
  for (int e = 0; e < 4; e++) {
    LevelMap m = lm;
    m.dmax = rg[e].x;                                      // per-frame display range (autoscale)
    m.dmin = rg[e].y;
    v[e] = map_level(x[e], m);
  }
  if (levels) {
    if (cnt == 4) *reinterpret_cast<uchar4 *>(levels + p0) = make_uchar4(v[0], v[1], v[2], v[3]);
    else for (int e = 0; e < cnt; e++) levels[p0 + e] = v[e];
  }
  if (rgb) {
    unsigned char px[12];
#pragma unroll
    for (int e = 0; e < 4; e++) {
      px[3 * e] = colortab[3 * v[e]];
      px[3 * e + 1] = colortab[3 * v[e] + 1];
      px[3 * e + 2] = colortab[3 * v[e] + 2];
    }
    if (cnt == 4) {
      uint32_t *o = reinterpret_cast<uint32_t *>(rgb + 3 * p0);      // 12 p0' bytes: 4-byte aligned
#pragma unroll
      for (int q = 0; q < 3; q++)
        o[q] = (uint32_t) px[4 * q] | ((uint32_t) px[4 * q + 1] << 8) | ((uint32_t) px[4 * q + 2] << 16) | ((uint32_t) px[4 * q + 3] << 24);
    } else {
      for (int e = 0; e < 3 * cnt; e++) rgb[3 * p0 + e] = px[e];
    }
  }
}

extern "C" int glb_launch_agc(const float *stats, long long nframes, long long first_frame, float overlap, int log_scale,
                              float *state, float *range, void *stream) {
  if (nframes <= 0) return GLB_OK;
  // (asking for most of an SM's shared memory, to keep the chain's CTA alone on its SM, changed nothing end to end)
  agc_kernel<<<1, 256, 0, (cudaStream_t) stream>>>(stats, nframes, first_frame, overlap, log_scale, state, range);
  CU(cudaGetLastError());
  g_launches++;
  return GLB_OK;
}

extern "C" int glb_launch_levels(const float *rows, long long stride, int nbins, long long nframes, const float *range,
                                 const float *fixed_range, int log_scale, float thr, const void *level_tables,
                                 const unsigned char *level_lut, const unsigned char *colortab, unsigned char *levels,
                                 unsigned char *rgb, void *stream) {
  if (nframes <= 0) return GLB_OK;
  if ((!range && !fixed_range) || (rgb && !colortab) || !level_tables) {
    glb_set_error("glb_launch_levels: missing range / palette / level tables");
    return GLB_EINVAL;
  }
  LevelMap lm;
  lm.thr = ((const LevelTables *) level_tables)->thr_f;
  lm.lut = (!range && log_scale) ? level_lut : nullptr;       // the look-up table is for ONE display range
  lm.log_scale = log_scale;
  lm.dmax = fixed_range ? fixed_range[0] : 0.f;
  lm.dmin = fixed_range ? fixed_range[1] : 0.f;
  lm.thr_level = thr;
  if (nbins < 1 || ((reinterpret_cast<uintptr_t>(levels) | reinterpret_cast<uintptr_t>(rgb)) & 3) ||
      (range && (reinterpret_cast<uintptr_t>(range) & 7))) {
    glb_set_error("glb_launch_levels: unaligned output or range");
    return GLB_EINVAL;
  }
  const long long ctas = ((nframes * nbins + 3) / 4 + 255) / 256;
  levels_kernel<<<(unsigned) ctas, 256, 0, (cudaStream_t) stream>>>(rows, stride, nbins, nframes, range, lm, colortab, levels, rgb);
  CU(cudaGetLastError());
  g_launches++;
  return GLB_OK;
}
