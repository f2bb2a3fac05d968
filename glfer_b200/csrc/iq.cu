// iq.cu -- two-sided spectrogram of complex (I/Q) input: rows[f][j] = |Z_f[(j + n/2) mod n]|^2 / n, Z_f the
// complex FFT of frame f's n tapered complex samples (include/glfer_b200.h, glfer_iq_*).
//
//   gram_iq_kernel<M, QSC>  the fused path for the regular geometry (complex hop h = (n/16) << s, n - h a
//                           multiple of h).  An interleaved (I, Q) frame of n complex samples is a frame of
//                           N = 2n floats of the TMA ring kernel (gram_ring_kernel, gram_common.cuh), and the
//                           ring kernel already transforms it as the M = n complex points (I, Q).  So this is
//                           the ring kernel at M = n -- same ring of hop blocks, same bulk copies, same taper
//                           multiply, same passes -- without block means and with another epilogue: instead of
//                           the real-FFT split (emit_bins_rt), |Z[k]|^2 goes straight to row position
//                           (k + n/2) mod n (iq_core.cuh).
//   everything else         the general spectrogram kernel's spectrum output on the 2n-float frames, then
//                           zoom_split_kernel (glb_launch_iq_gram_general, zoom.cu): the zoom's frame stage.
//
//   gram_iq_mtm_kernel<M, QSC>  multitaper rows on the same geometry: the frame stays in registers while each of
//                           the K' tapers runs the transform, and the powers are summed before the one row store.
//                           Multitaper launches of any other geometry take the general path once per taper.
//   gram_iq_ftest_kernel<M, QSC>  the same with Thomson's harmonic F-test: one more transform per frame (the hn
//                           taper, first), and the F row beside or instead of the multitaper row.
//
// LEV instantiations write 8-bit display levels (levels.cuh) instead of the float row: pixel n - 1 - j shows row
// position j (iq_core.cuh).  Separate instantiations, for the reason the real ring kernel has them (store_levels,
// gram_common.cuh): as a run-time branch the level mapping would cost the float-row path registers.  Launches with
// levels that the fused kernel does not serve write float rows into scratch and map them with levels_kernel.
//
// glb_launch_iq_gram picks the path from the geometry; glb_force_generic_kernel(1) forces the general one.
#include "gram_common.cuh"
#include "iq_core.cuh"

extern int g_force_generic;           // gram_kernels.cu
int glb_tables_get(const void *tables, int *n, const float2 **tw, const float2 **vtab);

// The taper carries taper_scale = 1 / (2 sqrt(2n)) as the zoom's (host/zoom.c), so |Z|^2 of the tapered frame is
// the contract's |Z|^2 / n divided by 8: the epilogue multiplies by 8, exactly.
constexpr float kIqPowerScale = 8.f;

// testing aid (glb_set_ring_groups): > 0 replaces the frame-group count of the fused launch policy, so that short runs
// put several frames into every group and reach the ring's steady state
static int g_ring_groups = 0;
static int g_last_frames_per_group = 0;
extern "C" void glb_set_ring_groups(int groups) { g_ring_groups = groups > 0 ? groups : 0; }
extern "C" int glb_last_frames_per_group(void) { return g_last_frames_per_group; }

template <int M, int QSC, bool LEV = false>
__global__ void __launch_bounds__(Geo<M>::THREADS, (RingGeo<M, false>::MINB)) gram_iq_kernel(const KParams p) {
  using GeoM = Geo<M>;
  constexpr int T = GeoM::T, G = GeoM::G;
  constexpr bool RT = RingGeo<M, false>::RT;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int g = threadIdx.x / T;
  const int t = threadIdx.x % T;
  const int qs = QSC >= 0 ? QSC : p.qs;
  const int hop = QSC >= 0 ? ((2 * T) << (QSC >= 0 ? QSC : 0)) : p.hop;   // floats: 2 complex hops
  const int nb = kPoints >> qs;
  const RingLayout L = ring_layout<M>(hop, nb);                  // the real kernel's layout (the mean slots stay unused)
  const int slots = L.slots;
  unsigned char *gbase = smem_raw + (size_t) g * L.group_bytes;
  float2 *buf = reinterpret_cast<float2 *>(gbase);
  float *ring = reinterpret_cast<float *>(gbase + L.ring_off);
  float *red = reinterpret_cast<float *>(gbase + L.red_off);
  float *mu = reinterpret_cast<float *>(gbase + L.mu_off);
  unsigned long long *mbar = reinterpret_cast<unsigned long long *>(gbase + L.mbar_off);
  const long long gid = (long long) blockIdx.x * G + g;
  const long long fb = gid * p.frames_per_group;
  const bool group_active = fb < p.nframes;
  const long long f_first = p.first_frame + fb;
  const long long b0 = f_first - (nb - 1);                       // oldest block of the first frame
  const unsigned blk_bytes = (unsigned) hop * 4u;
  unsigned phase_bits = 0;

  TwRegs tr;
  if constexpr (RT) load_tw_regs<M>(tr, t, p.tw, p.vtab);
  if (t == 0) {
    for (int sl = 0; sl < slots; sl++) mbar_init(&mbar[sl], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  const float2 *tw_mid = p.tw;
  if constexpr (!RT) {
    float2 *tws = reinterpret_cast<float2 *>(smem_raw + (size_t) G * L.group_bytes);
    constexpr int kMid = TwOffset<M, Plan<M>::NP - 1>::value;
    for (int i = threadIdx.x; i < kMid; i += GeoM::THREADS) tws[i] = p.tw[i];
    tw_mid = tws;
  }
  group_sync<M>(g);

  // prologue: the nb blocks of the first frame, zeros before the stream start
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
  for (int lb = 0; lb < nb; lb++) {
    if (group_active && b0 + lb >= 0) {
      mbar_wait(&mbar[lb], 0);
      phase_bits ^= 1u << lb;
    }
  }
  group_sync<M>(g);                                               // zero fill visible

  int slot_new = nb - 1;
  const int nact = group_active ? (int) ((p.nframes - fb < p.frames_per_group) ? p.nframes - fb : p.frames_per_group) : 0;
  float *row_ptr = p.rows + fb * p.row_stride;                   // (never dereferenced past nact)
  const float *next_src = p.samples + ((f_first + 1) * (long long) hop - p.origin);
  int ob[4];
  if constexpr (LEV) iq_pixel_bases<M>(t, ob);
  else iq_row_bases<M>(t, ob);
  unsigned char *lev_ptr = LEV ? p.levels + fb * p.lev_stride : nullptr;
  float mu_new = 0.f;
  for (int it = 0; it < p.frames_per_group; ++it, row_ptr += p.row_stride, next_src += hop) {
    const bool active = it < nact;
    const bool next_there = it + 1 < nact;
    const int slot_next = (slot_new + 1 == slots) ? 0 : slot_new + 1;
    if (it > 0 && active) {
      mbar_wait(&mbar[slot_new], (phase_bits >> slot_new) & 1u);
      phase_bits ^= 1u << slot_new;
    }
    auto request_next = [&]() {
      GLB_CHECK_SRC(p, next_src, hop);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_expect_tx(&mbar[slot_next], blk_bytes);
      tma_load_1d(ring + (size_t) slot_next * hop, next_src, blk_bytes, &mbar[slot_next]);
    };
    if (GLB_RING_EXTRA && next_there && t == 0) request_next();
    const int slot_oldest = GLB_RING_EXTRA ? ((slot_next + 1 == slots) ? 0 : slot_next + 1) : slot_next;
    float2 v[kPoints];
    {
      float2 x[kPoints];
      if constexpr (QSC >= 0) {
        ring_fetch<M, (QSC >= 0 ? QSC : 0)>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, false, false, red, 0.f, g);
      } else {
        switch (qs) {
          case 4: ring_fetch<M, 4>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, false, false, red, 0.f, g); break;
          case 3: ring_fetch<M, 3>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, false, false, red, 0.f, g); break;
          case 2: ring_fetch<M, 2>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, false, false, red, 0.f, g); break;
          case 1: ring_fetch<M, 1>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, false, false, red, 0.f, g); break;
          default: ring_fetch<M, 0>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, false, false, red, 0.f, g); break;
        }
      }
      apply_taper<M, true>(v, x, t, p, p.tapers);
    }
    if constexpr (RT) {
      pass_compute_rt<M, 0>(v, tr);
      group_sync<M>(g);                // (A) the previous transform's last pass has been read by all
      pass_scatter<M, 0>(v, t, buf);
    } else {
      group_sync<M>(g);
      pass_store<M, 0>(v, t, buf, p.tw);
    }
    // the frame is in registers: past (A) nobody reads the oldest ring slot any more
    if (!GLB_RING_EXTRA && next_there && t == 0) request_next();
    group_sync<M>(g);
    RingMidPasses<M, 1, RT>::run(v, t, buf, tw_mid, tr, g);
    float yv[17];
    yv[16] = 0.f;
    const bool w0 = t < 32;           // warp-uniform: only the warp that holds thread 0 pays for its re-ordering
    if constexpr (RT) {
      last_pass_rt<M>(v, t, buf, p.tw, tr);
    } else {
      TwRegs tl;
      load_last_regs<M>(tl, t, p.tw, p.vtab);
      last_pass_load<M>(v, t, buf);
      last_pass_compute_rt<M>(v, t, tl);
    }
    if (w0) iq_emit_power<M, true>(v, t, kIqPowerScale, yv);
    else iq_emit_power<M, false>(v, t, kIqPowerScale, yv);
    if constexpr (LEV) {
      if (active) {
#pragma unroll
        for (int slot = 0; slot < 17; slot++) {
          if (slot == 16) {
            if (t == 0) lev_ptr[M - 1] = map_level(yv[16], p.lm);
          } else if (slot != 1 || t != 0) {
            lev_ptr[iq_pixel_offset<M>(ob, slot)] = map_level(yv[slot], p.lm);
          }
        }
      }
      lev_ptr += p.lev_stride;
    } else if (active) {
      GLB_CHECK_ROW(p, row_ptr);
      GLB_CHECK_ROW(p, row_ptr + M - 1);
#pragma unroll
      for (int slot = 0; slot < 17; slot++) {
        if (slot == 16) {
          if (t == 0) st_row(row_ptr, yv[16]);
        } else if (slot != 1 || t != 0) {
          st_row(row_ptr + iq_slot_offset<M>(ob, slot), yv[slot]);
        }
      }
    }
    slot_new = slot_next;
    // no barrier here: (A) of the next transform orders these reads of `buf` before its stores
  }
}

// CTAs per SM the multitaper kernel is compiled for: RingGeo<M, true>::MINB (4 CTAs of 128 threads) where that is
// spill-free (n <= 256); one CTA less from n = 512 on, where the frame x[], the sums acc[] and the transform's
// registers no longer fit 128 registers (at 4 CTAs n = 512 ... 4096 spill 4 ... 484 bytes): 3 CTAs for n = 512 ... 2048
// (134 - 144 registers), 2 for n = 4096 (256 threads, 120 registers), 1 for n = 8192 (512 threads, 118 - 120)
template <int M> struct IqMtmGeo {
  static constexpr int MINB = M <= 256 ? RingGeo<M, true>::MINB : (M <= 2048 ? 3 : (M == 4096 ? 2 : 1));
};
// Multitaper rows: the frame loop of gram_iq_kernel with the multitaper loop of gram_ring_kernel.  The frame is
// fetched from the ring once and kept in registers (x) while each of the p.ntapers tapers ([2M] floats each at
// p.tapers) runs the multiply, the passes and the power epilogue; the powers are summed per slot in taper order
// (acc) and stored once per frame, with the stores of the periodogram's float rows.  A kernel of its own rather than
// a template flag of gram_iq_kernel, which keeps the periodogram kernels' instructions as they are.
template <int M, int QSC>
__global__ void __launch_bounds__(Geo<M>::THREADS, (IqMtmGeo<M>::MINB)) gram_iq_mtm_kernel(const KParams p) {
  using GeoM = Geo<M>;
  constexpr int T = GeoM::T, G = GeoM::G;
  constexpr bool RT = RingGeo<M, true>::RT;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int g = threadIdx.x / T;
  const int t = threadIdx.x % T;
  const int qs = QSC >= 0 ? QSC : p.qs;
  const int hop = QSC >= 0 ? ((2 * T) << (QSC >= 0 ? QSC : 0)) : p.hop;   // floats: 2 complex hops
  const int nb = kPoints >> qs;
  const RingLayout L = ring_layout<M>(hop, nb);                  // the real kernel's layout (the mean slots stay unused)
  const int slots = L.slots;
  unsigned char *gbase = smem_raw + (size_t) g * L.group_bytes;
  float2 *buf = reinterpret_cast<float2 *>(gbase);
  float *ring = reinterpret_cast<float *>(gbase + L.ring_off);
  float *red = reinterpret_cast<float *>(gbase + L.red_off);
  float *mu = reinterpret_cast<float *>(gbase + L.mu_off);
  unsigned long long *mbar = reinterpret_cast<unsigned long long *>(gbase + L.mbar_off);
  const long long gid = (long long) blockIdx.x * G + g;
  const long long fb = gid * p.frames_per_group;
  const bool group_active = fb < p.nframes;
  const long long f_first = p.first_frame + fb;
  const long long b0 = f_first - (nb - 1);                       // oldest block of the first frame
  const unsigned blk_bytes = (unsigned) hop * 4u;
  unsigned phase_bits = 0;

  TwRegs tr;
  if constexpr (RT) load_tw_regs<M>(tr, t, p.tw, p.vtab);
  if (t == 0) {
    for (int sl = 0; sl < slots; sl++) mbar_init(&mbar[sl], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  const float2 *tw_mid = p.tw;
  if constexpr (!RT) {
    float2 *tws = reinterpret_cast<float2 *>(smem_raw + (size_t) G * L.group_bytes);
    constexpr int kMid = TwOffset<M, Plan<M>::NP - 1>::value;
    for (int i = threadIdx.x; i < kMid; i += GeoM::THREADS) tws[i] = p.tw[i];
    tw_mid = tws;
  }
  group_sync<M>(g);

  // prologue: the nb blocks of the first frame, zeros before the stream start
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
  for (int lb = 0; lb < nb; lb++) {
    if (group_active && b0 + lb >= 0) {
      mbar_wait(&mbar[lb], 0);
      phase_bits ^= 1u << lb;
    }
  }
  group_sync<M>(g);                                               // zero fill visible

  int slot_new = nb - 1;
  const int nact = group_active ? (int) ((p.nframes - fb < p.frames_per_group) ? p.nframes - fb : p.frames_per_group) : 0;
  float *row_ptr = p.rows + fb * p.row_stride;                   // (never dereferenced past nact)
  const float *next_src = p.samples + ((f_first + 1) * (long long) hop - p.origin);
  int ob[4];
  iq_row_bases<M>(t, ob);
  float mu_new = 0.f;
  for (int it = 0; it < p.frames_per_group; ++it, row_ptr += p.row_stride, next_src += hop) {
    const bool active = it < nact;
    const bool next_there = it + 1 < nact;
    const int slot_next = (slot_new + 1 == slots) ? 0 : slot_new + 1;
    if (it > 0 && active) {
      mbar_wait(&mbar[slot_new], (phase_bits >> slot_new) & 1u);
      phase_bits ^= 1u << slot_new;
    }
    auto request_next = [&]() {
      GLB_CHECK_SRC(p, next_src, hop);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_expect_tx(&mbar[slot_next], blk_bytes);
      tma_load_1d(ring + (size_t) slot_next * hop, next_src, blk_bytes, &mbar[slot_next]);
    };
    if (GLB_RING_EXTRA && next_there && t == 0) request_next();
    const int slot_oldest = GLB_RING_EXTRA ? ((slot_next + 1 == slots) ? 0 : slot_next + 1) : slot_next;
    {
      float2 x[kPoints];
      if constexpr (QSC >= 0) {
        ring_fetch<M, (QSC >= 0 ? QSC : 0)>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, false, false, red, 0.f, g);
      } else {
        switch (qs) {
          case 4: ring_fetch<M, 4>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, false, false, red, 0.f, g); break;
          case 3: ring_fetch<M, 3>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, false, false, red, 0.f, g); break;
          case 2: ring_fetch<M, 2>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, false, false, red, 0.f, g); break;
          case 1: ring_fetch<M, 1>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, false, false, red, 0.f, g); break;
          default: ring_fetch<M, 0>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, false, false, red, 0.f, g); break;
        }
      }
      float acc[17];
#pragma unroll
      for (int i = 0; i < 17; i++) acc[i] = 0.f;
      for (int j = 0; j < p.ntapers; ++j) {
        float2 v[kPoints];
        apply_taper<M, true>(v, x, t, p, p.tapers + (size_t) j * GeoM::N);
        if constexpr (RT) {
          pass_compute_rt<M, 0>(v, tr);
          group_sync<M>(g);            // (A) the previous transform's last pass has been read by all
          pass_scatter<M, 0>(v, t, buf);
        } else {
          group_sync<M>(g);
          pass_store<M, 0>(v, t, buf, p.tw);
        }
        // the frame is in registers: past the first (A) nobody reads the oldest ring slot any more
        if (!GLB_RING_EXTRA && next_there && j == 0 && t == 0) request_next();
        group_sync<M>(g);
        RingMidPasses<M, 1, RT>::run(v, t, buf, tw_mid, tr, g);
        const bool w0 = t < 32;
        if constexpr (RT) {
          last_pass_rt<M>(v, t, buf, p.tw, tr);
        } else {
          TwRegs tl;
          load_last_regs<M>(tl, t, p.tw, p.vtab);
          last_pass_load<M>(v, t, buf);
          last_pass_compute_rt<M>(v, t, tl);
        }
        if (w0) iq_add_power<M, true>(v, t, kIqPowerScale, acc);
        else iq_add_power<M, false>(v, t, kIqPowerScale, acc);
      }
      if (active) {
        GLB_CHECK_ROW(p, row_ptr);
        GLB_CHECK_ROW(p, row_ptr + M - 1);
#pragma unroll
        for (int slot = 0; slot < 17; slot++) {
          if (slot == 16) {
            if (t == 0) st_row(row_ptr, acc[16]);
          } else if (slot != 1 || t != 0) {
            st_row(row_ptr + iq_slot_offset<M>(ob, slot), acc[slot]);
          }
        }
      }
    }
    slot_new = slot_next;
    // no barrier here: (A) of the next transform orders these reads of `buf` before its stores
  }
}

// The F-test's inputs: a second kernel argument, so that KParams -- and every kernel that takes it -- keeps its layout
struct IqFtestParams {
  float *ftest;               // [nframes][row_stride] F rows, or nullptr
  const float *hn;            // [2M] floats: hn[i] taper_scale on both floats of complex sample i
  const float2 *u0;           // [ntapers]: (U0_k, sqrt(lambda_k))
  float fnum;                 // (K' - 1) S
};

// CTAs per SM of the F-test kernel, and the shared memory of mu (the hn transform, 17 complex slots per thread, in a
// per-thread column).  The multitaper kernel's budget (IqMtmGeo) has no room for mu's 34 registers: kept in registers,
// mu spills 64 ... 368 bytes at every n under IqMtmGeo's bounds.  In shared memory only den (17 registers) is added, and
// n = 512 ... 8192 compile without spills at IqMtmGeo's bounds (161 - 167 registers at 3 CTAs, 123 - 124 at 2 and 1).
// n <= 256 still spill (72 - 168 bytes) at the multitaper kernel's 4 CTAs of 128 threads, so they take 3 (DESIGN §7.6).
template <int M> struct IqFtestGeo {
  static constexpr int MINB = M <= 256 ? 3 : IqMtmGeo<M>::MINB;
  static constexpr size_t MU_BYTES = (size_t) Geo<M>::THREADS * 17 * sizeof(float2);
};

// Multitaper rows and Thomson's harmonic F-test in one pass: the frame loop of gram_iq_mtm_kernel with one more
// transform per frame.  The frame is fetched from the ring once; the hn transform runs first and leaves mu per slot
// (iq_emit_mu), then each of the p.ntapers tapers runs the multiply, the passes and iq_add_ftest, which adds the power
// to acc exactly as gram_iq_mtm_kernel does (so the rows are bit-identical to it) and the residual to den.  Rows
// (p.rows) and F rows (fp.ftest) are stored once per frame, either may be absent.  A kernel of its own, as
// gram_iq_mtm_kernel is, so that the existing kernels keep their instructions.
template <int M, int QSC>
__global__ void __launch_bounds__(Geo<M>::THREADS, (IqFtestGeo<M>::MINB))
gram_iq_ftest_kernel(const KParams p, const IqFtestParams fp) {
  using GeoM = Geo<M>;
  constexpr int T = GeoM::T, G = GeoM::G;
  constexpr bool RT = RingGeo<M, true>::RT;
  constexpr int ZST = GeoM::THREADS;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int g = threadIdx.x / T;
  const int t = threadIdx.x % T;
  const int qs = QSC >= 0 ? QSC : p.qs;
  const int hop = QSC >= 0 ? ((2 * T) << (QSC >= 0 ? QSC : 0)) : p.hop;   // floats: 2 complex hops
  const int nb = kPoints >> qs;
  const RingLayout L = ring_layout<M>(hop, nb);
  const int slots = L.slots;
  unsigned char *gbase = smem_raw + (size_t) g * L.group_bytes;
  float2 *buf = reinterpret_cast<float2 *>(gbase);
  float *ring = reinterpret_cast<float *>(gbase + L.ring_off);
  float *red = reinterpret_cast<float *>(gbase + L.red_off);
  float *mu = reinterpret_cast<float *>(gbase + L.mu_off);
  unsigned long long *mbar = reinterpret_cast<unsigned long long *>(gbase + L.mbar_off);
  // mu of the hn transform, slot s of this thread at zmu_s[s * THREADS] (conflict-free: a warp reads 32 consecutive float2)
  float2 *zmu = reinterpret_cast<float2 *>(smem_raw + (size_t) G * L.group_bytes + (RT ? 0 : GeoM::TWS_BYTES)) +
                threadIdx.x;
  const long long gid = (long long) blockIdx.x * G + g;
  const long long fb = gid * p.frames_per_group;
  const bool group_active = fb < p.nframes;
  const long long f_first = p.first_frame + fb;
  const long long b0 = f_first - (nb - 1);
  const unsigned blk_bytes = (unsigned) hop * 4u;
  unsigned phase_bits = 0;

  TwRegs tr;
  if constexpr (RT) load_tw_regs<M>(tr, t, p.tw, p.vtab);
  if (t == 0) {
    for (int sl = 0; sl < slots; sl++) mbar_init(&mbar[sl], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  const float2 *tw_mid = p.tw;
  if constexpr (!RT) {
    float2 *tws = reinterpret_cast<float2 *>(smem_raw + (size_t) G * L.group_bytes);
    constexpr int kMid = TwOffset<M, Plan<M>::NP - 1>::value;
    for (int i = threadIdx.x; i < kMid; i += GeoM::THREADS) tws[i] = p.tw[i];
    tw_mid = tws;
  }
  group_sync<M>(g);

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
  for (int lb = 0; lb < nb; lb++) {
    if (group_active && b0 + lb >= 0) {
      mbar_wait(&mbar[lb], 0);
      phase_bits ^= 1u << lb;
    }
  }
  group_sync<M>(g);

  int slot_new = nb - 1;
  const int nact = group_active ? (int) ((p.nframes - fb < p.frames_per_group) ? p.nframes - fb : p.frames_per_group) : 0;
  long long ro = fb * p.row_stride;                              // row offset of the frame (rows and F rows)
  const float *next_src = p.samples + ((f_first + 1) * (long long) hop - p.origin);
  int ob[4];
  iq_row_bases<M>(t, ob);
  float mu_new = 0.f;
  for (int it = 0; it < p.frames_per_group; ++it, ro += p.row_stride, next_src += hop) {
    const bool active = it < nact;
    const bool next_there = it + 1 < nact;
    const int slot_next = (slot_new + 1 == slots) ? 0 : slot_new + 1;
    if (it > 0 && active) {
      mbar_wait(&mbar[slot_new], (phase_bits >> slot_new) & 1u);
      phase_bits ^= 1u << slot_new;
    }
    auto request_next = [&]() {
      GLB_CHECK_SRC(p, next_src, hop);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      mbar_expect_tx(&mbar[slot_next], blk_bytes);
      tma_load_1d(ring + (size_t) slot_next * hop, next_src, blk_bytes, &mbar[slot_next]);
    };
    if (GLB_RING_EXTRA && next_there && t == 0) request_next();
    const int slot_oldest = GLB_RING_EXTRA ? ((slot_next + 1 == slots) ? 0 : slot_next + 1) : slot_next;
    {
      float2 x[kPoints];
      if constexpr (QSC >= 0) {
        ring_fetch<M, (QSC >= 0 ? QSC : 0)>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, false, false, red, 0.f, g);
      } else {
        switch (qs) {
          case 4: ring_fetch<M, 4>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, false, false, red, 0.f, g); break;
          case 3: ring_fetch<M, 3>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, false, false, red, 0.f, g); break;
          case 2: ring_fetch<M, 2>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, false, false, red, 0.f, g); break;
          case 1: ring_fetch<M, 1>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, false, false, red, 0.f, g); break;
          default: ring_fetch<M, 0>(x, t, ring, hop, slot_oldest, slots, mu, mu_new, false, false, red, 0.f, g); break;
        }
      }
      float acc[17], den[17];
#pragma unroll
      for (int i = 0; i < 17; i++) acc[i] = den[i] = 0.f;
      // j = -1: the hn transform (mu), then the K' tapers
      for (int j = -1; j < p.ntapers; ++j) {
        float2 v[kPoints];
        apply_taper<M, true>(v, x, t, p, j < 0 ? fp.hn : p.tapers + (size_t) j * GeoM::N);
        if constexpr (RT) {
          pass_compute_rt<M, 0>(v, tr);
          group_sync<M>(g);            // (A) the previous transform's last pass has been read by all
          pass_scatter<M, 0>(v, t, buf);
        } else {
          group_sync<M>(g);
          pass_store<M, 0>(v, t, buf, p.tw);
        }
        if (!GLB_RING_EXTRA && next_there && j < 0 && t == 0) request_next();
        group_sync<M>(g);
        RingMidPasses<M, 1, RT>::run(v, t, buf, tw_mid, tr, g);
        const bool w0 = t < 32;
        if constexpr (RT) {
          last_pass_rt<M>(v, t, buf, p.tw, tr);
        } else {
          TwRegs tl;
          load_last_regs<M>(tl, t, p.tw, p.vtab);
          last_pass_load<M>(v, t, buf);
          last_pass_compute_rt<M>(v, t, tl);
        }
        if (j < 0) {
          if (w0) iq_emit_mu<M, true>(v, t, zmu, ZST);
          else iq_emit_mu<M, false>(v, t, zmu, ZST);
        } else {
          const float2 w = __ldg(fp.u0 + j);
          if (w0) iq_add_ftest<M, true>(v, t, kIqPowerScale, w.x, w.y, zmu, ZST, acc, den);
          else iq_add_ftest<M, false>(v, t, kIqPowerScale, w.x, w.y, zmu, ZST, acc, den);
        }
      }
      if (active && p.rows) {
        float *row_ptr = p.rows + ro;
#pragma unroll
        for (int slot = 0; slot < 17; slot++) {
          if (slot == 16) {
            if (t == 0) st_row(row_ptr, acc[16]);
          } else if (slot != 1 || t != 0) {
            st_row(row_ptr + iq_slot_offset<M>(ob, slot), acc[slot]);
          }
        }
      }
      if (active && fp.ftest) {
        float *f_ptr = fp.ftest + ro;
#pragma unroll
        for (int slot = 0; slot < 17; slot++) {
          if (slot == 16) {
            if (t == 0) st_row(f_ptr, iq_ftest_value(zmu[16 * ZST], den[16], fp.fnum));
          } else if (slot != 1 || t != 0) {
            st_row(f_ptr + iq_slot_offset<M>(ob, slot), iq_ftest_value(zmu[slot * ZST], den[slot], fp.fnum));
          }
        }
      }
    }
    slot_new = slot_next;
  }
}

// regular geometry, staged span covers every block of the launch, 16-byte aligned blocks: fused kernel.
// Returns 1 when launched, 0 when the launch is not served, < 0 on error.
template <int M>
static int launch_iq_fused(const KParams &kp, const IqFtestParams *fp, cudaStream_t st) {
  using GeoM = Geo<M>;
  const bool multi = kp.ntapers > 1;
  const bool rt = multi ? RingGeo<M, true>::RT : RingGeo<M, false>::RT;
  const int unit = 2 * GeoM::T;
  int qs = -1;
  for (int s2 = 0; s2 <= 4; s2++)
    if (kp.hop == (unit << s2)) qs = s2;
  if (qs < 0 || (kp.n_ov % kp.hop) != 0 || (kp.hop % 4) != 0 || (kp.origin % 4) != 0 ||
      (reinterpret_cast<uintptr_t>(kp.samples) & 15) != 0)
    return 0;
  const long long blk_lo = (kp.first_frame - kp.n_ov / kp.hop) * (long long) kp.hop;
  const long long blk_hi = (kp.first_frame + kp.nframes) * (long long) kp.hop;
  if (!(kp.origin <= (blk_lo > 0 ? blk_lo : 0) && blk_hi <= kp.origin + kp.count)) return 0;
  const RingLayout L = ring_layout<M>(kp.hop, kPoints >> qs);
  const size_t smem = (size_t) GeoM::G * L.group_bytes + (rt ? 0 : Geo<M>::TWS_BYTES) + (fp ? IqFtestGeo<M>::MU_BYTES : 0);   // fp: F-test
  if (smem > 227 * 1024) return 0;
  const bool lev = kp.levels != nullptr;
  void (*rk)(const KParams) =
      multi ? (qs == 3 ? gram_iq_mtm_kernel<M, 3> : (qs == 2 ? gram_iq_mtm_kernel<M, 2> : gram_iq_mtm_kernel<M, -1>))
      : lev ? (qs == 3 ? gram_iq_kernel<M, 3, true> : (qs == 2 ? gram_iq_kernel<M, 2, true> : gram_iq_kernel<M, -1, true>))
            : (qs == 3 ? gram_iq_kernel<M, 3> : (qs == 2 ? gram_iq_kernel<M, 2> : gram_iq_kernel<M, -1>));
  void (*fk)(const KParams, const IqFtestParams) =
      qs == 3 ? gram_iq_ftest_kernel<M, 3> : (qs == 2 ? gram_iq_ftest_kernel<M, 2> : gram_iq_ftest_kernel<M, -1>);
  int dev = 0, sms = 0;
  CU(cudaGetDevice(&dev));
  CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  static thread_local int occ_iq[4][5][64];
  int &occ = occ_iq[fp ? 3 : multi ? 2 : lev][qs][dev & 63];
  if (occ == 0) {
    if (fp) {
      CU(cudaFuncSetAttribute(fk, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fk, GeoM::THREADS, smem));
    } else {
      CU(cudaFuncSetAttribute(rk, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, rk, GeoM::THREADS, smem));
    }
    if (occ < 1) occ = -1;
  }
  if (occ < 1) return 0;
  // the launch policy of the real ring kernel (launch_gram_m): up to four waves of runs of >= 16 frames
  long long groups = (long long) sms * occ * GeoM::G;
  constexpr int kRingWaves = 4, kRingMinRun = 16;
  if (occ >= 2) {
    int waves = kRingWaves;
    while (waves > 1 && kp.nframes < groups * waves * kRingMinRun) waves--;
    groups *= waves;
  }
  if (g_ring_groups > 0) groups = g_ring_groups;
  if (groups > kp.nframes) groups = kp.nframes;
  if (groups < 1) groups = 1;
  KParams k = kp;
  k.qs = qs;
  k.frames_per_group = (int) ((kp.nframes + groups - 1) / groups);
  g_last_frames_per_group = k.frames_per_group;
  const long long used = (kp.nframes + k.frames_per_group - 1) / k.frames_per_group;
  const int ctas = (int) ((used + GeoM::G - 1) / GeoM::G);
  if (fp) fk<<<ctas, GeoM::THREADS, smem, st>>>(k, *fp);
  else rk<<<ctas, GeoM::THREADS, smem, st>>>(k);
  CU(cudaGetLastError());
  g_launches++;
  g_last_family = 2;
  return 1;
}

// (the multitaper kernel serves the same n as the periodogram's, n = 8192 included: 3.6x faster than the general
// path there, DESIGN §7.5)
static int iq_fused_n(int n) { return n >= 32 && n <= 8192 && (n & (n - 1)) == 0; }

static bool iq_fused_geometry(int n, int hop) {
  if (!iq_fused_n(n) || hop < 1 || hop > n || (n - hop) % hop != 0) return false;
  for (int s = 0; s <= 4; s++)
    if (hop == ((n / 16) << s)) return true;
  return false;
}

static bool iq_fused_allowed() { return g_force_generic == 0 && g_kernel_pref != 1; }

// the general path's scratch (glb_iq_gram_general_scratch_bytes, zoom.cu).  A multitaper launch reuses the one spectrum
// plane for every taper and the fused kernel serves it wherever it serves the periodogram, so the size does not depend
// on ntapers.
extern "C" long long glb_iq_gram_scratch_bytes(int n, int hop, long long nframes, int levels, int ntapers, int ftest) {
  (void) ntapers;
  if (nframes <= 0 || (iq_fused_allowed() && iq_fused_geometry(n, hop))) return 0;
  return glb_iq_gram_general_scratch_bytes(n, nframes, levels, ftest);
}

extern "C" int glb_launch_iq_gram(const glb_iq_gram_args *a, void *stream) {
  if (!a || !a->tables || !a->samples || !a->taper || (a->ftest ? a->levels != nullptr : !a->rows == !a->levels) ||
      a->n < 32 || a->n > 16384 || (a->n & (a->n - 1)) != 0 || a->hop < 1 || a->hop > a->n || a->origin < 0 ||
      a->count < 0 || a->first_frame < 0) {
    glb_set_error("glb_launch_iq_gram: invalid arguments (exactly one of rows and levels, or F rows with optional rows)");
    return GLB_EINVAL;
  }
  if (a->ntapers < 0 || a->ntapers > 32) {
    glb_set_error("glb_launch_iq_gram: ntapers must be in 0..32");
    return GLB_EINVAL;
  }
  if (a->ftest && (a->ntapers < 2 || !a->ftest_taper || !a->ftest_u0)) {
    glb_set_error("glb_launch_iq_gram: the F-test needs ntapers >= 2, ftest_taper and ftest_u0");
    return GLB_EINVAL;
  }
  if (a->levels && a->ntapers > 1) {
    glb_set_error("glb_launch_iq_gram: multitaper rows have no level output (map them with glb_launch_levels)");
    return GLB_EINVAL;
  }
  if (a->levels && (!a->level_tables || a->levels_stride != a->n)) {
    glb_set_error("glb_launch_iq_gram: levels need level_tables and levels_stride = n");
    return GLB_EINVAL;
  }
  if (a->nframes <= 0) return GLB_OK;
  int tn = 0;
  const float2 *tw = nullptr, *vtab = nullptr;
  if (glb_tables_get(a->tables, &tn, &tw, &vtab) != GLB_OK || tn != 2 * a->n) {
    glb_set_error("glb_launch_iq_gram: tables must be built for 2 n");
    return GLB_EINVAL;
  }
  if (iq_fused_allowed() && iq_fused_geometry(a->n, a->hop)) {
    KParams k;
    memset(&k, 0, sizeof k);
    k.samples = a->samples;
    k.origin = 2 * a->origin;
    k.count = 2 * a->count;
    k.tapers = a->taper;
    k.ntapers = a->ntapers > 1 ? a->ntapers : 1;
    k.hop = 2 * a->hop;
    k.n_ov = 2 * (a->n - a->hop);
    k.first_frame = a->first_frame;
    k.nframes = a->nframes;
    k.rows = a->rows;
    k.row_stride = a->n;
    if (a->levels) {
      k.levels = a->levels;
      k.lev_stride = a->levels_stride;
      k.lm.thr = ((const LevelTables *) a->level_tables)->thr_f;
      k.lm.lut = a->levels_log ? a->level_lut : nullptr;
      k.lm.log_scale = a->levels_log;
      k.lm.dmin = a->level_min;
      k.lm.dmax = a->level_max;
      k.lm.thr_level = a->level_thr;
    }
    k.tw = tw;
    k.vtab = vtab;
    IqFtestParams fp;
    fp.ftest = a->ftest;
    fp.hn = a->ftest_taper;
    fp.u0 = reinterpret_cast<const float2 *>(a->ftest_u0);
    fp.fnum = (float) ((double) (a->ntapers - 1) * (double) a->ftest_s);
    const IqFtestParams *fpp = a->ftest ? &fp : nullptr;
    cudaStream_t st = (cudaStream_t) stream;
    int rc = 0;
    switch (a->n) {
      case 32: rc = launch_iq_fused<32>(k, fpp, st); break;
      case 64: rc = launch_iq_fused<64>(k, fpp, st); break;
      case 128: rc = launch_iq_fused<128>(k, fpp, st); break;
      case 256: rc = launch_iq_fused<256>(k, fpp, st); break;
      case 512: rc = launch_iq_fused<512>(k, fpp, st); break;
      case 1024: rc = launch_iq_fused<1024>(k, fpp, st); break;
      case 2048: rc = launch_iq_fused<2048>(k, fpp, st); break;
      case 4096: rc = launch_iq_fused<4096>(k, fpp, st); break;
      case 8192: rc = launch_iq_fused<8192>(k, fpp, st); break;
      default: break;
    }
    if (rc != 0) return rc < 0 ? rc : GLB_OK;
  }
  if (!a->levels) return glb_launch_iq_gram_general(a, stream);
  // two passes: float rows into the scratch behind the spectrum, then the fixed-range mapping of the fused epilogue
  if (!a->scratch) {
    glb_set_error("glb_launch_iq_gram: needs scratch for the spectrum and rows (glb_iq_gram_scratch_bytes)");
    return GLB_EINVAL;
  }
  glb_iq_gram_args g = *a;
  g.rows = (float *) a->scratch + a->nframes * (long long) (a->n + 1) * 2;
  g.levels = nullptr;
  int rc = glb_launch_iq_gram_general(&g, stream);
  if (rc != GLB_OK) return rc;
  const float fixed[2] = {a->level_max, a->level_min};
  return glb_launch_levels(g.rows, a->n, a->n, a->nframes, nullptr, fixed, a->levels_log, a->level_thr, a->level_tables,
                           a->level_lut, nullptr, a->levels, nullptr, stream);
}
