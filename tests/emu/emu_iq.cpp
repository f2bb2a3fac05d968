// CPU emulation of the fused I/Q spectrogram kernel (gram_iq_kernel, csrc/iq.cu): runs every thread of one
// frame phase by phase through the same fft_core.cuh passes the kernel runs at M = n (register twiddles where
// RingGeo<M, false>::RT, the table mid passes at M = 4096) and its own epilogue (iq_core.cuh), with the exchange
// buffer as a plain array.  Checks the row against a long-double DFT, and that every row position 0..n-1 is
// written exactly once, at the fft-shifted index of its bin.  The input of size M is the one emu_fft.cpp uses
// at M (same seed), read as M complex samples.  Prints "n maxrel bad path".
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <cmath>
#include "../../glfer_b200/csrc/tables.hpp"
#include "../../glfer_b200/csrc/iq_core.cuh"

using namespace glb;

template <int M, int P> struct MidTable {
  static void run(std::vector<std::vector<float2>> &regs, float2 *buf, const float2 *tw) {
    constexpr int T = M / kPoints;
    if constexpr (P < Plan<M>::NP - 1) {
      for (int t = 0; t < T; t++) pass_load<M>(regs[t].data(), t, buf);
      for (int t = 0; t < T; t++) pass_store<M, P>(regs[t].data(), t, buf, tw);
      MidTable<M, P + 1>::run(regs, buf, tw);
    }
  }
};

template <int M, int P> struct MidRT {
  static void run(std::vector<std::vector<float2>> &regs, float2 *buf, std::vector<TwRegs> &tr) {
    constexpr int T = M / kPoints;
    if constexpr (P < Plan<M>::NP - 1) {
      for (int t = 0; t < T; t++) pass_load<M>(regs[t].data(), t, buf);
      for (int t = 0; t < T; t++) pass_compute_rt<M, P>(regs[t].data(), tr[t]);
      for (int t = 0; t < T; t++) pass_scatter<M, P>(regs[t].data(), t, buf);
      MidRT<M, P + 1>::run(regs, buf, tr);
    }
  }
};

template <int M> int check(unsigned seed) {
  constexpr int T = M / kPoints;
  constexpr bool RT = (M <= 2048) || (M == 8192);       // RingGeo<M, false>::RT (gram_common.cuh)
  std::vector<float> x(2 * M);
  srand(seed);
  for (auto &v : x) v = (float) rand() / RAND_MAX - 0.5f;
  auto tw = build_twiddles<M>();
  auto vtab = build_vtab(M);
  std::vector<std::vector<float2>> regs(T, std::vector<float2>(kPoints));
  std::vector<float4> buf4((BufSize<M>::value + 1) / 2 + 1);
  float2 *buf = reinterpret_cast<float2 *>(buf4.data());
  // ring_fetch: element q of thread t is complex sample t + T q
  for (int t = 0; t < T; t++)
    for (int q = 0; q < kPoints; q++) regs[t][q] = make_float2(x[2 * (t + T * q)], x[2 * (t + T * q) + 1]);
  std::vector<TwRegs> tr(T);
  if (RT) {
    for (int t = 0; t < T; t++) load_tw_regs<M>(tr[t], t, tw.data(), vtab.data());
    for (int t = 0; t < T; t++) pass_compute_rt<M, 0>(regs[t].data(), tr[t]);
    for (int t = 0; t < T; t++) pass_scatter<M, 0>(regs[t].data(), t, buf);
    MidRT<M, 1>::run(regs, buf, tr);
    for (int t = 0; t < T; t++) last_pass_rt<M>(regs[t].data(), t, buf, tw.data(), tr[t]);
  } else {
    for (int t = 0; t < T; t++) pass_store<M, 0>(regs[t].data(), t, buf, tw.data());
    MidTable<M, 1>::run(regs, buf, tw.data());
    for (int t = 0; t < T; t++) {
      TwRegs tl;
      load_last_regs<M>(tl, t, tw.data(), vtab.data());
      last_pass_load<M>(regs[t].data(), t, buf);
      last_pass_compute_rt<M>(regs[t].data(), t, tl);
    }
  }
  std::vector<double> row(M, -1.0);
  std::vector<int> hits(M, 0);
  int bad = 0;
  for (int t = 0; t < T; t++) {
    float yv[17];
    yv[16] = 0.f;
    if (t < 32) iq_emit_power<M, true>(regs[t].data(), t, 1.f, yv);
    else iq_emit_power<M, false>(regs[t].data(), t, 1.f, yv);
    int ob[4];
    iq_row_bases<M>(t, ob);
    for (int slot = 0; slot < 17; slot++) {
      if (!iq_slot_stored<M>(t, slot)) continue;
      const int pos = iq_slot_offset<M>(ob, slot);
      if (pos < 0 || pos >= M || pos != ((slot_bin<M>(t, slot) + M / 2) & (M - 1))) {
        bad++;
        continue;
      }
      hits[pos]++;
      row[pos] = yv[slot];
    }
  }
  // long-double DFT of the M complex samples, bins in fft-shifted order
  std::vector<long double> c(M), s(M);
  for (int i = 0; i < M; i++) {
    const long double a = -2.0L * 3.14159265358979323846264338327950288L * (long double) i / M;
    c[i] = cosl(a);
    s[i] = sinl(a);
  }
  std::vector<double> ref(M);
  double ref_ms = 0;
  for (int k = 0; k < M; k++) {
    long double sr = 0, si = 0;
    for (int i = 0; i < M; i++) {
      const int e = (int) (((long long) i * k) % M);
      const long double zr = x[2 * i], zi = x[2 * i + 1];
      sr += zr * c[e] - zi * s[e];
      si += zr * s[e] + zi * c[e];
    }
    ref[(k + M / 2) & (M - 1)] = (double) (sr * sr + si * si);
    ref_ms += (double) (sr * sr + si * si);
  }
  ref_ms /= M;
  double maxrel = 0;
  for (int j = 0; j < M; j++) {
    if (hits[j] != 1) bad++;
    const double rel = std::fabs(row[j] - ref[j]) / (ref[j] + 1e-6 * ref_ms);
    if (rel > maxrel) maxrel = rel;
  }
  printf("%d %.3e %d %s\n", M, maxrel, bad, RT ? "rt" : "table");
  return bad != 0 || maxrel > 1e-4;
}

int main() {
  // seeds: the ones emu_fft.cpp uses at the same M (register-twiddle variant where it has one)
  int rc = 0;
  rc |= check<32>(2);
  rc |= check<64>(22);
  rc |= check<128>(23);
  rc |= check<256>(24);
  rc |= check<512>(25);
  rc |= check<1024>(26);
  rc |= check<2048>(27);
  rc |= check<4096>(28);
  rc |= check<8192>(29);
  return rc;
}
