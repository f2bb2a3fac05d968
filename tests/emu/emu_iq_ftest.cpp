// CPU emulation of the harmonic F-test epilogue of the fused I/Q multitaper kernel (gram_iq_ftest_kernel,
// csrc/iq.cu): every thread of one frame runs the kernel's transform (the fft_core.cuh passes at M = n, as
// emu_iq.cpp runs them) once under hn and once under each of K' tapers, then iq_emit_mu / iq_add_ftest /
// iq_ftest_value (iq_core.cuh) with mu in a per-thread column of a shared array, as the kernel keeps it.  The tapers
// are uploaded as the host does, v_k / sqrt(lambda_k), with sl = sqrt(lambda_k) undoing that in the residual.
// Checks F at every row position against a long-double DFT restatement of the contract (include/glfer_b200.h), the
// rows against the sum of the tapered powers, and that every row position is written exactly once.
// The frame is a tone on a bin plus noise, so F spans small and large values.  Prints "n maxrel_F maxrel_row bad".
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <cmath>
#include <algorithm>
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

// the kernel's transform of the frame z (M complex) under the real taper w: regs[t] after the last pass
template <int M>
void transform(const std::vector<float> &z, const std::vector<float> &w, std::vector<std::vector<float2>> &regs) {
  constexpr int T = M / kPoints;
  constexpr bool RT = (M <= 2048) || (M == 8192);       // RingGeo<M, true>::RT (gram_common.cuh)
  static auto tw = build_twiddles<M>();
  static auto vtab = build_vtab(M);
  std::vector<float4> buf4((BufSize<M>::value + 1) / 2 + 1);
  float2 *buf = reinterpret_cast<float2 *>(buf4.data());
  for (int t = 0; t < T; t++)
    for (int q = 0; q < kPoints; q++) {
      const int i = t + T * q;                           // apply_taper: element q of thread t is sample t + T q
      regs[t][q] = mul2(make_float2(z[2 * i], z[2 * i + 1]), make_float2(w[i], w[i]));
    }
  if (RT) {
    std::vector<TwRegs> tr(T);
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
}

// long-double DFT of w z, fft-shifted (position j holds bin (j + M/2) mod M)
template <int M> void dft(const std::vector<float> &z, const std::vector<long double> &w, std::vector<long double> &re,
                          std::vector<long double> &im) {
  static std::vector<long double> c, s;
  if (c.empty()) {
    c.resize(M);
    s.resize(M);
    for (int i = 0; i < M; i++) {
      const long double a = -2.0L * 3.14159265358979323846264338327950288L * (long double) i / M;
      c[i] = cosl(a);
      s[i] = sinl(a);
    }
  }
  re.assign(M, 0);
  im.assign(M, 0);
  for (int k = 0; k < M; k++) {
    long double sr = 0, si = 0;
    for (int i = 0; i < M; i++) {
      const int e = (int) (((long long) i * k) % M);
      const long double zr = w[i] * z[2 * i], zi = w[i] * z[2 * i + 1];
      sr += zr * c[e] - zi * s[e];
      si += zr * s[e] + zi * c[e];
    }
    re[(k + M / 2) & (M - 1)] = sr;
    im[(k + M / 2) & (M - 1)] = si;
  }
}

template <int M> int check(unsigned seed) {
  constexpr int T = M / kPoints, K = 4;
  srand(seed);
  auto rnd = [] { return (float) rand() / RAND_MAX - 0.5f; };
  std::vector<float> z(2 * M);
  const int tone = M / 8 + 3;                              // bin of the line
  for (int i = 0; i < M; i++) {
    const double a = 2.0 * M_PI * tone * i / M;
    z[2 * i] = (float) (1.0 * cos(a)) + rnd();
    z[2 * i + 1] = (float) (1.0 * sin(a)) + rnd();
  }
  // K smooth positive tapers (not DPSS: the epilogue does not depend on which), their U0, S, hn and made-up eigenvalues
  std::vector<std::vector<long double>> v(K, std::vector<long double>(M));
  std::vector<long double> u0(K, 0), lam(K), hn(M, 0);
  long double S = 0;
  for (int k = 0; k < K; k++) {
    for (int i = 0; i < M; i++) v[k][i] = sinl(3.14159265358979323846L * (i + 0.5L) * (k + 1) / M) + 0.1L * (k == 0);
    for (int i = 0; i < M; i++) u0[k] += v[k][i];
    S += u0[k] * u0[k];
    lam[k] = 1.0L - 0.1L * k;
  }
  for (int i = 0; i < M; i++) {
    for (int k = 0; k < K; k++) hn[i] += u0[k] * v[k][i];
    hn[i] /= S;
  }
  // uploaded forms: hn, and v_k / sqrt(lambda_k)
  std::vector<float> hn_f(M);
  for (int i = 0; i < M; i++) hn_f[i] = (float) hn[i];
  std::vector<std::vector<float2>> regs(T, std::vector<float2>(kPoints));
  std::vector<float2> zmu(17 * T);                         // slot s of thread t at zmu[s T + t]
  std::vector<std::vector<float>> acc(T, std::vector<float>(17, 0.f)), den(T, std::vector<float>(17, 0.f));
  transform<M>(z, hn_f, regs);
  for (int t = 0; t < T; t++) {
    if (t < 32) iq_emit_mu<M, true>(regs[t].data(), t, zmu.data() + t, T);
    else iq_emit_mu<M, false>(regs[t].data(), t, zmu.data() + t, T);
  }
  for (int k = 0; k < K; k++) {
    std::vector<float> wk(M);
    const long double sl = sqrtl(lam[k]);
    for (int i = 0; i < M; i++) wk[i] = (float) (v[k][i] / sl);
    transform<M>(z, wk, regs);
    for (int t = 0; t < T; t++) {
      float a[17], d[17];
      std::copy(acc[t].begin(), acc[t].end(), a);
      std::copy(den[t].begin(), den[t].end(), d);
      if (t < 32) iq_add_ftest<M, true>(regs[t].data(), t, 1.f, (float) u0[k], (float) sl, zmu.data() + t, T, a, d);
      else iq_add_ftest<M, false>(regs[t].data(), t, 1.f, (float) u0[k], (float) sl, zmu.data() + t, T, a, d);
      std::copy(a, a + 17, acc[t].begin());
      std::copy(d, d + 17, den[t].begin());
    }
  }
  const float fnum = (float) ((double) (K - 1) * (double) S);
  std::vector<double> F(M, -1.0), row(M, -1.0);
  std::vector<int> hits(M, 0);
  int bad = 0;
  for (int t = 0; t < T; t++) {
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
      F[pos] = iq_ftest_value(zmu[slot * T + t], den[t][slot], fnum);
      row[pos] = acc[t][slot];
    }
  }
  // the contract in long double
  std::vector<long double> mr, mi, yr, yi, dsum(M, 0), psum(M, 0);
  dft<M>(z, hn, mr, mi);
  for (int k = 0; k < K; k++) {
    dft<M>(z, v[k], yr, yi);
    for (int j = 0; j < M; j++) {
      const long double rr = yr[j] - mr[j] * u0[k], ri = yi[j] - mi[j] * u0[k];
      dsum[j] += rr * rr + ri * ri;
      psum[j] += (yr[j] * yr[j] + yi[j] * yi[j]) / lam[k];
    }
  }
  double maxf = 0, maxr = 0, pmean = 0;
  for (int j = 0; j < M; j++) pmean += (double) psum[j] / M;
  for (int j = 0; j < M; j++) {
    if (hits[j] != 1) bad++;
    const long double fref = (K - 1) * (mr[j] * mr[j] + mi[j] * mi[j]) * S / dsum[j];
    maxf = std::max(maxf, (double) (fabsl(F[j] - fref) / fref));
    maxr = std::max(maxr, std::fabs(row[j] - (double) psum[j]) / ((double) psum[j] + 1e-6 * pmean));
  }
  // the line is where F is large
  if (!(F[(tone + M / 2) & (M - 1)] > 100.0)) bad++;
  printf("%d %.3e %.3e %d\n", M, maxf, maxr, bad);
  return bad != 0 || maxf > 1e-3 || maxr > 1e-4;
}

int main() {
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
