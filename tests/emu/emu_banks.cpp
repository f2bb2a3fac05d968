// Shared-memory wavefronts of every exchange access of the 16-point ring kernel (fft_core.cuh, the same
// index functions the GPU compiles), per frame, for the ring shapes with whole warps (M = 512, 1024, 2048):
// ring fetch, first-pass scatter, mid-pass loads and scatter, last-pass loads of both butterflies.  Per warp
// instruction: 32 lanes, 64-bit, bank = (byte address / 4) mod 32, counted over the whole warp (distinct
// 4-byte words per bank) and as two half-warps (distinct 8-byte words per bank pair).  Conflict-free = 2
// wavefronts per instruction.  Prints the accounting; exits non-zero on any conflict.
#include <algorithm>
#include <cstdio>
#include <map>
#include <set>
#include <vector>
#include "../../glfer_b200/csrc/tables.hpp"

using namespace glb;

static int wavefronts_warp(const int *e) {
  std::map<int, std::set<int>> words;
  for (int l = 0; l < 32; l++)
    for (int h = 0; h < 2; h++) words[(2 * e[l] + h) & 31].insert(2 * e[l] + h);
  size_t w = 0;
  for (auto &kv : words) w = std::max(w, kv.second.size());
  return (int) w;
}
static int wavefronts_halves(const int *e) {
  int tot = 0;
  for (int h = 0; h < 2; h++) {
    std::map<int, std::set<int>> pairs;
    for (int l = 16 * h; l < 16 * h + 16; l++) pairs[e[l] & 15].insert(e[l]);
    size_t w = 0;
    for (auto &kv : pairs) w = std::max(w, kv.second.size());
    tot += (int) w;
  }
  return tot;
}

static int g_bad = 0;
// one access site: idx(t, u) is the float2 entry thread t touches in unrolled access u
template <int M, class F> static long account(const char *name, int nu, F idx) {
  constexpr int T = M / kPoints;
  long warp = 0, halves = 0, instr = 0;
  for (int w = 0; w < T / 32; w++)
    for (int u = 0; u < nu; u++) {
      int e[32];
      for (int l = 0; l < 32; l++) e[l] = idx(32 * w + l, u);
      warp += wavefronts_warp(e);
      halves += wavefronts_halves(e);
      instr++;
    }
  const bool clean = warp == 2 * instr && halves == 2 * instr;
  printf("  %-20s %4ld instr  %5ld / %5ld wavefronts%s\n", name, instr, warp, halves, clean ? "" : "  BANK CONFLICT");
  g_bad += !clean;
  return warp;
}

template <int M> static void frame() {
  constexpr int T = M / kPoints, P1 = Plan<M>::NP - 2;     // P1: the pass that feeds the last one
  // 50 % overlap (the benchmark shapes): two ring blocks of M/2 float2 each, 8 entries per thread
  auto ring = [](int t, int u) { return (u >> 3) * (M / 2) + t + T * (u & 7); };
  printf("M = %d (N = %d), %d warps per frame; whole warp / two half-warps:\n", M, 2 * M, T / 32);
  long tot = 0;
  tot += account<M>("ring fetch", 16, ring);
  tot += account<M>("pass 0 scatter", 16, [](int t, int r) { return scatter_index<M, 0>(scatter_base<M, 0>(t, 0), r); });
  tot += account<M>("mid pass load", 16, [](int t, int q) { return ld_index<M>(t, q); });
  constexpr int S = kPoints / PlanRadix<M, P1>::R;
  tot += account<M>("mid pass scatter", 16, [](int t, int i) {
    const int u = i % S, r = i / S;
    return scatter_index<M, P1>(scatter_base<M, P1>(t, u), r);
  });
  tot += account<M>("last pass load A", 8, [](int t, int r) { return last_index<M>(t, r); });
  tot += account<M>("last pass load B", 8, [](int t, int r) { return last_index<M>(t == 0 ? T : 2 * T - t, r); });
  printf("  %-20s %ld wavefronts per frame\n", "total", tot);
}

int main() {
  frame<512>();
  frame<1024>();
  frame<2048>();
  printf("%s\n", g_bad ? "FAIL" : "OK");
  return g_bad != 0;
}
