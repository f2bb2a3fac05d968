// CPU check of the pixel addressing of the fused I/Q kernel's level epilogue (gram_iq_kernel<M, QSC, true>,
// csrc/iq.cu): runs iq_pixel_bases / iq_pixel_offset of iq_core.cuh for every thread and slot the kernel stores,
// n = 32 .. 8192.  Checks that
//   - every pixel 0..n-1 of a row is written exactly once;
//   - the pixel of bin k is n - 1 - ((k + n/2) mod n): the fft-shifted row position, highest frequency first;
//   - each store instruction of a warp writes consecutive bytes: per slot, the lanes of one frame group (32, or T
//     when a warp holds several groups) cover a run of consecutive pixels in lane order, except thread 0, whose
//     re-ordered registers (thread0_fixup) hold bins outside its warp's runs for slots 8..15 and skip slot 1.
// Prints "n bad_once bad_bin bad_warp" per size; exits non-zero on any failure.
#include <cstdio>
#include <vector>
#include "../../glfer_b200/csrc/tables.hpp"
#include "../../glfer_b200/csrc/iq_core.cuh"

using namespace glb;

template <int M> int check() {
  constexpr int T = M / kPoints;
  constexpr int W = T < 32 ? T : 32;                     // lanes of one frame group in a warp
  std::vector<int> hits(M, 0);
  std::vector<std::vector<int>> pix(T, std::vector<int>(17, -1));
  int bad_bin = 0, bad_once = 0, bad_warp = 0;
  for (int t = 0; t < T; t++) {
    int pb[4];
    iq_pixel_bases<M>(t, pb);
    for (int slot = 0; slot < 17; slot++) {
      if (!iq_slot_stored<M>(t, slot)) continue;
      const int px = iq_pixel_offset<M>(pb, slot);
      const int want = M - 1 - ((slot_bin<M>(t, slot) + M / 2) & (M - 1));
      if (px < 0 || px >= M || px != want) {
        bad_bin++;
        continue;
      }
      hits[px]++;
      pix[t][slot] = px;
    }
  }
  for (int j = 0; j < M; j++)
    if (hits[j] != 1) bad_once++;
  for (int w0 = 0; w0 < T; w0 += W) {
    for (int slot = 0; slot < 16; slot++) {
      std::vector<int> run;
      for (int t = w0; t < w0 + W; t++) {
        if (t == 0 && (slot == 1 || slot >= 8)) continue;  // thread 0's re-ordered bins (see above)
        run.push_back(pix[t][slot]);
      }
      const bool has_t0 = w0 == 0 && (slot == 1 || slot >= 8);
      if ((int) run.size() != (has_t0 ? W - 1 : W)) { bad_warp++; continue; }
      const int step = run.size() > 1 ? run[1] - run[0] : 1;
      if (step != 1 && step != -1) { bad_warp++; continue; }
      for (size_t i = 1; i < run.size(); i++)
        if (run[i] - run[i - 1] != step) { bad_warp++; break; }
    }
  }
  printf("%d %d %d %d\n", M, bad_once, bad_bin, bad_warp);
  return bad_once != 0 || bad_bin != 0 || bad_warp != 0;
}

int main() {
  int rc = 0;
  rc |= check<32>();
  rc |= check<64>();
  rc |= check<128>();
  rc |= check<256>();
  rc |= check<512>();
  rc |= check<1024>();
  rc |= check<2048>();
  rc |= check<4096>();
  rc |= check<8192>();
  return rc;
}
