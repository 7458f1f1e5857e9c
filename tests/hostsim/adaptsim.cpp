// adaptsim.cpp — TEST-ONLY host compilation of the adaptive-sampling decision (ptc_render_adaptive): the schedule and the
// per-pixel functions of pt_adaptive.h, compiled by g++ into libhostsim.so next to hostsim.cpp, and one decision step
// as the device runs it (k_adapt_decide, k_adapt_keep, k_adapt_leave, then a stable compaction).  Exports `adapt_sim_*`
// symbols only; the product never links or loads it.
#include <cstdint>
#include <vector>

#include "../../raytracer-rust_b200/csrc/pt_adaptive.h"

using namespace pt;

extern "C" {

int32_t adapt_sim_next_end(int32_t n, int32_t spp) { return adapt_next_end(n, spp); }

// One decision over the active list (ascending pixel indices) of a width x height frame at n samples against the
// snapshot at m.  V, Vp: W*H*3 fp32 film sums (only active pixels are read).  needs: W*H bytes, the map as the decision
// leaves it (active pixels written, the ones that leave cleared, the others untouched).  counts: W*H, n written for the
// pixels that leave.  next: the pixels that stay, ascending.  Returns their number.
int64_t adapt_sim_step(int32_t width, int32_t height, const float *V, const float *Vp, const uint32_t *list, int64_t n_list,
                       int32_t n, int32_t m, float threshold, uint8_t *needs, int32_t *counts, uint32_t *next) {
  for (int64_t i = 0; i < n_list; i++) {
    const uint32_t p = list[i];
    needs[p] = adapt_needs_more(V + (size_t)p * 3, Vp + (size_t)p * 3, n, m, threshold) ? 1u : 0u;
  }
  std::vector<uint8_t> keep((size_t)n_list);
  for (int64_t i = 0; i < n_list; i++) keep[(size_t)i] = adapt_keep(needs, width, height, list[i]) ? 1u : 0u;
  int64_t k = 0;
  for (int64_t i = 0; i < n_list; i++) {
    const uint32_t p = list[i];
    if (keep[(size_t)i]) {
      next[k++] = p;
    } else {
      needs[p] = 0u;
      counts[p] = n;
    }
  }
  return k;
}

}  // extern "C"
