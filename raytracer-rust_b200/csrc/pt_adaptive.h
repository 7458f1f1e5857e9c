// pt_adaptive.h — the sample schedule and the per-pixel decision of adaptive sampling (ptc_render_adaptive).
//
// Written once as PT_HD code: nvcc compiles it into the decision kernels (pt_wavefront.cuh), g++ into the test-only
// hostsim library (tests/hostsim/adaptsim.cpp), so that a test can predict every decision of the device bit for bit.
//
// Schedule: pass 0 renders samples [0, min_spp/2) of every pixel, pass 1 [min_spp/2, min_spp); every later pass renders
// [n, min(2n, spp)) of the pixels still active.  A pass is a sample RANGE, not the even or odd samples: an NEE shadow ray
// carries a distance, not its sample index, so a parity split would need the index smuggled through the pool and a
// second film; a range needs neither, because the film of a pixel rendered over [0, n) in pieces is, bit for bit, the
// film of a uniform render at n spp (Philox keyed on (pixel, sample), fixed-point film).
//
// Decision after a pass, on the fp32 film sums (film_value, as k_film_to_accum produces them): V now at n samples, Vp
// before the pass at m samples.  I = V / n, A = (V - Vp) / (n - m), and the error of Dammertz et al. 2009 (as Cycles
// uses it) e = (|I_r - A_r| + |I_g - A_g| + |I_b - A_b|) / (1e-4 + sqrt(I_r + I_g + I_b)).  A pixel needs more iff
// e >= threshold; a pixel with a non-finite channel never does (a film flag cannot be undone by more samples).  A pixel
// stays active iff it is active and an active pixel of its 3x3 neighbourhood (itself included) needs more; pixels that
// leave never return, so all active pixels share one sample count.
//
// Every operation below rounds once (--fmad=false / -ffp-contract=off, pt_hd.h), in the order written.
#pragma once
#include "pt_hd.h"

namespace pt {

// the end of the pass that follows a pass ending at n (n >= min_spp): samples [n, min(2n, spp))
PT_HD int adapt_next_end(int n, int spp) { return n < spp - n ? 2 * n : spp; }

// V, Vp: the three fp32 film sums of a pixel at n and at m < n samples
PT_HD bool adapt_needs_more(const float V[3], const float Vp[3], int n, int m, float threshold) {
  if (!isfinite(V[0]) || !isfinite(V[1]) || !isfinite(V[2])) return false;
  const float fn = (float)n, fd = (float)(n - m);
  float num = 0.0f, lum = 0.0f;
  for (int c = 0; c < 3; c++) {
    const float I = V[c] / fn, A = (V[c] - Vp[c]) / fd;
    num = num + fabsf(I - A);
    lum = lum + I;
  }
  const float e = num / (1e-4f + sqrtf(lum));
  return e >= threshold;
}

// needs: W*H bytes, 1 where an ACTIVE pixel needs more, 0 everywhere else
PT_HD bool adapt_keep(const uint8_t *needs, int width, int height, uint32_t pixel) {
  const int x = (int)(pixel % (uint32_t)width), y = (int)(pixel / (uint32_t)width);
  const int x0 = x > 0 ? x - 1 : 0, x1 = x + 1 < width ? x + 1 : x;
  const int y0 = y > 0 ? y - 1 : 0, y1 = y + 1 < height ? y + 1 : y;
  for (int yy = y0; yy <= y1; yy++)
    for (int xx = x0; xx <= x1; xx++)
      if (needs[(size_t)yy * (size_t)width + (size_t)xx]) return true;
  return false;
}

}  // namespace pt
