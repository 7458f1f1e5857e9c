// pt_denoise.h — the per-pixel arithmetic of the denoiser (ptc_render_denoised, ptc_denoise_image): first-hit albedo,
// the variance of a pixel's mean from two halves of its samples, and one level of a variance-guided edge-avoiding
// à-trous filter (Dammertz et al. 2010, with SVGF's variance propagation, Schied et al. 2017).
//
// Written once as PT_HD code: nvcc compiles it into the denoise kernels (pt_denoise.cuh), g++ into the test-only
// hostsim library (tests/hostsim/denoisesim.cpp), so that a test can predict the device's output bit for bit.  Only
// + - * /, sqrtf, fminf and fmaxf appear: with --fmad=false / -ffp-contract=off (pt_hd.h) each rounds once, the same way
// on both sides.  The edge-stopping functions are rational, 1 / (1 + d² / σ²), rather than exp(-d² / σ²), because the
// device's expf and glibc's differ in their last bits.
//
// Per-pixel data, float4 each: xv = (x.rgb, var) with x the demodulated radiance noisy / max(albedo, kDenoiseAlbedoMin)
// and var the variance of its mean luminance; ga = (albedo.rgb, 0); gn = (normal.xyz, 0).  A pixel whose x has a
// non-finite channel (every pixel whose noisy value has one) is NON-FINITE: as a neighbour it has weight 0, as a centre
// it passes through every level unchanged, and its output is its noisy value itself.
#pragma once
#include "pt_bsdf.h"
#include "pt_hd.h"

namespace pt {

constexpr float kDenoiseAlbedoMin = 1e-3f;  // demodulation floor: black albedo must not divide by zero
constexpr int kDenoiseMaxIterations = 10;

// Albedo of a first hit, the guide the filter keeps edges of and the factor it demodulates by: the diffuse or specular
// colour of the materials that have one, the checker colour at the hit point, and 1 for the rest (dielectric, emitter,
// null material; a miss is 1 too)
PT_HD V3 feature_albedo(const DMaterial &m, V3 pos) {
  switch (m.type) {
    case 0:  // Lambertian
    case 2:  // metal
    case 5:  // plastic
    case 6:  // rough conductor
      return v3(m.albedo[0], m.albedo[1], m.albedo[2]);
    case 1:
      return checker_value(m, pos);
    default:
      return v3(1.0f, 1.0f, 1.0f);
  }
}

PT_HD float denoise_lum(float r, float g, float b) { return 0.2126f * r + 0.7152f * g + 0.0722f * b; }
PT_HD bool denoise_finite3(float a, float b, float c) { return isfinite(a) && isfinite(b) && isfinite(c); }

// Variance of a pixel's mean luminance, demodulated, from its fp32 film sums Sh over samples [0, h) and Sn over [0, n):
// A = Sh / h and B = (Sn - Sh) / (n - h) are independent means of h and n - h samples, so (L(A') - L(B'))² h (n - h) / n²
// is an unbiased estimate of the variance of the mean of all n (A' = A / max(albedo, kDenoiseAlbedoMin), B' likewise).
// Equal halves: (L(A') - L(B'))² / 4.  0 where Sn has a non-finite channel.
PT_HD float denoise_variance(const float Sh[3], const float Sn[3], int h, int n, const float albedo[3]) {
  if (!denoise_finite3(Sn[0], Sn[1], Sn[2])) return 0.0f;
  const float ih = 1.0f / (float)h, ib = 1.0f / (float)(n - h);
  float a[3], b[3];
  for (int c = 0; c < 3; c++) {
    const float d = fmaxf(albedo[c], kDenoiseAlbedoMin);
    a[c] = Sh[c] * ih / d;
    b[c] = (Sn[c] - Sh[c]) * ib / d;
  }
  const float dl = denoise_lum(a[0], a[1], a[2]) - denoise_lum(b[0], b[1], b[2]);
  const float k = (float)h * (float)(n - h) / ((float)n * (float)n);
  return dl * dl * k;
}

// The filter's input of one pixel: x = noisy / max(albedo, kDenoiseAlbedoMin) per channel, with its variance
PT_HD float4 denoise_demodulate(const float noisy[3], float var, const float albedo[3]) {
  return make_float4(noisy[0] / fmaxf(albedo[0], kDenoiseAlbedoMin), noisy[1] / fmaxf(albedo[1], kDenoiseAlbedoMin),
                     noisy[2] / fmaxf(albedo[2], kDenoiseAlbedoMin), var);
}

struct DenoiseParams {
  float sl2;               // σ_l², which scales the prefiltered variance
  float inv_sn2, inv_sa2;  // 1 / σ² of normal and albedo
};
PT_HD DenoiseParams denoise_params(float sigma_luminance, float sigma_normal, float sigma_albedo) {
  DenoiseParams p;
  p.sl2 = sigma_luminance * sigma_luminance;
  p.inv_sn2 = 1.0f / (sigma_normal * sigma_normal);
  p.inv_sa2 = 1.0f / (sigma_albedo * sigma_albedo);
  return p;
}

PT_HD float denoise_dist2(float4 a, float4 b) {
  const float d0 = a.x - b.x, d1 = a.y - b.y, d2 = a.z - b.z;
  return d0 * d0 + d1 * d1 + d2 * d2;
}

// One à-trous level at pixel (x, y) of a width x height frame with tap spacing `step`: xv, ga, gn as above (xv the
// level's input).  First the level's own variance is prefiltered with (1 2 1)x(1 2 1) over the finite pixels of the 3x3
// neighbourhood inside the frame, normalised by the weights used: g.  Then 5x5 taps (dy outer, dx inner, -2..2) with
// B3-spline weights (1 4 6 4 1)/16 times the edge-stopping weights
//   w_l = 1 / (1 + (L(x_p) - L(x_q))² / (σ_l² g + 1e-10)),  w_n = 1 / (1 + |n_p - n_q|² · (1/σ_n²)),  w_a likewise for albedo;
// taps outside the frame and non-finite ones are skipped.  x' = Σ w x_q / Σ w, var' = Σ w² var_q / (Σ w)².  The centre's
// own weight is at least (6/16)², so Σ w > 0.
PT_HD float4 denoise_atrous_pixel(const float4 *xv, const float4 *ga, const float4 *gn, int width, int height, int x, int y,
                                  int step, const DenoiseParams &dp) {
  const size_t p = (size_t)y * (size_t)width + (size_t)x;
  const float4 c = ldg4(xv + p);
  if (!denoise_finite3(c.x, c.y, c.z)) return c;
  float gs = 0.0f, gk = 0.0f;
  for (int dy = -1; dy <= 1; dy++) {
    const int qy = y + dy;
    if (qy < 0 || qy >= height) continue;
    for (int dx = -1; dx <= 1; dx++) {
      const int qx = x + dx;
      if (qx < 0 || qx >= width) continue;
      const float4 q = ldg4(xv + (size_t)qy * (size_t)width + (size_t)qx);
      if (!denoise_finite3(q.x, q.y, q.z)) continue;
      const float k = (dx == 0 ? 2.0f : 1.0f) * (dy == 0 ? 2.0f : 1.0f);
      gs = gs + k * q.w;
      gk = gk + k;
    }
  }
  const float g = gs / gk;
  const float lp = denoise_lum(c.x, c.y, c.z);
  const float4 ap = ldg4(ga + p), np = ldg4(gn + p);
  const float lden = dp.sl2 * g + 1e-10f;
  const float kB3[5] = {0.0625f, 0.25f, 0.375f, 0.25f, 0.0625f};
  float sw = 0.0f, sr = 0.0f, sg = 0.0f, sb = 0.0f, sv = 0.0f;
  for (int dy = -2; dy <= 2; dy++) {
    const int qy = y + dy * step;
    if (qy < 0 || qy >= height) continue;
    for (int dx = -2; dx <= 2; dx++) {
      const int qx = x + dx * step;
      if (qx < 0 || qx >= width) continue;
      const size_t q = (size_t)qy * (size_t)width + (size_t)qx;
      const float4 v = ldg4(xv + q);
      if (!denoise_finite3(v.x, v.y, v.z)) continue;
      const float dl = lp - denoise_lum(v.x, v.y, v.z);
      const float wl = 1.0f / (1.0f + dl * dl / lden);
      const float wn = 1.0f / (1.0f + denoise_dist2(np, ldg4(gn + q)) * dp.inv_sn2);
      const float wa = 1.0f / (1.0f + denoise_dist2(ap, ldg4(ga + q)) * dp.inv_sa2);
      const float w = kB3[dy + 2] * kB3[dx + 2] * wl * wn * wa;
      sw = sw + w;
      sr = sr + w * v.x;
      sg = sg + w * v.y;
      sb = sb + w * v.z;
      sv = sv + w * w * v.w;
    }
  }
  return make_float4(sr / sw, sg / sw, sb / sw, sv / (sw * sw));
}

// The filter's output of one pixel: x remodulated by max(albedo, kDenoiseAlbedoMin); a non-finite pixel's noisy value
PT_HD void denoise_remodulate(float4 xv, const float noisy[3], const float albedo[3], float out[3]) {
  if (!denoise_finite3(xv.x, xv.y, xv.z)) {
    out[0] = noisy[0], out[1] = noisy[1], out[2] = noisy[2];
    return;
  }
  out[0] = xv.x * fmaxf(albedo[0], kDenoiseAlbedoMin);
  out[1] = xv.y * fmaxf(albedo[1], kDenoiseAlbedoMin);
  out[2] = xv.z * fmaxf(albedo[2], kDenoiseAlbedoMin);
}

}  // namespace pt
