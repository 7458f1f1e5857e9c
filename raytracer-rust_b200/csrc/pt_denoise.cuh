// pt_denoise.cuh — the kernels of ptc_render_denoised and ptc_denoise_image.  The per-pixel arithmetic is pt_denoise.h's;
// these kernels only move data.  One thread per pixel everywhere; k_atrous runs in 2-D blocks whose rows lie along x.
#pragma once
#include "pt_denoise.h"
#include "pt_wavefront.cuh"

namespace ptw {

constexpr int kAtrousBlockX = 32, kAtrousBlockY = 8;

// The first hits of one camera sample (slot i = pixel i, as the extend stage left them in the hook workspace) added to
// the per-pixel sums: albedo (pt_denoise.h: feature_albedo; a miss adds 1) and normal (the hit record's, as the shade
// stage reads it; a miss adds 0).  One thread per pixel and one addition per sample, so the sums are in sample order.
__global__ void k_feature_add(const float4 *__restrict__ hit0, const float4 *__restrict__ hit1, const DMaterial *__restrict__ materials,
                              uint32_t n_pixels, float *albedo_sum, float *normal_sum) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_pixels) return;
  const float4 h1 = hit1[p];
  const uint32_t bits = f2u(h1.w);
  V3 a = v3(1.0f, 1.0f, 1.0f), n = v3(0.0f, 0.0f, 0.0f);
  if (bits & kHitBit) {
    const float4 h0 = hit0[p];
    a = feature_albedo(materials[bits & kMatMask], v3(h0.x, h0.y, h0.z));
    n = v3(h1.x, h1.y, h1.z);
  }
  const size_t i = (size_t)p * 3;
  albedo_sum[i] = albedo_sum[i] + a.x, albedo_sum[i + 1] = albedo_sum[i + 1] + a.y, albedo_sum[i + 2] = albedo_sum[i + 2] + a.z;
  normal_sum[i] = normal_sum[i] + n.x, normal_sum[i + 1] = normal_sum[i + 1] + n.y, normal_sum[i + 2] = normal_sum[i + 2] + n.z;
}
// sums -> means, in place: x scale = 1.0f / feature_spp
__global__ void k_feature_mean(float *albedo, float *normal, size_t n, float scale) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  albedo[i] = albedo[i] * scale;
  normal[i] = normal[i] * scale;
}
// var[p] = denoise_variance of the fp32 film sums after samples [0, h) (sh, k_film_to_accum's) and [0, n) (the film)
__global__ void k_denoise_variance(const float *__restrict__ sh, Film film, uint32_t n_pixels, int32_t h, int32_t n,
                                   const float *__restrict__ albedo, float *var) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_pixels) return;
  const unsigned long long flags = film.flags[p];
  const size_t i = (size_t)p * 3;
  float Sh[3], Sn[3], a[3];
  for (int c = 0; c < 3; c++) Sh[c] = sh[i + c], Sn[c] = 0.0f + film_value(film.sum[i + c], flags, c), a[c] = albedo[i + c];
  var[p] = denoise_variance(Sh, Sn, h, n, a);
}
// the filter's packed input: xv = (noisy / max(albedo, floor), var), ga = (albedo, 0), gn = (normal, 0)
__global__ void k_denoise_prepare(const float *__restrict__ noisy, const float *__restrict__ var, const float *__restrict__ albedo,
                                  const float *__restrict__ normal, uint32_t n_pixels, float4 *xv, float4 *ga, float4 *gn) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_pixels) return;
  const size_t i = (size_t)p * 3;
  const float c[3] = {noisy[i], noisy[i + 1], noisy[i + 2]}, a[3] = {albedo[i], albedo[i + 1], albedo[i + 2]};
  xv[p] = denoise_demodulate(c, var[p], a);
  ga[p] = make_float4(a[0], a[1], a[2], 0.0f);
  gn[p] = make_float4(normal[i], normal[i + 1], normal[i + 2], 0.0f);
}
// one à-trous level with tap spacing `step`: xv -> out
__global__ void __launch_bounds__(kAtrousBlockX * kAtrousBlockY) k_atrous(const float4 *__restrict__ xv, const float4 *__restrict__ ga,
                                                                          const float4 *__restrict__ gn, int32_t width, int32_t height,
                                                                          int32_t step, DenoiseParams dp, float4 *__restrict__ out) {
  const int x = (int)(blockIdx.x * blockDim.x + threadIdx.x), y = (int)(blockIdx.y * blockDim.y + threadIdx.y);
  if (x >= width || y >= height) return;
  out[(size_t)y * (size_t)width + (size_t)x] = denoise_atrous_pixel(xv, ga, gn, width, height, x, y, step, dp);
}
// the last level's x remodulated (a non-finite pixel: its noisy value) -> rgb, and resolve_pixel of it at scale 1 -> packed
// (either may be nullptr)
__global__ void k_denoise_finish(const float4 *__restrict__ xv, const float *__restrict__ noisy, const float *__restrict__ albedo,
                                 uint32_t n_pixels, float *rgb, uint32_t *packed) {
  const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_pixels) return;
  const size_t i = (size_t)p * 3;
  const float c[3] = {noisy[i], noisy[i + 1], noisy[i + 2]}, a[3] = {albedo[i], albedo[i + 1], albedo[i + 2]};
  float o[3];
  denoise_remodulate(xv[p], c, a, o);
  if (rgb) rgb[i] = o[0], rgb[i + 1] = o[1], rgb[i + 2] = o[2];
  if (packed) packed[p] = resolve_pixel(o[0], o[1], o[2]);
}

}  // namespace ptw
