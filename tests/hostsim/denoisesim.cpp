// denoisesim.cpp — TEST-ONLY host compilation of the denoiser (ptc_render_denoised, ptc_denoise_image): the per-pixel
// functions of pt_denoise.h, compiled by g++ into libhostsim.so next to hostsim.cpp, driven the way the device kernels
// drive them (k_feature_add, k_denoise_variance, k_denoise_prepare, k_atrous, k_denoise_finish).  Exports
// `denoise_sim_*` symbols only; the product never links or loads it.
#include <cstdint>
#include <vector>

#include "../../include/ptcore.h"
#include "../../raytracer-rust_b200/csrc/pt_denoise.h"
#include "../../raytracer-rust_b200/csrc/pt_scene_host.h"

using namespace pt;

extern "C" {

// feature_albedo of n first hits: mats = the scene's materials (as added), mat[i] = the hit's material index or -1 for a
// miss (albedo 1), pos = n x 3 hit points; out = n x 3
int32_t denoise_sim_feature_albedo(const ptc_material *mats, int32_t n_mats, const int32_t *mat, const float *pos, int64_t n, float *out) {
  HostScene hs;
  for (int32_t k = 0; k < n_mats; k++) hs.add_material(&mats[k]);
  for (int64_t i = 0; i < n; i++) {
    V3 a = v3(1.0f, 1.0f, 1.0f);
    if (mat[i] >= 0) {
      if (mat[i] >= n_mats) return -1;
      a = feature_albedo(hs.materials[(size_t)mat[i]], v3(pos[i * 3], pos[i * 3 + 1], pos[i * 3 + 2]));
    }
    out[i * 3] = a.x, out[i * 3 + 1] = a.y, out[i * 3 + 2] = a.z;
  }
  return 0;
}

// denoise_variance of n pixels: Sh, Sn = n x 3 fp32 film sums after samples [0, h) and [0, spp), albedo n x 3
void denoise_sim_variance(const float *Sh, const float *Sn, int64_t n, int32_t h, int32_t spp, const float *albedo, float *out) {
  for (int64_t i = 0; i < n; i++) out[i] = denoise_variance(Sh + i * 3, Sn + i * 3, h, spp, albedo + i * 3);
}

// The whole filter on a width x height frame, as ptc_denoise_image runs it: rgb, albedo, normal W*H*3, var W*H ->
// out W*H*3.  iterations 1..kDenoiseMaxIterations.
void denoise_sim_filter(int32_t width, int32_t height, const float *rgb, const float *var, const float *albedo, const float *normal,
                        int32_t iterations, float sigma_luminance, float sigma_normal, float sigma_albedo, float *out) {
  const size_t n_px = (size_t)width * (size_t)height;
  std::vector<float4> xv[2] = {std::vector<float4>(n_px), std::vector<float4>(n_px)};
  std::vector<float4> ga(n_px), gn(n_px);
  for (size_t p = 0; p < n_px; p++) {
    xv[0][p] = denoise_demodulate(rgb + p * 3, var[p], albedo + p * 3);
    ga[p] = make_float4(albedo[p * 3], albedo[p * 3 + 1], albedo[p * 3 + 2], 0.0f);
    gn[p] = make_float4(normal[p * 3], normal[p * 3 + 1], normal[p * 3 + 2], 0.0f);
  }
  const DenoiseParams dp = denoise_params(sigma_luminance, sigma_normal, sigma_albedo);
  for (int i = 0; i < iterations; i++) {
    const std::vector<float4> &src = xv[i & 1];
    std::vector<float4> &dst = xv[(i + 1) & 1];
    for (int y = 0; y < height; y++)
      for (int x = 0; x < width; x++)
        dst[(size_t)y * width + x] = denoise_atrous_pixel(src.data(), ga.data(), gn.data(), width, height, x, y, 1 << i, dp);
  }
  const std::vector<float4> &fin = xv[iterations & 1];
  for (size_t p = 0; p < n_px; p++) denoise_remodulate(fin[p], rgb + p * 3, albedo + p * 3, out + p * 3);
}

}  // extern "C"
