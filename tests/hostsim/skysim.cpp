// skysim.cpp — TEST-ONLY host compilation of the sky-as-a-light code (PTC_FLAG_NEE_SKY): the tables HostScene::build_all
// builds and the sky_sample / sky_pdf device functions of pt_bsdf.h, compiled by g++ into libhostsim.so next to
// hostsim.cpp.  A sky_sim holds a scene with nothing but its HDR sky, flattened exactly as ptc_scene_commit flattens it.
// Exports `sky_sim_*` symbols only; the product never links or loads it.
#include <cstdint>
#include <cstring>
#include <string>

#include "../../raytracer-rust_b200/csrc/pt_bsdf.h"
#include "../../raytracer-rust_b200/csrc/pt_scene_host.h"

using namespace pt;

struct sky_sim {
  HostScene hs;
  DScene ds;
};

extern "C" {

// nullptr when the sky image is refused (see HostScene::set_sky)
sky_sim *sky_sim_create(const float *rgb, int32_t w, int32_t h) {
  try {
    sky_sim *s = new sky_sim();
    s->hs.set_sky(rgb, w, h);
    s->hs.build_all();
    memset(&s->ds, 0, sizeof(s->ds));
    s->ds.sky = s->hs.sky.data();
    s->ds.sky_w = s->hs.sky_w;
    s->ds.sky_h = s->hs.sky_h;
    s->ds.sky_dist = s->hs.sky_dist.empty() ? nullptr : s->hs.sky_dist.data();
    return s;
  } catch (std::exception &) {
    return nullptr;
  }
}
void sky_sim_destroy(sky_sim *s) { delete s; }

// the tables as built (SkyDist layout, pt_types.h): their size in floats (0 = no distribution), copied to `out` if given
int64_t sky_sim_dist(const sky_sim *s, float *out) {
  if (out) memcpy(out, s->hs.sky_dist.data(), s->hs.sky_dist.size() * sizeof(float));
  return (int64_t)s->hs.sky_dist.size();
}

// what ptc_sky_sample / ptc_sky_pdf compute on the device; -4 (PTC_E_STATE) without a distribution
int sky_sim_sample(const sky_sim *s, const float *u4, int64_t n, float *out_dir, float *out_pdf, float *out_rgb) {
  if (!s->ds.sky_dist) return -4;
  for (int64_t i = 0; i < n; i++) {
    const V3 d = sky_sample(s->ds, u4 + i * 4, out_pdf[i]);
    const V3 c = sky_color(s->ds, d);
    out_dir[i * 3] = d.x, out_dir[i * 3 + 1] = d.y, out_dir[i * 3 + 2] = d.z;
    out_rgb[i * 3] = c.x, out_rgb[i * 3 + 1] = c.y, out_rgb[i * 3 + 2] = c.z;
  }
  return 0;
}
int sky_sim_pdf(const sky_sim *s, const float *dirs, int64_t n, float *out_pdf) {
  if (!s->ds.sky_dist) return -4;
  for (int64_t i = 0; i < n; i++) out_pdf[i] = sky_pdf(s->ds, v3(dirs[i * 3], dirs[i * 3 + 1], dirs[i * 3 + 2]));
  return 0;
}

}  // extern "C"
