// lenssim.cpp — TEST-ONLY host compilation of the thin-lens camera (ptc_scene_set_lens): camera_get_ray_lens of
// pt_bsdf.h with the Philox jitter draw of ptc_primary_rays, compiled by g++ into libhostsim.so next to hostsim.cpp.
// Exports `sim_primary_rays_lens` only; the product never links or loads it.
#include <cstdint>
#include <cstring>

#include "../../include/ptcore.h"
#include "../../raytracer-rust_b200/csrc/pt_bsdf.h"
#include "../../raytracer-rust_b200/csrc/pt_philox.h"

using namespace pt;

extern "C" {

// ptc_primary_rays through the thin lens (R, F): u[0], u[1] of the jitter draw place the sample in the pixel, u[2], u[3]
// on the lens.  The first argument is unused (it mirrors sim_primary_rays, whose scene handle is unused too).
int sim_primary_rays_lens(void *, const ptc_camera *cam, const ptc_render_settings *st, int32_t sample, float R, float F,
                          float *out_o, float *out_d) {
  DCamera c;
  memcpy(&c, cam, sizeof(c));
  for (int y = 0; y < st->height; y++)
    for (int x = 0; x < st->width; x++) {
      const uint32_t pixel = (uint32_t)(y * st->width + x);
      const Uniforms4 j = philox_uniforms(st->seed, pixel, (uint32_t)sample, 0xffffffffu, 0u);
      const float u = ((float)x + j.u[0]) / (float)st->width;
      const float v = ((float)y + j.u[1]) / (float)st->height;
      const Ray r = camera_get_ray_lens(c, R, F, u, v, j.u[2], j.u[3]);
      out_o[pixel * 3 + 0] = r.o.x, out_o[pixel * 3 + 1] = r.o.y, out_o[pixel * 3 + 2] = r.o.z;
      out_d[pixel * 3 + 0] = r.d.x, out_d[pixel * 3 + 1] = r.d.y, out_d[pixel * 3 + 2] = r.d.z;
    }
  return 0;
}

}  // extern "C"
