// motionsim.cpp — TEST-ONLY host compilation of the motion-blur functions (ptc_scene_set_object_motion /
// ptc_scene_set_camera_motion): camera_at and the per-object shifted scan of pt_bsdf.h / pt_prims.h, compiled by g++ into
// libhostsim.so next to hostsim.cpp.  Exports `sim_camera_at`, `sim_primary_rays_motion` and `sim_intersect_motion`
// only; the product never links or loads it.
#include <cstdint>
#include <cstring>

#include "../../include/ptcore.h"
#include "../../raytracer-rust_b200/csrc/pt_bsdf.h"
#include "../../raytracer-rust_b200/csrc/pt_philox.h"
#include "../../raytracer-rust_b200/csrc/pt_prims.h"

using namespace pt;

struct sim_scene;

extern "C" {

const DScene *sim_scene_dscene(const sim_scene *s);  // hostsim.cpp

// the camera at shutter time tau
int sim_camera_at(const ptc_camera *c0, const ptc_camera *c1, float tau, ptc_camera *out) {
  DCamera a, b;
  memcpy(&a, c0, sizeof(a));
  memcpy(&b, c1, sizeof(b));
  const DCamera c = camera_at(a, b, tau);
  memcpy(out, &c, sizeof(c));
  return 0;
}

// ptc_primary_rays under camera motion: the jitter (block 0), tau (block 1), the camera at tau, then the thin lens (R, F)
// (R == 0: the pinhole); out_tau receives tau
int sim_primary_rays_motion(const ptc_camera *cam, const ptc_camera *end, const ptc_render_settings *st, int32_t sample, float R,
                            float F, float *out_o, float *out_d, float *out_tau) {
  DCamera c0, c1;
  memcpy(&c0, cam, sizeof(c0));
  memcpy(&c1, end, sizeof(c1));
  for (int y = 0; y < st->height; y++)
    for (int x = 0; x < st->width; x++) {
      const uint32_t pixel = (uint32_t)(y * st->width + x);
      const Uniforms4 j = philox_uniforms(st->seed, pixel, (uint32_t)sample, 0xffffffffu, 0u);
      const float tau = philox_uniforms(st->seed, pixel, (uint32_t)sample, 0xffffffffu, 1u).u[0];
      const float u = ((float)x + j.u[0]) / (float)st->width;
      const float v = ((float)y + j.u[1]) / (float)st->height;
      const Ray r = camera_get_ray_lens(camera_at(c0, c1, tau), R, F, u, v, j.u[2], j.u[3]);
      out_o[pixel * 3 + 0] = r.o.x, out_o[pixel * 3 + 1] = r.o.y, out_o[pixel * 3 + 2] = r.o.z;
      out_d[pixel * 3 + 0] = r.d.x, out_d[pixel * 3 + 1] = r.d.y, out_d[pixel * 3 + 2] = r.d.z;
      out_tau[pixel] = tau;
    }
  return 0;
}

// HittableList::hit at shutter times: object k (displacement disp[3k .. 3k + 2]) on the ray shifted by -tau D_k, in list
// order with a shrinking closest (strict <, each primitive's own interval), its hit moved by +tau D_k; a static object
// on the ray itself.  The straight-line statement of what k_extend_pre_motion / k_traverse / k_extend_post_motion do.
int sim_intersect_motion(const sim_scene *s, const float *disp, const float *origins, const float *dirs, const float *times,
                         int64_t n, float t_min, float t_max, ptc_hit *out) {
  const DScene *sc = sim_scene_dscene(s);
  if (!sc) return -4;
  for (int64_t i = 0; i < n; i++) {
    const Ray ray{v3(origins[i * 3], origins[i * 3 + 1], origins[i * 3 + 2]), v3(dirs[i * 3], dirs[i * 3 + 1], dirs[i * 3 + 2])};
    const float tau = times[i];
    float closest = t_max;
    Hit best;
    memset(&best, 0, sizeof(best));
    bool any = false;
    for (int k = 0; k < sc->n_objects; k++) {
      const DObject *ob = sc->objects + k;
      float4 D;
      D.x = disp[k * 3], D.y = disp[k * 3 + 1], D.z = disp[k * 3 + 2], D.w = 0.0f;
      const bool moves = motion_moves(D);
      const Ray r = moves ? motion_object_ray(ray, tau, D) : ray;
      Hit tmp;
      tmp.triangle = -1;
      bool hit;
      if (ob->type == OBJ_SPHERE) hit = hit_sphere(ob->f, r, t_min, closest, tmp);
      else if (ob->type == OBJ_QUAD) hit = hit_quad(ob->f, r, t_min, closest, tmp);
      else if (ob->type == OBJ_CUBE) hit = hit_cube(ob->f, r, t_min, closest, tmp);
      else if (ob->type == OBJ_MESH) hit = hit_mesh<false>(ob->f, sc->meshes[ob->mesh], r, t_min, closest, tmp, nullptr);
      else hit = hit_plane(ob->f, r, t_min, closest, tmp);
      if (hit) {
        if (moves) motion_hit_position(tmp, tau, D);
        any = true;
        closest = tmp.t;
        best = tmp;
        best.object = k;
        best.material = ob->material;
      }
    }
    ptc_hit &o = out[i];
    memset(&o, 0, sizeof(o));
    if (any) {
      o.object = best.object;
      o.triangle = best.triangle;
      o.t = best.t;
      o.position[0] = best.px, o.position[1] = best.py, o.position[2] = best.pz;
      o.normal[0] = best.nx, o.normal[1] = best.ny, o.normal[2] = best.nz;
      o.front_face = best.front_face;
      o.material = best.material;
    } else {
      o.object = -1, o.triangle = -1, o.material = -1;
    }
  }
  return 0;
}

}  // extern "C"
