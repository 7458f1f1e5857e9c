// emsim.cpp — TEST-ONLY host compilation of PTC_FLAG_NEE_EMITTERS: the tables HostScene::build_emitters builds, the
// emitter_sample / emitter_mis_pdf device functions of pt_bsdf.h, and the closest hit of pt_prims.h, compiled by g++ into
// libhostsim.so next to hostsim.cpp.  An em_sim holds a scene flattened exactly as ptc_scene_commit flattens it.
// Exports `em_sim_*` symbols only; the product never links or loads it.
#include <cstdint>
#include <cstring>
#include <string>

#include "../../raytracer-rust_b200/csrc/pt_bsdf.h"
#include "../../raytracer-rust_b200/csrc/pt_prims.h"
#include "../../raytracer-rust_b200/csrc/pt_scene_host.h"

using namespace pt;

struct em_sim {
  HostScene hs;
  std::vector<DMesh> dmeshes;
  DScene ds;  // ds_em of ptcore.cu: the object table and the light list of the mode
  EmitterTables et;
};

extern "C" {

em_sim *em_sim_scene_create(void) { return new em_sim(); }
void em_sim_scene_destroy(em_sim *s) { delete s; }

#define EM_TRY(expr)             \
  try {                          \
    return (expr);               \
  } catch (std::exception & e) { \
    return -1;                   \
  }
int em_sim_scene_add_material(em_sim *s, const ptc_material *m) { EM_TRY(s->hs.add_material(m)) }
int em_sim_scene_add_sphere(em_sim *s, const float c[3], float r, int mat) { EM_TRY(s->hs.add_sphere(c, r, mat)) }
int em_sim_scene_add_plane(em_sim *s, const float p[3], const float n[3], int mat) { EM_TRY(s->hs.add_plane(p, n, mat)) }
int em_sim_scene_add_quad(em_sim *s, const float b[3], const float e0[3], const float e1[3], const float n[3], float d, float i0,
                          float i1, int mat) {
  EM_TRY(s->hs.add_quad(b, e0, e1, n, d, i0, i1, mat))
}
int em_sim_scene_add_cube(em_sim *s, const float o2w[16], const float w2o[16], int mat) { EM_TRY(s->hs.add_cube(o2w, w2o, mat)) }
int em_sim_scene_add_mesh(em_sim *s, const float *tris, int64_t n, const float o2w[16], const float w2o[16], int mat) {
  EM_TRY(s->hs.add_mesh(tris, n, o2w, w2o, mat))
}
int em_sim_scene_set_sky_hdr(em_sim *s, const float *rgb, int32_t w, int32_t h) {
  try {
    s->hs.set_sky(rgb, w, h);
    return 0;
  } catch (std::exception &) {
    return -1;
  }
}

int em_sim_commit(em_sim *s) {
  try {
    s->hs.build_all();
    s->dmeshes.clear();
    for (auto &m : s->hs.meshes)
      s->dmeshes.push_back(make_dmesh(*m, reinterpret_cast<const float4 *>(m->nodes.data()),
                                      reinterpret_cast<const float4 *>(m->tri48.data()), m->normals.data()));
    memset(&s->ds, 0, sizeof(s->ds));
    s->ds.objects = s->hs.objects_em.data();
    s->ds.materials = s->hs.materials.data();
    s->ds.meshes = s->dmeshes.data();
    s->ds.lights = s->hs.lights_em.data();
    s->ds.n_lights = (int32_t)s->hs.lights_em.size();
    s->ds.n_objects = (int32_t)s->hs.objects_em.size();
    s->ds.n_materials = (int32_t)s->hs.materials.size();
    s->ds.n_meshes = (int32_t)s->dmeshes.size();
    s->et = EmitterTables{s->hs.em_sel_cdf.data(), s->hs.em_ent.data(), s->hs.em_ent_cdf.data()};
    return 0;
  } catch (std::exception &) {
    return -1;
  }
}

// the light list: n lights; per light (type, object, entry count), area, and the selection CDF [n + 1]
int32_t em_sim_lights(const em_sim *s, int32_t *type_obj_count, float *area, float *sel_cdf) {
  const int32_t n = (int32_t)s->hs.lights_em.size();
  for (int32_t k = 0; k < n && type_obj_count; k++) {
    const DLight &L = s->hs.lights_em[(size_t)k];
    uint32_t count = 0;
    if (emitter_area_sampled(L)) memcpy(&count, &L.f[1], 4);
    type_obj_count[k * 3] = L.type, type_obj_count[k * 3 + 1] = L.object, type_obj_count[k * 3 + 2] = (int32_t)count;
    area[k] = L.area;
  }
  if (sel_cdf && n) memcpy(sel_cdf, s->hs.em_sel_cdf.data(), (size_t)(n + 1) * 4);
  return n;
}
// light k's entry CDF ([count + 1]) and entries (count x 12 floats: v0, nrec.x, e1, nrec.y, e2, nrec.z); -1 for other lights
int64_t em_sim_entries(const em_sim *s, int32_t k, float *cdf, float *ent) {
  if (k < 0 || (size_t)k >= s->hs.lights_em.size() || !emitter_area_sampled(s->hs.lights_em[(size_t)k])) return -1;
  const DLight &L = s->hs.lights_em[(size_t)k];
  uint32_t first, count, coff;
  memcpy(&first, &L.f[0], 4), memcpy(&count, &L.f[1], 4), memcpy(&coff, &L.f[2], 4);
  if (cdf) memcpy(cdf, s->hs.em_ent_cdf.data() + coff, ((size_t)count + 1) * 4);
  if (ent) memcpy(ent, s->hs.em_ent.data() + (size_t)first * 3, (size_t)count * 48);
  return (int64_t)count;
}
// the hit bits' light id of every object in the mode's object table
void em_sim_light_ids(const em_sim *s, int32_t *ids) {
  for (size_t k = 0; k < s->hs.objects_em.size(); k++) ids[k] = (s->hs.objects_em[k].hit_bits >> 20) & 63;
}

// what ptc_light_sample / ptc_light_pdf compute on the device; -4 (PTC_E_STATE) without a sampled emitter.  The pdf's
// closest hit is pt_prims.h's straight-line scene_hit over the same object table (t_min as the renderer's, 1e-4).
int em_sim_sample(const em_sim *s, const float *x, const float *u4, int64_t n, float *point, float *pdf, float *pmis, int32_t *object,
                  int32_t *triangle) {
  if (s->ds.n_lights == 0) return -4;
  for (int64_t i = 0; i < n; i++) {
    const V3 xi = v3(x[i * 3], x[i * 3 + 1], x[i * 3 + 2]);
    const float *u = u4 + i * 4;
    EmitterSample es;
    const bool ok = emitter_sample(s->ds, s->et, xi, u[0], u[1], u[2], u[3], es);
    const V3 y = ok ? xi + es.wi * es.dist : v3(0, 0, 0);
    point[i * 3] = y.x, point[i * 3 + 1] = y.y, point[i * 3 + 2] = y.z;
    pdf[i] = ok ? es.pdf : 0.0f;
    pmis[i] = ok ? es.pmis : 0.0f;
    object[i] = ok ? s->ds.lights[es.light].object : -1;
    triangle[i] = ok && s->ds.lights[es.light].type == OBJ_MESH ? es.entry : -1;
  }
  return 0;
}
int em_sim_pdf(const em_sim *s, const float *o, const float *d, int64_t n, float *pdf) {
  if (s->ds.n_lights == 0) return -4;
  for (int64_t i = 0; i < n; i++) {
    const Ray ray{v3(o[i * 3], o[i * 3 + 1], o[i * 3 + 2]), v3(d[i * 3], d[i * 3 + 1], d[i * 3 + 2])};
    Hit h;
    float p = 0.0f;
    if (scene_hit<false>(s->ds, ray, kEps, INFINITY, h, nullptr)) {
      const uint32_t light = ((uint32_t)s->ds.objects[h.object].hit_bits >> 20) & 63u;
      if (light != 0u) {
        const DLight &L = s->ds.lights[light - 1u];
        const V3 pos = v3(h.px, h.py, h.pz);
        const float dl = emitter_area_sampled(L) ? length(pos - ray.o) : h.t;
        p = emitter_mis_pdf(L, emitter_select_prob(s->et, light - 1u), dl, fabsf(dot(v3(h.nx, h.ny, h.nz), normalized(ray.d))));
      }
    }
    pdf[i] = p;
  }
  return 0;
}

}  // extern "C"
