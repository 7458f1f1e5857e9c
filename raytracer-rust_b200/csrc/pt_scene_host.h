// pt_scene_host.h — host-side scene under construction: what the add_* calls of include/ptcore.h collect before
// ptc_scene_commit flattens it (object table in Scene.object_list order, material table, one MeshBuild per Mesh).
#pragma once
#include <algorithm>
#include <cmath>
#include <cstring>
#include <memory>
#include <stdexcept>
#include <vector>

#include "../../include/ptcore.h"
#include "pt_build.h"
#include "pt_types.h"

namespace pt {

// The one place that fills a DMesh, so the CUDA upload and the hostsim harness cannot drift apart.
inline DMesh make_dmesh(const MeshBuild &m, const float4 *nodes, const float4 *tris, const float4 *normals) {
  DMesh d;
  d.nodes = nodes;
  d.tris = tris;
  d.normals = normals;
  d.n_nodes = (int32_t)m.nodes.size();
  d.n_tris = (int32_t)m.tri48.size();
  for (int a = 0; a < 3; a++) d.root_lo[a] = m.root_lo[a], d.root_hi[a] = m.root_hi[a];
  return d;
}

struct HostScene {
  std::vector<DMaterial> materials;
  std::vector<DObject> objects;
  std::vector<std::unique_ptr<MeshBuild>> meshes;
  std::vector<float> sky;
  int32_t sky_w = 0, sky_h = 0;
  std::vector<DLight> lights;  // filled by build_all
  std::vector<float> sky_dist;  // filled by build_all: SkyDist of the sky, or empty

  int add_material(const ptc_material *m) {
    if (m->type < PTC_MAT_LAMBERT || m->type > PTC_MAT_NULL) throw std::invalid_argument("unknown material type");
    DMaterial d;
    memset(&d, 0, sizeof(d));
    d.type = m->type;
    d.distribution = m->distribution;
    d.fuzz = m->fuzz;
    d.ior = m->ior;
    d.roughness = m->roughness;
    d.inv_scale = m->inv_scale;
    for (int i = 0; i < 3; i++) {
      d.albedo[i] = m->albedo[i];
      d.off_color[i] = m->off_color[i];
      d.eta[i] = m->eta[i];
      d.k[i] = m->k[i];
    }
    materials.push_back(d);
    return (int)materials.size() - 1;
  }
  void check_material(int material) const {
    if (material < 0 || (size_t)material >= materials.size()) throw std::invalid_argument("material index out of range");
  }
  DObject blank(int32_t type, int material) const {
    check_material(material);
    DObject o;
    memset(&o, 0, sizeof(o));
    o.type = type;
    o.material = material;
    o.mesh = -1;
    return o;
  }
  int add_sphere(const float c[3], float radius, int material) {
    // Sphere::hit divides by the radius through Vec3's Div<f32>, which PANICS for |radius| < 1e-4 (src/vec3.rs:117-122,
    // src/objects/sphere.rs:45): the reference's render aborts at the first hit of such a sphere.  Nothing may unwind
    // across this boundary, so the sphere is refused when it is added.
    if (!(std::fabs(radius) >= 1e-4f)) throw std::invalid_argument("sphere radius below 1e-4: a hit would panic in the reference (vec3.rs:117-122)");
    DObject o = blank(OBJ_SPHERE, material);
    o.f[0] = c[0], o.f[1] = c[1], o.f[2] = c[2], o.f[3] = radius;
    objects.push_back(o);
    return (int)objects.size() - 1;
  }
  int add_plane(const float p1[3], const float n[3], int material) {
    DObject o = blank(OBJ_PLANE, material);
    for (int i = 0; i < 3; i++) o.f[i] = p1[i], o.f[3 + i] = n[i];
    objects.push_back(o);
    return (int)objects.size() - 1;
  }
  int add_quad(const float base[3], const float e0[3], const float e1[3], const float n[3], float d, float inv0,
               float inv1, int material) {
    DObject o = blank(OBJ_QUAD, material);
    for (int i = 0; i < 3; i++) o.f[i] = base[i], o.f[3 + i] = e0[i], o.f[6 + i] = e1[i], o.f[9 + i] = n[i];
    o.f[12] = d, o.f[13] = inv0, o.f[14] = inv1;
    objects.push_back(o);
    return (int)objects.size() - 1;
  }
  int add_cube(const float o2w[16], const float w2o[16], int material) {
    DObject o = blank(OBJ_CUBE, material);
    for (int i = 0; i < 16; i++) o.f[i] = w2o[i], o.f[16 + i] = o2w[i];
    objects.push_back(o);
    return (int)objects.size() - 1;
  }
  int add_mesh(const float *tris, int64_t n, const float o2w[16], const float w2o[16], int material) {
    if (n <= 0 || tris == nullptr) throw std::invalid_argument("mesh without triangles (mesh_object.rs:30-36)");
    DObject o = blank(OBJ_MESH, material);
    for (int i = 0; i < 16; i++) o.f[i] = w2o[i], o.f[16 + i] = o2w[i];
    auto mb = std::make_unique<MeshBuild>();
    mb->n = n;
    mb->tris.assign(tris, tris + (size_t)n * 12);
    o.mesh = (int32_t)meshes.size();
    meshes.push_back(std::move(mb));
    objects.push_back(o);
    return (int)objects.size() - 1;
  }
  void set_sky(const float *rgb, int32_t w, int32_t h) {
    if (w <= 0 || h <= 0 || rgb == nullptr) throw std::invalid_argument("bad sky image");
    sky.assign(rgb, rgb + (size_t)w * h * 3);
    sky_w = w;
    sky_h = h;
  }
  void build_all() {
    for (auto &m : meshes)
      if (!m->built) build_mesh(*m);
    for (auto &m : meshes)
      if (m->wide_depth + 2 > kTraversalStack) throw std::runtime_error("wide BVH deeper than the traversal stack");
    if (materials.size() > (size_t)1 << 20) throw std::runtime_error("more than 2^20 materials");
    // emitters next-event estimation can sample: emissive spheres and quads, in object order
    lights.clear();
    for (size_t k = 0; k < objects.size(); k++) {
      DObject &o = objects[k];
      const DMaterial &m = materials[(size_t)o.material];
      int32_t light_id = 0;
      const bool emits = m.type == PTC_MAT_EMISSIVE && (m.albedo[0] != 0.0f || m.albedo[1] != 0.0f || m.albedo[2] != 0.0f);
      if (emits && (o.type == OBJ_SPHERE || o.type == OBJ_QUAD) && (int)lights.size() < kMaxLights) {
        DLight l;
        memset(&l, 0, sizeof(l));
        l.type = o.type, l.object = (int32_t)k;
        if (o.type == OBJ_SPHERE) {
          for (int i = 0; i < 4; i++) l.f[i] = o.f[i];
          l.area = 4.0f * 3.14159265358979323846f * o.f[3] * o.f[3];
        } else {
          for (int i = 0; i < 12; i++) l.f[i] = o.f[i];
          const float *a = o.f + 3, *b = o.f + 6;
          const float cx = a[1] * b[2] - a[2] * b[1], cy = a[2] * b[0] - a[0] * b[2], cz = a[0] * b[1] - a[1] * b[0];
          l.area = std::sqrt(cx * cx + cy * cy + cz * cz);
        }
        for (int i = 0; i < 3; i++) l.emission[i] = m.albedo[i];
        if (l.area > 0.0f) {
          lights.push_back(l);
          light_id = (int32_t)lights.size();
        }
      }
      o.hit_bits = (m.type << 26) | (light_id << 20) | o.material;
    }
    build_sky_dist();
  }
  // the sky as a light (PTC_FLAG_NEE_SKY, layout in pt_types.h: SkyDist): cell weight = max(r, g, b) x solid angle, summed
  // in double in a fixed order; left empty without a sky or when every weight is 0
  void build_sky_dist() {
    sky_dist.clear();
    if (sky.empty()) return;
    const int32_t wc = sky_cells(sky_w), hc = sky_cells(sky_h);
    std::vector<float> d(sky_dist_size(sky_w, sky_h));
    const SkyDist v = sky_dist_view(d.data(), sky_w, sky_h);
    float *marg = d.data(), *cosv = marg + (v.cos - v.marg), *inv_sa = marg + (v.inv_sa - v.marg), *cond = marg + (v.cond - v.marg);
    const double pi = 3.14159265358979323846;
    std::vector<double> row_w((size_t)hc), cum((size_t)wc + 1);
    double total = 0.0;
    for (int32_t y = 0; y < hc; y++) {
      const double c0 = std::cos(pi * y / hc), c1 = std::cos(pi * (y + 1) / hc);
      const double sa = 2.0 * pi / wc * (c0 - c1);
      cosv[y] = (float)c0;
      inv_sa[y] = (float)(1.0 / sa);
      cum[0] = 0.0;
      for (int32_t x = 0; x < wc; x++) {
        const float *px = sky.data() + ((size_t)y * sky_w + x) * 3;
        double wgt = 0.0;
        if (!std::isnan(px[0]) && !std::isnan(px[1]) && !std::isnan(px[2])) {
          wgt = (double)std::max(px[0], std::max(px[1], px[2])) * sa;
          if (!std::isfinite(wgt) || wgt < 0.0) wgt = 0.0;
        }
        cum[(size_t)x + 1] = cum[(size_t)x] + wgt;
      }
      const double rw = cum[(size_t)wc];
      float *row = cond + (size_t)y * (size_t)(wc + 1);
      for (int32_t x = 0; x < wc; x++) row[x] = rw > 0.0 ? (float)(cum[(size_t)x] / rw) : (float)x / (float)wc;
      row[wc] = 1.0f;
      row_w[(size_t)y] = rw;
      total += rw;
    }
    cosv[hc] = -1.0f;
    if (!(total > 0.0) || !std::isfinite(total)) return;
    double c = 0.0;
    for (int32_t y = 0; y < hc; y++) {
      marg[y] = (float)(c / total);
      c += row_w[(size_t)y];
    }
    marg[hc] = 1.0f;
    sky_dist = std::move(d);
  }
};

}  // namespace pt
