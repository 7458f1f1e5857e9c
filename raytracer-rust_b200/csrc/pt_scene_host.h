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
#include "pt_math.h"
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
    build_emitters();
  }
  // PTC_FLAG_NEE_EMITTERS (layout in pt_types.h: EmitterTables): the first kMaxLights emissive spheres, quads, cubes and
  // meshes of finite positive power max(r, g, b) x area, in object order, and a copy of the object table whose hit_bits
  // carry these light ids.  Areas and weights are summed in double in a fixed order, then stored as float CDFs.
  std::vector<DObject> objects_em;
  std::vector<DLight> lights_em;
  std::vector<float> em_sel_cdf;  // [lights_em.size() + 1], or empty
  std::vector<float4> em_ent;
  std::vector<float> em_ent_cdf;
  void build_emitters() {
    objects_em = objects;
    lights_em.clear(), em_sel_cdf.clear(), em_ent.clear(), em_ent_cdf.clear();
    std::vector<double> power, area;
    std::vector<double> ent_area;
    for (size_t k = 0; k < objects.size(); k++) {
      DObject &o = objects_em[k];
      const DMaterial &m = materials[(size_t)o.material];
      o.hit_bits &= ~(63 << 20);
      if (m.type != PTC_MAT_EMISSIVE || o.type == OBJ_PLANE || (int)lights_em.size() >= kMaxLights) continue;
      // every channel finite (std::max would drop a NaN in the second argument), the largest positive
      if (!std::isfinite(m.albedo[0]) || !std::isfinite(m.albedo[1]) || !std::isfinite(m.albedo[2])) continue;
      const double radiance = std::max((double)m.albedo[0], std::max((double)m.albedo[1], (double)m.albedo[2]));
      if (!(radiance > 0.0)) continue;
      DLight l;
      memset(&l, 0, sizeof(l));
      l.type = o.type, l.object = (int32_t)k;
      for (int i = 0; i < 3; i++) l.emission[i] = m.albedo[i];
      double a = 0.0;
      const size_t first = em_ent.size() / 3;
      ent_area.clear();
      if (o.type == OBJ_SPHERE || o.type == OBJ_QUAD) {  // as in the PTC_FLAG_NEE list
        if (o.type == OBJ_SPHERE) {
          for (int i = 0; i < 4; i++) l.f[i] = o.f[i];
          l.area = 4.0f * 3.14159265358979323846f * o.f[3] * o.f[3];
        } else {
          for (int i = 0; i < 12; i++) l.f[i] = o.f[i];
          const float *ea = o.f + 3, *eb = o.f + 6;
          const float cx = ea[1] * eb[2] - ea[2] * eb[1], cy = ea[2] * eb[0] - ea[0] * eb[2], cz = ea[0] * eb[1] - ea[1] * eb[0];
          l.area = std::sqrt(cx * cx + cy * cy + cz * cz);
        }
        a = l.area;
      } else {
        const float *w2o = o.f, *o2w = o.f + 16;
        auto push = [&](V3 v0, V3 e1, V3 e2, V3 n_obj, double scale, bool live) {
          const V3 nrec = normalized(mat_t_vector(w2o, n_obj));
          em_ent.push_back(make_float4(v0.x, v0.y, v0.z, nrec.x));
          em_ent.push_back(make_float4(e1.x, e1.y, e1.z, nrec.y));
          em_ent.push_back(make_float4(e2.x, e2.y, e2.z, nrec.z));
          const double cx = (double)e1.y * e2.z - (double)e1.z * e2.y, cy = (double)e1.z * e2.x - (double)e1.x * e2.z,
                       cz = (double)e1.x * e2.y - (double)e1.y * e2.x;
          const double ar = live ? scale * std::sqrt(cx * cx + cy * cy + cz * cz) : 0.0;
          ent_area.push_back(std::isfinite(ar) ? ar : 0.0);
        };
        if (o.type == OBJ_CUBE) {  // faces of [-0.5, 0.5]^3: +-x, +-y, +-z, each base + two unit edges
          for (int ax = 0; ax < 3; ax++)
            for (int sgn = 0; sgn < 2; sgn++) {
              float b[3] = {-0.5f, -0.5f, -0.5f}, u[3] = {0, 0, 0}, v[3] = {0, 0, 0}, n[3] = {0, 0, 0};
              b[ax] = sgn ? 0.5f : -0.5f;
              u[(ax + 1) % 3] = 1.0f, v[(ax + 2) % 3] = 1.0f, n[ax] = sgn ? 1.0f : -1.0f;
              push(mat_point(o2w, v3(b[0], b[1], b[2])), mat_vector(o2w, v3(u[0], u[1], u[2])), mat_vector(o2w, v3(v[0], v[1], v[2])),
                   v3(n[0], n[1], n[2]), 1.0, true);
            }
        } else {  // every triangle in original order; a dead one (never hit) with weight 0
          const MeshBuild &mb = *meshes[(size_t)o.mesh];
          for (int64_t t = 0; t < mb.n; t++) {
            const float *q = mb.tris.data() + (size_t)t * 12;
            const V3 v0 = mat_point(o2w, v3(q[0], q[1], q[2]));
            const V3 e1 = mat_point(o2w, v3(q[3], q[4], q[5])) - v0, e2 = mat_point(o2w, v3(q[6], q[7], q[8])) - v0;
            push(v0, e1, e2, v3(q[9], q[10], q[11]), 0.5, !mb.dead[(size_t)t]);
          }
        }
        for (double x : ent_area) a += x;
        l.area = (float)a;
      }
      const double pw = radiance * a;
      if (!(a > 0.0) || !(l.area > 0.0f) || !std::isfinite(pw) || !std::isfinite(l.area)) {
        em_ent.resize(first * 3);
        continue;
      }
      if (o.type == OBJ_CUBE || o.type == OBJ_MESH) {
        // (DLight holds 32-bit offsets: entry and CDF tables of at most 2^32 - 1 floats each)
        if (em_ent.size() / 3 > 0xffffffffull || em_ent_cdf.size() + ent_area.size() + 1 > 0xffffffffull)
          throw std::runtime_error("emissive meshes too large for the PTC_FLAG_NEE_EMITTERS tables");
        const uint32_t first32 = (uint32_t)first, count = (uint32_t)ent_area.size(), coff = (uint32_t)em_ent_cdf.size();
        memcpy(&l.f[0], &first32, 4), memcpy(&l.f[1], &count, 4), memcpy(&l.f[2], &coff, 4);
        double c = 0.0;
        for (uint32_t i = 0; i < count; i++) {
          em_ent_cdf.push_back((float)(c / a));
          c += ent_area[i];
        }
        em_ent_cdf.push_back(1.0f);
      }
      lights_em.push_back(l);
      power.push_back(pw);
      o.hit_bits |= (int32_t)lights_em.size() << 20;
    }
    if (lights_em.empty()) return;
    double total = 0.0;
    for (double p : power) total += p;
    double c = 0.0;
    for (size_t i = 0; i < power.size(); i++) {
      em_sel_cdf.push_back((float)(c / total));
      c += power[i];
    }
    em_sel_cdf.push_back(1.0f);
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
