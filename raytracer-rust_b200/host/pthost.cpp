// pthost.cpp — C++ stand-in for the reference's Rust host side (see include/pthost.h).  Plain host code: no CUDA,
// no oracle.  Each function cites the reference code whose behaviour it mirrors (paths under /root/reference).
#include "../../include/pthost.h"

#include <dlfcn.h>
#include <zlib.h>

#include <algorithm>
#include <cctype>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <map>
#include <sstream>
#include <string>
#include <type_traits>
#include <vector>

#include "json.hpp"

namespace {

thread_local std::string g_err;
constexpr float EPSILON = 1e-4f;  // renderer.rs:17
constexpr float PI_F = 3.14159265358979323846f;

struct V {
  float x, y, z;
};
V operator+(V a, V b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
V operator-(V a, V b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
V operator*(V a, float s) { return {a.x * s, a.y * s, a.z * s}; }
float dot(V a, V b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
V cross(V a, V b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
float len2(V a) { return a.x * a.x + a.y * a.y + a.z * a.z; }
V normalized(V a) {  // vec3.rs:37-44
  float l = std::sqrt(len2(a));
  if (l < EPSILON) return a;
  return a * (1.0f / l);
}

// ---- glam 0.30.3 restated (source not vendored with the reference: parity unpinned) -------------------------
struct Quat {
  float x, y, z, w;
};
Quat qmul(Quat a, Quat b) {  // glam Quat::mul_quat (scalar path)
  return {a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y, a.w * b.y - a.x * b.z + a.y * b.w + a.z * b.x,
          a.w * b.z + a.x * b.y - a.y * b.x + a.z * b.w, a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z};
}
Quat quat_from_euler_yxz(float a, float b, float c) {  // Quat::from_euler(EulerRot::YXZ, a, b, c) = Ry(a) * Rx(b) * Rz(c)
  Quat qy{0, std::sin(a * 0.5f), 0, std::cos(a * 0.5f)};
  Quat qx{std::sin(b * 0.5f), 0, 0, std::cos(b * 0.5f)};
  Quat qz{0, 0, std::sin(c * 0.5f), std::cos(c * 0.5f)};
  return qmul(qmul(qy, qx), qz);
}
// Mat4::from_scale_rotation_translation: columns = rotation axes * scale, then translation
void mat_from_srt(V s, Quat q, V t, float m[16]) {
  const float x2 = q.x + q.x, y2 = q.y + q.y, z2 = q.z + q.z;
  const float xx = q.x * x2, xy = q.x * y2, xz = q.x * z2;
  const float yy = q.y * y2, yz = q.y * z2, zz = q.z * z2;
  const float wx = q.w * x2, wy = q.w * y2, wz = q.w * z2;
  const float xa[4] = {1.0f - (yy + zz), xy + wz, xz - wy, 0.0f};
  const float ya[4] = {xy - wz, 1.0f - (xx + zz), yz + wx, 0.0f};
  const float za[4] = {xz + wy, yz - wx, 1.0f - (xx + yy), 0.0f};
  for (int i = 0; i < 4; i++) {
    m[i] = xa[i] * s.x;
    m[4 + i] = ya[i] * s.y;
    m[8 + i] = za[i] * s.z;
  }
  m[12] = t.x, m[13] = t.y, m[14] = t.z, m[15] = 1.0f;
}
// Mat4::inverse: the cofactor expansion glam shares with GLM (m[col*4+row])
void mat_inverse(const float m[16], float out[16]) {
  auto M = [&](int c, int r) { return m[c * 4 + r]; };
  const float c00 = M(2, 2) * M(3, 3) - M(3, 2) * M(2, 3), c02 = M(1, 2) * M(3, 3) - M(3, 2) * M(1, 3),
              c03 = M(1, 2) * M(2, 3) - M(2, 2) * M(1, 3);
  const float c04 = M(2, 1) * M(3, 3) - M(3, 1) * M(2, 3), c06 = M(1, 1) * M(3, 3) - M(3, 1) * M(1, 3),
              c07 = M(1, 1) * M(2, 3) - M(2, 1) * M(1, 3);
  const float c08 = M(2, 1) * M(3, 2) - M(3, 1) * M(2, 2), c10 = M(1, 1) * M(3, 2) - M(3, 1) * M(1, 2),
              c11 = M(1, 1) * M(2, 2) - M(2, 1) * M(1, 2);
  const float c12 = M(2, 0) * M(3, 3) - M(3, 0) * M(2, 3), c14 = M(1, 0) * M(3, 3) - M(3, 0) * M(1, 3),
              c15 = M(1, 0) * M(2, 3) - M(2, 0) * M(1, 3);
  const float c16 = M(2, 0) * M(3, 2) - M(3, 0) * M(2, 2), c18 = M(1, 0) * M(3, 2) - M(3, 0) * M(1, 2),
              c19 = M(1, 0) * M(2, 2) - M(2, 0) * M(1, 2);
  const float c20 = M(2, 0) * M(3, 1) - M(3, 0) * M(2, 1), c22 = M(1, 0) * M(3, 1) - M(3, 0) * M(1, 1),
              c23 = M(1, 0) * M(2, 1) - M(2, 0) * M(1, 1);
  const float f0[4] = {c00, c00, c02, c03}, f1[4] = {c04, c04, c06, c07}, f2[4] = {c08, c08, c10, c11};
  const float f3[4] = {c12, c12, c14, c15}, f4[4] = {c16, c16, c18, c19}, f5[4] = {c20, c20, c22, c23};
  const float v0[4] = {M(1, 0), M(0, 0), M(0, 0), M(0, 0)}, v1[4] = {M(1, 1), M(0, 1), M(0, 1), M(0, 1)};
  const float v2[4] = {M(1, 2), M(0, 2), M(0, 2), M(0, 2)}, v3[4] = {M(1, 3), M(0, 3), M(0, 3), M(0, 3)};
  const float sa[4] = {1, -1, 1, -1}, sb[4] = {-1, 1, -1, 1};
  float inv[4][4];
  for (int i = 0; i < 4; i++) {
    inv[0][i] = ((v1[i] * f0[i] - v2[i] * f1[i]) + v3[i] * f2[i]) * sa[i];
    inv[1][i] = ((v0[i] * f0[i] - v2[i] * f3[i]) + v3[i] * f4[i]) * sb[i];
    inv[2][i] = ((v0[i] * f1[i] - v1[i] * f3[i]) + v3[i] * f5[i]) * sa[i];
    inv[3][i] = ((v0[i] * f2[i] - v1[i] * f4[i]) + v2[i] * f5[i]) * sb[i];
  }
  const float d0 = M(0, 0) * inv[0][0], d1 = M(0, 1) * inv[1][0], d2 = M(0, 2) * inv[2][0], d3 = M(0, 3) * inv[3][0];
  const float det = (d0 + d1) + (d2 + d3);
  const float rcp = 1.0f / det;
  for (int c = 0; c < 4; c++)
    for (int r = 0; r < 4; r++) out[c * 4 + r] = inv[c][r] * rcp;
}
V mat_point(const float m[16], V p) {  // (Mat4 * Vec4(p, 1)).truncate()
  return {((m[0] * p.x + m[4] * p.y) + m[8] * p.z) + m[12] * 1.0f, ((m[1] * p.x + m[5] * p.y) + m[9] * p.z) + m[13] * 1.0f,
          ((m[2] * p.x + m[6] * p.y) + m[10] * p.z) + m[14] * 1.0f};
}
float to_radians(float deg) { return deg * (PI_F / 180.0f); }  // f32::to_radians

void transform_from(V scale, V rot_deg, V pos, float o2w[16], float w2o[16]) {  // parser.rs:647-674
  Quat q = quat_from_euler_yxz(to_radians(rot_deg.y), to_radians(rot_deg.x), to_radians(rot_deg.z));
  mat_from_srt(scale, q, pos, o2w);
  mat_inverse(o2w, w2o);
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
struct pth_scene {
  std::vector<ptc_material> materials;
  std::vector<pth_object> objects;
  std::vector<std::vector<float>> meshes;  // n x 12 each
  std::vector<float> sky;
  int32_t sky_w = 0, sky_h = 0;
  ptc_camera camera;
  bool has_lens = false;  // PTH_LOAD_THIN_LENS: a "thinlens" camera's lens
  ptc_lens lens = {0.0f, 0.0f};
  int32_t width = 800, height = 600, spp = 16, max_depth = 10;  // parser.rs:255-258
  pth_scene() { memset(&camera, 0, sizeof(camera)); }
};

namespace {

ptc_material mat_blank(int type) {
  ptc_material m;
  memset(&m, 0, sizeof(m));
  m.type = type;
  return m;
}
ptc_material mat_lambert(float r, float g, float b) {  // Lambertian::new_solid
  ptc_material m = mat_blank(PTC_MAT_LAMBERT);
  m.albedo[0] = r, m.albedo[1] = g, m.albedo[2] = b;
  return m;
}
ptc_material mat_checker(const float on[3], const float off[3], float scale) {  // CheckerTexture::new, materials.rs:80-87
  ptc_material m = mat_blank(PTC_MAT_LAMBERT_CHECKER);
  for (int i = 0; i < 3; i++) m.albedo[i] = on[i], m.off_color[i] = off[i];
  m.inv_scale = std::fabs(scale) < 1e-6f ? 1.0f : 1.0f / scale;
  return m;
}
ptc_material mat_metal(const float a[3], float fuzz) {  // Metal::new clamps fuzz (material.rs:79-84)
  ptc_material m = mat_blank(PTC_MAT_METAL);
  for (int i = 0; i < 3; i++) m.albedo[i] = a[i];
  m.fuzz = fuzz < 0.0f ? 0.0f : (fuzz > 1.0f ? 1.0f : fuzz);
  return m;
}
ptc_material mat_dielectric(float ior) {
  ptc_material m = mat_blank(PTC_MAT_DIELECTRIC);
  m.ior = ior;
  return m;
}
ptc_material mat_emissive(float r, float g, float b) {
  ptc_material m = mat_blank(PTC_MAT_EMISSIVE);
  m.albedo[0] = r, m.albedo[1] = g, m.albedo[2] = b;
  return m;
}
ptc_material mat_plastic(const float a[3], float ior) {
  ptc_material m = mat_blank(PTC_MAT_PLASTIC);
  for (int i = 0; i < 3; i++) m.albedo[i] = a[i];
  m.ior = ior;
  return m;
}
// MetalType::ior_k, tungsten/materials.rs:116-152
bool metal_ior_k(const std::string &name_lower, float eta[3], float k[3]) {
  struct E {
    const char *n;
    float e[3], k[3];
  };
  static const E table[] = {
      {"cu", {0.200f, 1.090f, 1.420f}, {3.910f, 2.570f, 2.300f}}, {"au", {0.170f, 0.350f, 1.500f}, {3.140f, 2.300f, 1.920f}},
      {"ag", {0.155f, 0.145f, 0.135f}, {3.910f, 2.610f, 2.370f}}, {"al", {1.360f, 0.965f, 0.620f}, {7.570f, 6.690f, 5.440f}},
      {"ni", {1.920f, 1.920f, 1.920f}, {3.670f, 3.670f, 3.670f}}, {"ti", {2.740f, 2.740f, 2.740f}, {3.170f, 3.170f, 3.170f}},
      {"fe", {2.870f, 2.870f, 2.870f}, {3.140f, 3.140f, 3.140f}}, {"pb", {1.910f, 1.910f, 1.910f}, {3.180f, 3.180f, 3.180f}},
  };
  for (const E &e : table)
    if (name_lower == e.n) {
      for (int i = 0; i < 3; i++) eta[i] = e.e[i], k[i] = e.k[i];
      return true;
    }
  return false;
}
ptc_material mat_rough_conductor(const float a[3], float roughness, const std::string &metal_lower, int dist) {
  ptc_material m = mat_blank(PTC_MAT_ROUGH_CONDUCTOR);
  for (int i = 0; i < 3; i++) m.albedo[i] = a[i];
  m.roughness = std::fmax(roughness, 0.01f);  // RoughConductor::new, materials.rs:177
  if (!metal_ior_k(metal_lower, m.eta, m.k)) metal_ior_k("cu", m.eta, m.k);
  m.distribution = dist;
  return m;
}

std::string lower(std::string s) {
  for (auto &c : s) c = (char)std::tolower((unsigned char)c);
  return s;
}
bool ends_with(const std::string &s, const char *suf) {
  size_t n = strlen(suf);
  return s.size() >= n && s.compare(s.size() - n, n, suf) == 0;
}
std::string dir_of(const std::string &p) {
  size_t k = p.find_last_of('/');
  return k == std::string::npos ? std::string(".") : p.substr(0, k);
}

// serde: a struct {x,y,z} also deserialises from a 3-element sequence (Vec3Config, parser.rs:23-28)
bool parse_vec3(const pth::Json &j, V &out) {
  if (j.is_array()) {
    if (j.arr.size() != 3) return false;
    for (auto &e : j.arr)
      if (!e.is_number()) return false;
    out = {(float)j.arr[0].num, (float)j.arr[1].num, (float)j.arr[2].num};
    return true;
  }
  if (j.is_object()) {
    const pth::Json *x = j.find("x"), *y = j.find("y"), *z = j.find("z");
    if (!x || !y || !z || !x->is_number() || !y->is_number() || !z->is_number()) return false;
    out = {(float)x->num, (float)y->num, (float)z->num};
    return true;
  }
  return false;
}
bool parse_color(const pth::Json &j, float c[3]) {  // ColorConfig(f32,f32,f32): a 3-element sequence
  if (!j.is_array() || j.arr.size() != 3) return false;
  for (int i = 0; i < 3; i++) {
    if (!j.arr[i].is_number()) return false;
    c[i] = (float)j.arr[i].num;
  }
  return true;
}

struct Xform {
  bool has_pos = false, has_scale = false, scale_uniform = false, has_rot = false;
  V pos{0, 0, 0}, scale{1, 1, 1}, rot{0, 0, 0};
  float uniform = 1.0f;
};
// ObjectTransformConfig, parser.rs:128-133 (every field optional; ScaleConfig = f32 | vec3)
void parse_transform(const pth::Json &j, Xform &t) {
  if (!j.is_object()) throw std::runtime_error("transform: expected a map");
  if (const pth::Json *p = j.find("position"); p && !p->is_null()) {
    if (!parse_vec3(*p, t.pos)) throw std::runtime_error("transform.position: invalid Vec3");
    t.has_pos = true;
  }
  if (const pth::Json *s = j.find("scale"); s && !s->is_null()) {
    if (s->is_number()) {
      t.scale_uniform = true;
      t.uniform = (float)s->num;
      t.scale = {t.uniform, t.uniform, t.uniform};
    } else if (!parse_vec3(*s, t.scale)) {
      throw std::runtime_error("transform.scale: data did not match any variant of untagged enum ScaleConfig");
    }
    t.has_scale = true;
  }
  if (const pth::Json *r = j.find("rotation"); r && !r->is_null()) {
    if (!parse_vec3(*r, t.rot)) throw std::runtime_error("transform.rotation: invalid Vec3");
    t.has_rot = true;
  }
}

void camera_new(V position, V look_at, V up, float fov, float aspect, ptc_camera *c) {  // camera.rs:14-31
  V forward = normalized(look_at - position);
  V right = normalized(cross(forward, normalized(up)));
  V true_up = normalized(cross(right, forward));
  float fov_rad = fov * PI_F / 180.0f;
  float half_height = std::tan(fov_rad / 2.0f);
  float half_width = half_height * aspect;
  c->position[0] = position.x, c->position[1] = position.y, c->position[2] = position.z;
  c->forward[0] = forward.x, c->forward[1] = forward.y, c->forward[2] = forward.z;
  c->right[0] = right.x, c->right[1] = right.y, c->right[2] = right.z;
  c->true_up[0] = true_up.x, c->true_up[1] = true_up.y, c->true_up[2] = true_up.z;
  c->half_width = half_width;
  c->half_height = half_height;
}

pth_object obj_blank(int type, int material) {
  pth_object o;
  memset(&o, 0, sizeof(o));
  o.type = type;
  o.material = material;
  o.mesh = -1;
  return o;
}

// Quad::new_transformed, tungsten/objects/quad.rs:26-79
pth_object make_quad(const float m[16], int material) {
  pth_object o = obj_blank(PTH_QUAD, material);
  V base = mat_point(m, {-0.5f, 0.0f, -0.5f});
  V pb = mat_point(m, {0.5f, 0.0f, -0.5f});
  V pd = mat_point(m, {-0.5f, 0.0f, 0.5f});
  V e0 = pb - base, e1 = pd - base;
  V n = normalized(cross(e0, e1));
  float d = dot(n, base);
  float l0 = len2(e0), l1 = len2(e1);
  o.base[0] = base.x, o.base[1] = base.y, o.base[2] = base.z;
  o.edge0[0] = e0.x, o.edge0[1] = e0.y, o.edge0[2] = e0.z;
  o.edge1[0] = e1.x, o.edge1[1] = e1.y, o.edge1[2] = e1.z;
  o.normal[0] = n.x, o.normal[1] = n.y, o.normal[2] = n.z;
  o.d = d;
  o.inv_edge0_len_sq = l0 > EPSILON ? 1.0f / l0 : 0.0f;
  o.inv_edge1_len_sq = l1 > EPSILON ? 1.0f / l1 : 0.0f;
  return o;
}

// Triangle::new (mesh/triangle.rs:14-25) + the degenerate filter of Mesh::from_obj (mesh_object.rs:128-134)
bool push_triangle(std::vector<float> &out, V v0, V v1, V v2) {
  V e1 = v1 - v0, e2 = v2 - v0;
  V c = cross(e1, e2);
  if (len2(c) < EPSILON * EPSILON) return false;
  V n = normalized(c);
  const float rec[12] = {v0.x, v0.y, v0.z, v1.x, v1.y, v1.z, v2.x, v2.y, v2.z, n.x, n.y, n.z};
  out.insert(out.end(), rec, rec + 12);
  return true;
}

// Stand-in for tobj::load_obj(path, GPU_LOAD_OPTIONS) (tobj 4.0.3, not vendored: parity unpinned) as consumed by
// Mesh::from_obj (mesh_object.rs:59-139): positions + triangulated faces (fan 0,i,i+1), points/lines ignored,
// triangles in file order.
bool load_obj_triangles(const std::string &path, std::vector<float> &out, std::string &err) {
  std::ifstream f(path);
  if (!f) {
    err = "cannot open OBJ file: " + path;
    return false;
  }
  std::vector<V> verts;
  std::string line;
  std::vector<long> face;
  bool any_face = false;
  while (std::getline(f, line)) {
    const char *p = line.c_str();
    while (*p == ' ' || *p == '\t') p++;
    if (p[0] == 'v' && (p[1] == ' ' || p[1] == '\t')) {
      char *e;
      p += 2;
      float x = std::strtof(p, &e);
      p = e;
      float y = std::strtof(p, &e);
      p = e;
      float z = std::strtof(p, &e);
      verts.push_back({x, y, z});
    } else if (p[0] == 'f' && (p[1] == ' ' || p[1] == '\t')) {
      p += 2;
      face.clear();
      while (*p) {
        while (*p == ' ' || *p == '\t' || *p == '\r') p++;
        if (!*p) break;
        char *e;
        long idx = std::strtol(p, &e, 10);
        if (e == p) break;
        p = e;
        while (*p && *p != ' ' && *p != '\t' && *p != '\r') p++;  // skip /vt/vn
        if (idx < 0) idx = (long)verts.size() + idx;
        else idx -= 1;
        face.push_back(idx);
      }
      if (face.size() < 3) continue;  // ignore_points / ignore_lines
      any_face = true;
      for (size_t i = 1; i + 1 < face.size(); i++) {
        long a = face[0], b = face[i], c = face[i + 1];
        if (a < 0 || b < 0 || c < 0 || (size_t)a >= verts.size() || (size_t)b >= verts.size() || (size_t)c >= verts.size()) {
          fprintf(stderr, "Warning: Vertex index out of bounds in OBJ file '%s'. Skipping triangle.\n", path.c_str());
          continue;
        }
        push_triangle(out, verts[(size_t)a], verts[(size_t)b], verts[(size_t)c]);
      }
    }
  }
  if (!any_face) {
    err = "No models found in OBJ file: " + path;
    return false;
  }
  if (out.empty()) {
    err = "No valid, non-degenerate triangles loaded for mesh '" + path + "'";  // mesh_object.rs:30-36
    return false;
  }
  return true;
}

// Mesh::from_wo3 (mesh_object.rs:141-259).  A Tungsten .wo3 file is: u64 vertex count, 32-byte vertices (position,
// normal, uv), u64 triangle count, 16-byte triangles (v0, v1, v2: u32, material: i32).  The reference reads the
// triangles as consecutive 12-byte index triples (it never skips the material word, mesh_object.rs:188-190), so from the
// second record on its indices are taken from a shifted stream; triples with an index out of range are skipped
// (:201-215), the rest become (wrong) triangles.  `tungsten_stride` = false restates exactly that; true reads the file
// the way Tungsten wrote it (PTH_LOAD_WO3_STRIDE16).
bool load_wo3_triangles(const std::string &path, std::vector<float> &out, std::string &err, bool tungsten_stride) {
  std::ifstream f(path, std::ios::binary);
  if (!f) {
    err = "No such file or directory";
    return false;
  }
  std::vector<unsigned char> buf((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
  size_t pos = 0;
  auto rd_u64 = [&]() {
    uint64_t v = 0;
    memcpy(&v, &buf[pos], 8);
    pos += 8;
    return v;
  };
  if (buf.size() < 8) {
    err = "failed to fill whole buffer";
    return false;
  }
  const uint64_t nv = rd_u64();
  if (nv > (buf.size() - pos) / 32) {
    err = "failed to fill whole buffer";
    return false;
  }
  std::vector<V> verts((size_t)nv);
  for (uint64_t i = 0; i < nv; i++) {
    float q[3];
    memcpy(q, &buf[pos], 12);
    verts[(size_t)i] = V{q[0], q[1], q[2]};
    pos += 32;
  }
  if (buf.size() - pos < 8) {
    err = "failed to fill whole buffer";
    return false;
  }
  const uint64_t nt = rd_u64();
  const size_t stride = tungsten_stride ? 16 : 12;
  if (nt > (buf.size() - pos) / stride) {
    err = "failed to fill whole buffer";
    return false;
  }
  for (uint64_t i = 0; i < nt; i++) {
    uint32_t idx[3];
    memcpy(idx, &buf[pos], 12);
    pos += stride;
    if (idx[0] >= nv || idx[1] >= nv || idx[2] >= nv) continue;
    push_triangle(out, verts[idx[0]], verts[idx[1]], verts[idx[2]]);
  }
  if (out.empty()) {
    err = "[WO3_LOADER] No valid triangles in " + path;
    return false;
  }
  return true;
}

// Radiance .hdr (RGBE) -> linear f32 RGB, the job of image::open(..).into_rgb32f() (parser.rs:502-506; image 0.25.6
// is not vendored: parity unpinned).  Handles flat and new-style RLE scanlines, -Y +X orientation.
bool load_hdr(const std::string &path, std::vector<float> &rgb, int &w, int &h, std::string &err) {
  FILE *f = fopen(path.c_str(), "rb");
  if (!f) {
    err = "cannot open HDR file: " + path;
    return false;
  }
  char line[512];
  bool ok_magic = false;
  w = h = 0;
  while (fgets(line, sizeof(line), f)) {
    if (!ok_magic) {
      if (strncmp(line, "#?", 2) != 0) break;
      ok_magic = true;
      continue;
    }
    if (line[0] == '\n' || line[0] == '\r') {
      if (!fgets(line, sizeof(line), f)) break;
      if (sscanf(line, "-Y %d +X %d", &h, &w) != 2) w = h = 0;
      break;
    }
  }
  if (!ok_magic || w <= 0 || h <= 0) {
    fclose(f);
    err = "not a Radiance HDR file: " + path;
    return false;
  }
  rgb.assign((size_t)w * h * 3, 0.0f);
  std::vector<unsigned char> scan((size_t)w * 4);
  for (int y = 0; y < h; y++) {
    unsigned char hd[4];
    if (fread(hd, 1, 4, f) != 4) goto fail;
    if (hd[0] == 2 && hd[1] == 2 && (hd[2] & 0x80) == 0 && ((hd[2] << 8) | hd[3]) == w && w >= 8 && w < 32768) {
      for (int c = 0; c < 4; c++) {
        int x = 0;
        while (x < w) {
          int n = fgetc(f);
          if (n == EOF) goto fail;
          if (n > 128) {
            n -= 128;
            int v = fgetc(f);
            if (v == EOF || x + n > w) goto fail;
            for (int i = 0; i < n; i++) scan[(size_t)(x++) * 4 + c] = (unsigned char)v;
          } else {
            if (n == 0 || x + n > w) goto fail;
            for (int i = 0; i < n; i++) {
              int v = fgetc(f);
              if (v == EOF) goto fail;
              scan[(size_t)(x++) * 4 + c] = (unsigned char)v;
            }
          }
        }
      }
    } else {
      memcpy(scan.data(), hd, 4);
      if (w > 1 && fread(scan.data() + 4, 4, (size_t)w - 1, f) != (size_t)w - 1) goto fail;
    }
    for (int x = 0; x < w; x++) {
      const unsigned char *p = &scan[(size_t)x * 4];
      float *o = &rgb[((size_t)y * w + x) * 3];
      if (p[3] == 0) {
        o[0] = o[1] = o[2] = 0.0f;
      } else {
        const float s = std::exp2((float)p[3] - 128.0f - 8.0f);
        o[0] = (float)p[0] * s, o[1] = (float)p[1] * s, o[2] = (float)p[2] * s;
      }
    }
  }
  fclose(f);
  return true;
fail:
  fclose(f);
  err = "truncated or corrupt HDR file: " + path;
  return false;
}

int find_or_magenta(pth_scene *s, const std::map<std::string, int> &bsdfs, const std::string &name, const char *what) {
  auto it = bsdfs.find(name);
  if (it != bsdfs.end()) return it->second;
  fprintf(stderr, "Warning: BSDF '%s' not found for %s. Using default (magenta Lambertian) material.\n", name.c_str(), what);
  s->materials.push_back(mat_lambert(1.0f, 0.0f, 1.0f));  // Color::MAGENTA
  return (int)s->materials.size() - 1;
}

// AlbedoConfig (untagged: Solid(rgb) | GrayscaleSolid(f32) | Checker{..}), parser.rs:82-88,429-443
bool lambert_from_albedo(const pth::Json &a, ptc_material &out) {
  float c[3];
  if (parse_color(a, c)) {
    out = mat_lambert(c[0], c[1], c[2]);
    return true;
  }
  if (a.is_number()) {
    out = mat_lambert((float)a.num, (float)a.num, (float)a.num);
    return true;
  }
  if (a.is_object()) {
    const pth::Json *on = a.find("on_color"), *off = a.find("off_color");
    float onc[3], offc[3];
    if (on && off && parse_color(*on, onc) && parse_color(*off, offc)) {
      const pth::Json *ru = a.find("res_u"), *rv = a.find("res_v");
      float scale = 10.0f;
      if (ru && ru->is_number()) scale = (float)ru->num;
      else if (rv && rv->is_number()) scale = (float)rv->num;
      out = mat_checker(onc, offc, scale);
      return true;
    }
  }
  return false;
}

// MaterialTypeConfig for an inline Plane material: externally tagged, PascalCase (parser.rs:90-119,590-630)
ptc_material plane_inline_material(const pth::Json &j) {
  if (!j.is_object() || j.obj.size() != 1) throw std::runtime_error("plane.material: expected an externally tagged enum");
  const std::string &tag = j.obj[0].first;
  const pth::Json &b = j.obj[0].second;
  auto num = [&](const char *k) -> float {
    const pth::Json *v = b.find(k);
    if (!v || !v->is_number()) throw std::runtime_error(std::string("plane.material: missing field `") + k + "`");
    return (float)v->num;
  };
  auto col = [&](const char *k, float c[3]) {
    const pth::Json *v = b.find(k);
    if (!v || !parse_color(*v, c)) throw std::runtime_error(std::string("plane.material: missing field `") + k + "`");
  };
  if (tag == "Lambertian") {
    const pth::Json *a = b.find("albedo");
    ptc_material m;
    if (!a || !lambert_from_albedo(*a, m)) throw std::runtime_error("plane.material: invalid Lambertian albedo");
    return m;
  }
  if (tag == "Metal") {
    float c[3];
    col("albedo", c);
    return mat_metal(c, num("fuzz"));
  }
  if (tag == "Glass") return mat_dielectric(num("index_of_refraction"));
  if (tag == "Plastic") {
    float c[3];
    col("albedo", c);
    return mat_plastic(c, num("ior"));
  }
  if (tag == "RoughConductor") {
    float c[3];
    col("albedo", c);
    const pth::Json *mt = b.find("metal_type"), *ds = b.find("distribution");
    if (!mt || !mt->is_string() || !ds || !ds->is_string()) throw std::runtime_error("plane.material: invalid RoughConductor");
    int dist;
    if (ds->str == "Ggx") dist = PTC_DIST_GGX;
    else if (ds->str == "Beckmann") dist = PTC_DIST_BECKMANN;
    else throw std::runtime_error("plane.material: unknown variant `" + ds->str + "`");
    float e[3], k[3];
    if (!metal_ior_k(lower(mt->str), e, k) || !std::isupper((unsigned char)mt->str[0]))
      throw std::runtime_error("plane.material: unknown variant `" + mt->str + "`");
    return mat_rough_conductor(c, num("roughness"), lower(mt->str), dist);
  }
  if (tag == "Texture" || tag == "Light") {
    fprintf(stderr, "Warning: Unsupported inline material type for Plane. Defaulting to white Lambertian.\n");
    return mat_lambert(1.0f, 1.0f, 1.0f);
  }
  throw std::runtime_error("plane.material: unknown variant `" + tag + "`");
}

pth_scene *load_scene(const std::string &json_path, int flags) {
  std::ifstream f(json_path);
  if (!f) throw std::runtime_error("No such file or directory: " + json_path);
  std::stringstream ss;
  ss << f.rdbuf();
  const std::string text = ss.str();
  pth::Json doc = pth::JsonParser(text).parse();
  if (!doc.is_object()) throw std::runtime_error("scene: expected a map");
  const std::string scene_dir = dir_of(json_path);

  std::unique_ptr<pth_scene> s(new pth_scene());

  // ---- camera (required) + settings, parser.rs:255-304
  const pth::Json *cam = doc.find("camera");
  if (!cam || !cam->is_object()) throw std::runtime_error("missing field `camera`");
  const pth::Json *ct = cam->find("transform");
  if (!ct || !ct->is_object()) throw std::runtime_error("camera: missing field `transform`");
  V cpos, clook, cup;
  {
    const pth::Json *p = ct->find("position"), *l = ct->find("look_at"), *u = ct->find("up");
    if (!p || !parse_vec3(*p, cpos)) throw std::runtime_error("camera.transform: missing field `position`");
    if (!l || !parse_vec3(*l, clook)) throw std::runtime_error("camera.transform: missing field `look_at`");
    if (!u || !parse_vec3(*u, cup)) throw std::runtime_error("camera.transform: missing field `up`");
  }
  const pth::Json *fov = cam->find("fov");
  if (!fov || !fov->is_number()) throw std::runtime_error("camera: missing field `fov`");
  if (const pth::Json *res = cam->find("resolution"); res && !res->is_null()) {
    if (res->is_number()) {
      s->width = s->height = (int32_t)res->num;
    } else if (res->is_array() && res->arr.size() == 2 && res->arr[0].is_number() && res->arr[1].is_number()) {
      s->width = (int32_t)res->arr[0].num;
      s->height = (int32_t)res->arr[1].num;
    } else {
      throw std::runtime_error("camera.resolution: data did not match any variant of untagged enum ResolutionConfig");
    }
  }
  if (const pth::Json *r = doc.find("renderer"); r && r->is_object())
    if (const pth::Json *spp = r->find("spp"); spp && spp->is_number()) s->spp = (int32_t)spp->num;
  if (const pth::Json *i = doc.find("integrator"); i && i->is_object())
    if (const pth::Json *mb = i->find("max_bounces"); mb && mb->is_number()) s->max_depth = (int32_t)mb->num;
  float aspect = (float)s->width / (float)s->height;
  if (const pth::Json *a = cam->find("aspect"); a && a->is_number()) aspect = (float)a->num;
  camera_new(cpos, clook, cup, (float)fov->num, aspect, &s->camera);
  if (const pth::Json *ty = cam->find("type"); (flags & PTH_LOAD_THIN_LENS) && ty && ty->is_string() && ty->str == "thinlens") {
    // Tungsten's aperture_size is the lens radius.  Without focus_distance we focus on look_at (our rule, not Tungsten's).
    const pth::Json *ap = cam->find("aperture_size"), *fd = cam->find("focus_distance");
    s->lens.aperture_radius = ap && ap->is_number() ? (float)ap->num : 0.0f;
    const float dx = clook.x - cpos.x, dy = clook.y - cpos.y, dz = clook.z - cpos.z;
    s->lens.focus_distance = fd && fd->is_number() ? (float)fd->num : std::sqrt(dx * dx + dy * dy + dz * dz);
    s->has_lens = true;
    for (const char *k : {"aperture", "cateye", "catEye", "focus_pivot"})
      if (cam->find(k)) {
        fprintf(stderr, "Warning: thinlens camera: aperture textures, cat-eye and focus_pivot are not supported and are ignored.\n");
        break;
      }
  }

  // ---- bsdfs, parser.rs:308-495
  std::map<std::string, int> bsdfs;
  if (const pth::Json *bl = doc.find("bsdfs"); bl && !bl->is_null()) {
    if (!bl->is_array()) throw std::runtime_error("bsdfs: expected a sequence");
    for (const pth::Json &b : bl->arr) {
      if (!b.is_object()) throw std::runtime_error("bsdfs[]: expected a map");
      const pth::Json *name = b.find("name"), *type = b.find("type");
      if (!name || !name->is_string()) throw std::runtime_error("bsdfs[]: missing field `name`");
      if (!type || !type->is_string()) throw std::runtime_error("bsdfs[]: missing field `type`");
      const pth::Json *albedo = b.find("albedo");
      if (albedo && albedo->is_null()) albedo = nullptr;
      auto optf = [&](const char *k, float dflt) {
        const pth::Json *v = b.find(k);
        if (v && !v->is_null() && !v->is_number()) throw std::runtime_error(std::string("bsdfs[].") + k + ": invalid type");
        return (v && v->is_number()) ? (float)v->num : dflt;
      };
      ptc_material m;
      bool ok = true;
      const std::string &t = type->str;
      if (t == "lambert") {
        if (!albedo) {
          fprintf(stderr, "Skipping BSDF '%s': Lambertian BSDF missing albedo.\n", name->str.c_str());
          ok = false;
        } else if (!lambert_from_albedo(*albedo, m)) {
          fprintf(stderr, "Skipping BSDF '%s': failed to parse albedo as Color, f32, or Checker.\n", name->str.c_str());
          ok = false;
        }
      } else if (t == "plastic") {
        float c[3] = {0.8f, 0.8f, 0.8f};
        if (albedo) {
          float cc[3];
          if (parse_color(*albedo, cc)) memcpy(c, cc, sizeof(c));
          else if (albedo->is_number()) c[0] = c[1] = c[2] = (float)albedo->num;
          else fprintf(stderr, "Warning: Failed to parse albedo for Plastic BSDF '%s'. Using default albedo.\n", name->str.c_str());
        } else {
          fprintf(stderr, "Warning: Plastic BSDF '%s' missing albedo. Using default albedo.\n", name->str.c_str());
        }
        m = mat_plastic(c, optf("ior", 1.5f));
      } else if (t == "null") {
        m = mat_lambert(0.0f, 0.0f, 0.0f);
      } else if (t == "glass" || t == "dielectric") {
        m = mat_dielectric(optf("ior", 1.5f));
      } else if (t == "rough_conductor") {
        float c[3] = {1.0f, 1.0f, 1.0f};
        if (albedo) {
          float cc[3];
          if (parse_color(*albedo, cc)) memcpy(c, cc, sizeof(c));
          else if (albedo->is_number()) c[0] = c[1] = c[2] = (float)albedo->num;
        }
        std::string metal = "cu";
        if (const pth::Json *mj = b.find("material"); mj && mj->is_string()) {
          float e[3], k[3];
          if (metal_ior_k(lower(mj->str), e, k)) metal = lower(mj->str);
          else fprintf(stderr, "Warning: Unknown metal type '%s' for rough_conductor, defaulting to Cu.\n", mj->str.c_str());
        }
        int dist = PTC_DIST_GGX;
        if (const pth::Json *dj = b.find("distribution"); dj && dj->is_string()) {
          const std::string d = lower(dj->str);
          if (d == "ggx") dist = PTC_DIST_GGX;
          else if (d == "beckmann") dist = PTC_DIST_BECKMANN;
          else fprintf(stderr, "Warning: Unknown distribution '%s' for rough_conductor, defaulting to Ggx.\n", dj->str.c_str());
        }
        m = mat_rough_conductor(c, optf("roughness", 0.1f), metal, dist);
      } else {
        fprintf(stderr, "Warning: Unsupported BSDF type '%s' for BSDF named '%s'.\n", t.c_str(), name->str.c_str());
        ok = false;
      }
      if (ok) {
        s->materials.push_back(m);
        bsdfs[name->str] = (int)s->materials.size() - 1;  // HashMap::insert: a repeated name replaces the earlier entry
      }
    }
  }

  // ---- sky, parser.rs:497-521 (only .hdr textures are ever sampled, renderer.rs:40)
  if (const pth::Json *sky = doc.find("sky"); sky && sky->is_object())
    if (const pth::Json *tex = sky->find("texture"); tex && tex->is_string()) {
      const std::string p = scene_dir + "/" + tex->str;
      if (ends_with(tex->str, ".hdr")) {
        std::string err;
        int w, h;
        std::vector<float> rgb;
        if (load_hdr(p, rgb, w, h, err)) {
          s->sky = std::move(rgb);
          s->sky_w = w;
          s->sky_h = h;
        } else {
          fprintf(stderr, "Error loading HDR skybox image from 'sky' config '%s': %s. Using default background.\n", p.c_str(),
                  err.c_str());
        }
      }  // LDR skyboxes are loaded by the reference but never sampled (scene.rs:8 vs renderer.rs:40)
    }

  // ---- primitives (required), parser.rs:523-812
  const pth::Json *prims = doc.find("primitives");
  if (!prims || !prims->is_array()) throw std::runtime_error("missing field `primitives`");
  for (const pth::Json &p : prims->arr) {
    if (!p.is_object()) throw std::runtime_error("primitives[]: expected a map");
    const pth::Json *type = p.find("type");
    if (!type || !type->is_string()) throw std::runtime_error("primitives[]: missing field `type`");
    const std::string &t = type->str;
    auto need_bsdf = [&]() -> std::string {
      const pth::Json *b = p.find("bsdf");
      if (!b) throw std::runtime_error("primitives[]: missing field `bsdf`");
      if (!b->is_string()) throw std::runtime_error("primitives[].bsdf: invalid type, expected a string");
      return b->str;
    };
    auto need_transform = [&](Xform &x) {
      const pth::Json *tr = p.find("transform");
      if (!tr) throw std::runtime_error("primitives[]: missing field `transform`");
      parse_transform(*tr, x);
    };
    if (t == "sphere") {
      Xform x;
      need_transform(x);
      const std::string bsdf = need_bsdf();
      const pth::Json *power = p.find("power"), *radius = p.find("radius");
      const bool has_power = power && power->is_number();
      float r;
      if (radius && radius->is_number()) r = (float)radius->num;
      else if (x.has_scale) r = x.scale_uniform ? x.uniform : x.scale.x;
      else r = 1.0f;
      int mat;
      if (has_power) {  // parser.rs:566-576 (note the PI * PI)
        const float pv = (float)power->num;
        const float rad = r > 1e-6f ? pv / (4.0f * PI_F * PI_F * r * r) : 0.0f;
        s->materials.push_back(mat_emissive(rad, rad, rad));
        mat = (int)s->materials.size() - 1;
      } else {
        mat = find_or_magenta(s.get(), bsdfs, bsdf, "Sphere");
      }
      pth_object o = obj_blank(PTH_SPHERE, mat);
      o.center[0] = x.pos.x, o.center[1] = x.pos.y, o.center[2] = x.pos.z;
      o.radius = r;
      s->objects.push_back(o);
    } else if (t == "plane") {
      const pth::Json *pt = p.find("point"), *nm = p.find("normal"), *mt = p.find("material");
      V point, normal;
      if (!pt || !parse_vec3(*pt, point)) throw std::runtime_error("plane: missing field `point`");
      if (!nm || !parse_vec3(*nm, normal)) throw std::runtime_error("plane: missing field `normal`");
      if (!mt) throw std::runtime_error("plane: missing field `material`");
      s->materials.push_back(plane_inline_material(*mt));
      pth_object o = obj_blank(PTH_PLANE, (int)s->materials.size() - 1);
      V n = normalized(normal);  // Plane::new, plane.rs:16-22
      o.p1[0] = point.x, o.p1[1] = point.y, o.p1[2] = point.z;
      o.normal[0] = n.x, o.normal[1] = n.y, o.normal[2] = n.z;
      s->objects.push_back(o);
    } else if (t == "mesh") {
      Xform x;
      need_transform(x);
      const pth::Json *file = p.find("file");
      if (!file || !file->is_string()) throw std::runtime_error("mesh: missing field `file`");
      const std::string bsdf = need_bsdf();
      const int mat = find_or_magenta(s.get(), bsdfs, bsdf, "Mesh");
      const std::string path = scene_dir + "/" + file->str;
      std::vector<float> tris;
      std::string err;
      if (ends_with(file->str, ".wo3")) {  // parser.rs:683-686
        if (!load_wo3_triangles(path, tris, err, (flags & PTH_LOAD_WO3_STRIDE16) != 0)) {
          fprintf(stderr, "Error loading .wo3 mesh '%s': %s\n", path.c_str(), err.c_str());  // object skipped, parser.rs:696-698
          continue;
        }
      } else if (!load_obj_triangles(path, tris, err)) {
        fprintf(stderr, "Error loading .obj mesh '%s': %s\n", path.c_str(), err.c_str());  // object skipped, parser.rs:696-698
        continue;
      }
      pth_object o = obj_blank(PTH_MESH, mat);
      transform_from(x.scale, x.rot, x.pos, o.o2w, o.w2o);
      o.mesh = (int32_t)s->meshes.size();
      s->meshes.push_back(std::move(tris));
      s->objects.push_back(o);
    } else if (t == "quad") {
      Xform x;
      need_transform(x);
      const std::string bsdf = need_bsdf();
      int mat;
      const pth::Json *em = p.find("emission");
      if (em && !em->is_null()) {  // parser.rs:707-725
        float c[3];
        if (parse_color(*em, c)) {
          s->materials.push_back(mat_emissive(c[0], c[1], c[2]));
          mat = (int)s->materials.size() - 1;
        } else if (em->is_string()) {
          fprintf(stderr, "Warning: Textured emission for Quad ('%s') not fully supported yet. Treating as bright light.\n",
                  em->str.c_str());
          s->materials.push_back(mat_emissive(5.0f, 5.0f, 5.0f));
          mat = (int)s->materials.size() - 1;
        } else {
          fprintf(stderr, "Warning: Could not parse emission for Quad. Using default material.\n");
          auto it = bsdfs.find(bsdf);
          if (it != bsdfs.end()) mat = it->second;
          else {
            s->materials.push_back(mat_lambert(1.0f, 0.0f, 1.0f));
            mat = (int)s->materials.size() - 1;
          }
        }
      } else {
        mat = find_or_magenta(s.get(), bsdfs, bsdf, "Quad");
      }
      float o2w[16], w2o[16];
      transform_from(x.scale, x.rot, x.pos, o2w, w2o);
      s->objects.push_back(make_quad(o2w, mat));
    } else if (t == "cube") {
      Xform x;
      need_transform(x);
      const std::string bsdf = need_bsdf();
      const int mat = find_or_magenta(s.get(), bsdfs, bsdf, "Cube");
      pth_object o = obj_blank(PTH_CUBE, mat);
      transform_from(x.scale, x.rot, x.pos, o.o2w, o.w2o);  // Cube::new_transformed, cube.rs:20-29
      s->objects.push_back(o);
    } else if (t == "infinite_sphere" && (flags & PTH_LOAD_INFINITE_SPHERE_SKY)) {
      // Extension (SURVEY.md 8f-2): Tungsten's environment light becomes the sky the renderer already knows how to look
      // up (renderer.rs:38-63).  The primitive's rotation is ignored, like every orientation in that lookup.
      const pth::Json *em = p.find("emission");
      float c[3];
      if (em && em->is_string() && ends_with(em->str, ".hdr")) {
        const std::string hp = scene_dir + "/" + em->str;
        std::string err;
        int w, h;
        std::vector<float> rgb;
        if (load_hdr(hp, rgb, w, h, err)) s->sky = std::move(rgb), s->sky_w = w, s->sky_h = h;
        else fprintf(stderr, "Error loading HDR emission of infinite_sphere '%s': %s. Using default background.\n", hp.c_str(), err.c_str());
      } else if (em && parse_color(*em, c)) {
        s->sky.assign(c, c + 3);
        s->sky_w = s->sky_h = 1;
      }
    } else if (flags & PTH_LOAD_SKIP_UNKNOWN) {
      fprintf(stderr, "Warning: primitive of unknown type `%s` skipped\n", t.c_str());
    } else {
      // serde: unknown variant of the internally tagged ObjectConfigVariant fails the whole file (parser.rs:135-165)
      throw std::runtime_error("unknown variant `" + t + "`, expected one of `sphere`, `plane`, `mesh`, `quad`, `cube`");
    }
  }
  return s.release();
}

// ---- PNG (8-bit RGB, zlib deflate), the job of image::ImageBuffer::save in save_image (renderer.rs:125-179)
uint32_t crc_table[256];
bool crc_ready = false;
uint32_t crc32_png(const unsigned char *buf, size_t len, uint32_t crc) {
  if (!crc_ready) {
    for (uint32_t n = 0; n < 256; n++) {
      uint32_t c = n;
      for (int k = 0; k < 8; k++) c = (c & 1) ? 0xedb88320u ^ (c >> 1) : c >> 1;
      crc_table[n] = c;
    }
    crc_ready = true;
  }
  for (size_t i = 0; i < len; i++) crc = crc_table[(crc ^ buf[i]) & 0xff] ^ (crc >> 8);
  return crc;
}
void png_chunk(FILE *f, const char *type, const unsigned char *data, uint32_t len) {
  unsigned char hdr[8] = {(unsigned char)(len >> 24), (unsigned char)(len >> 16), (unsigned char)(len >> 8), (unsigned char)len,
                          (unsigned char)type[0],     (unsigned char)type[1],     (unsigned char)type[2],    (unsigned char)type[3]};
  fwrite(hdr, 1, 8, f);
  if (len) fwrite(data, 1, len, f);
  uint32_t c = crc32_png(hdr + 4, 4, 0xffffffffu);
  if (len) c = crc32_png(data, len, c);
  c ^= 0xffffffffu;
  unsigned char cb[4] = {(unsigned char)(c >> 24), (unsigned char)(c >> 16), (unsigned char)(c >> 8), (unsigned char)c};
  fwrite(cb, 1, 4, f);
}

// value noise for the synthetic height field (integer hash, bilinear, smoothstep)
uint32_t hash2(uint32_t x, uint32_t y, uint32_t seed) {
  uint32_t h = x * 0x8da6b343u ^ y * 0xd8163841u ^ seed * 0xcb1ab31fu;
  h ^= h >> 16;
  h *= 0x7feb352du;
  h ^= h >> 15;
  h *= 0x846ca68bu;
  h ^= h >> 16;
  return h;
}
float lattice(int x, int y, uint32_t seed) { return (float)(hash2((uint32_t)x, (uint32_t)y, seed) >> 8) * (1.0f / 16777216.0f); }
float value_noise(float x, float y, uint32_t seed) {
  const float fx = std::floor(x), fy = std::floor(y);
  const int ix = (int)fx, iy = (int)fy;
  float tx = x - fx, ty = y - fy;
  tx = tx * tx * (3.0f - 2.0f * tx);
  ty = ty * ty * (3.0f - 2.0f * ty);
  const float a = lattice(ix, iy, seed), b = lattice(ix + 1, iy, seed), c = lattice(ix, iy + 1, seed), d = lattice(ix + 1, iy + 1, seed);
  return (a + (b - a) * tx) + ((c + (d - c) * tx) - (a + (b - a) * tx)) * ty;
}

}  // namespace

// =============================================================================================================
extern "C" {

const char *pth_last_error(void) { return g_err.c_str(); }

pth_scene *pth_load_scene_from_json_ex(const char *json_path, int flags) {
  try {
    return load_scene(json_path, flags);
  } catch (std::exception &e) {
    g_err = e.what();
    return nullptr;
  }
}
pth_scene *pth_load_scene_from_json(const char *json_path) { return pth_load_scene_from_json_ex(json_path, 0); }
pth_scene *pth_scene_new(void) { return new pth_scene(); }
void pth_scene_free(pth_scene *s) { delete s; }

int32_t pth_scene_material_count(const pth_scene *s) { return (int32_t)s->materials.size(); }
int32_t pth_scene_object_count(const pth_scene *s) { return (int32_t)s->objects.size(); }
int32_t pth_scene_mesh_count(const pth_scene *s) { return (int32_t)s->meshes.size(); }
const ptc_material *pth_scene_materials(const pth_scene *s) { return s->materials.data(); }
const pth_object *pth_scene_objects(const pth_scene *s) { return s->objects.data(); }
int64_t pth_scene_mesh(const pth_scene *s, int32_t mesh, const float **tris) {
  if (mesh < 0 || (size_t)mesh >= s->meshes.size()) return -1;
  if (tris) *tris = s->meshes[(size_t)mesh].data();
  return (int64_t)(s->meshes[(size_t)mesh].size() / 12);
}
int pth_scene_sky(const pth_scene *s, const float **rgb, int32_t *w, int32_t *h) {
  if (s->sky.empty()) return 0;
  if (rgb) *rgb = s->sky.data();
  if (w) *w = s->sky_w;
  if (h) *h = s->sky_h;
  return 1;
}
void pth_scene_camera(const pth_scene *s, ptc_camera *c) { *c = s->camera; }
int pth_scene_lens(const pth_scene *s, ptc_lens *out) {
  if (!s->has_lens) return 0;
  if (out) *out = s->lens;
  return 1;
}
void pth_scene_settings(const pth_scene *s, int32_t *w, int32_t *h, int32_t *spp, int32_t *md) {
  if (w) *w = s->width;
  if (h) *h = s->height;
  if (spp) *spp = s->spp;
  if (md) *md = s->max_depth;
}

int pth_scene_push_material(pth_scene *s, const ptc_material *m) {
  ptc_material c = *m;
  if (c.type == PTC_MAT_METAL) c.fuzz = c.fuzz < 0.0f ? 0.0f : (c.fuzz > 1.0f ? 1.0f : c.fuzz);
  if (c.type == PTC_MAT_ROUGH_CONDUCTOR) c.roughness = std::fmax(c.roughness, 0.01f);
  s->materials.push_back(c);
  return (int)s->materials.size() - 1;
}
int pth_scene_push_sphere(pth_scene *s, const float c[3], float radius, int material) {
  pth_object o = obj_blank(PTH_SPHERE, material);
  memcpy(o.center, c, 12);
  o.radius = radius;
  s->objects.push_back(o);
  return (int)s->objects.size() - 1;
}
int pth_scene_push_plane(pth_scene *s, const float point[3], const float normal[3], int material) {
  pth_object o = obj_blank(PTH_PLANE, material);
  V n = normalized({normal[0], normal[1], normal[2]});
  memcpy(o.p1, point, 12);
  o.normal[0] = n.x, o.normal[1] = n.y, o.normal[2] = n.z;
  s->objects.push_back(o);
  return (int)s->objects.size() - 1;
}
int pth_scene_push_quad(pth_scene *s, const float scale[3], const float rot[3], const float pos[3], int material) {
  float o2w[16], w2o[16];
  transform_from({scale[0], scale[1], scale[2]}, {rot[0], rot[1], rot[2]}, {pos[0], pos[1], pos[2]}, o2w, w2o);
  s->objects.push_back(make_quad(o2w, material));
  return (int)s->objects.size() - 1;
}
int pth_scene_push_cube(pth_scene *s, const float scale[3], const float rot[3], const float pos[3], int material) {
  pth_object o = obj_blank(PTH_CUBE, material);
  transform_from({scale[0], scale[1], scale[2]}, {rot[0], rot[1], rot[2]}, {pos[0], pos[1], pos[2]}, o.o2w, o.w2o);
  s->objects.push_back(o);
  return (int)s->objects.size() - 1;
}
int pth_scene_push_mesh(pth_scene *s, const float *verts, int64_t nv, const int32_t *indices, int64_t nt, const float scale[3],
                        const float rot[3], const float pos[3], int material) {
  std::vector<float> tris;
  tris.reserve((size_t)nt * 12);
  for (int64_t i = 0; i < nt; i++) {
    const int32_t a = indices[i * 3], b = indices[i * 3 + 1], c = indices[i * 3 + 2];
    if (a < 0 || b < 0 || c < 0 || a >= nv || b >= nv || c >= nv) continue;  // mesh_object.rs:114-119
    push_triangle(tris, {verts[a * 3], verts[a * 3 + 1], verts[a * 3 + 2]}, {verts[b * 3], verts[b * 3 + 1], verts[b * 3 + 2]},
                  {verts[c * 3], verts[c * 3 + 1], verts[c * 3 + 2]});
  }
  if (tris.empty()) {
    g_err = "No valid, non-degenerate triangles loaded for mesh";
    return -1;
  }
  pth_object o = obj_blank(PTH_MESH, material);
  transform_from({scale[0], scale[1], scale[2]}, {rot[0], rot[1], rot[2]}, {pos[0], pos[1], pos[2]}, o.o2w, o.w2o);
  o.mesh = (int32_t)s->meshes.size();
  s->meshes.push_back(std::move(tris));
  s->objects.push_back(o);
  return (int)s->objects.size() - 1;
}
int pth_scene_push_obj(pth_scene *s, const char *obj_path, const float scale[3], const float rot[3], const float pos[3],
                       int material) {
  std::vector<float> tris;
  std::string err;
  if (!load_obj_triangles(obj_path, tris, err)) {
    g_err = err;
    return -1;
  }
  pth_object o = obj_blank(PTH_MESH, material);
  transform_from({scale[0], scale[1], scale[2]}, {rot[0], rot[1], rot[2]}, {pos[0], pos[1], pos[2]}, o.o2w, o.w2o);
  o.mesh = (int32_t)s->meshes.size();
  s->meshes.push_back(std::move(tris));
  s->objects.push_back(o);
  return (int)s->objects.size() - 1;
}
int pth_scene_set_sky_hdr_file(pth_scene *s, const char *hdr_path) {
  std::string err;
  int w, h;
  std::vector<float> rgb;
  if (!load_hdr(hdr_path, rgb, w, h, err)) {
    g_err = err;
    return -1;
  }
  s->sky = std::move(rgb);
  s->sky_w = w;
  s->sky_h = h;
  return 0;
}
int pth_scene_set_sky_rgb(pth_scene *s, const float *rgb, int32_t w, int32_t h) {
  s->sky.assign(rgb, rgb + (size_t)w * h * 3);
  s->sky_w = w;
  s->sky_h = h;
  return 0;
}
void pth_scene_set_camera(pth_scene *s, const float position[3], const float look_at[3], const float up[3], float vfov_deg,
                          float aspect) {
  camera_new({position[0], position[1], position[2]}, {look_at[0], look_at[1], look_at[2]}, {up[0], up[1], up[2]}, vfov_deg,
             aspect, &s->camera);
}
void pth_scene_set_settings(pth_scene *s, int32_t width, int32_t height, int32_t spp, int32_t max_depth) {
  s->width = width, s->height = height, s->spp = spp, s->max_depth = max_depth;
}

void pth_transform(const float scale[3], const float rot[3], const float pos[3], float o2w[16], float w2o[16]) {
  transform_from({scale[0], scale[1], scale[2]}, {rot[0], rot[1], rot[2]}, {pos[0], pos[1], pos[2]}, o2w, w2o);
}
void pth_camera_new(const float position[3], const float look_at[3], const float up[3], float vfov_deg, float aspect,
                    ptc_camera *out) {
  camera_new({position[0], position[1], position[2]}, {look_at[0], look_at[1], look_at[2]}, {up[0], up[1], up[2]}, vfov_deg,
             aspect, out);
}

// BASELINE config C5 (SURVEY.md §8d): cells x cells x 2 triangles over [-50,50]^2, y = 4 octaves of value noise.
pth_scene *pth_scene_synthetic(int32_t cells, uint32_t seed) {
  if (cells < 1) cells = 1;
  std::unique_ptr<pth_scene> s(new pth_scene());
  const int n = cells + 1;
  std::vector<float> verts((size_t)n * n * 3);
  for (int j = 0; j < n; j++)
    for (int i = 0; i < n; i++) {
      const float x = -50.0f + 100.0f * (float)i / (float)cells;
      const float z = -50.0f + 100.0f * (float)j / (float)cells;
      float y = 0.0f, amp = 6.0f, freq = 0.04f;
      for (int o = 0; o < 4; o++) {
        y += amp * value_noise(x * freq + 17.0f, z * freq + 31.0f, seed + (uint32_t)o);
        amp *= 0.5f;
        freq *= 2.0f;
      }
      float *v = &verts[((size_t)j * n + i) * 3];
      v[0] = x, v[1] = y, v[2] = z;
    }
  std::vector<int32_t> idx;
  idx.reserve((size_t)cells * cells * 6);
  for (int j = 0; j < cells; j++)
    for (int i = 0; i < cells; i++) {
      const int32_t a = j * n + i, b = a + 1, c = a + n, d = c + 1;
      const int32_t t[6] = {a, c, b, b, c, d};
      idx.insert(idx.end(), t, t + 6);
    }
  const float gray[3] = {0.7f, 0.7f, 0.7f};
  const int lam = pth_scene_push_material(s.get(), &(const ptc_material &)mat_lambert(gray[0], gray[1], gray[2]));
  ptc_material glass = mat_dielectric(1.5f);
  const int gl = pth_scene_push_material(s.get(), &glass);
  const float white[3] = {1.0f, 1.0f, 1.0f};
  ptc_material al = mat_rough_conductor(white, 0.1f, "al", PTC_DIST_GGX);
  const int alm = pth_scene_push_material(s.get(), &al);
  ptc_material light = mat_emissive(12.0f, 12.0f, 12.0f);
  const int lm = pth_scene_push_material(s.get(), &light);
  const float one[3] = {1, 1, 1}, zero[3] = {0, 0, 0};
  pth_scene_push_mesh(s.get(), verts.data(), (int64_t)n * n, idx.data(), (int64_t)cells * cells * 2, one, zero, zero, lam);
  const float sc[3] = {10.0f, 14.0f, 0.0f};
  pth_scene_push_sphere(s.get(), sc, 5.0f, gl);
  const float cs[3] = {8, 8, 8}, cr[3] = {0, 30, 0}, cp[3] = {-14.0f, 13.0f, 8.0f};
  pth_scene_push_cube(s.get(), cs, cr, cp, alm);
  const float qs[3] = {40, 1, 40}, qr[3] = {0, 0, 0}, qp[3] = {0.0f, 45.0f, 0.0f};
  pth_scene_push_quad(s.get(), qs, qr, qp, lm);
  const float cpos[3] = {60, 40, 60}, clook[3] = {0, 5, 0}, cup[3] = {0, 1, 0};
  pth_scene_set_settings(s.get(), 3840, 2160, 256, 16);
  pth_scene_set_camera(s.get(), cpos, clook, cup, 45.0f, 3840.0f / 2160.0f);
  return s.release();
}

// The product core is bound when first needed, not at link time: loading a scene description (tests of the loader, the
// CPU reference arm of bench.py) must not map the CUDA library.  libptcore.so is looked up next to this library.
namespace {
struct CoreApi {
  decltype(&::ptc_last_error) last_error = nullptr;
  decltype(&::ptc_scene_create) scene_create = nullptr;
  decltype(&::ptc_scene_destroy) scene_destroy = nullptr;
  decltype(&::ptc_scene_add_material) add_material = nullptr;
  decltype(&::ptc_scene_add_sphere) add_sphere = nullptr;
  decltype(&::ptc_scene_add_plane) add_plane = nullptr;
  decltype(&::ptc_scene_add_quad) add_quad = nullptr;
  decltype(&::ptc_scene_add_cube) add_cube = nullptr;
  decltype(&::ptc_scene_add_mesh) add_mesh = nullptr;
  decltype(&::ptc_scene_set_sky_hdr) set_sky_hdr = nullptr;
  decltype(&::ptc_scene_commit) commit = nullptr;
  decltype(&::ptc_render_u32) render_u32 = nullptr;
  decltype(&::ptc_scene_set_lens) set_lens = nullptr;
  bool ok = false;
  std::string err;
  CoreApi() {
    void *lib = nullptr;
    Dl_info info;
    if (dladdr((void *)&pth_last_error, &info) && info.dli_fname) {
      std::string dir(info.dli_fname);
      const size_t k = dir.rfind('/');
      dir = k == std::string::npos ? std::string(".") : dir.substr(0, k);
      lib = dlopen((dir + "/libptcore.so").c_str(), RTLD_NOW | RTLD_GLOBAL);
    }
    if (!lib) lib = dlopen("libptcore.so", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) {
      err = std::string("libptcore.so not found (the path tracer has no CPU fallback): ") + dlerror();
      return;
    }
    bool all = true;
    auto bind = [&](auto &fn, const char *name) {
      fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(dlsym(lib, name));
      if (!fn) all = false, err = std::string("libptcore.so does not export ") + name;
    };
    bind(last_error, "ptc_last_error"), bind(scene_create, "ptc_scene_create"), bind(scene_destroy, "ptc_scene_destroy");
    bind(add_material, "ptc_scene_add_material"), bind(add_sphere, "ptc_scene_add_sphere"), bind(add_plane, "ptc_scene_add_plane");
    bind(add_quad, "ptc_scene_add_quad"), bind(add_cube, "ptc_scene_add_cube"), bind(add_mesh, "ptc_scene_add_mesh");
    bind(set_sky_hdr, "ptc_scene_set_sky_hdr"), bind(commit, "ptc_scene_commit"), bind(render_u32, "ptc_render_u32");
    bind(set_lens, "ptc_scene_set_lens");
    ok = all;
  }
};
const CoreApi *core_api() {
  static const CoreApi api;
  if (!api.ok) {
    g_err = api.err;
    return nullptr;
  }
  return &api;
}
}  // namespace

ptc_scene *pth_build_ptc_scene(const pth_scene *s) {
  const CoreApi *api = core_api();
  if (!api) return nullptr;
  ptc_scene *c = api->scene_create();
  if (!c) {
    g_err = api->last_error();
    return nullptr;
  }
  auto fail = [&]() -> ptc_scene * {
    g_err = api->last_error();
    api->scene_destroy(c);
    return nullptr;
  };
  for (const ptc_material &m : s->materials)
    if (api->add_material(c, &m) < 0) return fail();
  for (const pth_object &o : s->objects) {
    int r = 0;
    switch (o.type) {
      case PTH_SPHERE: r = api->add_sphere(c, o.center, o.radius, o.material); break;
      case PTH_PLANE: r = api->add_plane(c, o.p1, o.normal, o.material); break;
      case PTH_QUAD:
        r = api->add_quad(c, o.base, o.edge0, o.edge1, o.normal, o.d, o.inv_edge0_len_sq, o.inv_edge1_len_sq, o.material);
        break;
      case PTH_CUBE: r = api->add_cube(c, o.o2w, o.w2o, o.material); break;
      case PTH_MESH: {
        const std::vector<float> &t = s->meshes[(size_t)o.mesh];
        r = api->add_mesh(c, t.data(), (int64_t)(t.size() / 12), o.o2w, o.w2o, o.material);
        break;
      }
      default: r = PTC_E_INVALID;
    }
    if (r < 0) return fail();
  }
  if (!s->sky.empty() && api->set_sky_hdr(c, s->sky.data(), s->sky_w, s->sky_h) < 0) return fail();
  if (s->has_lens && api->set_lens(c, &s->lens, 1) < 0) return fail();
  return c;
}

// render_scene (renderer.rs:67-123): everything between the two lines of that function is the GPU core.
int pth_render_scene(const pth_scene *s, int device, uint32_t *out_u32, ptc_stats *stats) {
  const CoreApi *api = core_api();
  if (!api) return PTC_E_INVALID;
  ptc_scene *c = pth_build_ptc_scene(s);
  if (!c) return PTC_E_INVALID;
  int r = api->commit(c, device);
  if (r == 0) {
    ptc_render_settings st;
    memset(&st, 0, sizeof(st));
    st.width = s->width, st.height = s->height, st.spp = s->spp, st.max_depth = s->max_depth;
    r = api->render_u32(c, &s->camera, &st, out_u32, stats);
  }
  if (r != 0) g_err = api->last_error();
  api->scene_destroy(c);
  return r;
}

int pth_save_png(const char *path, const uint32_t *buffer, int32_t width, int32_t height) {
  // renderer.rs:129-141: 0x00RRGGBB -> Rgb<u8>
  std::vector<unsigned char> raw((size_t)height * ((size_t)width * 3 + 1));
  for (int y = 0; y < height; y++) {
    unsigned char *row = &raw[(size_t)y * ((size_t)width * 3 + 1)];
    row[0] = 0;
    for (int x = 0; x < width; x++) {
      const uint32_t px = buffer[(size_t)y * width + x];
      row[1 + x * 3] = (unsigned char)((px >> 16) & 0xff);
      row[2 + x * 3] = (unsigned char)((px >> 8) & 0xff);
      row[3 + x * 3] = (unsigned char)(px & 0xff);
    }
  }
  uLongf zlen = compressBound((uLong)raw.size());
  std::vector<unsigned char> z(zlen);
  if (compress2(z.data(), &zlen, raw.data(), (uLong)raw.size(), 6) != Z_OK) {
    g_err = "zlib compress failed";
    return -1;
  }
  FILE *f = fopen(path, "wb");
  if (!f) {
    g_err = std::string("cannot open for writing: ") + path;
    return -1;
  }
  static const unsigned char sig[8] = {0x89, 'P', 'N', 'G', 0x0d, 0x0a, 0x1a, 0x0a};
  fwrite(sig, 1, 8, f);
  unsigned char ihdr[13] = {(unsigned char)(width >> 24), (unsigned char)(width >> 16), (unsigned char)(width >> 8),
                            (unsigned char)width,         (unsigned char)(height >> 24), (unsigned char)(height >> 16),
                            (unsigned char)(height >> 8), (unsigned char)height,         8, 2, 0, 0, 0};
  png_chunk(f, "IHDR", ihdr, 13);
  png_chunk(f, "IDAT", z.data(), (uint32_t)zlen);
  png_chunk(f, "IEND", nullptr, 0);
  fclose(f);
  return 0;
}

}  // extern "C"
