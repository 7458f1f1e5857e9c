// pt_types.h — flattened scene as the kernels see it (plain data, shared by the host builder and the kernels).
#pragma once
#include "pt_hd.h"

namespace pt {

enum ObjType : int32_t { OBJ_SPHERE = 0, OBJ_PLANE = 1, OBJ_QUAD = 2, OBJ_CUBE = 3, OBJ_MESH = 4 };

// One entry of Scene.object_list (src/hittable.rs:28-44), in insertion order.  48 floats of parameters:
//   sphere  f[0..2] center, f[3] radius                                   (src/objects/sphere.rs:8-12)
//   plane   f[0..2] p1, f[3..5] normal                                    (src/objects/plane.rs:9-13)
//   quad    f[0..2] base, f[3..5] edge0, f[6..8] edge1, f[9..11] normal,
//           f[12] d, f[13] inv_edge0_len_sq, f[14] inv_edge1_len_sq       (src/tungsten/objects/quad.rs:10-18)
//   cube    f[0..15] world_to_object, f[16..31] object_to_world           (src/objects/cube.rs:11-17)
//   mesh    like cube; `mesh` indexes the mesh table                      (src/mesh/mesh_object.rs:17-22)
struct alignas(16) DObject {
  int32_t type;
  int32_t material;
  int32_t mesh;
  int32_t hit_bits;  // filled at commit: DMaterial::type << 26 | light id << 20 | material — what the extend stage ORs into the
                     // hit record (the shade stage's sort key and the NEE light of the object ride along with the material)
  float f[32];
};
static_assert(sizeof(DObject) == 144, "DObject layout");

// Material table entry; field meaning as ptc_material (include/ptcore.h).
struct alignas(16) DMaterial {
  int32_t type;
  int32_t distribution;
  float fuzz, ior;
  float albedo[3];
  float roughness;
  float off_color[3];
  float inv_scale;
  float eta[3];
  float pad0;
  float k[3];
  float pad1;
};
static_assert(sizeof(DMaterial) == 80, "DMaterial layout");

// 8-wide BVH node with child boxes quantised to 8 bits in a per-node frame; 80 bytes = five 16-byte loads.
// (layout after Ylitie, Karras & Laine 2017, "Efficient Incoherent Ray Traversal on GPUs Through Compressed
// Wide BVHs")
//   q0: origin.x, origin.y, origin.z, [ex | ey<<8 | ez<<16 | imask<<24]   frame origin, per-axis scale exponents
//                                                                         (IEEE biased), imask bit s = slot s is an
//                                                                         inner node
//   q1: child_base, tri_base, meta[0..3], meta[4..7]                      meta[s]: 0 = empty; inner = 0x20 | (24+s);
//                                                                         leaf = (unary tri count)<<5 | tri offset
//   q2: qlo_x[0..7], qlo_y[0..7]
//   q3: qlo_z[0..7], qhi_x[0..7]
//   q4: qhi_y[0..7], qhi_z[0..7]
struct alignas(16) Node8 {
  float4 q[5];
};
static_assert(sizeof(Node8) == 80, "Node8 layout");

// Triangle record, 48 bytes = three 16-byte loads:
//   t0: v0.xyz,        original triangle index (as passed to add_mesh) bit-cast
//   t1: v1-v0 (edge1), position in the reference BVH's depth-first leaf order bit-cast (tie-break key)
//   t2: v2-v0 (edge2), 0
struct alignas(16) Tri48 {
  float4 t[3];
};

struct DMesh {
  const float4 *nodes;    // Node8 array, root = node 0
  const float4 *tris;     // Tri48 array in leaf order
  const float4 *normals;  // Triangle.normal by position in the reference's DFS leaf order, original index bit-cast in .w
  int32_t n_nodes, n_tris;
  float root_lo[3], root_hi[3];  // padded frame of the root node: a ray that misses it cannot hit any live triangle
};

// An emitter that next-event estimation can sample (PTC_FLAG_NEE; the reference has no light sampling): emissive spheres
// and quads.  Other emissive objects are found by BSDF sampling alone, like every emitter in the reference.
struct alignas(16) DLight {
  int32_t type;    // OBJ_SPHERE or OBJ_QUAD
  int32_t object;  // index in the object table
  float area;      // 4 pi r^2 / |edge0 x edge1|
  float pad;
  float f[12];     // sphere: center, radius | quad: base, edge0, edge1, normal
  float emission[3];
  float pad2;
};
constexpr int kMaxLights = 63;  // light id 1..63 in the hit record's 6 bits; further emitters are simply not sampled

// The HDR sky as a light (PTC_FLAG_NEE_SKY).  The reference's lookup (pt_bsdf.h: sky_texel) makes a w x h sky piecewise
// constant over Wc x Hc cells, Wc = max(w - 1, 1), Hc = max(h - 1, 1): cell (x, y) has the radiance of texel (x, y) and
// covers phi in [2 pi x / Wc, 2 pi (x + 1) / Wc), theta in [pi y / Hc, pi (y + 1) / Hc).  (The last texel column and row
// are looked up on a set of measure zero only: they have probability 0.)  DScene::sky_dist holds, as floats:
//   marg   [Hc + 1]         marginal CDF over the rows, 0 ... 1
//   cos    [Hc + 1]         cos(pi y / Hc): the theta bounds of the rows
//   inv_sa [Hc]             1 / solid angle of one cell of row y
//   cond   [Hc][Wc + 1]     conditional CDF over the columns of row y, 0 ... 1
// Built on the host (HostScene::build_all), from weights max(r, g, b) x solid angle summed in double.
struct SkyDist {
  const float *marg, *cos, *inv_sa, *cond;
  int32_t wc, hc;
};
PT_HD int32_t sky_cells(int32_t texels) { return texels > 1 ? texels - 1 : 1; }
PT_HD size_t sky_dist_size(int32_t w, int32_t h) {
  const size_t wc = (size_t)sky_cells(w), hc = (size_t)sky_cells(h);
  return 3 * hc + 2 + hc * (wc + 1);
}
PT_HD SkyDist sky_dist_view(const float *p, int32_t w, int32_t h) {
  SkyDist d;
  d.wc = sky_cells(w), d.hc = sky_cells(h);
  d.marg = p;
  d.cos = p + d.hc + 1;
  d.inv_sa = p + 2 * d.hc + 2;
  d.cond = p + 3 * d.hc + 2;
  return d;
}

struct DScene {
  const DObject *objects;
  const DMaterial *materials;
  const DMesh *meshes;
  const float *sky;  // w*h*3 floats or nullptr (Scene.skybox_hdr_image, src/scene.rs:9)
  const DLight *lights;
  int32_t n_objects, n_materials, n_meshes;
  int32_t sky_w, sky_h;
  int32_t n_lights;
  // PTC_FLAG_NEE_SKY: the sky as a light (pt_bsdf.h: sky_sample / sky_pdf); nullptr without a sky or with an all-zero one.
  // sky_dist_size(sky_w, sky_h) floats, see SkyDist.  (Last, and padded to 16 bytes: the kernels' other parameters keep
  // their offsets modulo 16, hence their 128-bit constant loads.)
  const float *sky_dist;
  int32_t pad[2];
};

// HitRecord (src/hittable.rs:10-16) + the ids the parity bar is stated on.
struct Hit {
  float t;
  float px, py, pz;
  float nx, ny, nz;
  int32_t object;    // -1 = miss
  int32_t triangle;  // original index, -1 for analytic primitives
  int32_t material;
  int32_t front_face;
};

// Traversal counters for the instrumented build of extend (PTC_FLAG_COUNTERS)
struct TraversalCounters {
  uint32_t nodes, tris, mesh_rays;
};

constexpr int kTraversalStack = 48;  // uint2 entries; ptc_scene_commit refuses BVHs that could need more

}  // namespace pt
