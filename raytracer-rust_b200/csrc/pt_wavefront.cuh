// pt_wavefront.cuh — the wavefront kernels of the B200 path-tracing core (included by ptcore.cu only).
//
// trace_ray's recursion  L = Le + f * trace(next)  (src/renderer.rs:19-65 of the reference) is unrolled into a
// SEGMENTED wavefront.  The path pool is cut into S segments of `cap` slots, S = resident blocks of the GPU; block b of
// every kernel owns segment b and nothing else:
//
//   k_extend_pre   analytic primitives of the object list up to the first mesh whose root-frame test passes; such a
//                  ray is PARKED as a task in the block's task segment (shared-memory cursor)
//   k_traverse     persistent warps over the block's tasks: each lane walks its own BVH one step at a time, idle lanes
//                  refetch from the block's cursor
//   k_extend_post  second half of Mesh::hit + rest of the object list for every task; may park again (next round)
//   k_shade        counting-sorts 2048-ray windows of the segment by material class (keys only, in shared memory), every
//                  warp shades 8 class-homogeneous 32-ray groups spread over the sorted window (gathered straight from
//                  global memory), survivors go to the front of the segment's OTHER ray buffer (ping-pong), then the
//                  block REGENERATES: tops the segment up with fresh camera paths (Philox jitter + Camera::get_ray)
//
// Consequences: no global compaction, no global queue cursor — the only same-address global atomics left are one
// `next_path` reservation and one ray-count add per block and iteration (per-warp atomics on single counters were 16-56 %
// of the stall samples of the previous design, profiles/r1_v3_*); a block never needs another block's data, so the
// launches of a render are ordered per SEGMENT, not per launch (stage_begin / stage_end below); the ray arrays are ping-ponged between two sets (k_shade reads one, writes the other); each block's working
// set stays in its own slice of memory; when the path supply runs out all segments drain together, so the tail needs
// no repacking either.  (A persistent one-kernel variant and a two-stream variant of this loop were measured slower on
// B200 and removed; DESIGN.md section 5 keeps the numbers.)
//
// Only Emissive surfaces and the sky carry radiance and both end the path (EmissiveLight::scatter is None), so a path
// contributes beta * Le exactly once, when it terminates: one 64-bit integer RED triple per path into the fixed-point film.
#pragma once
#include <cuda_runtime.h>

#include <type_traits>

#include "../../include/ptcore.h"
#include "pt_adaptive.h"
#include "pt_bsdf.h"
#include "pt_philox.h"
#include "pt_prims.h"

namespace ptw {
using namespace pt;

constexpr int kBlock = 256;    // threads per block of every stage kernel
constexpr int kSegPerSM = 4;   // segments (= resident blocks) per SM: 4 x 256 threads x <= 64 registers
constexpr uint32_t kRefillLanes = 8;
constexpr uint32_t kNoSteal = 0x80000000u;  // bit of k_traverse's `refill_lanes` argument: in-warp work stealing off (measurements)
constexpr unsigned long long kNoTriHit = ~0ull;  // a traversal warp fetches new tasks once this many lanes are idle

// Device-side control block of one render
struct Ctl {
  unsigned long long next_path;    // next camera path index to hand out
  unsigned long long total_paths;  // path index space of this call (padded tiles x samples)
  unsigned long long rays;         // extend items so far = trace_ray calls with depth > 0
  unsigned long long nodes, tris, mesh_rays;  // PTC_FLAG_COUNTERS
  uint32_t n_active;       // segments that are not yet empty for good (see stage_shade); 0 = the render is over
  uint32_t sync_timeouts;  // stage_begin gave up waiting for a segment's previous stage (must stay 0)
  uint32_t iterations[2];  // [0]: the last iteration that had a ray to extend
};

// A kernel launch covers segments [seg0, seg0 + gridDim.x).
struct SegRange {
  uint32_t seg0;   // first segment of this launch
  uint32_t n_seg;  // segments of the whole pool (stride of the task-count table)
  uint32_t half;   // (unused)
  uint32_t trav_seq, trav_parts;  // k_traverse only: sequence number of the launch, parts every segment's task list is cut into
  // Segment-level ordering of the launches of a render (stage_begin / stage_end below).  flags[seg] = number of the last
  // launch that finished this segment; flags[n_seg + seg] = 1 once the segment is empty for good; [2 * n_seg + seg]: see
  // trav_counter.  nullptr: stream order alone (ptc_intersect).
  uint32_t *flags;
  uint32_t stage_id;   // number of this launch, 1, 2, 3, ... within the render
  uint32_t flag_wait;  // 1: a block waits for ITS segment's flag to reach stage_id - 1; 0: for the whole preceding launch
  // k_traverse with trav_parts > 1 only: this launch's own hand-out counter (zeroed by the host before the render; a
  // counter per launch, so that launches far apart may overlap); flags[2 * n_seg + seg] counts the finished parts of a segment
  uint32_t *trav_counter;
};

struct RenderParams {
  DCamera cam;
  int32_t width, height;
  int32_t max_depth;
  int32_t sample_begin, n_samples;
  int32_t tiles_x, n_my_tiles, tile_mod, tile_rem;
  uint32_t row_mult;  // odd, coprime with n_my_tiles: scatters consecutive 32-pixel rows over the image (see k_shade)
  uint64_t seed;
  // ptc_render_adaptive's later passes: the pixels to start paths for (ascending; padded to a multiple of 32 by index
  // space only, entries >= n_list start no path); read by k_shade<Mode, true> only, nullptr otherwise
  const uint32_t *pixel_list;
  uint32_t n_list;
};

// ptc_render_batch: n views of one scene as ONE job.  The path index space is n_views stacked tile grids (local tile t
// -> view t / tiles_per_view, tile t % tiles_per_view); a pool entry's pixel word holds the global film index
// view * view_px + pixel.  Philox is keyed on the view's seed and the pixel within the view, so view k is, bit for bit,
// the single render of cams[k] with seeds[k].  Read by k_shade_batch only: a kernel argument of its own, so that the
// parameters of every other kernel keep their layout.
struct BatchTables {
  const DCamera *cams;    // [n_views]
  const uint64_t *seeds;  // [n_views]
  uint32_t view_px;       // width * height
  uint32_t tiles_per_view;
};

// ptc_scene_set_lens: (aperture radius, focus distance) per view (a single render is view 0).  Read by k_shade_lens and
// k_primary_rays_lens only: a trailing kernel argument of their own, like BatchTables.
struct LensTables {
  const float2 *lens;
};

// Motion blur (DESIGN.md 5l): the displacement D_k of every object over the shutter, the end camera of every view (a
// single render is view 0; nullptr: a static camera), and the shutter time of every ray of the two ray sets (`tau` is
// read, `ntau` written by k_shade; the host swaps them with the nray_* arrays).  Read by the *_motion kernels only: a
// trailing kernel argument of their own, like LensTables, so that Buffers, RenderParams, DObject and DScene keep their
// layout and every other kernel its instructions.
struct MotionTables {
  const float4 *disp;        // [n_objects]: D_k in .xyz
  const DCamera *end_cams;   // [views] or nullptr
  const float *tau;
  float *ntau;
};

// Path state, SoA of float4.  Segment b = slots [b * cap, b * cap + cnt[b]).
struct Buffers {
  float4 *ray_o;  // origin.xyz, pixel index
  float4 *ray_d;  // direction.xyz, sample index
  float4 *beta;   // throughput.rgb, bounce (segments already traced)
  float4 *hit0;   // position.xyz, t
  float4 *hit1;   // normal.xyz, [hit<<31 | front_face<<30 | material]
  uint32_t *cnt;  // [S]
  uint32_t cap;   // multiple of kBlock
  // the ray arrays the shade stage writes (survivors + regenerated paths); the host swaps the two sets every iteration
  float4 *nray_o, *nray_d, *nbeta;
  // PTC_FLAG_NEE only: solid-angle pdf with which the ray's direction was sampled (-1: camera ray / delta lobe), for the MIS
  // weight of an emitter it may hit; nullptr otherwise
  float *aux, *naux;
};

struct ExtendOut {
  Buffers b;
  int2 *ids;  // (object, triangle) per ray, only for ptc_intersect (nullptr in renders)
};

// Parked-ray tasks, [round & 1]; block b's tasks of round r = slots [b * cap, b * cap + cnt[r * S + b])
struct TaskQ {
  uint2 *ray[2];   // x = ray slot, y = object index of the mesh
  float4 *o[2];    // object-space origin, closest_so_far (the t_max Mesh::hit was called with)
  float4 *d[2];    // object-space direction (normalised twice, mesh_object.rs:287 + ray.rs:15)
  unsigned long long *res[2];  // traversal result: f2u(t) << 32 | reference DFS position of the triangle (kNoTriHit = none); set to
                               // kNoTriHit when the ray is parked, lowered with atomicMin by every lane that worked on the task
  uint32_t *cnt;   // [(rounds + 1) * S]
};

// The film a render accumulates into: FIXED-POINT radiance sums, so that the image does not depend on the order in which
// paths terminate (integer addition is associative): the same seed gives the same Vec<u32> bit for bit, run after run,
// for any pool size, any tile / sample sharding and — with the int64 reduce of ptc_multi_* — any number of GPUs, like the
// reference, whose per-pixel sum has a fixed order (renderer.rs:93-102).  (fp32 atomics, round 1, moved <1 % of the pixels
// by one display level from run to run.)  One sample's radiance is rounded to a multiple of 2^-28 (the fp32 RED it
// replaces rounded to an ulp of the running sum, ~2^-17 for a sum of 100) and must be below 2^24 in magnitude; anything
// larger, infinite or NaN sets a per-pixel flag field instead and comes out of the conversion as +-inf / NaN, which is
// what an fp32 sum would hold.  A sum holds 2^35: 2048 samples at the per-sample limit.
constexpr float kFilmScale = 268435456.0f;     // 2^28
constexpr float kFilmSampleMax = 16777216.0f;  // 2^24
struct Film {
  long long *sum;             // [W*H*3] radiance sums * 2^28
  unsigned long long *flags;  // [W*H] nine 7-bit fields: channel c NaN -> field c, +inf -> 3 + c, -inf -> 6 + c (fields ADD up in
                              // the multi-GPU reduce: > 0 means set, good for 127 devices)
};
__device__ __forceinline__ void film_add1(const Film &f, uint32_t pixel, int c, float v) {
  if (fabsf(v) < kFilmSampleMax) {
    atomicAdd(reinterpret_cast<unsigned long long *>(f.sum + (size_t)pixel * 3 + c), (unsigned long long)__float2ll_rn(v * kFilmScale));
  } else {
    const int field = (v != v) ? c : (v > 0.0f ? 3 + c : 6 + c);
    atomicOr(f.flags + pixel, 1ull << (7 * field));
  }
}
__device__ __forceinline__ void film_add(const Film &f, uint32_t pixel, V3 r) {
  film_add1(f, pixel, 0, r.x);
  film_add1(f, pixel, 1, r.y);
  film_add1(f, pixel, 2, r.z);
}
// fixed-point film -> fp32 radiance sum of channel c of a pixel (one rounding)
__device__ __forceinline__ float film_value(long long sum, unsigned long long flags, int c) {
  float v = (float)sum * (1.0f / kFilmScale);
  if (flags) {
    const bool nan = ((flags >> (7 * c)) & 127ull) != 0ull, pinf = ((flags >> (7 * (3 + c))) & 127ull) != 0ull,
               ninf = ((flags >> (7 * (6 + c))) & 127ull) != 0ull;
    if (nan || (pinf && ninf)) v = u2f(0x7fc00000u);
    else if (pinf) v = INFINITY;
    else if (ninf) v = -INFINITY;
  }
  return v;
}

// hit1.w: hit << 31 | front_face << 30 | material type << 26 (the shade stage's sort key) | light id << 20 | material index
constexpr uint32_t kHitBit = 0x80000000u, kFrontBit = 0x40000000u, kMatMask = 0x000fffffu;
constexpr int kTypeShift = 26, kLightShift = 20;  // DObject::hit_bits: type << 26 | NEE light id << 20 | material index
constexpr uint32_t kShadowBit = 0x80000000u;       // in a pool entry's pixel word: the entry is an NEE shadow ray (see stage_shade)
// PTC_FLAG_NEE_EMITTERS: in a shadow ray's bounce word (beta.w), the ray goes to a mesh or cube light, whose id is in the
// low 6 bits: it is unoccluded iff its closest hit is that light at the sampled point (see stage_shade)
constexpr uint32_t kPosTestBit = 0x80000000u;
// The hit point must lie within kPosTestTol x distance + kPosTestAbs x max|coordinate| of the sampled point: the two
// points differ by the rounding of the transforms (a few ulps of the coordinates) only, and two sheets of one emitter
// that are farther apart than this are told apart (10^-4 x distance: 0.2 mm at 2 m)
constexpr float kPosTestTol = 1e-4f, kPosTestAbs = 1e-5f;

__device__ __forceinline__ void write_hit(const ExtendOut &out, uint32_t i, const Hit &h) {
  out.b.hit0[i] = make_float4(h.px, h.py, h.pz, h.t);
  out.b.hit1[i] = make_float4(h.nx, h.ny, h.nz, u2f(kHitBit | (h.front_face ? kFrontBit : 0u) | ((uint32_t)h.material & ~(kHitBit | kFrontBit))));
  if (out.ids) out.ids[i] = make_int2(h.object, h.triangle);
}
__device__ __forceinline__ void write_miss(const ExtendOut &out, uint32_t i) {
  out.b.hit1[i] = make_float4(0.0f, 0.0f, 0.0f, u2f(0u));
  if (out.ids) out.ids[i] = make_int2(-1, -1);
}

// HittableList::hit (hittable.rs:46-57) over objects [k_begin, n): insertion order, shrinking t_max, each primitive's own
// interval convention.  Returns the index of the mesh the ray has to be parked at (its object-space ray in
// `park_ray`), or -1 when the scan is complete.  Every object sees exactly the `closest` it would have seen in the
// reference's sequential scan, so tie-breaking is untouched by the parking.
__device__ __forceinline__ int scan_objects(const DScene &sc, const DObject *objs, const Ray &ray, float t_min, float &closest,
                                            Hit &best, bool &improved, int k_begin, MeshRay &park_ray) {
  for (int k = k_begin; k < sc.n_objects; k++) {
    const DObject *ob = objs + k;
    const int type = ob->type;
    bool hit;
    if (type == OBJ_MESH) {
      const MeshRay mr = mesh_object_ray(ob->f, ray);
      if (!mesh_root_may_hit(sc.meshes[ob->mesh], mr, t_min, closest)) continue;  // same as Mesh::hit returning None
      park_ray = mr;
      return k;
    }
    // the primitives' tests write the record only when they accept the hit, so they can write straight into `best`
    if (type == OBJ_SPHERE) hit = hit_sphere(ob->f, ray, t_min, closest, best);
    else if (type == OBJ_QUAD) hit = hit_quad(ob->f, ray, t_min, closest, best);
    else if (type == OBJ_CUBE) hit = hit_cube_t(ob->f, ray, t_min, closest, best);  // normal: finish_hit, once per ray
    else hit = hit_plane(ob->f, ray, t_min, closest, best);
    if (hit) {
      improved = true;
      closest = best.t;
      best.object = k;
      best.triangle = -1;
      best.material = ob->hit_bits;  // type << 26 | light << 20 | index, see write_hit
    }
  }
  return -1;
}
// The same scan at shutter time tau (motion blur): object k is tested on the ray shifted by -tau D_k (disp, the table in
// shared or global memory), and a hit it reports moves by +tau D_k; an object with D_k == 0 sees `ray` itself.  A mesh
// is parked with the object-space ray of its shifted ray, so k_traverse needs nothing of the motion.
__device__ __forceinline__ int scan_objects_motion(const DScene &sc, const DObject *objs, const Ray &ray, float t_min, float &closest,
                                                   Hit &best, bool &improved, int k_begin, MeshRay &park_ray, const float4 *disp,
                                                   float tau) {
  for (int k = k_begin; k < sc.n_objects; k++) {
    const DObject *ob = objs + k;
    const int type = ob->type;
    const float4 D = disp[k];
    const bool moves = motion_moves(D);
    const Ray r = moves ? motion_object_ray(ray, tau, D) : ray;
    bool hit;
    if (type == OBJ_MESH) {
      const MeshRay mr = mesh_object_ray(ob->f, r);
      if (!mesh_root_may_hit(sc.meshes[ob->mesh], mr, t_min, closest)) continue;
      park_ray = mr;
      return k;
    }
    if (type == OBJ_SPHERE) hit = hit_sphere(ob->f, r, t_min, closest, best);
    else if (type == OBJ_QUAD) hit = hit_quad(ob->f, r, t_min, closest, best);
    else if (type == OBJ_CUBE) hit = hit_cube_t(ob->f, r, t_min, closest, best);
    else hit = hit_plane(ob->f, r, t_min, closest, best);
    if (hit) {
      if (moves) motion_hit_position(best, tau, D);
      improved = true;
      closest = best.t;
      best.object = k;
      best.triangle = -1;
      best.material = ob->hit_bits;
    }
  }
  return -1;
}

// Completes the record that won the scan (pt_prims.h: a cube hit carries its normal as "pending" through the scan).
// cube_finish_normal reads the ray's direction only, which the motion shift leaves as it is: a moving cube's record is
// completed with the same bits from the world ray as from its shifted one.
__device__ __forceinline__ void finish_hit(const DObject *objs, const Ray &ray, Hit &best) {
  if (best.front_face == kCubeNormalPending) cube_finish_normal(objs[best.object].f, ray, best);
}

// The object table is read by every lane for every ray; ray data streaming through L1 kept evicting it (the load of
// `ob->type` alone was 12 % of k_extend_pre's stall samples), so each block stages it into shared memory once.
// The stages are compiled twice, for the table in shared memory (kSharedObjs: loads are LDS, not generic LD) and, for
// scenes with more than kSmemObjects objects, in global memory.
constexpr int kSmemObjects = 24;
template <bool kSharedObjs>
__device__ __forceinline__ const DObject *stage_objects(const DScene &sc, DObject *s_objs) {
  if (!kSharedObjs) return sc.objects;
  const uint4 *src = reinterpret_cast<const uint4 *>(sc.objects);
  uint4 *dst = reinterpret_cast<uint4 *>(s_objs);
  const int n16 = sc.n_objects * (int)(sizeof(DObject) / 16);
  for (int i = threadIdx.x; i < n16; i += blockDim.x) dst[i] = src[i];
  return s_objs;  // visible after the caller's __syncthreads()
}
// ... and the motion kernels stage the displacement table next to it
template <bool kSharedObjs>
__device__ __forceinline__ const float4 *stage_disp(const DScene &sc, const float4 *disp, float4 *s_disp) {
  if constexpr (!kSharedObjs) {
    return disp;
  } else {
    for (int i = threadIdx.x; i < sc.n_objects; i += blockDim.x) s_disp[i] = disp[i];
    return s_disp;  // visible after the caller's __syncthreads()
  }
}

// Append the parked lanes of this warp to the block's task segment: ballot + one SHARED-memory atomic per warp.
__device__ __forceinline__ void park_tasks(uint32_t *s_ntask, const TaskQ &tq, int par, uint32_t seg_base, int park, uint32_t i,
                                           const MeshRay &mr, float closest) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t mask = __ballot_sync(0xffffffffu, park >= 0);
  if (mask == 0u) return;
  uint32_t slot0 = 0;
  if (lane == 0) slot0 = atomicAdd(s_ntask, (uint32_t)__popc(mask));
  slot0 = __shfl_sync(0xffffffffu, slot0, 0);
  if (park >= 0) {
    const uint32_t slot = seg_base + slot0 + (uint32_t)__popc(mask & ((1u << lane) - 1u));
    tq.ray[par][slot] = make_uint2(i, (uint32_t)park);
    tq.o[par][slot] = make_float4(mr.o.x, mr.o.y, mr.o.z, closest);
    tq.d[par][slot] = make_float4(mr.d.x, mr.d.y, mr.d.z, 0.0f);
    tq.res[par][slot] = kNoTriHit;
  }
}

// ---- the four stages, each written for ONE block working on ITS segment; the per-stage kernels below call them.
template <bool kSharedObjs>
__device__ __forceinline__ void stage_pre(uint32_t seg, uint32_t n_seg, const DScene &sc, const ExtendOut &out, const TaskQ &tq,
                                          float t_min, float t_max) {
  __shared__ uint32_t s_ntask;
  __shared__ __align__(16) DObject s_objs[kSmemObjects];
  const uint32_t tid = threadIdx.x;
  const uint32_t n = out.b.cnt[seg], seg_base = seg * out.b.cap;
  if (tid == 0) s_ntask = 0;
  const DObject *objs = kSharedObjs ? s_objs : sc.objects;
  stage_objects<kSharedObjs>(sc, s_objs);
  __syncthreads();
  for (uint32_t c0 = 0; c0 < n; c0 += (uint32_t)kBlock) {
    const uint32_t i = seg_base + c0 + tid;
    int park = -1;
    MeshRay mr;
    float closest = t_max;
    if (c0 + tid < n) {
      const float4 o4 = out.b.ray_o[i], d4 = out.b.ray_d[i];
      const Ray ray{v3(o4.x, o4.y, o4.z), v3(d4.x, d4.y, d4.z)};
      Hit best;
      bool improved = false;
      park = scan_objects(sc, objs, ray, t_min, closest, best, improved, 0, mr);  // renderer.rs:24
      if (improved) finish_hit(objs, ray, best);
      if (improved) write_hit(out, i, best);
      else write_miss(out, i);
    }
    park_tasks(&s_ntask, tq, 0, seg_base, park, i, mr, closest);
  }
  __syncthreads();
  if (tid == 0 && tq.cnt) tq.cnt[seg] = s_ntask;
  (void)n_seg;
}

// Motion blur: stage_pre with every ray at its own shutter time mt.tau[i] (scan_objects_motion)
template <bool kSharedObjs>
__device__ __forceinline__ void stage_pre_motion(uint32_t seg, uint32_t n_seg, const DScene &sc, const ExtendOut &out, const TaskQ &tq,
                                                 float t_min, float t_max, const MotionTables &mt) {
  __shared__ uint32_t s_ntask;
  __shared__ __align__(16) DObject s_objs[kSmemObjects];
  const uint32_t tid = threadIdx.x;
  const uint32_t n = out.b.cnt[seg], seg_base = seg * out.b.cap;
  if (tid == 0) s_ntask = 0;
  const DObject *objs = kSharedObjs ? s_objs : sc.objects;
  stage_objects<kSharedObjs>(sc, s_objs);
  __shared__ float4 s_disp[kSmemObjects];
  const float4 *disp = stage_disp<kSharedObjs>(sc, mt.disp, s_disp);
  __syncthreads();
  for (uint32_t c0 = 0; c0 < n; c0 += (uint32_t)kBlock) {
    const uint32_t i = seg_base + c0 + tid;
    int park = -1;
    MeshRay mr;
    float closest = t_max;
    if (c0 + tid < n) {
      const float4 o4 = out.b.ray_o[i], d4 = out.b.ray_d[i];
      const Ray ray{v3(o4.x, o4.y, o4.z), v3(d4.x, d4.y, d4.z)};
      Hit best;
      bool improved = false;
      park = scan_objects_motion(sc, objs, ray, t_min, closest, best, improved, 0, mr, disp, mt.tau[i]);  // renderer.rs:24
      if (improved) finish_hit(objs, ray, best);
      if (improved) write_hit(out, i, best);
      else write_miss(out, i);
    }
    park_tasks(&s_ntask, tq, 0, seg_base, park, i, mr, closest);
  }
  __syncthreads();
  if (tid == 0 && tq.cnt) tq.cnt[seg] = s_ntask;
  (void)n_seg;
}

// Persistent warps over the block's tasks; every lane walks its own BVH one step at a time and idle lanes refetch from
// the block's cursor.  Once the cursor is exhausted, idle lanes STEAL from busy ones of their warp: a donor hands over the
// bottom entry of its stack (the farthest pending node group) or, with an empty stack, the lowest-priority child of the
// group it is working on; the thief copies the donor's ray by shuffles and walks that subtree for the same task.  Every
// lane that finds a hit lowers the task's 64-bit result key (t, DFS position) with one atomicMin, so the result is the
// same closest hit whatever the split.  Why: a launch ends when its LAST traversal ends, and in the drain of a render
// (a few deep paths inside the glass sphere) a launch IS one or two 40-step traversals: 36-42 us per launch at ~0.8 us
// per dependent node step (profiles/r1_v4_launches.csv), the largest part of the per-iteration floor that limits strong
// scaling.  Split over the idle lanes the same walk is a few steps deep.
template <bool COUNT>
__device__ __forceinline__ void stage_traverse(uint32_t seg, uint32_t n_seg, Ctl *ctl, const DScene &sc, const TaskQ &tq, int round,
                                               float t_min, uint32_t cap, uint32_t refill_arg, uint32_t part = 0u, uint32_t parts = 1u) {
  __shared__ uint32_t s_cur;
  // tasks [first, first + n) of the segment: the whole list, or one of `parts` equal cuts of it
  const uint32_t n_all = tq.cnt[(uint32_t)round * n_seg + seg];
  const uint32_t first = (uint32_t)((unsigned long long)n_all * part / parts);
  const uint32_t n = (uint32_t)((unsigned long long)n_all * (part + 1u) / parts) - first, seg_base = seg * cap + first;
  const int par = round & 1;
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t lt_mask = (1u << lane) - 1u;
  const uint32_t refill_lanes = refill_arg & ~kNoSteal;
  const bool steal = (refill_arg & kNoSteal) == 0u;
  const uint32_t quota = (n >= (uint32_t)kBlock || !steal) ? 32u : max(1u, (n + (uint32_t)(kBlock / 32) - 1u) / (uint32_t)(kBlock / 32));
  if (threadIdx.x == 0) s_cur = 0;
  __syncthreads();
  TraversalCounters tc{0u, 0u, 0u};
  TravState s;
  DMesh mesh;  // the two pointers of the mesh this lane walks, kept in registers
  mesh.nodes = nullptr, mesh.tris = nullptr;
  uint2 stack[kTraversalStack];
  int sp = 0, sb = 0;  // live entries: [sb, sp)
  bool active = false;
  uint32_t task = 0;
  bool exhausted = n == 0u;
  s.ng = make_uint2(0u, 0u);
  for (;;) {
    const uint32_t idle = __ballot_sync(0xffffffffu, !active);
    if (!exhausted && (idle == 0xffffffffu || (uint32_t)__popc(idle) >= refill_lanes)) {
      // a block with few tasks (the drain of a render: a few dozen per segment) spreads them over all its warps instead
      // of filling the first two: the idle lanes next to every walker are what the stealing below splits long walks over
      const uint32_t cnt = min((uint32_t)__popc(idle), quota);
      uint32_t base = 0;
      if (lane == 0) base = atomicAdd(&s_cur, cnt);  // shared memory: the block's own cursor
      base = __shfl_sync(0xffffffffu, base, 0);
      const uint32_t my_rank = (uint32_t)__popc(idle & lt_mask);
      if (!active && my_rank < cnt) {
        const uint32_t j = base + my_rank;
        if (j < n) {
          const uint32_t slot = seg_base + j;
          const uint2 rk = tq.ray[par][slot];
          // the direction is read exactly once: a streaming load (evict-first) keeps it from pushing BVH nodes out of L1.
          // (ray / origin records are re-read by k_extend_post; streaming them too cost post what it saved here.)
          const float4 o4 = tq.o[par][slot], d4 = __ldcs(&tq.d[par][slot]);
          const DMesh *gm = sc.meshes + sc.objects[rk.y].mesh;
          mesh.nodes = gm->nodes;
          mesh.tris = gm->tris;
          trav_begin(s, v3(o4.x, o4.y, o4.z), v3(d4.x, d4.y, d4.z), t_min, o4.w);  // world t bounds, mesh_object.rs:289-291
          sp = sb = 0;
          task = slot;
          active = true;
          if (COUNT) tc.mesh_rays++;
        }
      }
      if (base + cnt >= n) exhausted = true;
    } else if (steal && exhausted && idle != 0u && idle != 0xffffffffu) {
      const bool can_give = active && (sp > sb || __popc(s.ng.y >> 24) >= 2);
      const uint32_t donors = __ballot_sync(0xffffffffu, can_give);
      if (donors != 0u) {
        const uint32_t pairs = (uint32_t)min(__popc(idle), __popc(donors));
        const bool give = can_give && (uint32_t)__popc(donors & lt_mask) < pairs;
        const uint32_t my_idle_rank = (uint32_t)__popc(idle & lt_mask);
        const bool take = !active && my_idle_rank < pairs;
        uint2 entry = make_uint2(0u, 0u);
        if (give) {
          if (sp > sb) {
            entry = stack[sb++];
          } else {  // split the group in hand: its lowest-priority pending child goes
            const uint32_t pend = s.ng.y & 0xFF000000u, bit = pend & (0u - pend);
            entry = make_uint2(s.ng.x, bit | (s.ng.y & 0xffu));
            s.ng.y &= ~bit;
          }
        }
        const int src = take ? (int)__fns(donors, 0u, (int)my_idle_rank + 1) : (int)lane;
        const float ox = __shfl_sync(0xffffffffu, s.o.x, src), oy = __shfl_sync(0xffffffffu, s.o.y, src), oz = __shfl_sync(0xffffffffu, s.o.z, src);
        const float dx = __shfl_sync(0xffffffffu, s.d.x, src), dy = __shfl_sync(0xffffffffu, s.d.y, src), dz = __shfl_sync(0xffffffffu, s.d.z, src);
        const float ix = __shfl_sync(0xffffffffu, s.idx, src), iy = __shfl_sync(0xffffffffu, s.idy, src), iz = __shfl_sync(0xffffffffu, s.idz, src);
        const float tmn = __shfl_sync(0xffffffffu, s.t_min, src), bt = __shfl_sync(0xffffffffu, s.best_t, src);
        const uint32_t bo = __shfl_sync(0xffffffffu, s.best_order, src), oi = __shfl_sync(0xffffffffu, s.octinv, src);
        const uint32_t ex = __shfl_sync(0xffffffffu, entry.x, src), ey = __shfl_sync(0xffffffffu, entry.y, src);
        const uint32_t tk = __shfl_sync(0xffffffffu, task, src);
        const unsigned long long pn = __shfl_sync(0xffffffffu, (unsigned long long)mesh.nodes, src);
        const unsigned long long ptri = __shfl_sync(0xffffffffu, (unsigned long long)mesh.tris, src);
        if (take) {
          s.o = v3(ox, oy, oz), s.d = v3(dx, dy, dz);
          s.idx = ix, s.idy = iy, s.idz = iz;
          s.t_min = tmn, s.best_t = bt, s.best_order = bo, s.octinv = oi;
          s.best_tri = 0xffffffffu;  // "nothing found by THIS lane": the donor's best only prunes
          s.ng = make_uint2(ex, ey);
          s.tg = make_uint2(0u, 0u), s.tg2 = make_uint2(0u, 0u);
          mesh.nodes = reinterpret_cast<const float4 *>(pn);
          mesh.tris = reinterpret_cast<const float4 *>(ptri);
          task = tk;
          sp = sb = 0;
          active = true;
        }
      }
    }
    if (__ballot_sync(0xffffffffu, active) == 0u) {
      if (exhausted) break;
      continue;
    }
    if (active) {
      // one node step AND one triangle test per turn: the node step does not wait for the lane's pending triangles
      if (!trav_has_node(s)) {
        if (sp > sb) {
          s.ng = stack[--sp];
        } else if (!trav_has_tri(s)) {
          if (s.best_tri != 0xffffffffu) atomicMin(&tq.res[par][task], ((unsigned long long)f2u(s.best_t) << 32) | (unsigned long long)s.best_order);
          active = false;
          s.ng.y = 0u;
        }
        if (sp == sb) sp = sb = 0;
      }
      if (active && trav_has_node(s) && s.tg2.y == 0u) trav_node<COUNT>(mesh, s, stack, sp, &tc);
      if (active && trav_has_tri(s)) trav_tri<COUNT>(mesh, s, &tc);
    }
  }
  if (COUNT) {
    atomicAdd(&ctl->nodes, (unsigned long long)tc.nodes);
    atomicAdd(&ctl->tris, (unsigned long long)tc.tris);
    atomicAdd(&ctl->mesh_rays, (unsigned long long)tc.mesh_rays);
  }
}

template <bool kSharedObjs>
__device__ __forceinline__ void stage_post(uint32_t seg, uint32_t n_seg, const DScene &sc, const ExtendOut &out, const TaskQ &tq,
                                           int round, float t_min, float t_max) {
  __shared__ uint32_t s_ntask;
  __shared__ __align__(16) DObject s_objs[kSmemObjects];
  const uint32_t tid = threadIdx.x;
  const uint32_t n = tq.cnt[(uint32_t)round * n_seg + seg], seg_base = seg * out.b.cap;
  const int par = round & 1;
  if (tid == 0) s_ntask = 0;
  const DObject *objs = kSharedObjs ? s_objs : sc.objects;
  stage_objects<kSharedObjs>(sc, s_objs);
  __syncthreads();
  for (uint32_t c0 = 0; c0 < n; c0 += (uint32_t)kBlock) {
    const uint32_t j = seg_base + c0 + tid;
    int park = -1;
    MeshRay mr;
    float closest = t_max;
    uint32_t i = 0;
    if (c0 + tid < n) {
      const uint2 rk = tq.ray[par][j];
      const unsigned long long res = tq.res[par][j];
      i = rk.x;
      const int k = (int)rk.y;
      const DObject *ob = objs + k;
      const bool tri_hit = res != kNoTriHit;
      const uint32_t order = (uint32_t)res;
      // the stage is bound by the latency of these gathers: issue all of them before the first use
      const float4 o4 = out.b.ray_o[i], d4 = out.b.ray_d[i];
      // closest_so_far travels with the task (the t_max the traversal ran with; == t_max when nothing was hit before the
      // mesh): a sequential 4-byte read instead of two gathered sectors of the hit record (hit0.w, hit1.w) per task
      closest = tq.o[par][j].w;
      float4 nq = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      if (tri_hit) nq = ldg4(sc.meshes[ob->mesh].normals + order);  // normal + original index, by DFS position
      const Ray ray{v3(o4.x, o4.y, o4.z), v3(d4.x, d4.y, d4.z)};
      Hit best;
      best.triangle = -1;
      bool improved = false;
      if (tri_hit) {
        const MeshRay omr = mesh_object_ray<false>(ob->f, ray);  // same inputs, same bits as in k_extend_pre
        MeshHit mh;
        mh.t = u2f((uint32_t)(res >> 32)), mh.tri = f2u(nq.w), mh.order = order;
        Hit tmp;
        if (mesh_finish(ob->f, nq, ray, omr, mh, t_min, closest, tmp)) {
          improved = true;
          closest = tmp.t;
          best = tmp;
          best.object = k;
          best.material = ob->hit_bits;  // type << 26 | light << 20 | index, see write_hit
        }
      }
      park = scan_objects(sc, objs, ray, t_min, closest, best, improved, k + 1, mr);
      if (improved) finish_hit(objs, ray, best);
      if (improved) write_hit(out, i, best);  // otherwise the record parked by the previous stage stands
    }
    park_tasks(&s_ntask, tq, par ^ 1, seg_base, park, i, mr, closest);
  }
  __syncthreads();
  if (tid == 0) tq.cnt[(uint32_t)(round + 1) * n_seg + seg] = s_ntask;
}

// Motion blur: stage_post with the ray at its shutter time mt.tau[i]; the mesh that parked it finishes on the shifted ray,
// as k_extend_pre_motion parked it
template <bool kSharedObjs>
__device__ __forceinline__ void stage_post_motion(uint32_t seg, uint32_t n_seg, const DScene &sc, const ExtendOut &out, const TaskQ &tq,
                                                  int round, float t_min, float t_max, const MotionTables &mt) {
  __shared__ uint32_t s_ntask;
  __shared__ __align__(16) DObject s_objs[kSmemObjects];
  const uint32_t tid = threadIdx.x;
  const uint32_t n = tq.cnt[(uint32_t)round * n_seg + seg], seg_base = seg * out.b.cap;
  const int par = round & 1;
  if (tid == 0) s_ntask = 0;
  const DObject *objs = kSharedObjs ? s_objs : sc.objects;
  stage_objects<kSharedObjs>(sc, s_objs);
  __shared__ float4 s_disp[kSmemObjects];
  const float4 *disp = stage_disp<kSharedObjs>(sc, mt.disp, s_disp);
  __syncthreads();
  for (uint32_t c0 = 0; c0 < n; c0 += (uint32_t)kBlock) {
    const uint32_t j = seg_base + c0 + tid;
    int park = -1;
    MeshRay mr;
    float closest = t_max;
    uint32_t i = 0;
    if (c0 + tid < n) {
      const uint2 rk = tq.ray[par][j];
      const unsigned long long res = tq.res[par][j];
      i = rk.x;
      const int k = (int)rk.y;
      const DObject *ob = objs + k;
      const bool tri_hit = res != kNoTriHit;
      const uint32_t order = (uint32_t)res;
      // the stage is bound by the latency of these gathers: issue all of them before the first use
      const float4 o4 = out.b.ray_o[i], d4 = out.b.ray_d[i];
      // closest_so_far travels with the task (the t_max the traversal ran with; == t_max when nothing was hit before the
      // mesh): a sequential 4-byte read instead of two gathered sectors of the hit record (hit0.w, hit1.w) per task
      closest = tq.o[par][j].w;
      float4 nq = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      if (tri_hit) nq = ldg4(sc.meshes[ob->mesh].normals + order);  // normal + original index, by DFS position
      const Ray ray{v3(o4.x, o4.y, o4.z), v3(d4.x, d4.y, d4.z)};
      const float tau = mt.tau[i];
      Hit best;
      best.triangle = -1;
      bool improved = false;
      if (tri_hit) {
        MeshHit mh;
        mh.t = u2f((uint32_t)(res >> 32)), mh.tri = f2u(nq.w), mh.order = order;
        Hit tmp;
        // the shifted ray the mesh was parked with, and its hit back at tau
        const float4 D = disp[k];
        const bool moves = motion_moves(D);
        const Ray r = moves ? motion_object_ray(ray, tau, D) : ray;
        const MeshRay omr = mesh_object_ray<false>(ob->f, r);  // same inputs, same bits as in k_extend_pre_motion
        const bool found = mesh_finish(ob->f, nq, r, omr, mh, t_min, closest, tmp);
        if (found && moves) motion_hit_position(tmp, tau, D);
        if (found) {
          improved = true;
          closest = tmp.t;
          best = tmp;
          best.object = k;
          best.material = ob->hit_bits;  // type << 26 | light << 20 | index, see write_hit
        }
      }
      park = scan_objects_motion(sc, objs, ray, t_min, closest, best, improved, k + 1, mr, disp, tau);
      if (improved) finish_hit(objs, ray, best);
      if (improved) write_hit(out, i, best);  // otherwise the record parked by the previous stage stands
    }
    park_tasks(&s_ntask, tq, par ^ 1, seg_base, park, i, mr, closest);
  }
  __syncthreads();
  if (tid == 0) tq.cnt[(uint32_t)(round + 1) * n_seg + seg] = s_ntask;
}

constexpr int kShadeClasses = 11;  // 0 = miss, 1 + material type (8 types), 9 = NEE shadow ray, 10 = no ray (tail of the last window)
constexpr int kShadeWindow = 2048;                   // rays one block sorts together
constexpr int kShadeGroups = kShadeWindow / kBlock;  // 32-ray groups each warp shades per window

// Block-wide exclusive offsets for a per-thread flag: ranks from the warp ballot, warp totals through shared memory.
// Returns this thread's offset (valid if `flag`); *total = number of flagged threads.  Two block barriers.
__device__ __forceinline__ uint32_t block_rank(bool flag, uint32_t *s_warp /* [kBlock/32 + 1] */, uint32_t *total) {
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t mask = __ballot_sync(0xffffffffu, flag);
  if (lane == 0) s_warp[warp] = (uint32_t)__popc(mask);
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t tot = 0;
    for (int w = 0; w < kBlock / 32; w++) {
      const uint32_t c = s_warp[w];
      s_warp[w] = tot;
      tot += c;
    }
    s_warp[kBlock / 32] = tot;
  }
  __syncthreads();
  *total = s_warp[kBlock / 32];
  return s_warp[warp] + (uint32_t)__popc(mask & ((1u << lane) - 1u));
}

// shade (+ regenerate): emitted + scatter (renderer.rs:26-36) or sky (renderer.rs:38-63) for every ray of the segment,
// survivors written to the front of the segment in the other ray buffer; then fresh camera paths (renderer.rs:96-99,
// camera.rs:33-42) fill the free slots.
//
// Rays arrive in no particular order, so a warp would see a mix of misses and of every material and run all of their
// code (measured: 11.5 of 32 lanes active).  The first remedy (round 1, v2) sorted 256-ray chunks staged in shared
// memory by TMA bulk copies; its profile showed 43 % of the stall samples on block barriers: the eight 32-ray groups of
// a chunk are homogeneous, hence of very different cost (a group of misses is a few instructions, a group of rough
// conductors several hundred), and every chunk ended with the whole block waiting for its most expensive group (the
// SIMT model in tests/hostsim/wfsim.cpp puts the barrier-synchronous cost at 2.3-3x the sum of the group costs).  Now:
//   * a WINDOW of 2048 rays is counting-sorted by (miss | material type) — keys only: one 16-byte load of hit1 per ray,
//     warp-aggregated shared-memory atomics for the position inside the class, two block barriers per window;
//   * warp w shades groups w, w + 8, ..., w + 56 of the sorted window: eight groups spread over all classes, so the
//     warps of a block carry nearly equal work and nobody waits; the larger window also leaves fewer mixed groups
//     (model: lane efficiency 0.77 -> 0.93 on C2);
//   * a thread gathers its ray (five 16-byte loads) straight from global memory.  The window is block-local (160 KB of
//     contiguous slots), so the other half of every 32-byte sector is consumed by a neighbour warp of the same block
//     out of L1/L2: no extra DRAM traffic, and no staging buffers, mbarriers or proxy fences;
//   * survivors are appended at a block-local cursor (one shared-memory atomic per warp) in the OTHER ray buffer:
//     with gathers in flight all over the window, compaction in place would overwrite rays that are still to be read.
//
// NEE = true (PTC_FLAG_NEE): next-event estimation with multiple importance sampling on top of the same loop.  At every
// hit whose material has a continuous lobe the stage also samples one emitter (uniformly chosen sphere / quad light,
// uniform point on it) and emits a SHADOW RAY: one more pool entry (pixel word tagged kShadowBit, the distance in the
// sample field, the MIS-weighted contribution in beta) that goes through the very same extend stages; the next shade adds
// its contribution to the film if nothing was hit before the light, and drops it.  An emitter reached by BSDF sampling is
// weighted with the power heuristic against the light pdf of that point (the sampling pdf travels with the ray in `aux`).
// The path count of a segment is capped at cap / 2 so that paths + their shadow rays always fit.  The estimator's
// expectation is the plain integrator's (tested): same image, less variance where the lights are small.
// Mode 2 (PTC_FLAG_NEE_SKY, the scene has a sky distribution): NEE also samples the HDR sky as an environment light.  The
// sky is chosen with probability p_sky = 0.5 when there are analytic lights (1 otherwise; each light then has (1 - p_sky) /
// n_lights), its direction is drawn from the sky's own distribution (pt_bsdf.h: sky_sample, Philox block 2) and the
// shadow ray has an infinite distance: any hit occludes.  A BSDF-sampled ray that misses is weighted with the power
// heuristic against p_sky * sky_pdf.  Mode 0 = plain, 1 = NEE.
// Modes 3 and 4 (PTC_FLAG_NEE_EMITTERS, without and with the sky): the lights are `sc.lights` = HostScene::lights_em,
// emissive meshes and cubes included, chosen by power from `et`'s selection CDF (u[0] of Philox block 1; with the sky,
// what is left of it after the sky's share), a triangle or cube face by area with u[3] (pt_bsdf.h: emitter_sample).  The
// extend stages ran on the object table whose hit_bits carry these light ids.  A mesh's t is not a distance
// (mesh_finish), so the shadow ray of a mesh or cube light is unoccluded iff its closest hit carries that light's id
// at the sampled point, to within rounding (kPosTestTol; a concave emitter occludes itself), and the hit-side MIS density
// uses |hit point - ray origin|.  Spheres and quads keep Mode 1 / 2's rules bit for bit.
// Returns the new ray count of the segment.
// `seg_done` (or nullptr): one word per segment, set when the segment is found empty with the path supply exhausted — it
// will never hold a ray again — and counted off ctl->n_active, once.
// (The path state is read with plain loads: launches overlap, see stage_begin, so it is not read-only while a k_shade runs.)
// Src: where regeneration starts paths.  kSrcTiles: the tiles of tile_mod / tile_rem; kSrcList: rp.pixel_list
// (ptc_render_adaptive's later passes); kSrcBatch: the stacked tile grids of `bt` (ptc_render_batch).  A template
// argument, so that the shade kernels of every other render compile to the instructions they had.
// Lens: camera paths start through the thin lens of `lt` (camera_get_ray_lens, with u[2], u[3] of the jitter draw);
// only regeneration changes.
// Motion: every ray carries its shutter time (mt.tau -> mt.ntau for survivors and shadow rays); regeneration draws it
// (Philox block 1 of the jitter counter), takes the camera at that time and then the lens of `lt` if lt.lens is set; a
// light of a moving object is sampled from x - tau D_L (nee_origin).
constexpr int kSrcTiles = 0, kSrcList = 1, kSrcBatch = 2;
struct MotionNone {};  // what stands for a value of the motion twins in every other instantiation
// The point a light is sampled from: x, or x - tau D of the light's object when it moves.  wi, dist and the pdfs come out
// as for the static light seen from the shifted point, which is the moving light seen from x at tau.
__device__ __forceinline__ V3 nee_origin(V3 x, const MotionTables &mt, int32_t object, float tau) {
  const float4 D = mt.disp[object];
  return motion_moves(D) ? motion_point(x, tau, D) : x;
}
template <int Mode, int Src, bool Lens = false, bool Motion = false>
__device__ __forceinline__ uint32_t stage_shade(uint32_t seg, uint32_t n_seg, uint32_t *seg_done, Ctl *ctl, const DScene &sc, const RenderParams &rp,
                                                const Buffers &b, const Film &film, const BatchTables &bt, const EmitterTables &et,
                                                const LensTables &lt = LensTables{}, const MotionTables *mt = nullptr) {
  constexpr bool List = Src == kSrcList, Batch = Src == kSrcBatch;
  __shared__ uint16_t s_perm[kShadeWindow];
  __shared__ uint32_t s_hist[2][16];
  __shared__ uint32_t s_warp[kBlock / 32 + 1];
  __shared__ unsigned long long s_first;
  __shared__ uint32_t s_avail, s_more, s_w, s_wp;
  constexpr bool NEE = Mode != 0, SKY = Mode == 2 || Mode == 4, EM = Mode >= 3;
  const uint32_t n = b.cnt[seg], seg_base = seg * b.cap;
  const uint32_t tid = threadIdx.x, lane = tid & 31u;
  const uint32_t lt_mask = (1u << lane) - 1u;
  if (tid == 0) s_w = 0u, s_wp = 0u;
  if (tid < 32u) s_hist[0][tid & 15u] = 0u, s_hist[1][tid & 15u] = 0u;
  __syncthreads();

  uint32_t parity = 0;
  for (uint32_t w0 = 0; w0 < n; w0 += (uint32_t)kShadeWindow, parity ^= 1u) {
    const uint32_t wn = n - w0 < (uint32_t)kShadeWindow ? n - w0 : (uint32_t)kShadeWindow;
    const uint32_t win_base = seg_base + w0;
    // ---- pass 1: class key and position inside the class for the thread's 8 rays
    uint32_t keypos[kShadeGroups];
#pragma unroll
    for (int r = 0; r < kShadeGroups; r++) {
      const uint32_t idx = (uint32_t)r * kBlock + tid;
      uint32_t key = kShadeClasses - 1;
      if (idx < wn) {
        const uint32_t bits = f2u(b.hit1[win_base + idx].w);
        key = (bits & kHitBit) ? 1u + ((bits >> kTypeShift) & 15u) : 0u;
        if (NEE && (f2u(b.ray_o[win_base + idx].w) & kShadowBit)) key = 9u;
      }
      const uint32_t peers = __match_any_sync(0xffffffffu, key);
      const int leader = __ffs((int)peers) - 1;
      uint32_t base = 0;
      if ((int)lane == leader) base = atomicAdd(&s_hist[parity][key], (uint32_t)__popc(peers));
      base = __shfl_sync(0xffffffffu, base, leader);
      keypos[r] = key | ((base + (uint32_t)__popc(peers & lt_mask)) << 4);
    }
    __syncthreads();
    if (tid < 16u) s_hist[parity ^ 1u][tid] = 0u;  // free since barrier 2 of the previous window, next used after barrier 2 below
    {
      const uint32_t h = lane < (uint32_t)kShadeClasses ? s_hist[parity][lane] : 0u;
      uint32_t incl = h;  // inclusive scan over the classes
#pragma unroll
      for (int d = 1; d < 16; d <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= (uint32_t)d) incl += v;
      }
      const uint32_t excl = incl - h;
#pragma unroll
      for (int r = 0; r < kShadeGroups; r++) {
        const uint32_t key = keypos[r] & 15u;
        const uint32_t off = __shfl_sync(0xffffffffu, excl, (int)key);
        if (key != (uint32_t)kShadeClasses - 1u) s_perm[off + (keypos[r] >> 4)] = (uint16_t)((uint32_t)r * kBlock + tid);
      }
    }
    __syncthreads();

    // ---- pass 2: the t-th thread of group g shades the (g * 256 + t)-th ray of the sorted window
#pragma unroll 1
    for (int g = 0; g < kShadeGroups; g++) {
      const uint32_t p = (uint32_t)g * kBlock + tid;
      if ((uint32_t)g * kBlock >= wn) break;
      bool alive = false, shadow = false;
      float4 no, nd, nb, so4, sd4, sb4;
      float npdf = -1.0f;
      std::conditional_t<Motion, float, MotionNone> tau{};  // the ray's shutter time: a float in the motion twins only
      if (p < wn) {
        const uint32_t i = win_base + (uint32_t)s_perm[p];
        const float4 o4 = b.ray_o[i], d4 = b.ray_d[i], b4 = b.beta[i];
        const float4 h1 = b.hit1[i];
        if constexpr (Motion) tau = mt->tau[i];
        const uint32_t pixel_word = f2u(o4.w), sample = f2u(d4.w), bounce = f2u(b4.w);
        const uint32_t pixel = NEE ? (pixel_word & ~kShadowBit) : pixel_word;  // the film index (global in a batch)
        // Philox key: the view's seed and the pixel within the view
        uint64_t seed = rp.seed;
        uint32_t key_pixel = pixel;
        if (Batch) {
          const uint32_t view = pixel / bt.view_px;
          seed = bt.seeds[view];
          key_pixel = pixel - view * bt.view_px;
        }
        const uint32_t bits = f2u(h1.w);
        const V3 beta = v3(b4.x, b4.y, b4.z);
        const V3 ray_d = v3(d4.x, d4.y, d4.z);
        V3 radiance = v3(0, 0, 0);
        bool add = false;
        if (NEE && (pixel_word & kShadowBit)) {
          // a shadow ray: beta is the MIS-weighted contribution, the sample field the distance to the light point.  The light
          // itself is hit at that distance; anything nearer (by more than the tolerance) occludes.
          const float t_light = d4.w;
          if (EM && (bounce & kPosTestBit)) {
            const float4 h0 = b.hit0[i];
            const V3 y = v3(o4.x, o4.y, o4.z) + ray_d * t_light;
            const float tol = kPosTestTol * t_light + kPosTestAbs * fmaxf(fabsf(y.x), fmaxf(fabsf(y.y), fabsf(y.z)));
            if ((bits & kHitBit) && ((bits >> kLightShift) & 63u) == (bounce & 63u) && length_squared(v3(h0.x, h0.y, h0.z) - y) <= tol * tol)
              radiance = beta, add = true;
          } else if (!(bits & kHitBit) || !(b.hit0[i].w < t_light * (1.0f - 2e-4f))) {
            radiance = beta, add = true;
          }
        } else if (!(bits & kHitBit)) {
          radiance = beta * sky_color(sc, ray_d);
          if (SKY) {  // power heuristic against the sky's light-sampling pdf (camera rays and delta lobes: weight 1)
            const float pb = b.aux[i];
            if (pb >= 0.0f) {
              const float pe = (sc.n_lights > 0 ? 0.5f : 1.0f) * sky_pdf(sc, ray_d);
              if (pe > 0.0f) radiance = radiance * (pb * pb / (pb * pb + pe * pe));
            }
          }
          add = true;
        } else {
          const float4 h0 = b.hit0[i];
          const DMaterial m = sc.materials[bits & kMatMask];
          const V3 pos = v3(h0.x, h0.y, h0.z), nrm = v3(h1.x, h1.y, h1.z);
          const V3 e = mat_emitted(m);
          if (e.x != 0.0f || e.y != 0.0f || e.z != 0.0f) {
            float w_mis = 1.0f;
            if (NEE) {  // power heuristic against the light-sampling pdf of this very point, if the emitter is a sampled light
              const float pb = b.aux[i];
              const uint32_t light = (bits >> kLightShift) & 63u;
              if (EM && pb >= 0.0f && light != 0u) {
                // selection probability by power, times 1 - p_sky when the sky is sampled too
                const DLight &L = sc.lights[light - 1u];
                const float dl = emitter_area_sampled(L) ? length(pos - v3(o4.x, o4.y, o4.z)) : h0.w;
                const float pl = emitter_mis_pdf(L, emitter_select_prob(et, light - 1u) * (SKY ? 0.5f : 1.0f), dl, fabsf(dot(nrm, ray_d)));
                w_mis = pb * pb / (pb * pb + pl * pl);
              } else if (!EM && pb >= 0.0f && light != 0u) {
                // selection probability 1 / n_lights, or (1 - p_sky) / n_lights when the sky is sampled too
                const float pl = light_pdf(sc.lights[light - 1u], h0.w, fabsf(dot(nrm, ray_d))) * ((SKY ? 0.5f : 1.0f) / (float)sc.n_lights);
                w_mis = pb * pb / (pb * pb + pl * pl);
              }
            }
            radiance = beta * e * w_mis;
            add = true;
          }
          const Uniforms4 u = philox_uniforms(seed, key_pixel, sample, bounce, 0u);
          Ray sc_ray;
          V3 att;
          if (mat_scatter(m, ray_d, pos, nrm, (bits & kFrontBit) != 0u, u.u, sc_ray, att)) {
            // trace_ray(scattered, depth - 1): depth 0 returns black (renderer.rs:20-22)
            if (bounce + 1u < (uint32_t)rp.max_depth) {
              alive = true;
              const V3 nbeta = beta * att;
              no = make_float4(sc_ray.o.x, sc_ray.o.y, sc_ray.o.z, o4.w);
              nd = make_float4(sc_ray.d.x, sc_ray.d.y, sc_ray.d.z, d4.w);
              nb = make_float4(nbeta.x, nbeta.y, nbeta.z, u2f(bounce + 1u));
              if (NEE) {
                npdf = mat_sampled_pdf(m, ray_d, pos, nrm, u.u, sc_ray.d);
                // light sampling: what the NEXT segment could find at an emitter (hence the same depth rule as the continuation)
                if (SKY) {
                  // one emitter: the sky with probability p_sky (own uniforms, Philox block 2; infinitely far, so any hit
                  // occludes), else a uniformly chosen analytic light with the rest of u[0]
                  const Uniforms4 ul = philox_uniforms(seed, key_pixel, sample, bounce, 1u);
                  const float p_sky = sc.n_lights > 0 ? 0.5f : 1.0f;
                  const V3 so = pos + nrm * kEps;
                  V3 wi, fcos, le;
                  float dist, pl, pb, pm;
                  uint32_t tag = bounce + 1u;
                  bool ok;
                  if (ul.u[0] < p_sky) {
                    const Uniforms4 us = philox_uniforms(seed, key_pixel, sample, bounce, 2u);
                    wi = sky_sample(sc, us.u, pl);
                    pl *= p_sky;
                    dist = INFINITY;
                    le = sky_color(sc, wi);
                    ok = pl > 0.0f;
                    pm = pl;
                  } else if (EM) {
                    EmitterSample es;
                    if constexpr (Motion) {  // the light is chosen once, and sampled from x - tau D of its object
                      const uint32_t pick = cdf_search(et.sel_cdf, (uint32_t)sc.n_lights, (ul.u[0] - p_sky) * 2.0f);
                      ok = emitter_sample_light(sc, et, pick, nee_origin(so, *mt, sc.lights[pick].object, tau), ul.u[1], ul.u[2], ul.u[3], es);
                    } else {
                      ok = emitter_sample(sc, et, so, (ul.u[0] - p_sky) * 2.0f, ul.u[1], ul.u[2], ul.u[3], es);
                    }
                    const DLight &L = sc.lights[es.light];
                    wi = es.wi, dist = es.dist, pl = es.pdf * 0.5f, pm = es.pmis * 0.5f;  // (1 - p_sky) x the light's own
                    le = v3(L.emission[0], L.emission[1], L.emission[2]);
                    if (emitter_area_sampled(L)) tag = kPosTestBit | (es.light + 1u);
                  } else {
                    const uint32_t li = min((uint32_t)((ul.u[0] - p_sky) * 2.0f * (float)sc.n_lights), (uint32_t)sc.n_lights - 1u);
                    const DLight L = sc.lights[li];
                    if constexpr (Motion) ok = light_sample(L, nee_origin(so, *mt, L.object, tau), ul.u[1], ul.u[2], wi, dist, pl);
                    else ok = light_sample(L, so, ul.u[1], ul.u[2], wi, dist, pl);
                    pl *= 0.5f / (float)sc.n_lights;  // (1 - p_sky) / n_lights, as where a BSDF-sampled ray hits the light
                    le = v3(L.emission[0], L.emission[1], L.emission[2]);
                    pm = pl;
                  }
                  if (ok && mat_eval_pdf(m, ray_d, pos, nrm, wi, fcos, pb) && (fcos.x > 0.0f || fcos.y > 0.0f || fcos.z > 0.0f)) {
                    const float w_mis = pm * pm / (pm * pm + pb * pb);
                    const V3 c = beta * fcos * le * (w_mis / pl);
                    shadow = true;
                    so4 = make_float4(so.x, so.y, so.z, u2f(pixel | kShadowBit));
                    sd4 = make_float4(wi.x, wi.y, wi.z, dist);
                    sb4 = make_float4(c.x, c.y, c.z, u2f(tag));
                  }
                } else if (EM && sc.n_lights > 0) {
                  const Uniforms4 ul = philox_uniforms(seed, key_pixel, sample, bounce, 1u);
                  const V3 so = pos + nrm * kEps;
                  EmitterSample es;
                  V3 fcos;
                  float pb;
                  bool ok;
                  if constexpr (Motion) {  // the light is chosen once, and sampled from x - tau D of its object
                    const uint32_t pick = cdf_search(et.sel_cdf, (uint32_t)sc.n_lights, ul.u[0]);
                    ok = emitter_sample_light(sc, et, pick, nee_origin(so, *mt, sc.lights[pick].object, tau), ul.u[1], ul.u[2], ul.u[3], es);
                  } else {
                    ok = emitter_sample(sc, et, so, ul.u[0], ul.u[1], ul.u[2], ul.u[3], es);
                  }
                  if (ok && mat_eval_pdf(m, ray_d, pos, nrm, es.wi, fcos, pb) &&
                      (fcos.x > 0.0f || fcos.y > 0.0f || fcos.z > 0.0f)) {
                    const DLight &L = sc.lights[es.light];
                    const float w_mis = es.pmis * es.pmis / (es.pmis * es.pmis + pb * pb);
                    const V3 c = beta * fcos * v3(L.emission[0], L.emission[1], L.emission[2]) * (w_mis / es.pdf);
                    shadow = true;
                    so4 = make_float4(so.x, so.y, so.z, u2f(pixel | kShadowBit));
                    sd4 = make_float4(es.wi.x, es.wi.y, es.wi.z, es.dist);
                    sb4 = make_float4(c.x, c.y, c.z, u2f(emitter_area_sampled(L) ? kPosTestBit | (es.light + 1u) : bounce + 1u));
                  }
                } else if (!EM && sc.n_lights > 0) {
                  const Uniforms4 ul = philox_uniforms(seed, key_pixel, sample, bounce, 1u);
                  const uint32_t li = min((uint32_t)(ul.u[0] * (float)sc.n_lights), (uint32_t)sc.n_lights - 1u);
                  const DLight L = sc.lights[li];
                  const V3 so = pos + nrm * kEps;
                  V3 wi, fcos;
                  float dist, pl, pb;
                  bool ok;
                  if constexpr (Motion) ok = light_sample(L, nee_origin(so, *mt, L.object, tau), ul.u[1], ul.u[2], wi, dist, pl);
                  else ok = light_sample(L, so, ul.u[1], ul.u[2], wi, dist, pl);
                  if (ok && mat_eval_pdf(m, ray_d, pos, nrm, wi, fcos, pb) &&
                      (fcos.x > 0.0f || fcos.y > 0.0f || fcos.z > 0.0f)) {
                    pl *= 1.0f / (float)sc.n_lights;
                    const float w_mis = pl * pl / (pl * pl + pb * pb);
                    const V3 c = beta * fcos * v3(L.emission[0], L.emission[1], L.emission[2]) * (w_mis / pl);
                    shadow = true;
                    so4 = make_float4(so.x, so.y, so.z, u2f(pixel | kShadowBit));
                    sd4 = make_float4(wi.x, wi.y, wi.z, dist);
                    sb4 = make_float4(c.x, c.y, c.z, u2f(bounce + 1u));
                  }
                }
              }
            }
          }
        }
        if (add) {
          film_add(film, pixel, radiance);
        }
      }
      // survivors (and, with NEE, their shadow rays): one shared-memory atomic per warp, no barrier
      const uint32_t amask = __ballot_sync(0xffffffffu, alive);
      const uint32_t smask = NEE ? __ballot_sync(0xffffffffu, shadow) : 0u;
      if ((amask | smask) != 0u) {
        uint32_t base = 0;
        if (lane == 0) {
          base = atomicAdd(&s_w, (uint32_t)(__popc(amask) + __popc(smask)));
          if (NEE) atomicAdd(&s_wp, (uint32_t)__popc(amask));
        }
        base = __shfl_sync(0xffffffffu, base, 0);
        if (alive) {
          const uint32_t slot = seg_base + base + (uint32_t)__popc(amask & lt_mask);
          b.nray_o[slot] = no;
          b.nray_d[slot] = nd;
          b.nbeta[slot] = nb;
          if (NEE) b.naux[slot] = npdf;
          if constexpr (Motion) mt->ntau[slot] = tau;
        }
        if (NEE && shadow) {
          const uint32_t slot = seg_base + base + (uint32_t)__popc(amask) + (uint32_t)__popc(smask & lt_mask);
          b.nray_o[slot] = so4;
          b.nray_d[slot] = sd4;
          b.nbeta[slot] = sb4;
          b.naux[slot] = -1.0f;
          if constexpr (Motion) mt->ntau[slot] = tau;
        }
      }
    }
    // no barrier here: the next window's pass 1 touches only the other histogram, and s_perm is rewritten after its
    // first barrier, which every thread reaches only after it has finished this loop
  }
  __syncthreads();
  uint32_t w = s_w;  // survivors written so far = write cursor inside the segment (same value in every thread)
  uint32_t wp = NEE ? s_wp : w;  // ... of which paths (the rest are shadow rays)

  // ---- regeneration: top the segment up with fresh camera paths.  Path index -> (sample, 32-pixel row of one of this
  // rank's 32x32 tiles, lane): a warp starts 32 horizontally adjacent pixels of one sample (coherent primary rays,
  // distinct film addresses), but consecutive rows are scattered over the image by a multiplicative bijection, so every
  // segment holds a uniform sample of the frame — segments are statically owned by blocks, and a segment that got all
  // the rays of the mesh's screen region would make its block the straggler of every traversal pass.  Pixels of partial
  // border tiles that fall outside the image start no path.  With a pixel list the 32-pixel rows are 32 consecutive
  // list entries instead, and the padding of the last row starts no path.
  const unsigned long long per_sample = List ? (unsigned long long)((rp.n_list + 31u) & ~31u) : (unsigned long long)rp.n_my_tiles * 1024ull;
  for (;;) {
    if (tid == 0) {
      const unsigned long long total = ctl->total_paths;
      // no more than a fair share of the whole job per block, in whole 32-pixel rows: a render smaller than the pool
      // would otherwise be swallowed by the first few segments and traced by that many blocks
      const unsigned long long share = ((total + n_seg - 1) / n_seg + 31ull) & ~31ull;
      // with NEE a path may add a shadow ray at every bounce: paths are capped at half the segment
      const uint32_t room = NEE ? min(b.cap - w, b.cap / 2u > wp ? b.cap / 2u - wp : 0u) : b.cap - w;
      const uint32_t free_slots = (uint32_t)min((unsigned long long)room, share);
      unsigned long long first = total;
      if (free_slots > 0 && ctl->next_path < total) first = atomicAdd(&ctl->next_path, (unsigned long long)free_slots);
      s_first = first;
      s_avail = first < total ? (uint32_t)min((unsigned long long)free_slots, total - first) : 0u;
      s_more = (first + free_slots < total) ? 1u : 0u;  // the supply is not exhausted yet
    }
    __syncthreads();
    const unsigned long long first_path = s_first;
    const uint32_t avail = s_avail;
    for (uint32_t j0 = 0; j0 < avail; j0 += (uint32_t)kBlock) {
      const uint32_t j = j0 + tid;
      bool valid = j < avail;
      uint32_t pixel = 0, sample = 0, view = 0;
      int x = 0, y = 0;
      if (valid) {
        const unsigned long long p = first_path + j;
        const uint32_t s = (uint32_t)(p / per_sample);
        const uint32_t r0 = (uint32_t)(p - (unsigned long long)s * per_sample);
        const uint32_t row = (uint32_t)(((unsigned long long)(r0 >> 5) * rp.row_mult) % (unsigned long long)(per_sample >> 5));
        const uint32_t r = (row << 5) | (r0 & 31u);
        if (List) {
          valid = r < rp.n_list;
          pixel = valid ? rp.pixel_list[r] : 0u;
          x = (int)(pixel % (uint32_t)rp.width);
          y = (int)(pixel / (uint32_t)rp.width);
        } else {
          const uint32_t local_tile = r >> 10, in_tile = r & 1023u;
          uint32_t tile = local_tile * (uint32_t)rp.tile_mod + (uint32_t)rp.tile_rem;
          if (Batch) {  // (tile_mod = 1, tile_rem = 0) the row scatter above runs over the rows of every view
            view = local_tile / bt.tiles_per_view;
            tile = local_tile - view * bt.tiles_per_view;
          }
          x = (int)((tile % (uint32_t)rp.tiles_x) * 32u + (in_tile & 31u));
          y = (int)((tile / (uint32_t)rp.tiles_x) * 32u + (in_tile >> 5));
          valid = x < rp.width && y < rp.height;
          pixel = (uint32_t)(y * rp.width + x);
        }
        sample = (uint32_t)rp.sample_begin + s;
      }
      uint32_t total;
      const uint32_t off = block_rank(valid, s_warp, &total);
      if (valid) {
        const uint32_t slot = seg_base + w + off;
        const Uniforms4 jit = philox_uniforms(Batch ? bt.seeds[view] : rp.seed, pixel, sample, 0xffffffffu, 0u);
        const float u = ((float)x + jit.u[0]) / (float)rp.width;   // renderer.rs:96
        const float v = ((float)y + jit.u[1]) / (float)rp.height;  // renderer.rs:97
        Ray ray;
        if constexpr (Motion) {
          // the shutter time: Philox block 1 of the jitter counter, never drawn otherwise
          const float tau = philox_uniforms(Batch ? bt.seeds[view] : rp.seed, pixel, sample, 0xffffffffu, 1u).u[0];
          DCamera cam = Batch ? bt.cams[view] : rp.cam;
          if (mt->end_cams) cam = camera_at(cam, mt->end_cams[Batch ? view : 0u], tau);
          if (lt.lens) {
            const float2 ln = lt.lens[Batch ? view : 0u];
            ray = camera_get_ray_lens(cam, ln.x, ln.y, u, v, jit.u[2], jit.u[3]);
          } else {
            ray = camera_get_ray(cam, u, v);
          }
          mt->ntau[slot] = tau;
        } else if (Lens) {
          const float2 ln = lt.lens[Batch ? view : 0u];
          ray = camera_get_ray_lens(Batch ? bt.cams[view] : rp.cam, ln.x, ln.y, u, v, jit.u[2], jit.u[3]);
        } else {
          ray = camera_get_ray(Batch ? bt.cams[view] : rp.cam, u, v);
        }
        b.nray_o[slot] = make_float4(ray.o.x, ray.o.y, ray.o.z, u2f(Batch ? view * bt.view_px + pixel : pixel));
        b.nray_d[slot] = make_float4(ray.d.x, ray.d.y, ray.d.z, u2f(sample));
        b.nbeta[slot] = make_float4(1.0f, 1.0f, 1.0f, u2f(0u));
        if (NEE) b.naux[slot] = -1.0f;
      }
      w += total;
      wp += total;
      __syncthreads();
    }
    // a batch that fell entirely on out-of-image pixels of border tiles must not look like "no paths left"
    const bool again = (w == 0u) && (s_more != 0u);
    __syncthreads();
    if (!again) break;
  }
  if (tid == 0) {
    b.cnt[seg] = w;
    // w == 0 here means the loop above ended on an exhausted supply: the segment is empty for good
    if (w == 0u && seg_done && seg_done[seg] == 0u) {
      seg_done[seg] = 1u;
      atomicSub(&ctl->n_active, 1u);
    }
  }
  return w;
}


// Launches as code switches, segments as the unit of ordering.
//
// Every stage launch of a render is a programmatic dependent launch (sm_90+): it may be scheduled before its predecessor
// in the stream has drained.  Round 1 then waited for the whole predecessor (griddepcontrol.wait) — and so every stage of
// every iteration ended with the GPU waiting for the one block that had drawn the longest walk: a constant 20-28 us per
// traversal launch, ~40 us per iteration, 1.1 ms of the 6.2 ms of C2's 1/8 share (tools/drain_trace.py).  But block b of a
// launch only ever needs what block b of the launch before it wrote: a block touches nothing outside its own segment.
// So a block now waits for ITS segment: flags[seg] is set to the launch's number by the block that finished the segment
// (release, after a block barrier) and awaited by the same-numbered block of the next launch (relaxed polling, one acquire
// fence, then a block barrier).  A segment whose traversal was slow falls behind while the others go on into the next stages and
// iterations, a different one is slow next time, and what is waited for is the SUM over a segment's stages, once, at the
// end of the render — what a persistent per-block loop would give, without four stages' code fighting for one
// instruction cache (DESIGN.md 5c).  No deadlock: a dependent launch's blocks are scheduled only when every block of
// the launch before it has started, so the block a waiting block depends on is always resident (or done) itself.
// A traversal whose blocks take (segment, part) items from a counter waits per ITEM and counts a segment's finished
// parts; the block that finishes the last one sets the flag.  A launch without flags, or with flag_wait = 0 (the first
// launch after the host's memsets), waits for the whole predecessor as before.
// Polling is RELAXED (coherent at gpu scope, i.e. served by L2) and the acquire is one fence after the flag has been seen:
// ld.acquire compiles to the load plus CCTL.IVALL, and a block spinning on that would wipe the L1 of its SM — the L1 the
// blocks it is waiting for, two slots over, are walking their BVH out of — a million times a second.
__device__ __forceinline__ uint32_t ld_relaxed_u32(const uint32_t *p) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void fence_acquire() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }
__device__ __forceinline__ void st_release_u32(uint32_t *p, uint32_t v) {
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// the block waits until the launch before this one has finished segment `seg` (no-op without flags / with flag_wait = 0)
__device__ __forceinline__ void segment_wait(const SegRange &sr, uint32_t seg, Ctl *ctl) {
  if (sr.flags == nullptr || sr.flag_wait == 0u) return;
  if (threadIdx.x == 0) {
    const uint32_t need = sr.stage_id - 1u;
    uint32_t spins = 0;
    while (ld_relaxed_u32(sr.flags + seg) < need) {
      if (++spins == (1u << 25)) {  // tens of seconds: cannot happen; the host reports it instead of hanging
        atomicAdd(&ctl->sync_timeouts, 1u);
        break;
      }
      __nanosleep(64);
    }
    fence_acquire();
  }
  __syncthreads();
}
__device__ __forceinline__ void stage_begin(const SegRange &sr, uint32_t seg, Ctl *ctl) {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (sr.flags == nullptr || sr.flag_wait == 0u) asm volatile("griddepcontrol.wait;" ::: "memory");
  else segment_wait(sr, seg, ctl);
}
// every thread of the block has finished the segment's stage
__device__ __forceinline__ void stage_end(const SegRange &sr, uint32_t seg) {
  if (sr.flags == nullptr) return;
  __syncthreads();
  if (threadIdx.x == 0) st_release_u32(sr.flags + seg, sr.stage_id);  // release at gpu scope: cumulative over the barrier
}

// ---- per-stage kernels: one block per segment --------------------------------------------------------------------
// `progress` (pinned host memory mapped into the device, or nullptr): one word per render the host polls instead of
// putting a copy of the control block between the launches of every drain iteration — `seq << 2 | supply exhausted << 1 |
// every segment empty for good`, as segment 0 finds it at the start of iteration seq.  One 4-byte store: never seen
// half-written.
__global__ void __launch_bounds__(kBlock, kSegPerSM) k_extend_pre(Ctl *ctl, SegRange sr, DScene sc, ExtendOut out, TaskQ tq, float t_min,
                                                                  float t_max, volatile uint32_t *progress, uint32_t seq) {
  const uint32_t seg = sr.seg0 + blockIdx.x;
  stage_begin(sr, seg, ctl);
  if (threadIdx.x == 0) {  // bookkeeping, per segment: rays = extend items = trace_ray calls with depth > 0
    const uint32_t n = out.b.cnt[seg];
    if (n) {
      atomicAdd(&ctl->rays, (unsigned long long)n);
      atomicMax(&ctl->iterations[0], seq);
    }
    if (progress && blockIdx.x == 0) {
      *progress = seq << 2 | (ctl->next_path >= ctl->total_paths ? 2u : 0u) | (ctl->n_active == 0u ? 1u : 0u);
      __threadfence_system();
    }
  }
  if (sc.n_objects <= kSmemObjects) stage_pre<true>(seg, sr.n_seg, sc, out, tq, t_min, t_max);
  else stage_pre<false>(seg, sr.n_seg, sc, out, tq, t_min, t_max);
  stage_end(sr, seg);
}
// Motion blur: k_extend_pre with every ray at its shutter time mt.tau (stage_pre_motion); the same bookkeeping
__global__ void __launch_bounds__(kBlock, kSegPerSM) k_extend_pre_motion(Ctl *ctl, SegRange sr, DScene sc, ExtendOut out, TaskQ tq, float t_min,
                                                                         float t_max, volatile uint32_t *progress, uint32_t seq,
                                                                         MotionTables mt) {
  const uint32_t seg = sr.seg0 + blockIdx.x;
  stage_begin(sr, seg, ctl);
  if (threadIdx.x == 0) {
    const uint32_t n = out.b.cnt[seg];
    if (n) {
      atomicAdd(&ctl->rays, (unsigned long long)n);
      atomicMax(&ctl->iterations[0], seq);
    }
    if (progress && blockIdx.x == 0) {
      *progress = seq << 2 | (ctl->next_path >= ctl->total_paths ? 2u : 0u) | (ctl->n_active == 0u ? 1u : 0u);
      __threadfence_system();
    }
  }
  if (sc.n_objects <= kSmemObjects) stage_pre_motion<true>(seg, sr.n_seg, sc, out, tq, t_min, t_max, mt);
  else stage_pre_motion<false>(seg, sr.n_seg, sc, out, tq, t_min, t_max, mt);
  stage_end(sr, seg);
}
template <bool COUNT>
__global__ void __launch_bounds__(kBlock, kSegPerSM) k_traverse(Ctl *ctl, SegRange sr, DScene sc, TaskQ tq, int round, float t_min,
                                                                uint32_t cap, uint32_t refill_lanes) {
  if (sr.trav_parts <= 1u) {
    stage_begin(sr, sr.seg0 + blockIdx.x, ctl);
    stage_traverse<COUNT>(sr.seg0 + blockIdx.x, sr.n_seg, ctl, sc, tq, round, t_min, cap, refill_lanes);
    stage_end(sr, sr.seg0 + blockIdx.x);
    return;
  }
  // Heavy meshes, bulk of the render (the host decides): every segment's task list is cut into `trav_parts` items and
  // the items beyond the first per block are handed out by a counter — a block whose walks were short takes another
  // item instead of idling until the slowest block of the launch is done (C5: 5-10 % of every traversal launch).
  // Ownership of the SEGMENT is irrelevant here: a traversal only reads its task and lowers that task's result key.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (sr.flags == nullptr || sr.flag_wait == 0u) asm volatile("griddepcontrol.wait;" ::: "memory");
  __shared__ uint32_t s_item;  // the item in hand lives in shared memory: nothing of the hand-out stays in registers during a walk
  if (threadIdx.x == 0) s_item = blockIdx.x;
  __syncthreads();
  for (;;) {
    {
      const uint32_t item = s_item;
      if (item >= sr.n_seg * sr.trav_parts) break;
      const uint32_t seg = sr.seg0 + item % sr.n_seg;
      segment_wait(sr, seg, ctl);
      stage_traverse<COUNT>(seg, sr.n_seg, ctl, sc, tq, round, t_min, cap, refill_lanes, item / sr.n_seg, sr.trav_parts);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      if (sr.flags) {  // the last part of a segment to finish publishes the segment (the results are L2 atomics; fenced anyway)
        const uint32_t seg = sr.seg0 + s_item % sr.n_seg;
        __threadfence();
        if (atomicInc(sr.flags + 2u * sr.n_seg + seg, sr.trav_parts - 1u) == sr.trav_parts - 1u) {
          __threadfence();
          st_release_u32(sr.flags + seg, sr.stage_id);
        }
      }
      s_item = gridDim.x + atomicAdd(sr.trav_counter, 1u);
    }
    __syncthreads();
  }
}
__global__ void __launch_bounds__(kBlock, kSegPerSM) k_extend_post(Ctl *ctl, SegRange sr, DScene sc, ExtendOut out, TaskQ tq, int round,
                                                                   float t_min, float t_max) {
  stage_begin(sr, sr.seg0 + blockIdx.x, ctl);
  if (sc.n_objects <= kSmemObjects) stage_post<true>(sr.seg0 + blockIdx.x, sr.n_seg, sc, out, tq, round, t_min, t_max);
  else stage_post<false>(sr.seg0 + blockIdx.x, sr.n_seg, sc, out, tq, round, t_min, t_max);
  stage_end(sr, sr.seg0 + blockIdx.x);
}
// Motion blur: k_extend_post with every ray at its shutter time mt.tau (stage_post_motion)
__global__ void __launch_bounds__(kBlock, kSegPerSM) k_extend_post_motion(Ctl *ctl, SegRange sr, DScene sc, ExtendOut out, TaskQ tq, int round,
                                                                          float t_min, float t_max, MotionTables mt) {
  stage_begin(sr, sr.seg0 + blockIdx.x, ctl);
  if (sc.n_objects <= kSmemObjects) stage_post_motion<true>(sr.seg0 + blockIdx.x, sr.n_seg, sc, out, tq, round, t_min, t_max, mt);
  else stage_post_motion<false>(sr.seg0 + blockIdx.x, sr.n_seg, sc, out, tq, round, t_min, t_max, mt);
  stage_end(sr, sr.seg0 + blockIdx.x);
}
// Mode: 0 = plain, 1 = PTC_FLAG_NEE, 2 = PTC_FLAG_NEE | PTC_FLAG_NEE_SKY on a scene with a sky distribution.  List: paths
// start from rp.pixel_list (stage_shade).
template <int Mode, bool List = false>
__global__ void __launch_bounds__(kBlock, kSegPerSM) k_shade(Ctl *ctl, SegRange sr, DScene sc, RenderParams rp, Buffers b, Film film) {
  stage_begin(sr, sr.seg0 + blockIdx.x, ctl);
  stage_shade<Mode, List ? kSrcList : kSrcTiles>(sr.seg0 + blockIdx.x, sr.n_seg, sr.flags ? sr.flags + sr.n_seg : nullptr, ctl, sc, rp, b,
                                                 film, BatchTables{}, EmitterTables{});
  stage_end(sr, sr.seg0 + blockIdx.x);
}
// ptc_render_batch: paths of every view of `bt` (stage_shade, kSrcBatch); rp.tile_mod = 1, rp.n_my_tiles = views x tiles
template <int Mode>
__global__ void __launch_bounds__(kBlock, kSegPerSM) k_shade_batch(Ctl *ctl, SegRange sr, DScene sc, RenderParams rp, Buffers b, Film film,
                                                                   BatchTables bt) {
  stage_begin(sr, sr.seg0 + blockIdx.x, ctl);
  stage_shade<Mode, kSrcBatch>(sr.seg0 + blockIdx.x, sr.n_seg, sr.flags ? sr.flags + sr.n_seg : nullptr, ctl, sc, rp, b, film, bt,
                               EmitterTables{});
  stage_end(sr, sr.seg0 + blockIdx.x);
}
// PTC_FLAG_NEE_EMITTERS: Mode 3 (NEE + emitters) or 4 (NEE + sky + emitters), paths from any Src; the emitter tables are a
// kernel argument of these instantiations only, so that the parameters of every other kernel keep their layout
template <int Mode, int Src>
__global__ void __launch_bounds__(kBlock, kSegPerSM) k_shade_em(Ctl *ctl, SegRange sr, DScene sc, RenderParams rp, Buffers b, Film film,
                                                                BatchTables bt, EmitterTables et) {
  stage_begin(sr, sr.seg0 + blockIdx.x, ctl);
  stage_shade<Mode, Src>(sr.seg0 + blockIdx.x, sr.n_seg, sr.flags ? sr.flags + sr.n_seg : nullptr, ctl, sc, rp, b, film, bt, et);
  stage_end(sr, sr.seg0 + blockIdx.x);
}
// ptc_scene_set_lens with a nonzero aperture: Mode 0-4, paths from any Src, through the thin lens of `lt`.  The lens table
// is a trailing argument of these instantiations only (see k_shade_em).
template <int Mode, int Src>
__global__ void __launch_bounds__(kBlock, kSegPerSM) k_shade_lens(Ctl *ctl, SegRange sr, DScene sc, RenderParams rp, Buffers b, Film film,
                                                                  BatchTables bt, EmitterTables et, LensTables lt) {
  stage_begin(sr, sr.seg0 + blockIdx.x, ctl);
  stage_shade<Mode, Src, true>(sr.seg0 + blockIdx.x, sr.n_seg, sr.flags ? sr.flags + sr.n_seg : nullptr, ctl, sc, rp, b, film, bt, et, lt);
  stage_end(sr, sr.seg0 + blockIdx.x);
}
// Motion blur (an object moves, or a camera differs from its end camera): Mode 0-4, paths from any Src, every ray at its
// shutter time; the lens of `lt` if lt.lens is set (nullptr: a pinhole).  The tables are trailing arguments of these
// instantiations only (see k_shade_em).
template <int Mode, int Src>
__global__ void __launch_bounds__(kBlock, kSegPerSM) k_shade_motion(Ctl *ctl, SegRange sr, DScene sc, RenderParams rp, Buffers b, Film film,
                                                                    BatchTables bt, EmitterTables et, LensTables lt, MotionTables mt) {
  stage_begin(sr, sr.seg0 + blockIdx.x, ctl);
  stage_shade<Mode, Src, false, true>(sr.seg0 + blockIdx.x, sr.n_seg, sr.flags ? sr.flags + sr.n_seg : nullptr, ctl, sc, rp, b, film, bt, et,
                                      lt, &mt);
  stage_end(sr, sr.seg0 + blockIdx.x);
}

// accum[i] += fp32(film sum i): the end of ptc_render_accumulate (which ADDS into the caller's fp32 film), and
// ptc_render_adaptive's snapshot
__global__ void k_film_to_accum(Film film, size_t n_pixels, float *accum) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pixels * 3) return;
  const size_t px = i / 3;
  accum[i] += film_value(film.sum[i], film.flags[px], (int)(i - px * 3));
}
// renderer.rs:112-120 + color.rs:87-93 on a caller's fp32 film (ptc_resolve_device / ptc_resolve_u32)
__global__ void k_resolve(const float *rgb, size_t n_pixels, float scale, uint32_t *out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_pixels) out[i] = resolve_pixel(rgb[i * 3] * scale, rgb[i * 3 + 1] * scale, rgb[i * 3 + 2] * scale);
}
// The end of every render that returns an image: rgb = film sum x scale (renderer.rs:103; counts != nullptr: x 1 / the
// pixel's own count, ptc_render_adaptive), packed = resolve_pixel of that (renderer.rs:112-120 + color.rs:87-93).
// 0.0f + the sum is what k_film_to_accum leaves in a zeroed fp32 film, so the result is bit for bit that film x scale,
// then k_resolve.  Either output may be nullptr.
__global__ void k_resolve_film(Film film, size_t n_pixels, float scale, const int32_t *counts, float *rgb, uint32_t *packed) {
  const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_pixels) return;
  if (counts) scale = 1.0f / (float)counts[p];
  const unsigned long long flags = film.flags[p];
  float c[3];
  for (int k = 0; k < 3; k++) c[k] = (0.0f + film_value(film.sum[p * 3 + k], flags, k)) * scale;
  if (rgb) rgb[p * 3] = c[0], rgb[p * 3 + 1] = c[1], rgb[p * 3 + 2] = c[2];
  if (packed) packed[p] = resolve_pixel(c[0], c[1], c[2]);
}

// ---- ptc_render_adaptive (pt_adaptive.h): decision and dilation ------------------------------------------------
// every pixel active, none needing more, every final count spp until the pixel leaves earlier
__global__ void k_adapt_init(uint32_t n_pixels, int32_t spp, uint32_t *list, uint8_t *needs, int32_t *counts) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_pixels) return;
  list[i] = i, needs[i] = 0u, counts[i] = spp;
}
// needs[p] = the decision of every active pixel p at n samples against its snapshot vp at m; vp <- the film now
__global__ void k_adapt_decide(Film film, const uint32_t *list, uint32_t n_list, int32_t n, int32_t m, float threshold, float *vp,
                               uint8_t *needs) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_list) return;
  const uint32_t p = list[i];
  const unsigned long long flags = film.flags[p];
  float V[3], P[3];
  for (int c = 0; c < 3; c++) V[c] = film_value(film.sum[(size_t)p * 3 + c], flags, c), P[c] = vp[(size_t)p * 3 + c];
  needs[p] = adapt_needs_more(V, P, n, m, threshold) ? 1u : 0u;
  for (int c = 0; c < 3; c++) vp[(size_t)p * 3 + c] = V[c];
}
// keep[i] = list entry i stays active (3x3 dilation of needs over the active set)
__global__ void k_adapt_keep(const uint32_t *list, uint32_t n_list, const uint8_t *needs, int32_t width, int32_t height, uint8_t *keep) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_list) keep[i] = adapt_keep(needs, width, height, list[i]) ? 1u : 0u;
}
// a pixel that leaves keeps its count n and stops counting as needing more (after every k_adapt_keep read of needs)
__global__ void k_adapt_leave(const uint32_t *list, uint32_t n_list, const uint8_t *keep, int32_t n, uint8_t *needs, int32_t *counts) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_list || keep[i]) return;
  const uint32_t p = list[i];
  needs[p] = 0u, counts[p] = n;
}

// ---- parity hooks: the same device functions / kernels, driven by caller-provided inputs ---------------------
// ptc_intersect runs the very kernels the renderer uses (k_extend_*); these two only repack inputs / outputs.
__global__ void k_pack_rays(const float *o, const float *d, size_t n, float4 *ro, float4 *rd) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  ro[i] = make_float4(o[i * 3], o[i * 3 + 1], o[i * 3 + 2], 0.0f);
  rd[i] = make_float4(d[i * 3], d[i * 3 + 1], d[i * 3 + 2], 0.0f);
}
__global__ void k_unpack_hits(const float4 *hit0, const float4 *hit1, const int2 *ids, size_t n, ptc_hit *out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  ptc_hit r;
  memset(&r, 0, sizeof(r));
  const float4 h1 = hit1[i];
  const uint32_t bits = f2u(h1.w);
  if (bits & kHitBit) {
    const float4 h0 = hit0[i];
    const int2 id = ids[i];
    r.object = id.x, r.triangle = id.y;
    r.t = h0.w;
    r.position[0] = h0.x, r.position[1] = h0.y, r.position[2] = h0.z;
    r.normal[0] = h1.x, r.normal[1] = h1.y, r.normal[2] = h1.z;
    r.front_face = (bits & kFrontBit) ? 1 : 0;
    r.material = (int32_t)(bits & kMatMask);
  } else {
    r.object = -1, r.triangle = -1, r.material = -1;
  }
  out[i] = r;
}

__global__ void k_primary_rays(RenderParams rp, uint32_t sample, float *out_o, float *out_d) {
  const uint32_t pixel = blockIdx.x * blockDim.x + threadIdx.x;
  if (pixel >= (uint32_t)(rp.width * rp.height)) return;
  const int x = (int)(pixel % (uint32_t)rp.width), y = (int)(pixel / (uint32_t)rp.width);
  const Uniforms4 jit = philox_uniforms(rp.seed, pixel, sample, 0xffffffffu, 0u);
  const float u = ((float)x + jit.u[0]) / (float)rp.width;
  const float v = ((float)y + jit.u[1]) / (float)rp.height;
  const Ray ray = camera_get_ray(rp.cam, u, v);
  out_o[pixel * 3 + 0] = ray.o.x, out_o[pixel * 3 + 1] = ray.o.y, out_o[pixel * 3 + 2] = ray.o.z;
  out_d[pixel * 3 + 0] = ray.d.x, out_d[pixel * 3 + 1] = ray.d.y, out_d[pixel * 3 + 2] = ray.d.z;
}
// the same through the thin lens lt.lens[0]: ptc_primary_rays and ptc_render_denoised's feature pass under a lens see
// exactly the camera rays k_shade_lens starts
__global__ void k_primary_rays_lens(RenderParams rp, uint32_t sample, float *out_o, float *out_d, LensTables lt) {
  const uint32_t pixel = blockIdx.x * blockDim.x + threadIdx.x;
  if (pixel >= (uint32_t)(rp.width * rp.height)) return;
  const int x = (int)(pixel % (uint32_t)rp.width), y = (int)(pixel / (uint32_t)rp.width);
  const Uniforms4 jit = philox_uniforms(rp.seed, pixel, sample, 0xffffffffu, 0u);
  const float u = ((float)x + jit.u[0]) / (float)rp.width;
  const float v = ((float)y + jit.u[1]) / (float)rp.height;
  const float2 ln = lt.lens[0];
  const Ray ray = camera_get_ray_lens(rp.cam, ln.x, ln.y, u, v, jit.u[2], jit.u[3]);
  out_o[pixel * 3 + 0] = ray.o.x, out_o[pixel * 3 + 1] = ray.o.y, out_o[pixel * 3 + 2] = ray.o.z;
  out_d[pixel * 3 + 0] = ray.d.x, out_d[pixel * 3 + 1] = ray.d.y, out_d[pixel * 3 + 2] = ray.d.z;
}
// ... and at the shutter time: the camera at tau (mt.end_cams[0], if any), then the lens lt.lens[0] (if any), exactly as
// k_shade_motion starts its paths; out_tau (or nullptr) receives tau.  ptc_primary_rays and the denoiser's feature pass
// of a motion render.
__global__ void k_primary_rays_motion(RenderParams rp, uint32_t sample, float *out_o, float *out_d, float *out_tau, LensTables lt,
                                      MotionTables mt) {
  const uint32_t pixel = blockIdx.x * blockDim.x + threadIdx.x;
  if (pixel >= (uint32_t)(rp.width * rp.height)) return;
  const int x = (int)(pixel % (uint32_t)rp.width), y = (int)(pixel / (uint32_t)rp.width);
  const Uniforms4 jit = philox_uniforms(rp.seed, pixel, sample, 0xffffffffu, 0u);
  const float u = ((float)x + jit.u[0]) / (float)rp.width;
  const float v = ((float)y + jit.u[1]) / (float)rp.height;
  const float tau = philox_uniforms(rp.seed, pixel, sample, 0xffffffffu, 1u).u[0];
  const DCamera cam = mt.end_cams ? camera_at(rp.cam, mt.end_cams[0], tau) : rp.cam;
  Ray ray;
  if (lt.lens) {
    const float2 ln = lt.lens[0];
    ray = camera_get_ray_lens(cam, ln.x, ln.y, u, v, jit.u[2], jit.u[3]);
  } else {
    ray = camera_get_ray(cam, u, v);
  }
  out_o[pixel * 3 + 0] = ray.o.x, out_o[pixel * 3 + 1] = ray.o.y, out_o[pixel * 3 + 2] = ray.o.z;
  out_d[pixel * 3 + 0] = ray.d.x, out_d[pixel * 3 + 1] = ray.d.y, out_d[pixel * 3 + 2] = ray.d.z;
  if (out_tau) out_tau[pixel] = tau;
}
// ptc_ray_times: the shutter time of camera sample `sample` of every pixel
__global__ void k_ray_times(uint64_t seed, uint32_t n_pixels, uint32_t sample, float *out_tau) {
  const uint32_t pixel = blockIdx.x * blockDim.x + threadIdx.x;
  if (pixel < n_pixels) out_tau[pixel] = philox_uniforms(seed, pixel, sample, 0xffffffffu, 1u).u[0];
}

__global__ void k_scatter(DMaterial m, const float *dirs, const float *pos, const float *nrm, const int32_t *front,
                          const float *u4, size_t n, int32_t *scattered, float *out_o, float *out_d, float *att_out,
                          float *emitted) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Ray sr{v3(0, 0, 0), v3(0, 0, 0)};
  V3 att = v3(0, 0, 0);
  const V3 e = mat_emitted(m);
  const float u[4] = {u4[i * 4], u4[i * 4 + 1], u4[i * 4 + 2], u4[i * 4 + 3]};
  const bool ok = mat_scatter(m, v3(dirs[i * 3], dirs[i * 3 + 1], dirs[i * 3 + 2]), v3(pos[i * 3], pos[i * 3 + 1], pos[i * 3 + 2]),
                              v3(nrm[i * 3], nrm[i * 3 + 1], nrm[i * 3 + 2]), front[i] != 0, u, sr, att);
  scattered[i] = ok ? 1 : 0;
  out_o[i * 3] = sr.o.x, out_o[i * 3 + 1] = sr.o.y, out_o[i * 3 + 2] = sr.o.z;
  out_d[i * 3] = sr.d.x, out_d[i * 3 + 1] = sr.d.y, out_d[i * 3 + 2] = sr.d.z;
  att_out[i * 3] = att.x, att_out[i * 3 + 1] = att.y, att_out[i * 3 + 2] = att.z;
  emitted[i * 3] = e.x, emitted[i * 3 + 1] = e.y, emitted[i * 3 + 2] = e.z;
}

// PTC_FLAG_NEE_SKY parity hooks: sky_sample / sky_pdf as the shade stage runs them
__global__ void k_sky_sample(DScene sc, const float *u4, size_t n, float *dirs, float *pdf, float *rgb) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float u[4] = {u4[i * 4], u4[i * 4 + 1], u4[i * 4 + 2], u4[i * 4 + 3]};
  float p;
  const V3 d = sky_sample(sc, u, p);
  const V3 c = sky_color(sc, d);
  dirs[i * 3] = d.x, dirs[i * 3 + 1] = d.y, dirs[i * 3 + 2] = d.z;
  pdf[i] = p;
  rgb[i * 3] = c.x, rgb[i * 3 + 1] = c.y, rgb[i * 3 + 2] = c.z;
}
__global__ void k_sky_pdf(DScene sc, const float *dirs, size_t n, float *pdf) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) pdf[i] = sky_pdf(sc, v3(dirs[i * 3], dirs[i * 3 + 1], dirs[i * 3 + 2]));
}

// PTC_FLAG_NEE_EMITTERS parity hooks: emitter_sample as the shade stage runs it (u4 = Philox block 1's uniforms), and the
// MIS density the shade stage gives a BSDF ray whose closest hit (extend kernels, hit0 / hit1) is a sampled emitter
__global__ void k_light_sample(DScene sc, EmitterTables et, const float *x, const float *u4, size_t n, float *point, float *pdf,
                               int32_t *object, int32_t *triangle) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const V3 xi = v3(x[i * 3], x[i * 3 + 1], x[i * 3 + 2]);
  EmitterSample es;
  const bool ok = emitter_sample(sc, et, xi, u4[i * 4], u4[i * 4 + 1], u4[i * 4 + 2], u4[i * 4 + 3], es);
  const V3 y = ok ? xi + es.wi * es.dist : v3(0, 0, 0);
  point[i * 3] = y.x, point[i * 3 + 1] = y.y, point[i * 3 + 2] = y.z;
  pdf[i] = ok ? es.pdf : 0.0f;
  object[i] = ok ? sc.lights[es.light].object : -1;
  triangle[i] = ok && sc.lights[es.light].type == OBJ_MESH ? es.entry : -1;
}
__global__ void k_light_pdf(DScene sc, EmitterTables et, const float *o, const float *d, const float4 *hit0, const float4 *hit1, size_t n,
                            float *pdf) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 h0 = hit0[i], h1 = hit1[i];
  const uint32_t bits = f2u(h1.w), light = (bits >> kLightShift) & 63u;
  float p = 0.0f;
  if ((bits & kHitBit) && light != 0u) {
    const DLight &L = sc.lights[light - 1u];
    const V3 pos = v3(h0.x, h0.y, h0.z), ray_d = normalized(v3(d[i * 3], d[i * 3 + 1], d[i * 3 + 2]));
    const float dl = emitter_area_sampled(L) ? length(pos - v3(o[i * 3], o[i * 3 + 1], o[i * 3 + 2])) : h0.w;
    p = emitter_mis_pdf(L, emitter_select_prob(et, light - 1u), dl, fabsf(dot(v3(h1.x, h1.y, h1.z), ray_d)));
  }
  pdf[i] = p;
}

__global__ void k_philox(U4 c, uint32_t k0, uint32_t k1, uint32_t *out) {
  const U4 r = philox4x32_10(c, k0, k1);
  out[0] = r.x, out[1] = r.y, out[2] = r.z, out[3] = r.w;
}

// segment counts for a flat array of n rays laid out at slots [0, n): segment b holds min(cap, n - b * cap)
__global__ void k_fill_counts(uint32_t *cnt, uint32_t n_seg, uint32_t cap, uint32_t n) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n_seg) return;
  const unsigned long long lo = (unsigned long long)b * cap;
  cnt[b] = lo >= n ? 0u : (uint32_t)min((unsigned long long)cap, (unsigned long long)n - lo);
}

}  // namespace ptw
