/* ptcore.h — C ABI of the B200 path-tracing core (libptcore.so).
 *
 * Drop-in boundary for the hot path of jackra1n/raytracer-rust: the body of
 *     pub fn render_scene(scene: &Scene, camera: &Camera, render_settings: &RenderSettings) -> Vec<u32>
 * (src/renderer.rs:67-123, called once from src/main.rs:57) and everything it calls
 * (trace_ray src/renderer.rs:19-65, HittableList::hit src/hittable.rs:46-57, the `hit` of every
 * primitive, the BVH, every Material::scatter/emitted).  The reference has no FFI of its own; these
 * are the entry points an `extern "C"` block in a `ptcore-sys` crate binds (see INTEGRATION.md).
 *
 * Conventions
 *  - every function returns 0 on success or a negative PTC_E_* code; nothing unwinds or aborts across
 *    the boundary; ptc_last_error() gives the thread-local message of the last failure.
 *  - the caller owns every input and output buffer; inputs are copied during the add_* call.
 *  - matrices are 16 floats, column-major, exactly glam::Mat4::to_cols_array().
 *  - the ORDER of add_* calls is the order of Scene.object_list and is semantically significant
 *    (closest-hit tie-breaking, hittable.rs:50-55).  add_* return the object / material index.
 *  - a scene handle is not thread-safe; one render in flight per handle.
 *  - there is NO CPU fallback: without a CUDA device commit/render/intersect fail with PTC_E_CUDA.
 */
#ifndef PTCORE_H
#define PTCORE_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define PTC_ABI_VERSION 1

enum {
  PTC_OK = 0,
  PTC_E_INVALID = -1, /* bad argument / bad handle state */
  PTC_E_CUDA = -2,    /* CUDA runtime error or no device */
  PTC_E_NOMEM = -3,
  PTC_E_STATE = -4    /* call order violated (e.g. render before commit) */
};

/* Material tags (one per `impl Material`) */
enum {
  PTC_MAT_LAMBERT = 0,         /* Lambertian, AlbedoKind::Solid      src/material.rs:29-71 */
  PTC_MAT_LAMBERT_CHECKER = 1, /* Lambertian, AlbedoKind::Checked    src/material.rs:38-46, tungsten/materials.rs:72-100 */
  PTC_MAT_METAL = 2,           /* Metal                              src/material.rs:73-110 */
  PTC_MAT_DIELECTRIC = 3,      /* Dielectric                         src/material.rs:112-167 */
  PTC_MAT_EMISSIVE = 4,        /* EmissiveLight                      src/material.rs:169-192 */
  PTC_MAT_PLASTIC = 5,         /* PlasticMaterial                    src/tungsten/materials.rs:12-70 */
  PTC_MAT_ROUGH_CONDUCTOR = 6, /* RoughConductor                     src/tungsten/materials.rs:154-377 */
  PTC_MAT_NULL = 7             /* NullMaterial                       src/material.rs:229-252 */
};
enum { PTC_DIST_GGX = 0, PTC_DIST_BECKMANN = 1 }; /* MicrofacetDistribution, tungsten/materials.rs:148-152 */

/* What `Material::describe()` forwards: the struct fields as the Rust constructors left them. */
typedef struct ptc_material {
  int32_t type;
  float albedo[3];    /* Lambertian/Metal/Plastic/RoughConductor albedo; EmissiveLight.color; checker on_color */
  float off_color[3]; /* CheckerTexture.off_color */
  float inv_scale;    /* CheckerTexture.inv_scale */
  float fuzz;         /* Metal.fuzz (already clamped by Metal::new) */
  float ior;          /* Dielectric.refractive_index / PlasticMaterial.ior */
  float roughness;    /* RoughConductor.roughness (already >= 0.01) */
  float eta[3];       /* MetalType::ior_k().0 */
  float k[3];         /* MetalType::ior_k().1 */
  int32_t distribution;
} ptc_material;

/* Camera fields, src/camera.rs:4-11 */
typedef struct ptc_camera {
  float position[3], forward[3], right[3], true_up[3];
  float half_width, half_height;
} ptc_camera;

/* RenderSettings (src/tungsten/parser.rs:191-197) + what a sharded GPU run needs. */
typedef struct ptc_render_settings {
  int32_t width, height;
  int32_t spp;          /* samples_per_pixel of the whole job (the 1/spp of renderer.rs:85 uses this) */
  int32_t max_depth;    /* renderer.rs:101 */
  uint64_t seed;        /* Philox key (the reference seeds a per-row StdRng with y, renderer.rs:91) */
  int32_t sample_begin; /* this call renders samples [sample_begin, sample_end); 0,0 = [0, spp) */
  int32_t sample_end;
  int32_t tile_mod;     /* pixel sharding: only 32x32 tiles with tile_index % tile_mod == tile_rem; 0 = all */
  int32_t tile_rem;
  int32_t pool_paths;   /* path-pool slots; 0 = default: the whole job in flight at once when that fits a quarter of the free
                           device memory (224 B per slot with meshes), else 48 Mi slots */
  int32_t flags;        /* PTC_FLAG_* */
} ptc_render_settings;

enum {
  PTC_FLAG_COUNTERS = 1, /* run the instrumented extend kernel: fills nodes_visited / tris_tested (slower) */
  PTC_FLAG_TIMING = 2,   /* record CUDA events around every extend / shade launch: fills extend_ms / shade_ms */
  PTC_FLAG_NEE = 4,      /* next-event estimation + multiple importance sampling (SURVEY.md 8f-4; the Tungsten scenes ask for
                            it with "enable_mis", which the reference's IntegratorConfig ignores, src/tungsten/parser.rs:167-171).
                            OFF by default: the default integrator is the reference's, sample for sample.  With the flag every
                            non-specular hit also samples one emissive sphere / quad through a shadow ray, and emitters found
                            by BSDF sampling are weighted with the power heuristic.  Same expected image, far less noise where
                            emitters are small (veach-mis).  stats.rays then counts the shadow rays too. */
  PTC_FLAG_NEE_SKY = 8   /* with PTC_FLAG_NEE only (alone: PTC_E_INVALID): NEE also samples the HDR sky as an environment light,
                            importance-sampled by its radiance over the cells of the reference's equirectangular lookup, with
                            the power heuristic against BSDF sampling (the Tungsten scenes' "enable_light_sampling").  Same
                            expected image, less noise under a sky with bright spots (the teapot's envmap).  On a scene
                            without an HDR sky, or with an all-zero one, it changes nothing: the image is PTC_FLAG_NEE's. */
};

/* HitRecord (src/hittable.rs:10-16) plus the ids the parity bar is stated on. */
typedef struct ptc_hit {
  int32_t object;   /* index in object_list, -1 = miss */
  int32_t triangle; /* index in Mesh.triangles as passed to add_mesh, -1 for analytic primitives */
  float t;
  float position[3];
  float normal[3];
  int32_t front_face;
  int32_t material;
} ptc_hit;

typedef struct ptc_stats {
  uint64_t paths;          /* camera paths started */
  uint64_t rays;           /* extend-queue items = trace_ray calls with depth > 0 */
  uint64_t iterations;     /* wavefront iterations: the last one in which any pool segment had a ray to extend */
  uint64_t kernel_launches;
  double render_ms;        /* CUDA-event time of the whole render on the render stream */
  double extend_ms;        /* sum of CUDA-event times of the extend kernel launches (PTC_FLAG_TIMING) */
  double shade_ms;         /* ... of the shade kernel launches                        (PTC_FLAG_TIMING) */
  uint64_t extend_launches;/* number of extend launches those times cover */
  uint64_t nodes_visited;  /* wide-BVH nodes popped   (only with PTC_FLAG_COUNTERS) */
  uint64_t tris_tested;    /* triangles tested        (only with PTC_FLAG_COUNTERS) */
  uint64_t mesh_rays;      /* ray x mesh-instance traversals (only with PTC_FLAG_COUNTERS) */
  double pre_ms, traverse_ms, post_ms; /* the three kernels of the extend stage (PTC_FLAG_TIMING); extend_ms = their sum */
  double regen_ms;         /* always 0: path regeneration is part of the shade kernel (kept for ABI v1 layout) */
} ptc_stats;

typedef struct ptc_mesh_info {
  int64_t triangles;       /* as passed to add_mesh */
  int64_t live_triangles;  /* not under a flat node of the reference's BVH (src/acceleration/aabb.rs:40) */
  int64_t ref_nodes, ref_leaves; /* shape of the restated reference build (src/acceleration/bvh.rs:15-76) */
  int32_t ref_depth;
  int64_t wide_nodes;      /* 80-byte 8-wide nodes in the device BVH */
  int32_t wide_depth;
  int64_t node_bytes, triangle_bytes;
} ptc_mesh_info;

typedef struct ptc_scene ptc_scene;

const char *ptc_last_error(void);
int ptc_abi_version(void);
int ptc_device_count(void);

ptc_scene *ptc_scene_create(void);
void ptc_scene_destroy(ptc_scene *);

int ptc_scene_add_material(ptc_scene *, const ptc_material *);
/* Sphere { center, radius, material }                      src/objects/sphere.rs:8-12 */
int ptc_scene_add_sphere(ptc_scene *, const float center[3], float radius, int material);
/* Plane { p1, normal (already normalised), material }      src/objects/plane.rs:9-13 */
int ptc_scene_add_plane(ptc_scene *, const float p1[3], const float normal[3], int material);
/* Quad { base, edge0, edge1, normal, d, inv_edge0_len_sq, inv_edge1_len_sq }  src/tungsten/objects/quad.rs:10-18 */
int ptc_scene_add_quad(ptc_scene *, const float base[3], const float edge0[3], const float edge1[3],
                       const float normal[3], float d, float inv_edge0_len_sq, float inv_edge1_len_sq, int material);
/* Cube { object_to_world, world_to_object }                src/objects/cube.rs:11-17 */
int ptc_scene_add_cube(ptc_scene *, const float object_to_world[16], const float world_to_object[16], int material);
/* Mesh { triangles, object_to_world, world_to_object }     src/mesh/mesh_object.rs:17-22
 * tris = n x 12 floats: Triangle { v0, v1, v2, normal } (src/mesh/triangle.rs:5-11), object space. */
int ptc_scene_add_mesh(ptc_scene *, const float *tris, int64_t n, const float object_to_world[16],
                       const float world_to_object[16], int material);
/* Scene.skybox_hdr_image (src/scene.rs:9): w*h*3 linear floats, row-major, top row first */
int ptc_scene_set_sky_hdr(ptc_scene *, const float *rgb, int32_t w, int32_t h);

/* Host half of commit only (reference-BVH dead mask -> SAH -> 8-wide quantised BVH); needs no device.  Optional:
 * ptc_scene_commit runs it if it has not been run. */
int ptc_scene_build(ptc_scene *);
/* Flatten + build + upload to CUDA device `device`.  Fails with PTC_E_CUDA when there is no device. */
int ptc_scene_commit(ptc_scene *, int device);
/* Same with options.  PTC_COMMIT_FAST_BUILD: flatten the meshes entirely on the device — the reference's own median-split
 * tree (src/acceleration/bvh.rs:15-76), which has to be restated anyway for the dead-triangle mask, doubles as the
 * traversal tree: 2 M triangles commit in ~0.2 s instead of ~1 s, the render is ~20 % slower than through the default
 * SAH tree (host-built from the device-restated mask).  Results (hit records, images) are identical either way.
 * PTC_COMMIT_DEVICE_SAH: flatten the meshes entirely on the device AND build the default's traversal tree there — the
 * binned SAH tree and 8-wide collapse of the host builder, decision for decision, for meshes of every size (same wide
 * nodes and leaves, same node and triangle tests per ray).  Meshes of 2^27
 * triangles or more, and a non-default PTC_REF_TIE, still take the host builder; PTC_COLLAPSE=greedy applies to the host
 * builder only.  Combined with PTC_COMMIT_FAST_BUILD: PTC_E_INVALID. */
enum { PTC_COMMIT_FAST_BUILD = 1, PTC_COMMIT_DEVICE_SAH = 2 };
int ptc_scene_commit_ex(ptc_scene *, int device, int flags);
/* Path-pool slots the last render on this handle used (what pool_paths = 0 resolved to). */
int64_t ptc_scene_last_pool_slots(const ptc_scene *);
int ptc_scene_mesh_info(const ptc_scene *, int object, ptc_mesh_info *info, uint8_t *dead /* n or NULL */,
                        int32_t *order /* n or NULL */);

/* render_scene up to `image_data` (renderer.rs:83-106): out_rgb = W*H*3 floats on the HOST, linear mean
 * radiance (sum over this call's samples / spp).  Includes the device->host copy. */
int ptc_render(ptc_scene *, const ptc_camera *, const ptc_render_settings *, float *out_rgb, ptc_stats *stats);
/* render_scene as a whole (renderer.rs:67-123): out_u32 = W*H pixels 0x00RRGGBB on the HOST, row-major, top row first —
 * the Vec<u32> the reference returns.  The film is resolved on the device; only W*H*4 bytes cross PCIe. */
int ptc_render_u32(ptc_scene *, const ptc_camera *, const ptc_render_settings *, uint32_t *out_u32, ptc_stats *stats);
/* Same, device-resident: ADDS this call's radiance sum (not divided by spp) into d_accum (W*H*3 floats in
 * device memory of the scene's device), ordered on `cuda_stream` (a cudaStream_t; NULL = the legacy default stream,
 * so work the caller queued on stream 0 — zeroing d_accum, waiting for a collective — is ordered before the render).
 * Returns after the work is enqueued AND finished (the wavefront loop polls its queue counters). */
int ptc_render_accumulate(ptc_scene *, const ptc_camera *, const ptc_render_settings *, float *d_accum,
                          void *cuda_stream, ptc_stats *stats);
/* Adaptive sampling: every pixel is rendered until its noise estimate converges, at most settings->spp samples.
 * Schedule: samples [0, min_spp/2) and [min_spp/2, min_spp) of every pixel, then [n, min(2n, spp)) of the pixels still
 * active.  After each pass from m to n samples a pixel with fp32 film sum V (Vp before the pass) NEEDS MORE iff
 * e = sum_c |V_c/n - (V_c-Vp_c)/(n-m)| / (1e-4 + sqrt(sum_c V_c/n)) >= threshold (Dammertz et al. 2009) and every channel
 * of V is finite; it stays active iff some active pixel of its 3x3 neighbourhood (itself included) needs more.  A pixel
 * that leaves never returns.  Philox is keyed on (pixel, sample) and the film sums are fixed-point, so every pixel ends
 * with exactly the film, the image and the packed value of a uniform render at its own sample count.
 * settings: sample_begin = sample_end = 0 and tile_mod = 0, else PTC_E_INVALID; flags as in ptc_render.  Single device:
 * ptc_multi_* has no adaptive variant.  Outputs are host buffers, each may be NULL: out_rgb W*H*3 linear mean radiance
 * (the pixel's sum / its own count), out_u32 W*H 0x00RRGGBB as ptc_render_u32, out_spp W*H samples each pixel received.
 * stats: paths = sum of the counts; rays, iterations, launches and stage times summed over the passes; render_ms from
 * the first pass to the end of the resolve (device events).  The ptc_adaptive arguments are checked before the scene's
 * state: PTC_E_INVALID for bad ones even on an uncommitted scene. */
typedef struct ptc_adaptive {
  int32_t min_spp; /* every pixel gets at least this many samples; even, >= 2, <= settings->spp */
  float threshold; /* a pixel keeps sampling while its error estimate is >= threshold; 0 = never stop early, +inf = stop at min_spp */
} ptc_adaptive;
int ptc_render_adaptive(ptc_scene *, const ptc_camera *, const ptc_render_settings *, const ptc_adaptive *, float *out_rgb,
                        uint32_t *out_u32, int32_t *out_spp, ptc_stats *stats);
/* Film resolve, renderer.rs:112-120 + color.rs:87-93: out = pack(sqrt(rgb * scale)).  Device and host buffers. */
int ptc_resolve_device(const float *d_rgb, int64_t n_pixels, float scale, uint32_t *d_out, void *cuda_stream);
int ptc_resolve_u32(ptc_scene *, const float *rgb, int64_t n_pixels, float scale, uint32_t *out);

/* In-process multi-GPU, for a single-process host like the reference's binary (SURVEY.md 8e): the scene is replicated
 * on every device of `devices` (devices[0] = the device `primary` was committed on; the host-side flattening is not
 * repeated), one host thread per device renders its shard — a balanced sample range or the interleaved 32x32 tiles
 * with index % n == i, Philox keyed on the global pixel / sample so the shards are invisible — and the fixed-point films
 * (int64 radiance sums, then the NaN / inf flag words) are summed onto devices[0] by two ncclReduce calls over NVLink, so
 * the image is the one-GPU image bit for bit.  devices[0] then resolves the film (1/spp, and the packing for
 * ptc_multi_render_u32) and copies the image to the host.
 * The one-process-per-GPU route (ptc_render_accumulate + torch.distributed, bench.py) stays available.
 * NCCL is loaded at run time (libnccl.so.2) by ptc_multi_create for n > 1 only. */
typedef struct ptc_multi ptc_multi;
enum { PTC_SHARD_SAMPLES = 0, PTC_SHARD_TILES = 1 };
int ptc_multi_create(ptc_scene *primary, const int *devices, int n, ptc_multi **out);
void ptc_multi_destroy(ptc_multi *);
/* out_rgb as in ptc_render.  stats: paths / rays / launches summed over the devices, render_ms = host wall clock of the
 * whole call.  settings->tile_mod must be 0. */
int ptc_multi_render(ptc_multi *, const ptc_camera *, const ptc_render_settings *, int shard_mode, float *out_rgb,
                     ptc_stats *stats);
/* out_u32 as in ptc_render_u32 (resolved on devices[0]) */
int ptc_multi_render_u32(ptc_multi *, const ptc_camera *, const ptc_render_settings *, int shard_mode, uint32_t *out_u32,
                         ptc_stats *stats);

/* Parity hooks (host buffers in and out; each runs the SAME device functions the render kernels use). */
/* HittableList::hit for n caller-provided rays (directions used as given). */
int ptc_intersect(ptc_scene *, const float *origins, const float *dirs, int64_t n, float t_min, float t_max,
                  ptc_hit *out, ptc_stats *stats);
/* Camera::get_ray + the Philox jitter for sample `sample` of every pixel: out_o/out_d = W*H*3 floats. */
int ptc_primary_rays(ptc_scene *, const ptc_camera *, const ptc_render_settings *, int32_t sample, float *out_o,
                     float *out_d);
/* Material::emitted + Material::scatter for n (ray_dir, position, normal, front_face, u[4]) tuples.
 * scattered[i] = 1/0; out_origin/out_dir/attenuation/emitted = n x 3 floats. */
int ptc_scatter(ptc_scene *, int material, const float *ray_dirs, const float *positions, const float *normals,
                const int32_t *front_face, const float *u4, int64_t n, int32_t *scattered, float *out_origin,
                float *out_dir, float *attenuation, float *emitted);
/* The HDR sky as a light (PTC_FLAG_NEE_SKY): n directions drawn from u4 (n x 4 uniforms in [0, 1)), their solid-angle
 * pdf and the sky's radiance along them (out_dir / out_rgb n x 3 floats, out_pdf n floats); and the pdf of n directions.
 * PTC_E_STATE when the committed scene has no sky distribution (no HDR sky, or an all-zero one). */
int ptc_sky_sample(ptc_scene *, const float *u4, int64_t n, float *out_dir, float *out_pdf, float *out_rgb);
int ptc_sky_pdf(ptc_scene *, const float *dirs, int64_t n, float *out_pdf);
/* Philox4x32-10 known-answer hook (runs on the device). */
int ptc_philox(ptc_scene *, const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);

#ifdef __cplusplus
}
#endif
#endif
