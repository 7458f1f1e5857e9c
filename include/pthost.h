/* pthost.h — host-side surface of the renderer, kept as the reference has it (libpthost.so).
 *
 * The north star keeps the reference's host side (Tungsten-style JSON loading, Camera, the
 * Hittable/Material abstractions, PNG output) in Rust and swaps only the body of render_scene for the
 * C ABI in ptcore.h.  This image has no Rust toolchain, so this library is the C++ stand-in for that host
 * side: same entry points, same argument meaning, same error behaviour as
 *     load_scene_from_json   src/tungsten/parser.rs:245-815
 *     Mesh::from_obj         src/mesh/mesh_object.rs:59-139
 *     Camera::new            src/camera.rs:14-31
 *     Quad::new_transformed  src/tungsten/objects/quad.rs:26-79
 *     render_scene           src/renderer.rs:67-123   (forwards to ptc_render + ptc_resolve_u32)
 *     save_image             src/renderer.rs:125-179
 * It is plain host code: no CUDA, no oracle.  It is what tests and bench.py use to build scene
 * descriptions that are then fed, unchanged, both to libptcore (product) and to the oracle (checker).
 */
#ifndef PTHOST_H
#define PTHOST_H
#include <stdint.h>
#include "ptcore.h"
#ifdef __cplusplus
extern "C" {
#endif

enum { PTH_SPHERE = 0, PTH_PLANE = 1, PTH_QUAD = 2, PTH_CUBE = 3, PTH_MESH = 4 };

/* One entry of Scene.object_list with the already-derived fields of the Rust struct. */
typedef struct pth_object {
  int32_t type;     /* PTH_* */
  int32_t material; /* index into the material table */
  int32_t mesh;     /* index into the mesh table (PTH_MESH) or -1 */
  int32_t pad;
  float center[3];  /* Sphere.center */
  float radius;     /* Sphere.radius */
  float p1[3];      /* Plane.p1 */
  float normal[3];  /* Plane.normal / Quad.normal */
  float base[3], edge0[3], edge1[3]; /* Quad */
  float d, inv_edge0_len_sq, inv_edge1_len_sq;
  float o2w[16], w2o[16]; /* Cube / Mesh, column-major */
} pth_object;

typedef struct pth_scene pth_scene;

const char *pth_last_error(void);

/* load_scene_from_json: returns NULL on error (message in pth_last_error), like the Err(..) of parser.rs:247. */
pth_scene *pth_load_scene_from_json(const char *json_path);
/* Extensions beyond the reference's loader (SURVEY.md 8f-2), all OFF in pth_load_scene_from_json:
 *   INFINITE_SPHERE_SKY  `"type": "infinite_sphere"` (not a variant of ObjectConfigVariant, parser.rs:136-165: the
 *                        reference rejects the whole file, e.g. its own tungsten/teapot/scene.json) becomes the sky
 *   WO3_STRIDE16         read .wo3 triangles with Tungsten's 16-byte records; without it the reader restates the
 *                        reference's 12-byte mis-read (mesh_object.rs:188-190) index for index
 *   SKIP_UNKNOWN         other unknown primitive types are skipped with a warning instead of failing the file
 *   THIN_LENS            a camera of `"type": "thinlens"` gets a lens (pth_scene_lens): aperture_size is the lens radius,
 *                        focus_distance the focus distance, or |look_at - position| when the key is missing (our rule);
 *                        aperture textures, cat-eye and focus_pivot are ignored with a warning.  Without the flag the
 *                        camera is a pinhole, as in the reference */
enum { PTH_LOAD_INFINITE_SPHERE_SKY = 1, PTH_LOAD_WO3_STRIDE16 = 2, PTH_LOAD_SKIP_UNKNOWN = 4, PTH_LOAD_THIN_LENS = 8 };
pth_scene *pth_load_scene_from_json_ex(const char *json_path, int flags);
/* An empty scene to be filled programmatically (tests, synthetic scenes). */
pth_scene *pth_scene_new(void);
void pth_scene_free(pth_scene *);

int32_t pth_scene_material_count(const pth_scene *);
int32_t pth_scene_object_count(const pth_scene *);
int32_t pth_scene_mesh_count(const pth_scene *);
const ptc_material *pth_scene_materials(const pth_scene *);
const pth_object *pth_scene_objects(const pth_scene *);
/* n x 12 floats (v0,v1,v2,normal), object space, degenerate triangles already filtered */
int64_t pth_scene_mesh(const pth_scene *, int32_t mesh, const float **tris);
int pth_scene_sky(const pth_scene *, const float **rgb, int32_t *w, int32_t *h);
void pth_scene_camera(const pth_scene *, ptc_camera *);
/* 1 and *out = the camera's lens when the scene has one (PTH_LOAD_THIN_LENS), 0 for a pinhole (out untouched) */
int pth_scene_lens(const pth_scene *, ptc_lens *out);
/* RenderSettings: width, height, samples_per_pixel, max_depth (parser.rs:255-292) */
void pth_scene_settings(const pth_scene *, int32_t *width, int32_t *height, int32_t *spp, int32_t *max_depth);

/* programmatic construction (same derivations as the loader) */
int pth_scene_push_material(pth_scene *, const ptc_material *);
int pth_scene_push_sphere(pth_scene *, const float center[3], float radius, int material);
int pth_scene_push_plane(pth_scene *, const float point[3], const float normal[3], int material); /* Plane::new normalises */
int pth_scene_push_quad(pth_scene *, const float scale[3], const float rot_deg[3], const float pos[3], int material);
int pth_scene_push_cube(pth_scene *, const float scale[3], const float rot_deg[3], const float pos[3], int material);
/* verts: nv x 3, indices: nt x 3; builds Triangle::new + degenerate filter */
int pth_scene_push_mesh(pth_scene *, const float *verts, int64_t nv, const int32_t *indices, int64_t nt,
                        const float scale[3], const float rot_deg[3], const float pos[3], int material);
int pth_scene_push_obj(pth_scene *, const char *obj_path, const float scale[3], const float rot_deg[3],
                       const float pos[3], int material);
int pth_scene_set_sky_hdr_file(pth_scene *, const char *hdr_path);
/* w*h*3 linear floats, row-major, top row first (what into_rgb32f() yields, parser.rs:504) */
int pth_scene_set_sky_rgb(pth_scene *, const float *rgb, int32_t w, int32_t h);
void pth_scene_set_camera(pth_scene *, const float position[3], const float look_at[3], const float up[3], float vfov_deg,
                          float aspect);
void pth_scene_set_settings(pth_scene *, int32_t width, int32_t height, int32_t spp, int32_t max_depth);

/* BASELINE config C5: procedural height field (cells x cells x 2 triangles over [-50,50]^2, 4 octaves of
 * integer-hash value noise, seed 0x5EED) + glass sphere + GGX-Al cube + emissive quad; camera (60,40,60)->(0,5,0). */
pth_scene *pth_scene_synthetic(int32_t cells, uint32_t seed);

/* Transform = Mat4::from_scale_rotation_translation(scale, Quat::from_euler(YXZ, ry, rx, rz), pos) and its inverse
 * (parser.rs:647-674). */
void pth_transform(const float scale[3], const float rot_deg[3], const float pos[3], float o2w[16], float w2o[16]);
/* Camera::new (camera.rs:14-31) */
void pth_camera_new(const float position[3], const float look_at[3], const float up[3], float vfov_deg, float aspect,
                    ptc_camera *out);

/* Feed the description to the product core in object_list order (what the Rust `describe()` walk does), and the lens if
 * the scene has one (ptc_scene_set_lens). */
ptc_scene *pth_build_ptc_scene(const pth_scene *);
/* render_scene (renderer.rs:67-123): Vec<u32> 0x00RRGGBB, row-major, top row first, on device `device`. */
int pth_render_scene(const pth_scene *, int device, uint32_t *out_u32, ptc_stats *stats);
/* save_image (renderer.rs:125-179) minus the timestamped file name: writes an 8-bit RGB PNG. */
int pth_save_png(const char *path, const uint32_t *buffer, int32_t width, int32_t height);

#ifdef __cplusplus
}
#endif
#endif
