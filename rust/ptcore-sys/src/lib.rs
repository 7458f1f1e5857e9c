//! UNVERIFIED (no Rust toolchain in the build image): `extern "C"` declarations of include/ptcore.h, one to one.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

pub const PTC_OK: c_int = 0;
pub const PTC_E_INVALID: c_int = -1;
pub const PTC_E_CUDA: c_int = -2;
pub const PTC_E_NOMEM: c_int = -3;
pub const PTC_E_STATE: c_int = -4;

/// ptc_scene_commit_ex flags
pub const PTC_COMMIT_FAST_BUILD: c_int = 1;
pub const PTC_COMMIT_DEVICE_SAH: c_int = 2;

/// ptc_render_settings.flags
pub const PTC_FLAG_COUNTERS: i32 = 1;
pub const PTC_FLAG_TIMING: i32 = 2;
pub const PTC_FLAG_NEE: i32 = 4;
/// with PTC_FLAG_NEE only: NEE also samples the HDR sky as an environment light
pub const PTC_FLAG_NEE_SKY: i32 = 8;

pub const PTC_MAT_LAMBERT: i32 = 0;
pub const PTC_MAT_LAMBERT_CHECKER: i32 = 1;
pub const PTC_MAT_METAL: i32 = 2;
pub const PTC_MAT_DIELECTRIC: i32 = 3;
pub const PTC_MAT_EMISSIVE: i32 = 4;
pub const PTC_MAT_PLASTIC: i32 = 5;
pub const PTC_MAT_ROUGH_CONDUCTOR: i32 = 6;
pub const PTC_MAT_NULL: i32 = 7;
pub const PTC_DIST_GGX: i32 = 0;
pub const PTC_DIST_BECKMANN: i32 = 1;

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct ptc_material {
    pub type_: i32,
    pub albedo: [f32; 3],
    pub off_color: [f32; 3],
    pub inv_scale: f32,
    pub fuzz: f32,
    pub ior: f32,
    pub roughness: f32,
    pub eta: [f32; 3],
    pub k: [f32; 3],
    pub distribution: i32,
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct ptc_camera {
    pub position: [f32; 3],
    pub forward: [f32; 3],
    pub right: [f32; 3],
    pub true_up: [f32; 3],
    pub half_width: f32,
    pub half_height: f32,
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct ptc_render_settings {
    pub width: i32,
    pub height: i32,
    pub spp: i32,
    pub max_depth: i32,
    pub seed: u64,
    pub sample_begin: i32,
    pub sample_end: i32,
    pub tile_mod: i32,
    pub tile_rem: i32,
    pub pool_paths: i32,
    pub flags: i32,
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct ptc_stats {
    pub paths: u64,
    pub rays: u64,
    pub iterations: u64,
    pub kernel_launches: u64,
    pub render_ms: f64,
    pub extend_ms: f64,
    pub shade_ms: f64,
    pub extend_launches: u64,
    pub nodes_visited: u64,
    pub tris_tested: u64,
    pub mesh_rays: u64,
    pub pre_ms: f64,
    pub traverse_ms: f64,
    pub post_ms: f64,
    pub regen_ms: f64,
}

/// ptc_render_adaptive's parameters: min_spp even, >= 2, <= spp; threshold >= 0 (0: never stop early, +inf: stop at min_spp)
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct ptc_adaptive {
    pub min_spp: i32,
    pub threshold: f32,
}

#[repr(C)]
pub struct ptc_scene {
    _private: [u8; 0],
}

extern "C" {
    pub fn ptc_last_error() -> *const c_char;
    pub fn ptc_abi_version() -> c_int;
    pub fn ptc_device_count() -> c_int;
    pub fn ptc_scene_create() -> *mut ptc_scene;
    pub fn ptc_scene_destroy(s: *mut ptc_scene);
    pub fn ptc_scene_add_material(s: *mut ptc_scene, m: *const ptc_material) -> c_int;
    pub fn ptc_scene_add_sphere(s: *mut ptc_scene, center: *const f32, radius: f32, material: c_int) -> c_int;
    pub fn ptc_scene_add_plane(s: *mut ptc_scene, p1: *const f32, normal: *const f32, material: c_int) -> c_int;
    pub fn ptc_scene_add_quad(s: *mut ptc_scene, base: *const f32, edge0: *const f32, edge1: *const f32, normal: *const f32,
                              d: f32, inv_edge0_len_sq: f32, inv_edge1_len_sq: f32, material: c_int) -> c_int;
    pub fn ptc_scene_add_cube(s: *mut ptc_scene, object_to_world: *const f32, world_to_object: *const f32, material: c_int) -> c_int;
    pub fn ptc_scene_add_mesh(s: *mut ptc_scene, tris: *const f32, n: i64, object_to_world: *const f32,
                              world_to_object: *const f32, material: c_int) -> c_int;
    pub fn ptc_scene_set_sky_hdr(s: *mut ptc_scene, rgb: *const f32, w: i32, h: i32) -> c_int;
    pub fn ptc_scene_build(s: *mut ptc_scene) -> c_int;
    pub fn ptc_scene_last_pool_slots(s: *const ptc_scene) -> i64;
    pub fn ptc_scene_commit(s: *mut ptc_scene, device: c_int) -> c_int;
    /// flags: PTC_COMMIT_FAST_BUILD (flatten meshes entirely on the device: quick commit, slower traversal) or
    /// PTC_COMMIT_DEVICE_SAH (flatten them on the device into the default SAH tree: quick commit, same traversal)
    pub fn ptc_scene_commit_ex(s: *mut ptc_scene, device: c_int, flags: c_int) -> c_int;
    pub fn ptc_render(s: *mut ptc_scene, cam: *const ptc_camera, st: *const ptc_render_settings, out_rgb: *mut f32,
                      stats: *mut ptc_stats) -> c_int;
    pub fn ptc_render_u32(s: *mut ptc_scene, cam: *const ptc_camera, st: *const ptc_render_settings, out_u32: *mut u32,
                          stats: *mut ptc_stats) -> c_int;
    /// adaptive sampling, one device (include/ptcore.h); every output may be null
    pub fn ptc_render_adaptive(s: *mut ptc_scene, cam: *const ptc_camera, st: *const ptc_render_settings, ad: *const ptc_adaptive,
                               out_rgb: *mut f32, out_u32: *mut u32, out_spp: *mut i32, stats: *mut ptc_stats) -> c_int;
    pub fn ptc_render_accumulate(s: *mut ptc_scene, cam: *const ptc_camera, st: *const ptc_render_settings, d_accum: *mut f32,
                                 cuda_stream: *mut c_void, stats: *mut ptc_stats) -> c_int;
    pub fn ptc_resolve_u32(s: *mut ptc_scene, rgb: *const f32, n_pixels: i64, scale: f32, out: *mut u32) -> c_int;
    /// the HDR sky as a light (PTC_FLAG_NEE_SKY): sample / pdf hooks; PTC_E_STATE without a sky distribution
    pub fn ptc_sky_sample(s: *mut ptc_scene, u4: *const f32, n: i64, out_dir: *mut f32, out_pdf: *mut f32, out_rgb: *mut f32) -> c_int;
    pub fn ptc_sky_pdf(s: *mut ptc_scene, dirs: *const f32, n: i64, out_pdf: *mut f32) -> c_int;
    pub fn ptc_resolve_device(d_rgb: *const f32, n_pixels: i64, scale: f32, d_out: *mut u32, cuda_stream: *mut c_void) -> c_int;

    // in-process multi-GPU: one host thread per device inside the library, one ncclReduce of the film (include/ptcore.h)
    pub fn ptc_multi_create(primary: *mut ptc_scene, devices: *const c_int, n: c_int, out: *mut *mut ptc_multi) -> c_int;
    pub fn ptc_multi_destroy(m: *mut ptc_multi);
    pub fn ptc_multi_render_u32(m: *mut ptc_multi, cam: *const ptc_camera, st: *const ptc_render_settings, shard_mode: c_int,
                                out_u32: *mut u32, stats: *mut ptc_stats) -> c_int;
    pub fn ptc_multi_render(m: *mut ptc_multi, cam: *const ptc_camera, st: *const ptc_render_settings, shard_mode: c_int,
                            out_rgb: *mut f32, stats: *mut ptc_stats) -> c_int;
}

#[repr(C)]
pub struct ptc_multi {
    _private: [u8; 0],
}
pub const PTC_SHARD_SAMPLES: c_int = 0;
pub const PTC_SHARD_TILES: c_int = 1;
