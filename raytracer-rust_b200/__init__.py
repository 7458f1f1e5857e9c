"""raytracer-rust_b200 — Python surface over the two C-ABI libraries of this repo.

  libptcore.so  (include/ptcore.h)  the product: hand-written CUDA for sm_100a behind the drop-in boundary of the
                                    reference's `render_scene` (src/renderer.rs:67-123).  No CPU fallback.
  libpthost.so  (include/pthost.h)  C++ stand-in for the reference's Rust host side: `load_scene_from_json`
                                    (src/tungsten/parser.rs:245-815), `Camera::new`, `Quad::new_transformed`,
                                    `Mesh::from_obj`, `save_image`.

This module is plumbing (ctypes + numpy): it mirrors the reference's host API names so tests read like the
reference's call sites (`load_scene_from_json`, `render_scene`, `save_image`).  The directory name carries the
reference's hyphen, so import it through `ptload.load()` (repo root) or importlib, not with a plain `import`.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
REPO_ROOT = os.path.dirname(_HERE)

PTC_OK, PTC_E_INVALID, PTC_E_CUDA, PTC_E_NOMEM, PTC_E_STATE = 0, -1, -2, -3, -4
MAT_LAMBERT, MAT_LAMBERT_CHECKER, MAT_METAL, MAT_DIELECTRIC, MAT_EMISSIVE, MAT_PLASTIC, MAT_ROUGH_CONDUCTOR, MAT_NULL = range(8)
DIST_GGX, DIST_BECKMANN = 0, 1
FLAG_COUNTERS, FLAG_TIMING, FLAG_NEE, FLAG_NEE_SKY = 1, 2, 4, 8
COMMIT_FAST_BUILD = 1
COMMIT_DEVICE_SAH = 2
LOAD_INFINITE_SPHERE_SKY, LOAD_WO3_STRIDE16, LOAD_SKIP_UNKNOWN = 1, 2, 4
OBJ_SPHERE, OBJ_PLANE, OBJ_QUAD, OBJ_CUBE, OBJ_MESH = range(5)


class Material(C.Structure):  # ptc_material
    _fields_ = [("type", C.c_int32), ("albedo", C.c_float * 3), ("off_color", C.c_float * 3), ("inv_scale", C.c_float),
                ("fuzz", C.c_float), ("ior", C.c_float), ("roughness", C.c_float), ("eta", C.c_float * 3),
                ("k", C.c_float * 3), ("distribution", C.c_int32)]


class Camera(C.Structure):  # ptc_camera == src/camera.rs:4-11
    _fields_ = [("position", C.c_float * 3), ("forward", C.c_float * 3), ("right", C.c_float * 3),
                ("true_up", C.c_float * 3), ("half_width", C.c_float), ("half_height", C.c_float)]


class RenderSettings(C.Structure):  # ptc_render_settings
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("spp", C.c_int32), ("max_depth", C.c_int32),
                ("seed", C.c_uint64), ("sample_begin", C.c_int32), ("sample_end", C.c_int32), ("tile_mod", C.c_int32),
                ("tile_rem", C.c_int32), ("pool_paths", C.c_int32), ("flags", C.c_int32)]


class Adaptive(C.Structure):  # ptc_adaptive
    _fields_ = [("min_spp", C.c_int32), ("threshold", C.c_float)]


class Hit(C.Structure):  # ptc_hit
    _fields_ = [("object", C.c_int32), ("triangle", C.c_int32), ("t", C.c_float), ("position", C.c_float * 3),
                ("normal", C.c_float * 3), ("front_face", C.c_int32), ("material", C.c_int32)]


HIT_DTYPE = np.dtype([("object", "<i4"), ("triangle", "<i4"), ("t", "<f4"), ("position", "<f4", 3), ("normal", "<f4", 3),
                      ("front_face", "<i4"), ("material", "<i4")])
assert HIT_DTYPE.itemsize == C.sizeof(Hit)


class Stats(C.Structure):  # ptc_stats
    _fields_ = [("paths", C.c_uint64), ("rays", C.c_uint64), ("iterations", C.c_uint64), ("kernel_launches", C.c_uint64),
                ("render_ms", C.c_double), ("extend_ms", C.c_double), ("shade_ms", C.c_double),
                ("extend_launches", C.c_uint64), ("nodes_visited", C.c_uint64), ("tris_tested", C.c_uint64),
                ("mesh_rays", C.c_uint64), ("pre_ms", C.c_double), ("traverse_ms", C.c_double), ("post_ms", C.c_double),
                ("regen_ms", C.c_double)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class MeshInfo(C.Structure):  # ptc_mesh_info
    _fields_ = [("triangles", C.c_int64), ("live_triangles", C.c_int64), ("ref_nodes", C.c_int64), ("ref_leaves", C.c_int64),
                ("ref_depth", C.c_int32), ("wide_nodes", C.c_int64), ("wide_depth", C.c_int32), ("node_bytes", C.c_int64),
                ("triangle_bytes", C.c_int64)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class HostObject(C.Structure):  # pth_object
    _fields_ = [("type", C.c_int32), ("material", C.c_int32), ("mesh", C.c_int32), ("pad", C.c_int32),
                ("center", C.c_float * 3), ("radius", C.c_float), ("p1", C.c_float * 3), ("normal", C.c_float * 3),
                ("base", C.c_float * 3), ("edge0", C.c_float * 3), ("edge1", C.c_float * 3), ("d", C.c_float),
                ("inv_edge0_len_sq", C.c_float), ("inv_edge1_len_sq", C.c_float), ("o2w", C.c_float * 16),
                ("w2o", C.c_float * 16)]


_F = C.POINTER(C.c_float)
_vp = C.c_void_p


def _fptr(a):
    return a.ctypes.data_as(_F)


def _f32(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float32)
    if shape is not None:
        a = a.reshape(shape)
    return a


class PtcError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"ptcore error {code}: {msg}")
        self.code = code


_core = None
_host = None


def core_path():
    return os.path.join(_HERE, "libptcore.so")


def host_path():
    return os.path.join(_HERE, "libpthost.so")


def core():
    """Load libptcore.so (the CUDA core).  Raises if it has not been built: there is nothing to fall back to."""
    global _core
    if _core is not None:
        return _core
    p = core_path()
    if not os.path.exists(p):
        raise ImportError(f"{p} is missing: build it first (`make`, or __graft_entry__.build()); "
                          "the path tracer has no CPU fallback")
    L = C.CDLL(p, mode=C.RTLD_GLOBAL)
    L.ptc_last_error.restype = C.c_char_p
    L.ptc_scene_create.restype = _vp
    L.ptc_scene_destroy.argtypes = [_vp]
    L.ptc_scene_destroy.restype = None
    L.ptc_scene_add_material.argtypes = [_vp, C.POINTER(Material)]
    L.ptc_scene_add_sphere.argtypes = [_vp, _F, C.c_float, C.c_int]
    L.ptc_scene_add_plane.argtypes = [_vp, _F, _F, C.c_int]
    L.ptc_scene_add_quad.argtypes = [_vp, _F, _F, _F, _F, C.c_float, C.c_float, C.c_float, C.c_int]
    L.ptc_scene_add_cube.argtypes = [_vp, _F, _F, C.c_int]
    L.ptc_scene_add_mesh.argtypes = [_vp, _F, C.c_int64, _F, _F, C.c_int]
    L.ptc_scene_set_sky_hdr.argtypes = [_vp, _F, C.c_int32, C.c_int32]
    L.ptc_scene_build.argtypes = [_vp]
    L.ptc_scene_commit.argtypes = [_vp, C.c_int]
    L.ptc_scene_commit_ex.argtypes = [_vp, C.c_int, C.c_int]
    L.ptc_scene_mesh_info.argtypes = [_vp, C.c_int, C.POINTER(MeshInfo), _vp, _vp]
    L.ptc_scene_last_pool_slots.argtypes = [_vp]
    L.ptc_scene_last_pool_slots.restype = C.c_int64
    L.ptc_render.argtypes = [_vp, C.POINTER(Camera), C.POINTER(RenderSettings), _F, C.POINTER(Stats)]
    L.ptc_render_u32.argtypes = [_vp, C.POINTER(Camera), C.POINTER(RenderSettings), _vp, C.POINTER(Stats)]
    L.ptc_render_adaptive.argtypes = [_vp, C.POINTER(Camera), C.POINTER(RenderSettings), C.POINTER(Adaptive), _F, _vp, _vp,
                                      C.POINTER(Stats)]
    L.ptc_render_accumulate.argtypes = [_vp, C.POINTER(Camera), C.POINTER(RenderSettings), _vp, _vp, C.POINTER(Stats)]
    L.ptc_resolve_device.argtypes = [_vp, C.c_int64, C.c_float, _vp, _vp]
    L.ptc_resolve_u32.argtypes = [_vp, _F, C.c_int64, C.c_float, _vp]
    L.ptc_intersect.argtypes = [_vp, _F, _F, C.c_int64, C.c_float, C.c_float, _vp, C.POINTER(Stats)]
    L.ptc_primary_rays.argtypes = [_vp, C.POINTER(Camera), C.POINTER(RenderSettings), C.c_int32, _F, _F]
    L.ptc_scatter.argtypes = [_vp, C.c_int, _F, _F, _F, _vp, _F, C.c_int64, _vp, _F, _F, _F, _F]
    L.ptc_philox.argtypes = [_vp, _vp, _vp, _vp]
    L.ptc_sky_sample.argtypes = [_vp, _F, C.c_int64, _F, _F, _F]
    L.ptc_sky_pdf.argtypes = [_vp, _F, C.c_int64, _F]
    L.ptc_multi_create.argtypes = [_vp, C.POINTER(C.c_int), C.c_int, C.POINTER(_vp)]
    L.ptc_multi_destroy.argtypes = [_vp]
    L.ptc_multi_destroy.restype = None
    L.ptc_multi_render.argtypes = [_vp, C.POINTER(Camera), C.POINTER(RenderSettings), C.c_int, _F, C.POINTER(Stats)]
    L.ptc_multi_render_u32.argtypes = [_vp, C.POINTER(Camera), C.POINTER(RenderSettings), C.c_int, _vp, C.POINTER(Stats)]
    _core = L
    return L


def host():
    global _host
    if _host is not None:
        return _host
    p = host_path()  # binds libptcore.so itself, when a scene is first handed to the core (pth_build_ptc_scene)
    if not os.path.exists(p):
        raise ImportError(f"{p} is missing: build it first (`make`, or __graft_entry__.build())")
    L = C.CDLL(p)
    L.pth_last_error.restype = C.c_char_p
    L.pth_load_scene_from_json.argtypes = [C.c_char_p]
    L.pth_load_scene_from_json.restype = _vp
    L.pth_load_scene_from_json_ex.argtypes = [C.c_char_p, C.c_int]
    L.pth_load_scene_from_json_ex.restype = _vp
    L.pth_scene_new.restype = _vp
    L.pth_scene_free.argtypes = [_vp]
    L.pth_scene_free.restype = None
    for n in ("pth_scene_material_count", "pth_scene_object_count", "pth_scene_mesh_count"):
        getattr(L, n).argtypes = [_vp]
        getattr(L, n).restype = C.c_int32
    L.pth_scene_materials.argtypes = [_vp]
    L.pth_scene_materials.restype = C.POINTER(Material)
    L.pth_scene_objects.argtypes = [_vp]
    L.pth_scene_objects.restype = C.POINTER(HostObject)
    L.pth_scene_mesh.argtypes = [_vp, C.c_int32, C.POINTER(_F)]
    L.pth_scene_mesh.restype = C.c_int64
    L.pth_scene_sky.argtypes = [_vp, C.POINTER(_F), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    L.pth_scene_camera.argtypes = [_vp, C.POINTER(Camera)]
    L.pth_scene_camera.restype = None
    L.pth_scene_settings.argtypes = [_vp] + [C.POINTER(C.c_int32)] * 4
    L.pth_scene_settings.restype = None
    L.pth_scene_push_material.argtypes = [_vp, C.POINTER(Material)]
    L.pth_scene_push_sphere.argtypes = [_vp, _F, C.c_float, C.c_int]
    L.pth_scene_push_plane.argtypes = [_vp, _F, _F, C.c_int]
    L.pth_scene_push_quad.argtypes = [_vp, _F, _F, _F, C.c_int]
    L.pth_scene_push_cube.argtypes = [_vp, _F, _F, _F, C.c_int]
    L.pth_scene_push_mesh.argtypes = [_vp, _F, C.c_int64, _vp, C.c_int64, _F, _F, _F, C.c_int]
    L.pth_scene_push_obj.argtypes = [_vp, C.c_char_p, _F, _F, _F, C.c_int]
    L.pth_scene_set_sky_hdr_file.argtypes = [_vp, C.c_char_p]
    L.pth_scene_set_sky_rgb.argtypes = [_vp, _F, C.c_int32, C.c_int32]
    L.pth_scene_set_camera.argtypes = [_vp, _F, _F, _F, C.c_float, C.c_float]
    L.pth_scene_set_camera.restype = None
    L.pth_scene_set_settings.argtypes = [_vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32]
    L.pth_scene_set_settings.restype = None
    L.pth_scene_synthetic.argtypes = [C.c_int32, C.c_uint32]
    L.pth_scene_synthetic.restype = _vp
    L.pth_transform.argtypes = [_F, _F, _F, _F, _F]
    L.pth_transform.restype = None
    L.pth_camera_new.argtypes = [_F, _F, _F, C.c_float, C.c_float, C.POINTER(Camera)]
    L.pth_camera_new.restype = None
    L.pth_build_ptc_scene.argtypes = [_vp]
    L.pth_build_ptc_scene.restype = _vp
    L.pth_render_scene.argtypes = [_vp, C.c_int, _vp, C.POINTER(Stats)]
    L.pth_save_png.argtypes = [C.c_char_p, _vp, C.c_int32, C.c_int32]
    _host = L
    return L


def device_count():
    return core().ptc_device_count()


def _ck(rc):
    if rc < 0:
        raise PtcError(rc, core().ptc_last_error().decode())
    return rc


# ---------------------------------------------------------------------------------------------------------------
# Material constructors with the reference constructors' derivations (Metal::new, CheckerTexture::new,
# RoughConductor::new, MetalType::ior_k)
METALS = {  # src/tungsten/materials.rs:116-152
    "cu": ((0.200, 1.090, 1.420), (3.910, 2.570, 2.300)), "au": ((0.170, 0.350, 1.500), (3.140, 2.300, 1.920)),
    "ag": ((0.155, 0.145, 0.135), (3.910, 2.610, 2.370)), "al": ((1.360, 0.965, 0.620), (7.570, 6.690, 5.440)),
    "ni": ((1.920,) * 3, (3.670,) * 3), "ti": ((2.740,) * 3, (3.170,) * 3), "fe": ((2.870,) * 3, (3.140,) * 3),
    "pb": ((1.910,) * 3, (3.180,) * 3),
}


def lambertian(albedo):
    m = Material(type=MAT_LAMBERT)
    m.albedo[:] = albedo
    return m


def checker(on_color, off_color, scale):
    m = Material(type=MAT_LAMBERT_CHECKER)
    m.albedo[:] = on_color
    m.off_color[:] = off_color
    s = np.float32(scale)
    m.inv_scale = 1.0 if abs(s) < 1e-6 else float(np.float32(1.0) / s)
    return m


def metal(albedo, fuzz):
    m = Material(type=MAT_METAL)
    m.albedo[:] = albedo
    m.fuzz = min(max(fuzz, 0.0), 1.0)
    return m


def dielectric(ior):
    return Material(type=MAT_DIELECTRIC, ior=ior)


def emissive(color):
    m = Material(type=MAT_EMISSIVE)
    m.albedo[:] = color
    return m


def plastic(albedo, ior=1.5):
    m = Material(type=MAT_PLASTIC, ior=ior)
    m.albedo[:] = albedo
    return m


def rough_conductor(albedo, roughness, metal_type="cu", distribution=DIST_GGX):
    m = Material(type=MAT_ROUGH_CONDUCTOR, roughness=max(roughness, 0.01), distribution=distribution)
    m.albedo[:] = albedo
    eta, k = METALS[metal_type.lower()]
    m.eta[:] = eta
    m.k[:] = k
    return m


def null_material():
    return Material(type=MAT_NULL)


# ---------------------------------------------------------------------------------------------------------------
class Scene:
    """Host-side scene description = what `load_scene_from_json` returns: (Scene, Camera, RenderSettings)."""

    def __init__(self, handle=None):
        self._h = handle if handle is not None else host().pth_scene_new()
        if not self._h:
            raise RuntimeError(host().pth_last_error().decode())

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                host().pth_scene_free(self._h)
                self._h = None
        except Exception:
            pass

    # ---- read side
    @property
    def materials(self):
        n = host().pth_scene_material_count(self._h)
        p = host().pth_scene_materials(self._h)
        out = []
        for i in range(n):
            m = Material()
            C.memmove(C.byref(m), C.byref(p[i]), C.sizeof(Material))
            out.append(m)
        return out

    @property
    def objects(self):
        n = host().pth_scene_object_count(self._h)
        p = host().pth_scene_objects(self._h)
        out = []
        for i in range(n):
            o = HostObject()
            C.memmove(C.byref(o), C.byref(p[i]), C.sizeof(HostObject))
            out.append(o)
        return out

    def mesh(self, index):
        ptr = _F()
        n = host().pth_scene_mesh(self._h, index, C.byref(ptr))
        if n < 0:
            raise IndexError(index)
        return np.ctypeslib.as_array(ptr, shape=(n, 12)).copy()

    @property
    def sky(self):
        ptr, w, h = _F(), C.c_int32(), C.c_int32()
        if not host().pth_scene_sky(self._h, C.byref(ptr), C.byref(w), C.byref(h)):
            return None
        return np.ctypeslib.as_array(ptr, shape=(h.value, w.value, 3)).copy()

    @property
    def camera(self):
        c = Camera()
        host().pth_scene_camera(self._h, C.byref(c))
        return c

    @property
    def settings(self):
        v = [C.c_int32() for _ in range(4)]
        host().pth_scene_settings(self._h, *[C.byref(x) for x in v])
        return tuple(x.value for x in v)  # width, height, spp, max_depth

    # ---- write side (same derivations as the loader)
    def _ck(self, rc):
        if rc < 0:
            raise RuntimeError(host().pth_last_error().decode())
        return rc

    def add_material(self, m):
        return self._ck(host().pth_scene_push_material(self._h, C.byref(m)))

    def add_sphere(self, center, radius, material):
        return self._ck(host().pth_scene_push_sphere(self._h, _fptr(_f32(center)), radius, material))

    def add_plane(self, point, normal, material):
        return self._ck(host().pth_scene_push_plane(self._h, _fptr(_f32(point)), _fptr(_f32(normal)), material))

    def add_quad(self, material, scale=(1, 1, 1), rotation=(0, 0, 0), position=(0, 0, 0)):
        return self._ck(host().pth_scene_push_quad(self._h, _fptr(_f32(scale)), _fptr(_f32(rotation)), _fptr(_f32(position)), material))

    def add_cube(self, material, scale=(1, 1, 1), rotation=(0, 0, 0), position=(0, 0, 0)):
        return self._ck(host().pth_scene_push_cube(self._h, _fptr(_f32(scale)), _fptr(_f32(rotation)), _fptr(_f32(position)), material))

    def add_mesh(self, verts, indices, material, scale=(1, 1, 1), rotation=(0, 0, 0), position=(0, 0, 0)):
        v = _f32(verts, (-1, 3))
        idx = np.ascontiguousarray(indices, dtype=np.int32).reshape(-1, 3)
        return self._ck(host().pth_scene_push_mesh(self._h, _fptr(v), len(v), idx.ctypes.data, len(idx), _fptr(_f32(scale)),
                                                   _fptr(_f32(rotation)), _fptr(_f32(position)), material))

    def add_obj(self, path, material, scale=(1, 1, 1), rotation=(0, 0, 0), position=(0, 0, 0)):
        return self._ck(host().pth_scene_push_obj(self._h, os.fsencode(path), _fptr(_f32(scale)), _fptr(_f32(rotation)),
                                                  _fptr(_f32(position)), material))

    def set_sky(self, rgb):
        a = _f32(rgb)
        h, w = a.shape[0], a.shape[1]
        self._ck(host().pth_scene_set_sky_rgb(self._h, _fptr(a), w, h))

    def set_sky_hdr_file(self, path):
        self._ck(host().pth_scene_set_sky_hdr_file(self._h, os.fsencode(path)))

    def set_camera(self, position, look_at, up, vfov_deg, aspect):
        host().pth_scene_set_camera(self._h, _fptr(_f32(position)), _fptr(_f32(look_at)), _fptr(_f32(up)), vfov_deg, aspect)

    def set_settings(self, width, height, spp, max_depth):
        host().pth_scene_set_settings(self._h, width, height, spp, max_depth)

    def render_settings(self, **over):
        w, h, spp, md = self.settings
        st = RenderSettings(width=w, height=h, spp=spp, max_depth=md)
        for k, v in over.items():
            setattr(st, k, v)
        return st

    def to_core(self):
        """Walk object_list and feed it to the CUDA core through the C ABI (what the Rust `describe()` walk does)."""
        h = host().pth_build_ptc_scene(self._h)
        if not h:
            raise RuntimeError(host().pth_last_error().decode())
        return CoreScene(h)


def load_scene_from_json(path, flags=0):
    """src/tungsten/parser.rs:245 — returns the host Scene (camera and render settings ride along).  `flags` = LOAD_*
    extensions of include/pthost.h (0 = the reference's behaviour, including its failures)."""
    h = host().pth_load_scene_from_json_ex(os.fsencode(path), int(flags))
    if not h:
        raise RuntimeError(host().pth_last_error().decode())
    return Scene(h)


def synthetic_scene(cells=1000, seed=0x5EED):
    """BASELINE config C5: cells x cells x 2 triangle height field + glass sphere + GGX-Al cube + emissive quad."""
    return Scene(host().pth_scene_synthetic(cells, seed))


def transform(scale, rotation_deg, position):
    o2w, w2o = np.zeros(16, np.float32), np.zeros(16, np.float32)
    host().pth_transform(_fptr(_f32(scale)), _fptr(_f32(rotation_deg)), _fptr(_f32(position)), _fptr(o2w), _fptr(w2o))
    return o2w, w2o


def camera_new(position, look_at, up, vfov_deg, aspect):
    c = Camera()
    host().pth_camera_new(_fptr(_f32(position)), _fptr(_f32(look_at)), _fptr(_f32(up)), vfov_deg, aspect, C.byref(c))
    return c


def save_image(path, buffer_u32, width, height):
    """src/renderer.rs:125-179 minus the timestamped name."""
    b = np.ascontiguousarray(buffer_u32, dtype=np.uint32)
    if host().pth_save_png(os.fsencode(path), b.ctypes.data, width, height) != 0:
        raise RuntimeError(host().pth_last_error().decode())


SHARD_SAMPLES, SHARD_TILES = 0, 1


class MultiScene:
    """A ptc_multi handle: one process, one host thread per GPU, one NCCL reduce of the film (include/ptcore.h)."""

    def __init__(self, primary, devices):
        self._primary = primary  # keeps the ptc_scene alive
        devs = (C.c_int * len(devices))(*devices)
        h = _vp()
        _ck(core().ptc_multi_create(primary._h, devs, len(devices), C.byref(h)))
        self._h = h
        self.devices = list(devices)

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                core().ptc_multi_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def render(self, camera, settings, shard=SHARD_SAMPLES):
        out = np.empty((settings.height, settings.width, 3), np.float32)
        st = Stats()
        _ck(core().ptc_multi_render(self._h, C.byref(camera), C.byref(settings), shard, _fptr(out), C.byref(st)))
        return out, st

    def render_u32(self, camera, settings, shard=SHARD_SAMPLES):
        out = np.empty(settings.height * settings.width, np.uint32)
        st = Stats()
        _ck(core().ptc_multi_render_u32(self._h, C.byref(camera), C.byref(settings), shard, out.ctypes.data, C.byref(st)))
        return out, st


# ---------------------------------------------------------------------------------------------------------------
class CoreScene:
    """A ptc_scene handle: the flattened scene on one B200."""

    def __init__(self, handle):
        self._h = handle
        self.device = None

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                core().ptc_scene_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def build(self):
        _ck(core().ptc_scene_build(self._h))
        return self

    def commit(self, device=0, fast_build=False, device_sah=False):
        """fast_build: PTC_COMMIT_FAST_BUILD — flatten the meshes entirely on the device (quick commit, slower traversal).
        device_sah: PTC_COMMIT_DEVICE_SAH — flatten them on the device into the default's SAH tree (quick commit, same tree)."""
        flags = (COMMIT_FAST_BUILD if fast_build else 0) | (COMMIT_DEVICE_SAH if device_sah else 0)
        _ck(core().ptc_scene_commit_ex(self._h, device, flags))
        self.device = device
        return self

    def last_pool_slots(self):
        return int(core().ptc_scene_last_pool_slots(self._h))

    def mesh_info(self, obj):
        info = MeshInfo()
        _ck(core().ptc_scene_mesh_info(self._h, obj, C.byref(info), None, None))
        dead = np.zeros(info.triangles, np.uint8)
        order = np.zeros(info.triangles, np.int32)
        _ck(core().ptc_scene_mesh_info(self._h, obj, C.byref(info), dead.ctypes.data, order.ctypes.data))
        return info, dead, order

    def render(self, camera, settings):
        """-> (W*H*3 float32 linear mean radiance = `image_data` of renderer.rs:83, Stats)."""
        out = np.empty((settings.height, settings.width, 3), np.float32)
        st = Stats()
        _ck(core().ptc_render(self._h, C.byref(camera), C.byref(settings), _fptr(out), C.byref(st)))
        return out, st

    def render_u32(self, camera, settings):
        """-> (H*W uint32 0x00RRGGBB = the Vec<u32> of renderer.rs:67-123, Stats); resolved on the device."""
        out = np.empty(settings.height * settings.width, np.uint32)
        st = Stats()
        _ck(core().ptc_render_u32(self._h, C.byref(camera), C.byref(settings), out.ctypes.data, C.byref(st)))
        return out, st

    def render_adaptive(self, camera, settings, min_spp, threshold):
        """Adaptive sampling (ptc_render_adaptive): every pixel gets min_spp samples, then more, doubling, up to
        settings.spp while the noise estimate of its 3x3 neighbourhood is >= threshold.  -> (rgb [H,W,3] float32 linear
        mean radiance, u32 [H*W] 0x00RRGGBB, spp [H,W] int32 samples per pixel, Stats); each pixel is the uniform render
        at its own count."""
        rgb = np.empty((settings.height, settings.width, 3), np.float32)
        u32 = np.empty(settings.height * settings.width, np.uint32)
        spp = np.empty((settings.height, settings.width), np.int32)
        st = Stats()
        ad = Adaptive(min_spp, threshold)
        _ck(core().ptc_render_adaptive(self._h, C.byref(camera), C.byref(settings), C.byref(ad), _fptr(rgb), u32.ctypes.data,
                                       spp.ctypes.data, C.byref(st)))
        return rgb, u32, spp, st

    def multi(self, devices):
        """In-process multi-GPU (ptc_multi_*): this committed scene replicated on `devices` (devices[0] = its own)."""
        return MultiScene(self, devices)

    def render_accumulate(self, camera, settings, d_accum_ptr, stream_ptr=None):
        st = Stats()
        _ck(core().ptc_render_accumulate(self._h, C.byref(camera), C.byref(settings), d_accum_ptr, stream_ptr, C.byref(st)))
        return st

    def resolve_u32(self, rgb, scale=1.0):
        a = _f32(rgb).reshape(-1, 3)
        out = np.empty(len(a), np.uint32)
        _ck(core().ptc_resolve_u32(self._h, _fptr(a), len(a), scale, out.ctypes.data))
        return out

    def intersect(self, origins, dirs, t_min=1e-4, t_max=float("inf")):
        o, d = _f32(origins, (-1, 3)), _f32(dirs, (-1, 3))
        out = np.zeros(len(o), HIT_DTYPE)
        st = Stats()
        _ck(core().ptc_intersect(self._h, _fptr(o), _fptr(d), len(o), t_min, t_max, out.ctypes.data, C.byref(st)))
        return out, st

    def primary_rays(self, camera, settings, sample):
        n = settings.width * settings.height
        o, d = np.empty((n, 3), np.float32), np.empty((n, 3), np.float32)
        _ck(core().ptc_primary_rays(self._h, C.byref(camera), C.byref(settings), sample, _fptr(o), _fptr(d)))
        return o, d

    def scatter(self, material, ray_dirs, positions, normals, front_face, u4):
        d, p, nn, u = _f32(ray_dirs, (-1, 3)), _f32(positions, (-1, 3)), _f32(normals, (-1, 3)), _f32(u4, (-1, 4))
        ff = np.ascontiguousarray(front_face, dtype=np.int32)
        n = len(d)
        sc = np.zeros(n, np.int32)
        oo, od, att, em = (np.zeros((n, 3), np.float32) for _ in range(4))
        _ck(core().ptc_scatter(self._h, material, _fptr(d), _fptr(p), _fptr(nn), ff.ctypes.data, _fptr(u), n, sc.ctypes.data,
                               _fptr(oo), _fptr(od), _fptr(att), _fptr(em)))
        return sc, oo, od, att, em

    def sky_sample(self, u4):
        """The HDR sky as a light (FLAG_NEE_SKY): u4 = n x 4 uniforms in [0, 1) -> (directions n x 3, solid-angle pdf n,
        sky radiance along them n x 3), by the shade stage's own device functions."""
        u = _f32(u4, (-1, 4))
        n = len(u)
        d, pdf, rgb = np.empty((n, 3), np.float32), np.empty(n, np.float32), np.empty((n, 3), np.float32)
        _ck(core().ptc_sky_sample(self._h, _fptr(u), n, _fptr(d), _fptr(pdf), _fptr(rgb)))
        return d, pdf, rgb

    def sky_pdf(self, dirs):
        """Solid-angle pdf with which FLAG_NEE_SKY samples each direction of dirs (n x 3)."""
        d = _f32(dirs, (-1, 3))
        pdf = np.empty(len(d), np.float32)
        _ck(core().ptc_sky_pdf(self._h, _fptr(d), len(d), _fptr(pdf)))
        return pdf

    def philox(self, ctr, key):
        c = np.asarray(ctr, np.uint32)
        k = np.asarray(key, np.uint32)
        out = np.zeros(4, np.uint32)
        _ck(core().ptc_philox(self._h, c.ctypes.data, k.ctypes.data, out.ctypes.data))
        return out


def render_scene(scene, device=0, **over):
    """src/renderer.rs:67 — `render_scene(&scene, &camera, &render_settings) -> Vec<u32>` on one B200.

    Returns (buffer_u32 [H*W] 0x00RRGGBB row-major top row first, linear image [H,W,3], Stats)."""
    cs = scene.to_core().commit(device)
    st = scene.render_settings(**over)
    img, stats = cs.render(scene.camera, st)
    return cs.resolve_u32(img), img, stats
