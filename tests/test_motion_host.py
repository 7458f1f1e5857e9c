"""Motion blur (ptc_scene_set_object_motion / ptc_scene_set_camera_motion) without a device.

  * the host build of camera_at against a float64 restatement of the model in ptcore.h, and the bitwise rule for an end
    camera equal to its start camera;
  * the host build of the per-object shifted scan (hostsim: sim_intersect_motion) against ptc_intersect's host build on
    the shifted ray, and against a float64 restatement of a moving sphere;
  * the setters' argument checks, that a refused call leaves the previous state, and the motion rules of the render calls
    on an uncommitted scene;
  * the Python wrapper and the Rust declarations.
"""
import ctypes as C
import math
import os
import re

import numpy as np
import pytest

from bindings import sim_lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_F = C.POINTER(C.c_float)


def _cam_fields(c):
    return np.array(list(c.position) + list(c.forward) + list(c.right) + list(c.true_up) + [c.half_width, c.half_height],
                    np.float64)


def _camera_at(pt, c0, c1, tau):
    L = sim_lib()
    L.sim_camera_at.argtypes = [C.c_void_p, C.c_void_p, C.c_float, C.c_void_p]
    out = pt.Camera()
    assert L.sim_camera_at(C.addressof(c0), C.addressof(c1), tau, C.addressof(out)) == 0
    return out


def test_camera_at_is_the_componentwise_lerp(pt):
    c0 = pt.camera_new((0.3, 1.2, 4.0), (0.0, 0.5, 0.0), (0, 1, 0), 40.0, 1.5)
    c1 = pt.camera_new((2.3, 0.7, 3.0), (0.5, 0.2, -1.0), (0.1, 1, 0), 55.0, 1.5)  # moves, turns and zooms
    a, b = _cam_fields(c0), _cam_fields(c1)
    for tau in (0.0, 0.25, 0.5, 0.999, np.float32(1.0) - np.float32(2 ** -24)):
        got = _cam_fields(_camera_at(pt, c0, c1, float(tau)))
        want = a + float(tau) * (b - a)
        assert np.all(np.abs(got - want) <= 4e-7 * np.maximum(np.abs(a), np.abs(b)) + 1e-30), (tau, got - want)
    # float32 statement of c0 + tau (c1 - c0): bit for bit
    a32, b32 = a.astype(np.float32), b.astype(np.float32)
    tau = np.float32(0.37)
    want32 = a32 + tau * (b32 - a32)
    assert _cam_fields(_camera_at(pt, c0, c1, float(tau))).astype(np.float32).tobytes() == want32.tobytes()


def test_equal_end_camera_is_the_start_camera_bit_for_bit(pt):
    c0 = pt.camera_new((0.3, 1.2, 4.0), (0.0, 0.5, 0.0), (0, 1, 0), 40.0, 1.5)
    c0.right[2] = -0.0  # c0 + tau * 0 would turn a -0 into +0: the rule returns c0 itself
    c1 = pt.Camera.from_buffer_copy(c0)
    for tau in (0.0, 0.3, 0.999):
        assert bytes(_camera_at(pt, c0, c1, tau)) == bytes(c0)
    c1.half_width = np.nextafter(np.float32(c0.half_width), np.float32(2))  # one ulp off: the lerp
    assert bytes(_camera_at(pt, c0, c1, 0.5)) != bytes(c0)


def _sim_scene(pt, build):
    L = sim_lib()
    s = L.sim_scene_create()
    build(L, s)
    assert L.sim_scene_commit(s, 0) == 0
    return L, s


def _mixed(L, s, pt):
    """a sphere, a quad, a cube, a plane and a two-triangle mesh, listed in that order"""
    m = L.sim_scene_add_material(s, C.byref(pt.lambertian((0.5, 0.5, 0.5))))
    f3 = lambda *v: (C.c_float * len(v))(*v)
    L.sim_scene_add_sphere(s, f3(0.0, 0.0, -3.0), C.c_float(0.8), m)
    L.sim_scene_add_quad(s, f3(-1.0, -1.0, -5.0), f3(2.0, 0.0, 0.0), f3(0.0, 2.0, 0.0), f3(0.0, 0.0, 1.0), C.c_float(-5.0),
                         C.c_float(0.25), C.c_float(0.25), m)
    o2w = np.array([[0.6, 0, 0, 1.2], [0, 0.6, 0, 0.1], [0, 0, 0.6, -2.5], [0, 0, 0, 1]], np.float32)
    w2o = np.linalg.inv(o2w.astype(np.float64)).astype(np.float32)
    L.sim_scene_add_cube(s, o2w.ctypes.data_as(_F), w2o.ctypes.data_as(_F), m)
    L.sim_scene_add_plane(s, f3(0.0, -1.5, 0.0), f3(0.0, 1.0, 0.0), m)
    tris = np.array([[-1.5, -0.5, -4.0], [-0.5, -0.5, -4.0], [-1.0, 0.6, -4.2],
                     [-1.5, -0.5, -4.0], [-1.0, 0.6, -4.2], [-1.8, 0.4, -3.6]], np.float32)
    eye = np.eye(4, dtype=np.float32)
    L.sim_scene_add_mesh(s, tris.ctypes.data_as(_F), 2, eye.ctypes.data_as(_F), eye.ctypes.data_as(_F), m)
    return 5


def _rays(n, seed):
    rng = np.random.default_rng(seed)
    o = np.zeros((n, 3), np.float32) + rng.normal(0, 0.2, (n, 3)).astype(np.float32)
    d = np.stack([rng.uniform(-0.7, 0.7, n), rng.uniform(-0.6, 0.4, n), -np.ones(n)], 1).astype(np.float32)
    t = rng.random(n).astype(np.float32)
    t[:3] = (0.0, 1.0, 0.5)
    return o, d, t


def _sim_intersect_motion(pt, L, s, disp, o, d, t):
    L.sim_intersect_motion.argtypes = [C.c_void_p, _F, _F, _F, _F, C.c_int64, C.c_float, C.c_float, C.c_void_p]
    out = np.zeros(len(o), pt.HIT_DTYPE)
    dd = np.ascontiguousarray(disp, np.float32)
    assert L.sim_intersect_motion(s, dd.ctypes.data_as(_F), o.ctypes.data_as(_F), d.ctypes.data_as(_F), t.ctypes.data_as(_F),
                                  len(o), 1e-4, np.inf, out.ctypes.data) == 0
    return out


def _sim_intersect(pt, L, s, o, d):
    out = np.zeros(len(o), pt.HIT_DTYPE)
    st = pt.Stats()
    assert L.sim_intersect(s, o.ctypes.data_as(_F), d.ctypes.data_as(_F), len(o), C.c_float(1e-4), C.c_float(np.inf),
                           out.ctypes.data, C.byref(st)) == 0
    return out


def test_zero_displacement_is_the_static_scan(pt):
    L, s = _sim_scene(pt, lambda L, s: _mixed(L, s, pt))
    o, d, t = _rays(4000, 1)
    got = _sim_intersect_motion(pt, L, s, np.zeros((5, 3)), o, d, t)
    want = _sim_intersect(pt, L, s, o, d)
    assert (want["object"] >= 0).sum() > 1000
    assert got.tobytes() == want.tobytes()
    # -0 components are "static" too
    got = _sim_intersect_motion(pt, L, s, np.full((5, 3), -0.0), o, d, t)
    assert got.tobytes() == want.tobytes()
    L.sim_scene_destroy(s)


def test_common_displacement_is_the_static_scan_of_the_shifted_ray(pt):
    """Every object moved by the same D: the record is the static scan of (o - tau D, d) (float32 arithmetic, bit for
    bit) with its position + tau D."""
    L, s = _sim_scene(pt, lambda L, s: _mixed(L, s, pt))
    o, d, t = _rays(4000, 2)
    D = np.array([0.31, -0.12, 0.45], np.float32)
    got = _sim_intersect_motion(pt, L, s, np.tile(D, (5, 1)), o, d, t)
    ts = t[:, None]
    want = _sim_intersect(pt, L, s, (o - ts * D).astype(np.float32), d)
    hit = want["object"] >= 0
    want["position"][hit] = (want["position"][hit] + ts[hit] * D).astype(np.float32)
    assert hit.sum() > 1000 and set(np.unique(want["object"][hit])) == {0, 1, 2, 3, 4}
    assert got.tobytes() == want.tobytes()
    L.sim_scene_destroy(s)


def test_distinct_displacements_combine_single_object_results_in_list_order(pt):
    L, s = _sim_scene(pt, lambda L, s: _mixed(L, s, pt))
    o, d, t = _rays(3000, 3)
    disp = np.array([[0.4, 0, 0], [0, 0.3, 0], [0, 0, 0], [-0.2, 0.1, 0.3], [0.5, -0.5, 0.1]], np.float32)
    got = _sim_intersect_motion(pt, L, s, disp, o, d, t)
    # the same scan object by object: object k alone is the scan with every other object moved a million units away
    # (rays at tau < 1e-3, where "away" is still near, are left out)
    singles = []
    for k in range(5):
        far = np.tile(np.float32([0, 1e6, 0]), (5, 1))
        far[k] = disp[k]
        singles.append(_sim_intersect_motion(pt, L, s, far, o, d, t))
    for i in np.nonzero(t >= 1e-3)[0]:
        best = None
        for k in range(5):
            h = singles[k][i]
            if h["object"] == k and (best is None or h["t"] < best["t"]):
                best = h
        if best is None:
            assert got[i]["object"] == -1
        else:
            assert got[i].tobytes() == best.tobytes(), i
    L.sim_scene_destroy(s)


def test_moving_sphere_against_float64(pt):
    """A sphere translated by tau D is hit where the float64 ray-sphere intersection with centre c + tau D says."""
    c, r = np.array([0.0, 0.0, -3.0]), 0.8
    L, s = _sim_scene(pt, lambda L, s: L.sim_scene_add_sphere(
        s, (C.c_float * 3)(*c), C.c_float(r), L.sim_scene_add_material(s, C.byref(pt.lambertian((0.5, 0.5, 0.5))))))
    o, d, t = _rays(3000, 4)
    D = np.array([0.9, -0.4, 0.2], np.float32)
    got = _sim_intersect_motion(pt, L, s, D[None, :], o, d, t)
    o64, d64 = o.astype(np.float64), d.astype(np.float64)
    cc = c + t.astype(np.float64)[:, None] * D
    oc = o64 - cc
    a = (d64 * d64).sum(1)
    hb = (oc * d64).sum(1)
    disc = hb * hb - a * ((oc * oc).sum(1) - r * r)
    hit = disc > 1e-6 * a
    tt = (-hb - np.sqrt(np.where(hit, disc, 0))) / a
    solid = hit & (disc > 1e-3)
    assert solid.sum() > 500
    assert (got["object"][solid] == 0).all()
    assert np.allclose(got["t"][solid], tt[solid], rtol=2e-5, atol=2e-5)
    p = o64 + tt[:, None] * d64
    assert np.allclose(got["position"][solid], p[solid], atol=5e-5)
    assert (got["object"][~hit & (disc < -1e-3)] == -1).all()
    L.sim_scene_destroy(s)


def test_primary_rays_at_tau_start_from_the_camera_at_tau(pt):
    L = sim_lib()
    L.sim_primary_rays_motion.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_float, _F, _F, _F]
    c0 = pt.camera_new((0.0, 1.0, 4.0), (0.0, 0.5, 0.0), (0, 1, 0), 40.0, 1.5)
    c1 = pt.camera_new((1.0, 1.0, 4.0), (1.0, 0.5, 0.0), (0, 1, 0), 40.0, 1.5)
    st = pt.RenderSettings(width=21, height=13, spp=1, max_depth=1, seed=77)
    n = 21 * 13
    o, d, tau = np.empty((n, 3), np.float32), np.empty((n, 3), np.float32), np.empty(n, np.float32)
    assert L.sim_primary_rays_motion(C.addressof(c0), C.addressof(c1), C.addressof(st), 2, 0.0, 1.0, o.ctypes.data_as(_F),
                                     d.ctypes.data_as(_F), tau.ctypes.data_as(_F)) == 0
    assert (tau >= 0).all() and (tau < 1).all() and tau.std() > 0.2
    # a pure translation: origins on the segment, directions those of the static camera
    assert np.allclose(o[:, 0], tau, atol=1e-6) and np.allclose(o[:, 1:], [1.0, 4.0])
    po, pd = np.empty((n, 3), np.float32), np.empty((n, 3), np.float32)
    L.sim_primary_rays(None, C.addressof(c0), C.addressof(st), 2, po.ctypes.data_as(_F), pd.ctypes.data_as(_F))
    assert np.allclose(d, pd, atol=1e-6)
    # tau is u[0] of Philox block 1 of the jitter counter
    ctr = (C.c_uint32 * 4)(5, 2, 0xFFFFFFFF, 1)
    key = (C.c_uint32 * 2)(77, 0)
    out = (C.c_uint32 * 4)()
    L.sim_philox(None, ctr, key, out)
    assert tau[5] == np.float32((out[0] >> 8) / 16777216.0)


# ---- the C ABI --------------------------------------------------------------------------------------------------
def _scene(pt):
    s = pt.Scene()
    m = s.add_material(pt.lambertian((0.5, 0.5, 0.5)))
    s.add_sphere((0, 0, -1), 0.5, m)
    s.add_sphere((1, 0, -1), 0.5, m)
    s.set_camera((0, 0, 0), (0, 0, -1), (0, 1, 0), 60.0, 1.0)
    s.set_settings(8, 6, 16, 4)
    return s


def _obj(pt, cs, k, d):
    return pt.core().ptc_scene_set_object_motion(cs._h, k, (C.c_float * 3)(*d))


def _cams(pt, cams):
    arr = (pt.Camera * max(len(cams), 1))(*cams)
    return arr


def _set_cams(pt, cs, cams):
    return pt.core().ptc_scene_set_camera_motion(cs._h, _cams(pt, cams) if cams else None, len(cams))


def _render(pt, cs, s):
    out = np.empty((6, 8, 3), np.float32)
    return pt.core().ptc_render(cs._h, C.byref(s.camera), C.byref(s.render_settings()), out.ctypes.data_as(_F), None)


def _batch(pt, cs, s, n_views):
    arr = (pt.Camera * n_views)(*[s.camera] * n_views)
    out = np.empty(n_views * 48, np.uint32)
    return pt.core().ptc_render_batch(cs._h, arr, n_views, None, C.byref(s.render_settings()), None, out.ctypes.data, None)


@pytest.mark.parametrize("k, d", [(-1, (0.1, 0, 0)), (2, (0.1, 0, 0)), (0, (math.nan, 0, 0)), (1, (0, math.inf, 0)),
                                  (0, (0, 0, -math.inf))])
def test_bad_object_motion_is_refused(pt, k, d):
    s = _scene(pt)
    cs = s.to_core()
    assert _obj(pt, cs, 0, (0.5, 0.0, 0.0)) == 0
    assert _obj(pt, cs, k, d) == pt.PTC_E_INVALID
    assert pt.core().ptc_scene_set_object_motion(cs._h, 0, None) == pt.PTC_E_INVALID
    assert pt.core().ptc_scene_set_object_motion(None, 0, (C.c_float * 3)(0, 0, 0)) == pt.PTC_E_INVALID
    assert _obj(pt, cs, 1, (0.0, 0.0, 0.0)) == 0 and _obj(pt, cs, 1, (-0.0, 1e-30, 0.0)) == 0


def test_bad_end_cameras_are_refused_and_change_nothing(pt):
    s = _scene(pt)
    cs = s.to_core()
    cam = s.camera
    assert _set_cams(pt, cs, [cam, cam]) == 0
    for field, bad in (("half_width", math.nan), ("half_height", math.inf), ("position", math.nan), ("true_up", -math.inf)):
        c = pt.Camera.from_buffer_copy(cam)
        if field in ("half_width", "half_height"):
            setattr(c, field, bad)
        else:
            getattr(c, field)[1] = bad
        assert _set_cams(pt, cs, [cam, c]) == pt.PTC_E_INVALID, field
        # the previous two end cameras still apply: a single-camera call refuses them, a batch of two takes them
        assert _render(pt, cs, s) == pt.PTC_E_INVALID
        assert _batch(pt, cs, s, 2) == pt.PTC_E_STATE
        assert _batch(pt, cs, s, 3) == pt.PTC_E_INVALID
    assert pt.core().ptc_scene_set_camera_motion(cs._h, _cams(pt, [cam]), -1) == pt.PTC_E_INVALID
    assert pt.core().ptc_scene_set_camera_motion(cs._h, None, 1) == pt.PTC_E_INVALID
    assert pt.core().ptc_scene_set_camera_motion(None, None, 0) == pt.PTC_E_INVALID
    assert _render(pt, cs, s) == pt.PTC_E_INVALID  # still two end cameras
    assert _set_cams(pt, cs, []) == 0  # reset: a static camera, NULL allowed
    assert _render(pt, cs, s) == pt.PTC_E_STATE


def test_motion_rules_of_every_call_on_an_uncommitted_scene(pt):
    s = _scene(pt)
    cs = s.to_core()
    core, st, cam = pt.core(), s.render_settings(), s.camera
    f3 = np.empty(48 * 3, np.float32)
    u32 = np.empty(48, np.uint32)
    fp, up = f3.ctypes.data_as(_F), u32.ctypes.data

    def single_calls():
        return {
            "render": _render(pt, cs, s),
            "u32": core.ptc_render_u32(cs._h, C.byref(cam), C.byref(st), up, None),
            "accumulate": core.ptc_render_accumulate(cs._h, C.byref(cam), C.byref(st), C.c_void_p(16), None, None),
            "adaptive": core.ptc_render_adaptive(cs._h, C.byref(cam), C.byref(st), C.byref(pt.Adaptive(2, 0.01)), fp, up, None, None),
            "progressive": core.ptc_render_progressive(cs._h, C.byref(cam), C.byref(st), C.byref(pt.ProgressiveSettings(1, 0)),
                                                       pt.PREVIEW_FN(), None, fp, up, None, None),
            "denoised": core.ptc_render_denoised(cs._h, C.byref(cam), C.byref(st), C.byref(pt.Denoise(1, 3, 4.0, 0.1, 0.1)),
                                                 fp, up, None, None, None, None, None),
            "primary_rays": core.ptc_primary_rays(cs._h, C.byref(cam), C.byref(st), 0, fp, fp),
        }

    moved = pt.Camera.from_buffer_copy(cam)
    moved.position[0] += 0.5
    assert _obj(pt, cs, 1, (0.2, 0.0, 0.0)) == 0
    for ends in ([], [cam], [moved]):
        assert _set_cams(pt, cs, ends) == 0
        assert set(single_calls().values()) == {pt.PTC_E_STATE}, len(ends)
        assert _batch(pt, cs, s, 1) == pt.PTC_E_STATE and _batch(pt, cs, s, 4) == pt.PTC_E_STATE
    assert _set_cams(pt, cs, [moved, cam, moved]) == 0
    got = single_calls()
    assert set(got.values()) == {pt.PTC_E_INVALID}, got
    assert _batch(pt, cs, s, 3) == pt.PTC_E_STATE
    assert _batch(pt, cs, s, 2) == pt.PTC_E_INVALID and _batch(pt, cs, s, 4) == pt.PTC_E_INVALID
    arr = (pt.Camera * 2)(cam, cam)
    assert core.ptc_render_batch_accumulate(cs._h, arr, 2, None, C.byref(st), C.c_void_p(16), None, None) == pt.PTC_E_INVALID
    # the parity hooks need a committed scene
    o = np.zeros((1, 3), np.float32)
    t = np.zeros(1, np.float32)
    hits = np.zeros(1, pt.HIT_DTYPE)
    assert core.ptc_intersect_at(cs._h, o.ctypes.data_as(_F), o.ctypes.data_as(_F), t.ctypes.data_as(_F), 1, 1e-4, np.inf,
                                 hits.ctypes.data, None) == pt.PTC_E_STATE
    assert core.ptc_ray_times(cs._h, C.byref(st), 0, fp) == pt.PTC_E_STATE


def test_motion_set_after_commit_is_accepted_without_a_device(pt):
    """The setters are handle state: they need no device, before or after commit (commit itself needs one, so here the
    scene is only built; the setters do not look at the device state at all)."""
    s = _scene(pt)
    cs = s.to_core()
    assert pt.core().ptc_scene_build(cs._h) == 0
    assert _obj(pt, cs, 0, (0.1, 0.2, 0.3)) == 0
    assert _set_cams(pt, cs, [s.camera]) == 0
    assert _obj(pt, cs, 0, (0.0, 0.0, 0.0)) == 0 and _set_cams(pt, cs, []) == 0


def test_python_wrappers(pt):
    s = _scene(pt)
    cs = s.to_core()
    assert cs.set_object_motion(1, (0.1, 0.0, 0.0)) is cs
    with pytest.raises(pt.PtcError):
        cs.set_object_motion(5, (0.1, 0.0, 0.0))
    with pytest.raises(pt.PtcError):
        cs.set_object_motion(0, (float("nan"), 0.0, 0.0))
    assert cs.set_camera_motion(s.camera) is cs
    cs.set_camera_motion([s.camera, s.camera])
    assert _render(pt, cs, s) == pt.PTC_E_INVALID
    cs.set_camera_motion()
    assert _render(pt, cs, s) == pt.PTC_E_STATE


def test_header_and_rust_declarations(pt):
    hdr = open(os.path.join(ROOT, "include", "ptcore.h")).read()
    for name in ("ptc_scene_set_object_motion", "ptc_scene_set_camera_motion", "ptc_intersect_at", "ptc_ray_times"):
        assert re.search(r"\b%s\s*\(" % name, hdr), name
    rs = open(os.path.join(ROOT, "rust", "ptcore-sys", "src", "lib.rs")).read()
    for name in ("ptc_scene_set_object_motion", "ptc_scene_set_camera_motion"):
        assert re.search(r"pub fn %s\(" % name, rs), name
