"""Thin-lens depth of field (ptc_scene_set_lens) without a device.

  * the host build of camera_get_ray_lens (hostsim) against a float64 numpy restatement of the model in ptcore.h;
  * ptc_scene_set_lens's argument checks, and that a refused call leaves the previous lens in force;
  * the lens rules of the render calls on an uncommitted scene: a wrong lens count is PTC_E_INVALID, good arguments
    PTC_E_STATE;
  * the loader's PTH_LOAD_THIN_LENS, and the Python wrapper and Rust declarations.
"""
import ctypes as C
import json
import math
import os
import re

import numpy as np
import pytest

from bindings import sim_lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_F = C.POINTER(C.c_float)


# ---- float64 restatement of the model ------------------------------------------------------------------------
def _philox(ctr, k0, k1):
    """Philox4x32-10 on arrays of counters (uint64 holding uint32 values), as pt_philox.h."""
    c = [np.asarray(x, np.uint64) & 0xFFFFFFFF for x in ctr]
    k0, k1 = np.uint64(k0), np.uint64(k1)
    m = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & m
        hi1, lo1 = p1 >> np.uint64(32), p1 & m
        c = [(hi1 ^ c[1] ^ k0) & m, lo1, (hi0 ^ c[3] ^ k1) & m, lo0]
        k0 = (k0 + np.uint64(0x9E3779B9)) & m
        k1 = (k1 + np.uint64(0xBB67AE85)) & m
    return c


def _uniforms(seed, pixel, sample):
    r = _philox([pixel, np.full_like(pixel, sample), np.full_like(pixel, 0xFFFFFFFF), np.zeros_like(pixel)],
                seed & 0xFFFFFFFF, seed >> 32)
    return [(x >> np.uint64(8)).astype(np.float64) / 16777216.0 for x in r]


def _unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def model_rays(cam, w, h, seed, sample, R, F):
    """(origins, directions, degenerate mask) of every pixel, float64, as include/ptcore.h states the model."""
    pixel = np.arange(w * h, dtype=np.uint64)
    x, y = (pixel % np.uint64(w)).astype(np.float64), (pixel // np.uint64(w)).astype(np.float64)
    u0, u1, u2, u3 = _uniforms(seed, pixel, sample)
    u, v = (x + u0) / w, (y + u1) / h
    pos, fwd = np.array(cam.position, np.float64), np.array(cam.forward, np.float64)
    rgt, up = np.array(cam.right, np.float64), np.array(cam.true_up, np.float64)
    off = rgt * ((2 * u - 1) * cam.half_width)[:, None] + up * ((1 - 2 * v) * cam.half_height)[:, None]
    d = _unit(fwd + off)
    o = np.broadcast_to(pos, d.shape).copy()
    if R == 0:
        return o, d, np.zeros(len(d), bool)
    a, b = 2 * u2 - 1, 2 * u3 - 1
    with np.errstate(divide="ignore", invalid="ignore"):
        first = np.abs(a) > np.abs(b)
        r = np.where(first, a, b)
        phi = np.where(first, (math.pi / 4) * (b / a), math.pi / 2 - (math.pi / 4) * (a / b))
        zero = (a == 0) & (b == 0)
        r, phi = np.where(zero, 0.0, r), np.where(zero, 0.0, phi)
        dx, dy = r * np.cos(phi), r * np.sin(phi)
        fh, rh, uh = fwd / np.linalg.norm(fwd), rgt / np.linalg.norm(rgt), up / np.linalg.norm(up)
        cd = d @ fh
        o2 = o + R * (dx[:, None] * rh + dy[:, None] * uh)
        P = o + d * (F / cd)[:, None]
        d2 = _unit(P - o2)
        bad = ~(cd > 0) | ~np.isfinite(o2).all(axis=1) | ~np.isfinite(d2).all(axis=1)
    o2[bad], d2[bad] = o[bad], d[bad]
    return o2, d2, bad


def _sim_rays(pt, cam, w, h, seed, sample, R, F):
    L = sim_lib()
    L.sim_primary_rays_lens.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_float, _F, _F]
    st = pt.RenderSettings(width=w, height=h, spp=1, max_depth=1, seed=seed)
    o, d = np.empty((w * h, 3), np.float32), np.empty((w * h, 3), np.float32)
    assert L.sim_primary_rays_lens(None, C.addressof(cam), C.addressof(st), sample, R, F, o.ctypes.data_as(_F),
                                   d.ctypes.data_as(_F)) == 0
    return o, d


def _within(got, want, rel=2e-6):
    """componentwise within rel x the largest component of each vector"""
    tol = rel * np.abs(want).max(axis=1, keepdims=True)
    return np.abs(got.astype(np.float64) - want) <= tol


def _cam(pt, position, forward, right, up, hw, hh):
    c = pt.Camera()
    c.position[:], c.forward[:], c.right[:], c.true_up[:] = position, forward, right, up
    c.half_width, c.half_height = hw, hh
    return c


def _cameras(pt):
    return {
        "look-at": pt.camera_new((0.3, 1.2, 4.0), (0.0, 0.5, 0.0), (0, 1, 0), 40.0, 1.5),
        "far-from-origin": pt.camera_new((120.0, -35.0, 410.0), (118.0, -30.0, 400.0), (0, 1, 0), 65.0, 0.75),
        # Camera::new's forward is not normalised (look_at - position): the model normalises f^, r^ and u^
        "non-unit-forward": _cam(pt, (1.0, 2.0, 3.0), (0.0, 0.0, -3.5), (2.0, 0.0, 0.0), (0.0, 0.5, 0.0), 0.6, 0.4),
        "tilted": pt.camera_new((-2.0, 3.0, -1.0), (1.0, -1.0, 2.5), (0.2, 1, 0.1), 90.0, 1.0),
    }


@pytest.mark.parametrize("name", ["look-at", "far-from-origin", "non-unit-forward", "tilted"])
@pytest.mark.parametrize("R, F", [(0.05, 2.0), (0.7, 13.0), (2.5, 0.4)])
def test_hostsim_lens_rays_match_the_model(pt, name, R, F):
    cam = _cameras(pt)[name]
    for sample in (0, 5):
        o, d = _sim_rays(pt, cam, 37, 23, 0x1234_5678_9ABC, sample, R, F)
        wo, wd, bad = model_rays(cam, 37, 23, 0x1234_5678_9ABC, sample, R, F)
        assert not bad.any()
        assert _within(o, wo).all() and _within(d, wd).all(), (np.abs(o - wo).max(), np.abs(d - wd).max())
        assert not np.array_equal(o, np.broadcast_to(np.float32(cam.position), o.shape))  # the origins moved


def test_zero_aperture_is_the_pinhole_ray_itself(pt):
    L = sim_lib()
    for cam in _cameras(pt).values():
        st = pt.RenderSettings(width=29, height=17, spp=1, max_depth=1, seed=99)
        po, pd = np.empty((29 * 17, 3), np.float32), np.empty((29 * 17, 3), np.float32)
        assert L.sim_primary_rays(None, C.addressof(cam), C.addressof(st), 3, po.ctypes.data_as(_F), pd.ctypes.data_as(_F)) == 0
        o, d = _sim_rays(pt, cam, 29, 17, 99, 3, 0.0, 5.0)
        assert o.tobytes() == po.tobytes() and d.tobytes() == pd.tobytes()
        wo, wd, _ = model_rays(cam, 29, 17, 99, 3, 0.0, 5.0)
        assert _within(d, wd).all()


def test_degenerate_cameras_fall_back_to_the_pinhole_ray(pt):
    L = sim_lib()
    cams = [
        # right = -forward: the pinhole direction turns away from f^ for ndc_x > 1/3
        _cam(pt, (0.0, 0.0, 0.0), (0.0, 0.0, -1.0), (0.0, 0.0, 1.0), (0.0, 1.0, 0.0), 3.0, 1.0),
        # forward = 0: f^ is not finite
        _cam(pt, (1.0, 1.0, 1.0), (0.0, 0.0, 0.0), (1.0, 0.0, 0.0), (0.0, 1.0, 0.0), 1.0, 1.0),
    ]
    for k, cam in enumerate(cams):
        st = pt.RenderSettings(width=16, height=8, spp=1, max_depth=1, seed=5)
        po, pd = np.empty((128, 3), np.float32), np.empty((128, 3), np.float32)
        L.sim_primary_rays(None, C.addressof(cam), C.addressof(st), 0, po.ctypes.data_as(_F), pd.ctypes.data_as(_F))
        o, d = _sim_rays(pt, cam, 16, 8, 5, 0, 0.3, 2.0)
        _, _, bad = model_rays(cam, 16, 8, 5, 0, 0.3, 2.0)
        assert bad.any()
        if k == 1:
            assert bad.all()
        finite = np.isfinite(pd).all(axis=1)
        assert o[bad].tobytes() == po[bad].tobytes()
        assert d[bad & finite].tobytes() == pd[bad & finite].tobytes()
        if k == 0:
            assert (~bad).any() and not np.array_equal(o[~bad], po[~bad])


def test_blur_radius_formula(pt):
    """A point at depth z on the axis projects, through every lens point, onto a circle of radius R |1/z - 1/F| (in
    half_width units) around the image centre: the consequence DESIGN.md 5k documents, restated from the model."""
    cam = _cam(pt, (0.0, 0.0, 0.0), (0.0, 0.0, -1.0), (1.0, 0.0, 0.0), (0.0, 1.0, 0.0), 0.5, 0.5)
    R, F, z = 0.2, 2.0, 5.0
    phi = np.linspace(0, 2 * np.pi, 64, endpoint=False)
    lens = R * np.stack([np.cos(phi), np.sin(phi), np.zeros_like(phi)], 1)
    # the lens ray through lens point q that meets the point (0, 0, -z) starts toward the focus plane point P(q);
    # its pinhole direction d is P / |P|; its image-plane offset is d_xy / (-d_z)
    Pz = (np.array([0.0, 0.0, -z]) - lens) * (F / z) + lens
    img = Pz[:, :2] / F
    assert np.allclose(np.linalg.norm(img, axis=1), R * abs(1 / z - 1 / F))


# ---- the C ABI --------------------------------------------------------------------------------------------------
def _scene(pt):
    s = pt.Scene()
    s.add_sphere((0, 0, -1), 0.5, s.add_material(pt.lambertian((0.5, 0.5, 0.5))))
    s.set_camera((0, 0, 0), (0, 0, -1), (0, 1, 0), 60.0, 1.0)
    s.set_settings(8, 6, 16, 4)
    return s


def _set(pt, cs, pairs):
    arr = (pt.Lens * max(len(pairs), 1))(*[pt.Lens(r, f) for r, f in pairs])
    return pt.core().ptc_scene_set_lens(cs._h, arr, len(pairs))


def _render(pt, cs, s):
    out = np.empty((6, 8, 3), np.float32)
    return pt.core().ptc_render(cs._h, C.byref(s.camera), C.byref(s.render_settings()), out.ctypes.data_as(_F), None)


def _batch(pt, cs, s, n_views):
    arr = (pt.Camera * n_views)(*[s.camera] * n_views)
    out = np.empty(n_views * 48, np.uint32)
    return pt.core().ptc_render_batch(cs._h, arr, n_views, None, C.byref(s.render_settings()), None, out.ctypes.data, None)


@pytest.mark.parametrize("r, f", [(math.nan, 1.0), (math.inf, 1.0), (-0.1, 1.0), (-math.inf, 1.0), (0.1, 0.0), (0.1, -2.0),
                                  (0.1, math.nan), (0.1, math.inf)])
def test_bad_lenses_are_refused_and_change_nothing(pt, r, f):
    s = _scene(pt)
    cs = s.to_core()
    assert _set(pt, cs, [(0.1, 2.0), (0.2, 3.0)]) == 0
    assert _set(pt, cs, [(0.1, 2.0), (r, f)]) == pt.PTC_E_INVALID
    # the previous two lenses still apply: a single-camera call refuses them, a batch of two takes them
    assert _render(pt, cs, s) == pt.PTC_E_INVALID
    assert _batch(pt, cs, s, 2) == pt.PTC_E_STATE
    assert _batch(pt, cs, s, 3) == pt.PTC_E_INVALID


def test_negative_count_and_null_lenses_are_refused(pt):
    s = _scene(pt)
    cs = s.to_core()
    assert _set(pt, cs, [(0.1, 2.0), (0.2, 3.0)]) == 0
    assert pt.core().ptc_scene_set_lens(cs._h, (pt.Lens * 1)(pt.Lens(0.1, 1.0)), -1) == pt.PTC_E_INVALID
    assert pt.core().ptc_scene_set_lens(cs._h, None, 1) == pt.PTC_E_INVALID
    assert pt.core().ptc_scene_set_lens(None, None, 0) == pt.PTC_E_INVALID
    assert _render(pt, cs, s) == pt.PTC_E_INVALID  # still two lenses
    assert pt.core().ptc_scene_set_lens(cs._h, None, 0) == 0  # reset: a pinhole, NULL allowed
    assert _render(pt, cs, s) == pt.PTC_E_STATE


def test_lens_rules_of_every_call_on_an_uncommitted_scene(pt):
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

    for lenses in ([], [(0.0, 1.0)], [(0.3, 2.0)]):
        assert _set(pt, cs, lenses) == 0
        assert set(single_calls().values()) == {pt.PTC_E_STATE}, lenses
        assert _batch(pt, cs, s, 1) == pt.PTC_E_STATE and _batch(pt, cs, s, 4) == pt.PTC_E_STATE
    assert _set(pt, cs, [(0.3, 2.0), (0.0, 2.0), (0.1, 5.0)]) == 0
    got = single_calls()
    assert set(got.values()) == {pt.PTC_E_INVALID}, got
    assert _batch(pt, cs, s, 3) == pt.PTC_E_STATE
    assert _batch(pt, cs, s, 2) == pt.PTC_E_INVALID and _batch(pt, cs, s, 4) == pt.PTC_E_INVALID
    arr = (pt.Camera * 2)(cam, cam)
    assert core.ptc_render_batch_accumulate(cs._h, arr, 2, None, C.byref(st), C.c_void_p(16), None, None) == pt.PTC_E_INVALID


def test_python_set_lens_forms(pt):
    s = _scene(pt)
    cs = s.to_core()
    cs.set_lens(0.1, 2.0)
    with pytest.raises(pt.PtcError):
        cs.set_lens(-1.0, 2.0)
    cs.set_lens([(0.1, 2.0), (0.2, 4.0)])
    with pytest.raises(pt.PtcError) as e:
        cs.render(s.camera, s.render_settings())
    assert e.value.code == pt.PTC_E_INVALID
    cs.set_lens()
    with pytest.raises(pt.PtcError) as e:
        cs.render(s.camera, s.render_settings())
    assert e.value.code == pt.PTC_E_STATE


def test_rust_crate_declares_the_lens():
    src = open(os.path.join(ROOT, "rust", "ptcore-sys", "src", "lib.rs")).read()
    assert re.search(r"pub struct ptc_lens \{\s*pub aperture_radius: f32,\s*pub focus_distance: f32,\s*\}", src)
    assert re.search(r"pub fn ptc_scene_set_lens\(s: \*mut ptc_scene, lenses: \*const ptc_lens, n: i32\) -> c_int;", src)


# ---- the loader -------------------------------------------------------------------------------------------------
def _write(tmp_path, doc, name="scene.json"):
    p = tmp_path / name
    p.write_text(json.dumps(doc))
    return str(p)


CAM = {"transform": {"position": [0, 1, 5], "look_at": [0, 1, 1], "up": [0, 1, 0]}, "fov": 40, "resolution": [64, 48]}
BSDFS = [{"name": "w", "type": "lambert", "albedo": 0.5}]
PRIMS = [{"type": "sphere", "transform": {"position": [0, 1, 0]}, "bsdf": "w"}]


def test_thinlens_camera_is_a_pinhole_without_the_flag(pt, tmp_path):
    thin = dict(CAM, type="thinlens", focus_distance=3.0, aperture_size=0.25)
    a = pt.load_scene_from_json(_write(tmp_path, {"camera": CAM, "bsdfs": BSDFS, "primitives": PRIMS}, "a.json"))
    b = pt.load_scene_from_json(_write(tmp_path, {"camera": thin, "bsdfs": BSDFS, "primitives": PRIMS}, "b.json"))
    assert a.lens is None and b.lens is None
    assert bytes(a.camera) == bytes(b.camera) and a.settings == b.settings
    assert [bytes(o) for o in a.objects] == [bytes(o) for o in b.objects]
    assert [bytes(m) for m in a.materials] == [bytes(m) for m in b.materials]


def test_thinlens_camera_with_the_flag(pt, tmp_path, capfd):
    thin = dict(CAM, type="thinlens", focus_distance=3.0, aperture_size=0.25)
    s = pt.load_scene_from_json(_write(tmp_path, {"camera": thin, "bsdfs": BSDFS, "primitives": PRIMS}), pt.LOAD_THIN_LENS)
    assert s.lens == (pytest.approx(0.25), pytest.approx(3.0))
    plain = pt.load_scene_from_json(_write(tmp_path, {"camera": CAM, "bsdfs": BSDFS, "primitives": PRIMS}, "p.json"), pt.LOAD_THIN_LENS)
    assert plain.lens is None and bytes(plain.camera) == bytes(s.camera)
    # no focus_distance: |look_at - position| (our rule)
    s = pt.load_scene_from_json(_write(tmp_path, {"camera": dict(CAM, type="thinlens", aperture_size=0.1), "bsdfs": BSDFS, "primitives": PRIMS}),
                                pt.LOAD_THIN_LENS)
    assert s.lens == (pytest.approx(0.1), pytest.approx(4.0))
    assert "Warning" not in capfd.readouterr().err
    # other thinlens keys are ignored, with one warning
    extra = dict(CAM, type="thinlens", aperture_size=0.1, focus_distance=2.0, aperture="disk.png", catEye=0.5, focus_pivot="x")
    s = pt.load_scene_from_json(_write(tmp_path, {"camera": extra, "bsdfs": BSDFS, "primitives": PRIMS}), pt.LOAD_THIN_LENS)
    assert s.lens == (pytest.approx(0.1), pytest.approx(2.0))
    assert capfd.readouterr().err.count("Warning") == 1
