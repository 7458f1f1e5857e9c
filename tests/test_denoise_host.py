"""The denoiser (ptc_render_denoised, ptc_denoise_image) without a device.

  * the filter: the g++ build of pt_denoise.h (tests/hostsim/denoisesim.cpp) agrees with a float32 numpy restatement
    of the formulas to 1e-6 relative, for random images of several sizes and every level count 1..10; non-finite
    centres pass through and no finite pixel becomes non-finite; zero albedo; a pixel with no neighbour in the frame;
  * feature_albedo of every material type, and of a miss;
  * the variance from two halves is (A - B)^2 / 4 for equal halves, and h (n - h) / n^2 (A - B)^2 in general;
  * the ABI: ptc_denoise has the same layout in C and in ctypes, and the Rust crate declares it and both functions;
  * bad arguments are refused before the scene's state is looked at; good ones on an uncommitted scene are a state error.
"""
import ctypes as C
import os
import re
import subprocess
import zlib

import numpy as np
import pytest

from bindings import sim_lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_F = C.POINTER(C.c_float)
_vp = C.c_void_p


def _lib():
    L = sim_lib()
    L.denoise_sim_feature_albedo.argtypes = [_vp, C.c_int32, _vp, _F, C.c_int64, _F]
    L.denoise_sim_feature_albedo.restype = C.c_int32
    L.denoise_sim_variance.argtypes = [_F, _F, C.c_int64, C.c_int32, C.c_int32, _F, _F]
    L.denoise_sim_variance.restype = None
    L.denoise_sim_filter.argtypes = [C.c_int32, C.c_int32, _F, _F, _F, _F, C.c_int32, C.c_float, C.c_float, C.c_float, _F]
    L.denoise_sim_filter.restype = None
    return L


def _p(a):
    return a.ctypes.data_as(_F)


def sim_filter(rgb, var, albedo, normal, iterations, sl=4.0, sn=0.1, sa=0.1):
    h, w = rgb.shape[:2]
    rgb, var, albedo, normal = (np.ascontiguousarray(a, np.float32) for a in (rgb, var, albedo, normal))
    out = np.empty((h, w, 3), np.float32)
    _lib().denoise_sim_filter(w, h, _p(rgb), _p(var), _p(albedo), _p(normal), iterations, sl, sn, sa, _p(out))
    return out


def sim_variance(Sh, Sn, h, n, albedo):
    Sh, Sn, albedo = (np.ascontiguousarray(a, np.float32).reshape(-1, 3) for a in (Sh, Sn, albedo))
    out = np.empty(len(Sh), np.float32)
    _lib().denoise_sim_variance(_p(Sh), _p(Sn), len(Sh), h, n, _p(albedo), _p(out))
    return out


def sim_feature_albedo(materials, mat_idx, pos):
    mats = (materials[0].__class__ * max(len(materials), 1))(*materials)
    idx = np.ascontiguousarray(mat_idx, np.int32)
    pos = np.ascontiguousarray(pos, np.float32).reshape(-1, 3)
    out = np.empty((len(idx), 3), np.float32)
    assert _lib().denoise_sim_feature_albedo(C.addressof(mats), len(materials), idx.ctypes.data, _p(pos), len(idx), _p(out)) == 0
    return out


# ---- numpy restatement (float32, the header's order of operations) ----------------------------------------------
f32 = np.float32


def np_lum(x):
    return f32(0.2126) * x[..., 0] + f32(0.7152) * x[..., 1] + f32(0.0722) * x[..., 2]


def np_filter(rgb, var, albedo, normal, iterations, sl=4.0, sn=0.1, sa=0.1):
    rgb, var, albedo, normal = (np.asarray(a, np.float32) for a in (rgb, var, albedo, normal))
    h, w = rgb.shape[:2]
    d = np.maximum(albedo, f32(1e-3))
    with np.errstate(all="ignore"):
        x = rgb / d
        v = var.copy()
        sl2 = f32(sl) * f32(sl)
        isn2, isa2 = f32(1) / (f32(sn) * f32(sn)), f32(1) / (f32(sa) * f32(sa))
        b3 = np.array([1, 4, 6, 4, 1], np.float32) / f32(16)

        def shifted(a, dy, dx, fill):
            """a[y + dy, x + dx] where that is in the frame, else fill; and the in-frame mask"""
            out = np.full_like(a, fill)
            m = np.zeros((h, w), bool)
            if abs(dy) >= h or abs(dx) >= w:
                return out, m
            ys, yd = slice(max(0, -dy), min(h, h - dy)), slice(max(0, dy), min(h, h + dy))
            xs, xd = slice(max(0, -dx), min(w, w - dx)), slice(max(0, dx), min(w, w + dx))
            out[ys, xs] = a[yd, xd]
            m[ys, xs] = True
            return out, m

        for i in range(iterations):
            step = 1 << i
            fin = np.isfinite(x).all(axis=2)
            gs, gk = np.zeros((h, w), np.float32), np.zeros((h, w), np.float32)
            for dy in (-1, 0, 1):
                for dx in (-1, 0, 1):
                    vq, m = shifted(v, dy, dx, 0)
                    fq, _ = shifted(fin, dy, dx, False)
                    use = m & fq
                    k = f32((2 if dx == 0 else 1) * (2 if dy == 0 else 1))
                    gs = np.where(use, gs + k * vq, gs)
                    gk = np.where(use, gk + k, gk)
            g = gs / gk
            lp = np_lum(x)
            lden = sl2 * g + f32(1e-10)
            sw = np.zeros((h, w), np.float32)
            sx = np.zeros((h, w, 3), np.float32)
            sv = np.zeros((h, w), np.float32)
            for dy in range(-2, 3):
                for dx in range(-2, 3):
                    xq, m = shifted(x, dy * step, dx * step, 0)
                    vq, _ = shifted(v, dy * step, dx * step, 0)
                    aq, _ = shifted(albedo, dy * step, dx * step, 0)
                    nq, _ = shifted(normal, dy * step, dx * step, 0)
                    fq, _ = shifted(fin, dy * step, dx * step, False)
                    use = m & fq
                    dl = lp - np_lum(xq)
                    wl = f32(1) / (f32(1) + dl * dl / lden)
                    dn = normal - nq
                    da = albedo - aq
                    wn = f32(1) / (f32(1) + ((dn[..., 0] * dn[..., 0] + dn[..., 1] * dn[..., 1]) + dn[..., 2] * dn[..., 2]) * isn2)
                    wa = f32(1) / (f32(1) + ((da[..., 0] * da[..., 0] + da[..., 1] * da[..., 1]) + da[..., 2] * da[..., 2]) * isa2)
                    wt = (((b3[dy + 2] * b3[dx + 2]) * wl) * wn) * wa
                    sw = np.where(use, sw + wt, sw)
                    sx = np.where(use[..., None], sx + wt[..., None] * xq, sx)
                    sv = np.where(use, sv + (wt * wt) * vq, sv)
            nx = sx / sw[..., None]
            nv = sv / (sw * sw)
            x = np.where(fin[..., None], nx, x)
            v = np.where(fin, nv, v)
        fin = np.isfinite(x).all(axis=2)
        return np.where(fin[..., None], x * d, rgb).astype(np.float32)


def _inputs(rng, h, w):
    rgb = rng.gamma(1.5, 0.4, (h, w, 3)).astype(np.float32)
    var = (rng.random((h, w)) ** 3 * 0.5).astype(np.float32)
    albedo = rng.uniform(0.0, 1.0, (h, w, 3)).astype(np.float32)
    albedo[rng.random((h, w)) < 0.2] = 1.0  # misses and dielectrics
    n = rng.normal(size=(h, w, 3)).astype(np.float32)
    n /= np.linalg.norm(n, axis=2, keepdims=True).astype(np.float32)
    n[rng.random((h, w)) < 0.1] = 0.0  # misses
    # regions with equal guides, so that the luminance term decides
    albedo[: h // 2, : w // 2] = albedo[0, 0]
    n[: h // 2, : w // 2] = n[0, 0]
    return rgb, var, albedo, n.astype(np.float32)


def _close(a, b, rel=1e-6):
    fa, fb = np.isfinite(a), np.isfinite(b)
    assert np.array_equal(fa, fb)
    assert np.array_equal(a[~fa], b[~fb], equal_nan=True)
    assert np.all(np.abs(a[fa] - b[fa]) <= rel * np.maximum(np.abs(b[fa]), 1e-30) + 1e-30), np.max(np.abs(a[fa] - b[fa]))


@pytest.mark.parametrize("h, w", [(1, 1), (3, 7), (48, 64)])
@pytest.mark.parametrize("iterations", list(range(1, 11)))
def test_filter_matches_numpy(h, w, iterations):
    rng = np.random.default_rng(zlib.crc32(repr((h, w, iterations)).encode()))
    rgb, var, albedo, normal = _inputs(rng, h, w)
    a = sim_filter(rgb, var, albedo, normal, iterations)
    b = np_filter(rgb, var, albedo, normal, iterations)
    _close(a, b)
    assert np.isfinite(a).all()


@pytest.mark.parametrize("sl, sn, sa", [(4.0, 0.1, 0.1), (0.5, 1.0, 2.0), (100.0, 0.01, 0.05)])
def test_filter_matches_numpy_at_other_sigmas(sl, sn, sa):
    rng = np.random.default_rng(7)
    rgb, var, albedo, normal = _inputs(rng, 20, 24)
    _close(sim_filter(rgb, var, albedo, normal, 4, sl, sn, sa), np_filter(rgb, var, albedo, normal, 4, sl, sn, sa))


def test_non_finite_centres_pass_through():
    rng = np.random.default_rng(3)
    rgb, var, albedo, normal = _inputs(rng, 16, 20)
    bad = [(0, 0, 0, np.nan), (5, 7, 1, np.inf), (15, 19, 2, -np.inf), (8, 3, 0, np.nan), (8, 3, 1, np.inf), (2, 9, 1, np.nan)]
    for y, x, c, val in bad:
        rgb[y, x, c] = val
    for k in (1, 3, 5):
        out = sim_filter(rgb, var, albedo, normal, k)
        _close(out, np_filter(rgb, var, albedo, normal, k))
        mask = ~np.isfinite(rgb).all(axis=2)
        # the non-finite pixels are their noisy values, finite channels included, bit for bit
        assert np.array_equal(out[mask].view(np.uint32), rgb[mask].view(np.uint32))
        assert np.isfinite(out[~mask]).all()


def test_zero_albedo():
    rng = np.random.default_rng(5)
    rgb, var, albedo, normal = _inputs(rng, 12, 10)
    albedo[:, :5] = 0.0
    albedo[3, 7] = (0.0, 0.5, 0.0)
    for k in (1, 2, 5):
        out = sim_filter(rgb, var, albedo, normal, k)
        _close(out, np_filter(rgb, var, albedo, normal, k))
        assert np.isfinite(out).all()


def test_constant_image_is_a_fixed_point():
    # equal values everywhere: every weighted mean is the value again (up to rounding of the weights' sum)
    h, w = 9, 11
    rgb = np.full((h, w, 3), 0.25, np.float32)
    albedo = np.full((h, w, 3), 0.5, np.float32)
    normal = np.zeros((h, w, 3), np.float32)
    normal[..., 2] = 1.0
    out = sim_filter(rgb, np.full((h, w), 0.01, np.float32), albedo, normal, 5)
    assert np.allclose(out, 0.25, rtol=1e-6, atol=0)


def test_pixel_without_neighbours_in_the_frame():
    # 1 x 1: only the centre; and a 1-pixel-wide column at step 2^i > height: only the centre too at the later levels
    rgb = np.array([[[0.3, 1.5, 7.0]]], np.float32)
    var = np.array([[2.0]], np.float32)
    albedo = np.array([[[0.5, 0.0, 1.0]]], np.float32)
    normal = np.array([[[0.0, 1.0, 0.0]]], np.float32)
    for k in range(1, 11):
        out = sim_filter(rgb, var, albedo, normal, k)
        want = (rgb / np.maximum(albedo, np.float32(1e-3))) * np.maximum(albedo, np.float32(1e-3))
        assert np.array_equal(out, want)
    # a finite pixel whose every neighbour is non-finite keeps its value
    rgb = np.full((3, 3, 3), np.nan, np.float32)
    rgb[1, 1] = (0.2, 0.4, 0.6)
    out = sim_filter(rgb, np.ones((3, 3), np.float32), np.ones((3, 3, 3), np.float32), np.zeros((3, 3, 3), np.float32), 3)
    assert np.array_equal(out[1, 1], rgb[1, 1]) and np.isnan(out).sum() == 8 * 3


def test_feature_albedo_table(pt):
    mats = [pt.lambertian((0.1, 0.2, 0.3)), pt.checker((0.9, 0.8, 0.7), (0.05, 0.06, 0.07), 1.0), pt.metal((0.4, 0.5, 0.6), 0.1),
            pt.dielectric(1.5), pt.emissive((5.0, 6.0, 7.0)), pt.plastic((0.25, 0.35, 0.45)),
            pt.rough_conductor((0.7, 0.6, 0.5), 0.3), pt.null_material()]
    assert [m.type for m in mats] == list(range(8))
    pos = np.array([[0.5, 0.5, 0.5], [0.5, 0.5, 0.5], [1.5, 0.5, 0.5]] + [[0.5, 0.5, 0.5]] * 7, np.float32)  # checker: on, off
    idx = np.array([0, 1, 1, 2, 3, 4, 5, 6, 7, -1], np.int32)
    got = sim_feature_albedo(mats, idx, pos)
    want = np.array([(0.1, 0.2, 0.3), (0.9, 0.8, 0.7), (0.05, 0.06, 0.07), (0.4, 0.5, 0.6), (1, 1, 1), (1, 1, 1),
                     (0.25, 0.35, 0.45), (0.7, 0.6, 0.5), (1, 1, 1), (1, 1, 1)], np.float32)
    assert np.array_equal(got, want)


def test_variance_of_equal_halves():
    rng = np.random.default_rng(11)
    for n in (2, 8, 64, 1000):
        h = n // 2
        Sh = rng.uniform(0, 3, (500, 3)).astype(np.float32) * f32(h)
        Sn = Sh + rng.uniform(0, 3, (500, 3)).astype(np.float32) * f32(n - h)
        ones = np.ones((500, 3), np.float32)
        got = sim_variance(Sh, Sn, h, n, ones)
        A = Sh * (f32(1) / f32(h))
        B = (Sn - Sh) * (f32(1) / f32(n - h))
        dl = np_lum(A) - np_lum(B)
        assert np.array_equal(got, (dl * dl) / f32(4))


def test_variance_of_unequal_halves_and_demodulation():
    rng = np.random.default_rng(12)
    h, n = 3, 7
    Sh = rng.uniform(0, 3, (300, 3)).astype(np.float32)
    Sn = Sh + rng.uniform(0, 3, (300, 3)).astype(np.float32)
    alb = rng.uniform(0, 1, (300, 3)).astype(np.float32)
    alb[:20] = 0.0
    Sn[5, 1] = np.inf
    Sn[6, 0] = np.nan
    got = sim_variance(Sh, Sn, h, n, alb)
    d = np.maximum(alb, f32(1e-3))
    with np.errstate(all="ignore"):
        A = Sh * (f32(1) / f32(h)) / d
        B = (Sn - Sh) * (f32(1) / f32(n - h)) / d
        dl = np_lum(A) - np_lum(B)
        want = dl * dl * (f32(h) * f32(n - h) / (f32(n) * f32(n)))
    want[~np.isfinite(Sn).all(axis=1)] = 0.0
    assert np.array_equal(got, want.astype(np.float32))
    assert got[5] == 0.0 and got[6] == 0.0


def test_denoise_struct_layout(pt, tmp_path):
    src = tmp_path / "sz.c"
    fields = ("feature_spp", "iterations", "sigma_luminance", "sigma_normal", "sigma_albedo")
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "ptcore.h"\nint main(){printf("%zu' + " %zu" * len(fields) +
                   '\\n",sizeof(ptc_denoise)' + "".join(f",offsetof(ptc_denoise,{f})" for f in fields) + ");return 0;}\n")
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    want = [C.sizeof(pt.Denoise)] + [getattr(pt.Denoise, f).offset for f in fields]
    assert got == want == [20, 0, 4, 8, 12, 16]


def test_rust_crate_declares_it():
    src = open(os.path.join(ROOT, "rust", "ptcore-sys", "src", "lib.rs")).read()
    assert re.search(r"pub struct ptc_denoise \{\s*pub feature_spp: i32,\s*pub iterations: i32,\s*pub sigma_luminance: f32,\s*"
                     r"pub sigma_normal: f32,\s*pub sigma_albedo: f32,\s*\}", src)
    assert re.search(r"pub fn ptc_render_denoised\(s: \*mut ptc_scene, cam: \*const ptc_camera, st: \*const ptc_render_settings, "
                     r"dn: \*const ptc_denoise,\s*out_rgb: \*mut f32, out_u32: \*mut u32, out_noisy_rgb: \*mut f32, out_albedo: \*mut f32,\s*"
                     r"out_normal: \*mut f32, out_variance: \*mut f32, stats: \*mut ptc_stats\) -> c_int;", src)
    assert re.search(r"pub fn ptc_denoise_image\(s: \*mut ptc_scene, dn: \*const ptc_denoise, width: i32, height: i32, rgb: \*const f32, "
                     r"variance: \*const f32,\s*albedo: \*const f32, normal: \*const f32, out_rgb: \*mut f32\) -> c_int;", src)


def _scene(pt):
    s = pt.Scene()
    s.add_sphere((0, 0, -1), 0.5, s.add_material(pt.lambertian((0.5, 0.5, 0.5))))
    s.set_camera((0, 0, 0), (0, 0, -1), (0, 1, 0), 60.0, 1.0)
    s.set_settings(8, 6, 16, 4)
    return s


def test_wrapper_passes_arguments(pt, monkeypatch):
    s = _scene(pt)
    seen = []

    def fake(h, cam, settings, dn, rgb, u32, noisy, albedo, normal, var, stats):
        d = dn._obj
        seen.append((settings._obj.spp, d.feature_spp, d.iterations, round(d.sigma_luminance, 6), round(d.sigma_normal, 6),
                     round(d.sigma_albedo, 6), all(bool(p) for p in (rgb, u32, noisy, albedo, normal, var))))
        return 0

    monkeypatch.setattr(pt.core(), "ptc_render_denoised", fake)
    cs = s.to_core()
    rgb, u32, noisy, albedo, normal, var, stats = cs.render_denoised(s.camera, s.render_settings())
    assert seen[-1] == (16, 4, 5, 4.0, 0.1, 0.1, True)  # feature_spp None -> min(spp, 4)
    assert rgb.shape == noisy.shape == albedo.shape == normal.shape == (6, 8, 3) and var.shape == (6, 8)
    assert u32.shape == (48,) and u32.dtype == np.uint32 and isinstance(stats, pt.Stats)
    cs.render_denoised(s.camera, s.render_settings(spp=2))
    assert seen[-1][:2] == (2, 2)
    cs.render_denoised(s.camera, s.render_settings(), feature_spp=7, iterations=3, sigma_luminance=2.0, sigma_normal=0.5,
                       sigma_albedo=0.25)
    assert seen[-1] == (16, 7, 3, 2.0, 0.5, 0.25, True)


_GOOD = dict(feature_spp=2, iterations=5, sigma_luminance=4.0, sigma_normal=0.1, sigma_albedo=0.1)
_BAD = [
    ({"spp": 1}, {}), ({"spp": 0}, {}),                                                            # spp < 2
    ({}, {"feature_spp": 0}), ({}, {"feature_spp": 17}), ({}, {"feature_spp": -1}),                  # feature_spp outside [1, spp]
    ({}, {"iterations": 0}), ({}, {"iterations": 11}), ({}, {"iterations": -3}),                    # iterations outside 1..10
    ({}, {"sigma_luminance": 0.0}), ({}, {"sigma_normal": -1.0}), ({}, {"sigma_albedo": float("nan")}),
    ({}, {"sigma_luminance": float("inf")}), ({}, {"sigma_normal": float("nan")}), ({}, {"sigma_albedo": 0.0}),
    ({"sample_begin": 0, "sample_end": 8}, {}), ({"sample_begin": 2, "sample_end": 8}, {}),
    ({"tile_mod": 2, "tile_rem": 1}, {}), ({"flags": 8}, {}), ({"width": 0}, {}), ({"width": 32768, "height": 32768}, {}),
]


@pytest.mark.parametrize("over, dn", _BAD)
def test_bad_arguments_are_refused_without_a_device(pt, over, dn):
    s = _scene(pt)
    cs = s.to_core()  # not committed: the arguments are checked first
    with pytest.raises(pt.PtcError) as e:
        cs.render_denoised(s.camera, s.render_settings(**over), **dict(_GOOD, **dn))
    assert e.value.code == pt.PTC_E_INVALID


@pytest.mark.parametrize("dn", [d for o, d in _BAD if d and "feature_spp" not in d])
def test_bad_filter_arguments_are_refused_without_a_device(pt, dn):
    s = _scene(pt)
    img = np.zeros((4, 5, 3), np.float32)
    kw = {k: v for k, v in dict(_GOOD, **dn).items() if k != "feature_spp"}
    with pytest.raises(pt.PtcError) as e:
        s.to_core().denoise_image(img, np.zeros((4, 5), np.float32), img, img, **kw)
    assert e.value.code == pt.PTC_E_INVALID


def test_null_arguments_are_refused(pt):
    s = _scene(pt)
    cs = s.to_core()
    dn = pt.Denoise(2, 5, 4.0, 0.1, 0.1)
    st = s.render_settings()
    core = pt.core()
    for args in ((None, C.byref(s.camera), C.byref(st), C.byref(dn)), (cs._h, None, C.byref(st), C.byref(dn)),
                 (cs._h, C.byref(s.camera), None, C.byref(dn)), (cs._h, C.byref(s.camera), C.byref(st), None)):
        assert core.ptc_render_denoised(*args, None, None, None, None, None, None, None) == pt.PTC_E_INVALID
    buf = np.zeros(3, np.float32)
    p = buf.ctypes.data_as(_F)
    assert core.ptc_denoise_image(cs._h, C.byref(dn), 1, 1, p, p, p, None, p) == pt.PTC_E_INVALID
    assert core.ptc_denoise_image(cs._h, None, 1, 1, p, p, p, p, p) == pt.PTC_E_INVALID
    assert core.ptc_denoise_image(cs._h, C.byref(dn), 0, 1, p, p, p, p, p) == pt.PTC_E_INVALID


@pytest.mark.parametrize("spp, feature_spp, iterations", [(2, 1, 1), (16, 16, 10), (5, 3, 5)])
def test_uncommitted_scene_is_a_state_error(pt, spp, feature_spp, iterations):
    s = _scene(pt)
    cs = s.to_core()
    with pytest.raises(pt.PtcError) as e:
        cs.render_denoised(s.camera, s.render_settings(spp=spp), feature_spp=feature_spp, iterations=iterations)
    assert e.value.code == pt.PTC_E_STATE
    img = np.zeros((2, 3, 3), np.float32)
    with pytest.raises(pt.PtcError) as e:
        cs.denoise_image(img, np.zeros((2, 3), np.float32), img, img, iterations=iterations)
    assert e.value.code == pt.PTC_E_STATE
