"""Batch rendering (ptc_render_batch, ptc_render_batch_accumulate) without a device.

  * the Rust crate declares both functions;
  * the wrapper passes its arguments and returns view-major images of the right shapes;
  * bad arguments are refused before the scene's state is looked at; good ones on an uncommitted scene are a state error.
"""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _scene(pt):
    s = pt.Scene()
    s.add_sphere((0, 0, -1), 0.5, s.add_material(pt.lambertian((0.5, 0.5, 0.5))))
    s.set_camera((0, 0, 0), (0, 0, -1), (0, 1, 0), 60.0, 1.0)
    s.set_settings(8, 6, 16, 4)
    return s


def test_rust_crate_declares_them():
    src = open(os.path.join(ROOT, "rust", "ptcore-sys", "src", "lib.rs")).read()
    assert re.search(r"pub fn ptc_render_batch\(s: \*mut ptc_scene, cams: \*const ptc_camera, n_views: i32, seeds: \*const u64, "
                     r"st: \*const ptc_render_settings,\s*out_rgb: \*mut f32, out_u32: \*mut u32, stats: \*mut ptc_stats\) -> c_int;", src)
    assert re.search(r"pub fn ptc_render_batch_accumulate\(s: \*mut ptc_scene, cams: \*const ptc_camera, n_views: i32, "
                     r"seeds: \*const u64,\s*st: \*const ptc_render_settings, d_accum: \*mut f32, cuda_stream: \*mut c_void,\s*"
                     r"stats: \*mut ptc_stats\) -> c_int;", src)


def test_wrapper_shapes_and_arguments(pt, monkeypatch):
    s = _scene(pt)
    st = s.render_settings()
    cams = [s.camera] * 3
    seen = []

    class Fake:
        def ptc_render_batch(self, h, c, n, seeds, settings, rgb, u32, stats):
            sd = None if seeds is None else list(np.ctypeslib.as_array((C.c_uint64 * n).from_address(seeds)))
            seen.append(("batch", n, c[2].position[2], sd, settings._obj.width, bool(rgb), bool(u32)))
            return 0

        def ptc_render_batch_accumulate(self, h, c, n, seeds, settings, d_accum, stream, stats):
            seen.append(("accumulate", n, seeds is None, d_accum, stream))
            return 0

    monkeypatch.setattr(pt, "core", lambda: Fake())
    cs = pt.CoreScene(None)
    rgb, u32, stats = cs.render_batch(cams, st, seeds=[5, 6, 7])
    assert rgb.shape == (3, st.height, st.width, 3) and rgb.dtype == np.float32
    assert u32.shape == (3, st.height * st.width) and u32.dtype == np.uint32
    assert isinstance(stats, pt.Stats)
    assert pt.CoreScene._batch_args(cams, None)[2] is None
    cs.render_batch_accumulate(cams[:2], st, 1234, 99)
    assert seen == [("batch", 3, 0.0, [5, 6, 7], 8, True, True), ("accumulate", 2, True, 1234, 99)]
    with pytest.raises(ValueError):
        cs.render_batch(cams, st, seeds=[1, 2])


def _batch(pt, cs, cams, st, n=None, seeds=None, rgb=True, u32=True):
    n = len(cams) if n is None else n
    arr = (pt.Camera * max(len(cams), 1))(*cams) if cams is not None else None
    k = max(n, 1)
    out_rgb = np.empty(k * st.width * st.height * 3, np.float32) if rgb else None
    out_u32 = np.empty(k * st.width * st.height, np.uint32) if u32 else None
    sd = np.asarray(seeds, np.uint64) if seeds is not None else None
    return pt.core().ptc_render_batch(cs._h, arr, n, None if sd is None else sd.ctypes.data, C.byref(st),
                                      None if out_rgb is None else out_rgb.ctypes.data_as(C.POINTER(C.c_float)),
                                      None if out_u32 is None else out_u32.ctypes.data, None)


@pytest.mark.parametrize("case", ["n0", "n-1", "null-cams", "no-output", "tile_mod", "too-large", "nee-sky-alone", "spp0"])
def test_bad_arguments_are_refused_without_a_device(pt, case):
    s = _scene(pt)
    cs = s.to_core()  # not committed: the arguments are checked first
    cams = [s.camera, s.camera]
    over, kw = {}, {}
    if case == "n0":
        kw["n"] = 0
    elif case == "n-1":
        kw["n"] = -1
    elif case == "null-cams":
        cams = None
        kw["n"] = 2
    elif case == "no-output":
        kw.update(rgb=False, u32=False)
    elif case == "tile_mod":
        over = dict(tile_mod=2, tile_rem=1)
    elif case == "too-large":
        # 2 views of 33 x 32 pad to 2 x 64 x 32 pixels; 2^30 / 2048 + 1 views of that are over the limit
        over = dict(width=33, height=32)
        kw["n"] = (1 << 30) // (64 * 32) + 1
    elif case == "nee-sky-alone":
        over = dict(flags=pt.FLAG_NEE_SKY)
    elif case == "spp0":
        over = dict(spp=0)
    st = s.render_settings(**over)
    if case == "too-large":
        # no buffers for 2^19 views: the size is refused before any output is touched, so tiny ones stand in for them
        arr = (pt.Camera * 2)(*cams)
        rc = pt.core().ptc_render_batch(cs._h, arr, kw["n"], None, C.byref(st), (C.c_float * 3)(), (C.c_uint32 * 1)(), None)
    else:
        rc = _batch(pt, cs, cams, st, **kw)
    assert rc == pt.PTC_E_INVALID, pt.core().ptc_last_error()
    if case in ("n0", "null-cams", "tile_mod", "too-large"):  # the accumulate route shares the checks
        arr = (pt.Camera * 2)(*[s.camera] * 2) if cams is not None else None
        rc = pt.core().ptc_render_batch_accumulate(cs._h, arr, kw.get("n", 2), None, C.byref(st), C.c_void_p(16), None, None)
        assert rc == pt.PTC_E_INVALID


def test_the_largest_batch_is_not_refused_for_its_size(pt):
    s = _scene(pt)
    cs = s.to_core()
    st = s.render_settings(width=33, height=32)
    arr = (pt.Camera * 2)(s.camera, s.camera)
    n = (1 << 30) // (64 * 32)  # exactly 2^30 padded pixels: valid, so the uncommitted scene is what fails
    assert pt.core().ptc_render_batch(cs._h, arr, n, None, C.byref(st), (C.c_float * 3)(), None, None) == pt.PTC_E_STATE


def test_null_accumulate_buffer_and_handle_are_refused(pt):
    s = _scene(pt)
    st = s.render_settings()
    arr = (pt.Camera * 1)(s.camera)
    core = pt.core()
    assert core.ptc_render_batch_accumulate(s.to_core()._h, arr, 1, None, C.byref(st), None, None, None) == pt.PTC_E_INVALID
    assert core.ptc_render_batch(None, arr, 1, None, C.byref(st), None, (C.c_uint32 * 48)(), None) == pt.PTC_E_INVALID


@pytest.mark.parametrize("rgb, u32, seeds", [(True, True, None), (True, False, [1, 2]), (False, True, [3, 4])])
def test_uncommitted_scene_is_a_state_error(pt, rgb, u32, seeds):
    s = _scene(pt)
    cs = s.to_core()
    assert _batch(pt, cs, [s.camera, s.camera], s.render_settings(), seeds=seeds, rgb=rgb, u32=u32) == pt.PTC_E_STATE
    arr = (pt.Camera * 2)(s.camera, s.camera)
    assert pt.core().ptc_render_batch_accumulate(cs._h, arr, 2, None, C.byref(s.render_settings()), C.c_void_p(16), None,
                                                 None) == pt.PTC_E_STATE
    with pytest.raises(pt.PtcError) as e:
        cs.render_batch([s.camera], s.render_settings(), seeds=seeds[:1] if seeds else None)
    assert e.value.code == pt.PTC_E_STATE
