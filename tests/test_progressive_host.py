"""Progressive rendering (ptc_render_progressive) without a device.

  * the ABI: ptc_progressive has the same layout in C and in ctypes, and the Rust crate declares it, the callback type
    and the function;
  * the wrapper passes its arguments and wraps the Python callback;
  * bad arguments are refused before the scene's state is looked at; good ones on an uncommitted scene are a state error.
"""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_progressive_struct_layout(pt, tmp_path):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "ptcore.h"\nint main(){printf("%zu %zu %zu\\n",'
                   "sizeof(ptc_progressive),offsetof(ptc_progressive,first_spp),offsetof(ptc_progressive,max_pass_spp));"
                   "ptc_preview_fn f = 0; (void)f; return 0;}\n")
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    want = [C.sizeof(pt.ProgressiveSettings), pt.ProgressiveSettings.first_spp.offset, pt.ProgressiveSettings.max_pass_spp.offset]
    assert got == want == [8, 0, 4]


def test_rust_crate_declares_it():
    src = open(os.path.join(ROOT, "rust", "ptcore-sys", "src", "lib.rs")).read()
    assert re.search(r"pub struct ptc_progressive \{\s*pub first_spp: i32,\s*pub max_pass_spp: i32,\s*\}", src)
    assert re.search(r"pub type ptc_preview_fn = Option<unsafe extern \"C\" fn\(\*mut c_void, i32, i32, \*const u32\) -> i32>;", src)
    assert re.search(r"pub fn ptc_render_progressive\(s: \*mut ptc_scene, cam: \*const ptc_camera, st: \*const ptc_render_settings, "
                     r"pg: \*const ptc_progressive,\s*on_preview: ptc_preview_fn, user: \*mut c_void, out_rgb: \*mut f32, "
                     r"out_u32: \*mut u32,\s*out_samples: \*mut i32, stats: \*mut ptc_stats\) -> c_int;", src)


def _scene(pt):
    s = pt.Scene()
    s.add_sphere((0, 0, -1), 0.5, s.add_material(pt.lambertian((0.5, 0.5, 0.5))))
    s.set_camera((0, 0, 0), (0, 0, -1), (0, 1, 0), 60.0, 1.0)
    s.set_settings(8, 6, 16, 4)
    return s


def test_wrapper_passes_arguments(pt, monkeypatch):
    s = _scene(pt)
    st = s.render_settings()
    seen, shown = [], []

    def fake(h, cam, settings, pg, on_preview, user, rgb, u32, samples, stats):
        p = pg._obj
        seen.append((settings._obj.width, settings._obj.height, settings._obj.spp, p.first_spp, p.max_pass_spp,
                     bool(on_preview), user, bool(rgb), bool(u32)))
        if on_preview:  # call the wrapped callback as the library would, with an image of its own
            img = (C.c_uint32 * 48)(*range(48))
            assert on_preview(None, 0, 2, img) == 0
            img[0] = 7  # the callback got a copy
            assert on_preview(None, 1, 4, img) == 1
        samples._obj.value = 4
        return 0

    monkeypatch.setattr(pt.core(), "ptc_render_progressive", fake)
    cs = s.to_core()

    def cb(k, n, u32):
        shown.append((k, n, u32))
        return k == 1

    rgb, u32, samples, stats = cs.render_progressive(s.camera, st, 2, 3, on_preview=cb)
    assert seen == [(8, 6, 16, 2, 3, True, None, True, True)]
    assert [(k, n) for k, n, _ in shown] == [(0, 2), (1, 4)]
    assert shown[0][2].dtype == np.uint32 and np.array_equal(shown[0][2], np.arange(48))
    assert shown[1][2][0] == 7
    assert rgb.shape == (6, 8, 3) and rgb.dtype == np.float32
    assert u32.shape == (48,) and u32.dtype == np.uint32
    assert samples == 4 and isinstance(stats, pt.Stats)

    rgb, u32, samples, stats = cs.render_progressive(s.camera, st)  # defaults: first_spp 1, doubling, no callback
    assert seen[-1] == (8, 6, 16, 1, 0, False, None, True, True)


def test_exception_in_callback_stops_and_is_reraised(pt, monkeypatch):
    s = _scene(pt)
    returned = []

    def fake(h, cam, settings, pg, on_preview, user, rgb, u32, samples, stats):
        returned.append(on_preview(None, 0, 1, (C.c_uint32 * 48)()))
        return 0

    def boom(k, n, u32):
        raise KeyError("from the callback")

    monkeypatch.setattr(pt.core(), "ptc_render_progressive", fake)
    with pytest.raises(KeyError, match="from the callback"):
        s.to_core().render_progressive(s.camera, s.render_settings(), on_preview=boom)
    assert returned == [1]  # the library was told to stop


@pytest.mark.parametrize("first_spp, max_pass_spp, over", [
    (0, 0, {}), (-1, 0, {}), (17, 0, {}), (1, -1, {}),                      # first_spp outside [1, spp], negative cap
    (1, 0, {"sample_begin": 0, "sample_end": 8}), (1, 0, {"sample_begin": 2, "sample_end": 8}),
    (1, 0, {"tile_mod": 2, "tile_rem": 1}), (1, 0, {"flags": 8}),          # sample range, tile_mod, NEE_SKY without NEE
    (1, 0, {"spp": 0}), (1, 0, {"width": 0}), (1, 0, {"width": 32768, "height": 32768}),  # check_render_args
])
def test_bad_arguments_are_refused_without_a_device(pt, first_spp, max_pass_spp, over):
    s = _scene(pt)
    cs = s.to_core()  # not committed: the arguments are checked first
    with pytest.raises(pt.PtcError) as e:
        cs.render_progressive(s.camera, s.render_settings(**over), first_spp, max_pass_spp, on_preview=lambda *a: 0)
    assert e.value.code == pt.PTC_E_INVALID


def test_null_handle_and_settings_are_refused(pt):
    s = _scene(pt)
    pg = pt.ProgressiveSettings(1, 0)
    st = s.render_settings()
    core, null_fn = pt.core(), pt.PREVIEW_FN()
    cs = s.to_core()
    for args in ((None, C.byref(s.camera), C.byref(st), C.byref(pg)), (cs._h, C.byref(s.camera), C.byref(st), None),
                 (cs._h, None, C.byref(st), C.byref(pg)), (cs._h, C.byref(s.camera), None, C.byref(pg))):
        assert core.ptc_render_progressive(*args, null_fn, None, None, None, None, None) == pt.PTC_E_INVALID


@pytest.mark.parametrize("first_spp, max_pass_spp, with_callback", [(1, 0, False), (16, 0, True), (3, 4, True)])
def test_uncommitted_scene_is_a_state_error(pt, first_spp, max_pass_spp, with_callback):
    s = _scene(pt)
    called = []
    with pytest.raises(pt.PtcError) as e:
        s.to_core().render_progressive(s.camera, s.render_settings(), first_spp, max_pass_spp,
                                       on_preview=(lambda *a: called.append(a)) if with_callback else None)
    assert e.value.code == pt.PTC_E_STATE
    assert called == []
