"""Progressive rendering (ptc_render_progressive) on the B200.

Philox is keyed on the global (pixel, sample) and the film sums are fixed-point, so the film after the passes up to n
samples is, bit for bit, the film of a uniform render at n spp.  Hence, exactly (rgb compared as uint32 bit patterns, so
NaN and inf count):
  * every preview is render_u32 at its sample count, and the final images are render / render_u32 at spp — on the
    Cornell box, a shrunk semesterbild (mesh, depth 30), a shrunk teapot (C3s, NEE | NEE_SKY), a shrunk veach-mis (NEE),
    emitters beyond the fixed-point range, and max_depth 0;
  * the (pass, samples) sequence follows the schedule;
  * a stop at pass k gives k + 1 callbacks and the uniform render at n_k, and leaves the scene as it was;
  * the callback runs on the calling thread while the device renders the next pass;
  * an exception in the callback propagates; the pool size and repetition change nothing; no callback = render.
"""
import ctypes as C
import os
import threading
import time

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCENES = os.path.join(ROOT, "scenes")


def _case(pt, name):
    """-> (scene, render-settings keywords, progressive keywords)"""
    if name in ("cornell", "depth-0"):
        s = pt.load_scene_from_json(os.path.join(SCENES, "cornell-box", "scene.json"))
        return s, dict(width=64, height=48, spp=12, max_depth=0 if name == "depth-0" else 8, seed=3), dict(first_spp=1)
    if name == "semesterbild":
        s = pt.load_scene_from_json(os.path.join(SCENES, "semesterbild.json"))
        return s, dict(width=96, height=72, spp=10, max_depth=30, seed=7), dict(first_spp=3, max_pass_spp=2)
    if name == "teapot":
        s = pt.load_scene_from_json(os.path.join(SCENES, "teapot", "scene.json"), pt.LOAD_INFINITE_SPHERE_SKY | pt.LOAD_WO3_STRIDE16)
        return s, dict(width=128, height=72, spp=8, max_depth=16, seed=5, flags=pt.FLAG_NEE | pt.FLAG_NEE_SKY), dict(first_spp=1)
    if name == "veach-mis":
        s = pt.load_scene_from_json(os.path.join(SCENES, "veach-mis", "scene.json"))
        return s, dict(width=160, height=90, spp=16, max_depth=16, seed=11, flags=pt.FLAG_NEE), dict(first_spp=2)
    # test_gpu_film_resolve.py: radiance beyond the film's range
    s = pt.Scene()
    m = s.add_material(pt.emissive((3e7 if name == "emitter-3e7" else float("inf"), 1.0, 0.0)))
    s.add_sphere((0, 0, 0), 1.0, m)
    s.set_camera((0, 0, 4), (0, 0, 0), (0, 1, 0), 30.0, 1.0)
    return s, dict(width=16, height=16, spp=8, max_depth=3), dict(first_spp=1)


def _schedule(first_spp, max_pass_spp, spp):
    ns = [first_spp]
    while ns[-1] < spp:
        n = ns[-1]
        ns.append(min(n + (n if max_pass_spp == 0 else min(n, max_pass_spp)), spp))
    return ns


def _bits(rgb):
    return np.ascontiguousarray(rgb).view(np.uint32)


def _progressive(cs, s, st, stop_at=None, **kw):
    """-> (previews [(pass, samples, u32)], rgb, u32, samples, Stats)"""
    shown = []

    def cb(k, n, img):
        shown.append((k, n, img))
        return k == stop_at

    return (shown, *cs.render_progressive(s.camera, st, on_preview=cb, **kw))


@pytest.mark.parametrize("name", ["cornell", "semesterbild", "teapot", "veach-mis", "emitter-3e7", "emitter-inf", "depth-0"])
def test_every_preview_is_the_uniform_render_at_its_samples(pt, name):
    s, base, prog = _case(pt, name)
    cs = s.to_core().commit(0)
    st = s.render_settings(**base)
    shown, rgb, u32, n, stats = _progressive(cs, s, st, **prog)
    ns = _schedule(prog["first_spp"], prog.get("max_pass_spp", 0), st.spp)
    assert [(k, m) for k, m, _ in shown] == list(enumerate(ns))
    for k, m, img in shown:
        ref, _ = cs.render_u32(s.camera, s.render_settings(**dict(base, spp=m)))
        assert np.array_equal(img, ref), (k, m)
    ref_rgb, ref_stats = cs.render(s.camera, st)
    ref_u32, _ = cs.render_u32(s.camera, st)
    assert n == st.spp
    assert np.array_equal(_bits(rgb), _bits(ref_rgb))
    assert np.array_equal(u32, ref_u32) and np.array_equal(shown[-1][2], ref_u32)
    assert stats.paths == ref_stats.paths and stats.rays == ref_stats.rays
    assert stats.kernel_launches >= len(ns) and (stats.render_ms > 0 or name == "depth-0")
    if name.startswith("emitter"):
        assert np.isposinf(rgb[8, 8, 0]) and (u32[8 * 16 + 8] >> 16) == 255
    if name == "depth-0":
        assert not u32.any() and not rgb.any() and stats.paths == 0


_tiny = {}


def _tiny_scene(pt):
    if not _tiny:
        s = pt.load_scene_from_json(os.path.join(SCENES, "cornell-box", "scene.json"))
        _tiny["s"], _tiny["cs"] = s, s.to_core().commit(0)
    return _tiny["s"], _tiny["cs"]


@pytest.mark.parametrize("first_spp, max_pass_spp, spp, want", [
    (1, 0, 256, [1, 2, 4, 8, 16, 32, 64, 128, 256]),
    (3, 0, 100, [3, 6, 12, 24, 48, 96, 100]),
    (1, 4, 16, [1, 2, 4, 8, 12, 16]),
    (5, 0, 5, [5]),                     # first_spp = spp: one pass
    (7, 0, 7, [7]),
    (1, 0, 37, [1, 2, 4, 8, 16, 32, 37]),
    (2, 3, 11, [2, 4, 7, 10, 11]),
])
def test_schedule(pt, first_spp, max_pass_spp, spp, want):
    s, cs = _tiny_scene(pt)
    st = s.render_settings(width=16, height=16, spp=spp, max_depth=2, seed=1)
    shown, _, u32, n, stats = _progressive(cs, s, st, first_spp=first_spp, max_pass_spp=max_pass_spp)
    assert want == _schedule(first_spp, max_pass_spp, spp)
    assert [(k, m) for k, m, _ in shown] == list(enumerate(want))
    assert n == spp and stats.paths == 16 * 16 * spp


@pytest.mark.parametrize("stop_at", [0, 2])
def test_stop(pt, stop_at):
    s, base, _ = _case(pt, "cornell")
    base = dict(base, spp=32)
    cs = s.to_core().commit(0)
    st = s.render_settings(**base)
    ns = _schedule(1, 0, 32)
    shown, rgb, u32, n, stats = _progressive(cs, s, st, stop_at=stop_at, first_spp=1)
    assert len(shown) == stop_at + 1 and n == ns[stop_at]
    at_n = s.render_settings(**dict(base, spp=n))
    ref_rgb, _ = cs.render(s.camera, at_n)
    ref_u32, _ = cs.render_u32(s.camera, at_n)
    assert np.array_equal(_bits(rgb), _bits(ref_rgb)) and np.array_equal(u32, ref_u32)
    # every pass rendered counts, the one in flight at the stop (finished and discarded) included
    assert stats.paths in (64 * 48 * ns[stop_at], 64 * 48 * ns[stop_at + 1]), stats.paths

    # the scene is as it was: a render equals a fresh scene's, and a second progressive call shows the same previews
    after, _ = cs.render_u32(s.camera, st)
    fresh, _ = s.to_core().commit(0).render_u32(s.camera, st)
    assert np.array_equal(after, fresh)
    again, _, u32_full, n_full, _ = _progressive(cs, s, st, first_spp=1)
    assert n_full == 32 and np.array_equal(u32_full, fresh)
    for (k, m, img), (k2, m2, img2) in zip(shown, again):
        assert (k, m) == (k2, m2) and np.array_equal(img, img2)


def test_callback_runs_on_the_calling_thread(pt):
    s, cs = _tiny_scene(pt)
    idents = []
    cs.render_progressive(s.camera, s.render_settings(width=32, height=32, spp=16, max_depth=4),
                          on_preview=lambda k, n, img: idents.append(threading.get_ident()))
    assert len(idents) == 5 and set(idents) == {threading.get_ident()}


def test_device_renders_while_the_callback_runs(pt):
    # pass 1 (samples [128, 256) of C4's frame) renders while callback 0 sleeps, so callback 1 follows at once
    s = pt.load_scene_from_json(os.path.join(SCENES, "veach-mis", "scene.json"))
    cs = s.to_core().commit(0)
    st = s.render_settings(spp=512, seed=2)
    _, one_pass = cs.render_u32(s.camera, s.render_settings(spp=128, seed=2))
    assert one_pass.render_ms > 10.0, one_pass.render_ms  # (else the test would not show anything)
    times = []

    def cb(k, n, img):
        times.append(("enter", k, time.perf_counter()))
        if k == 0:
            time.sleep(0.3)
        times.append(("leave", k, time.perf_counter()))
        return k == 1

    _, _, n, stats = cs.render_progressive(s.camera, st, first_spp=128, on_preview=cb)
    assert n == 256 and [(e, k) for e, k, _ in times] == [("enter", 0), ("leave", 0), ("enter", 1), ("leave", 1)]
    gap_ms = (times[2][2] - times[1][2]) * 1e3
    assert gap_ms < 5.0, (gap_ms, one_pass.render_ms)


def test_exception_in_the_callback_propagates(pt):
    s, base, _ = _case(pt, "cornell")
    cs = s.to_core().commit(0)
    st = s.render_settings(**base)
    before, _ = cs.render_u32(s.camera, st)
    calls = []

    def cb(k, n, img):
        calls.append(k)
        if k == 1:
            raise ValueError("preview window closed")

    with pytest.raises(ValueError, match="preview window closed"):
        cs.render_progressive(s.camera, st, on_preview=cb)
    assert calls == [0, 1]
    after, _ = cs.render_u32(s.camera, st)
    assert np.array_equal(before, after)
    _, _, u32, n, _ = _progressive(cs, s, st)
    assert n == st.spp and np.array_equal(u32, before)


def test_pool_size_repetition_and_no_callback(pt):
    s, base, _ = _case(pt, "semesterbild")
    cs = s.to_core().commit(0)
    st = s.render_settings(**base)
    a = _progressive(cs, s, st, first_spp=1)
    b = _progressive(cs, s, st, first_spp=1)
    c = _progressive(cs, s, s.render_settings(**dict(base, pool_paths=4096)), first_spp=1)
    for x in (b, c):
        assert [(k, m) for k, m, _ in x[0]] == [(k, m) for k, m, _ in a[0]]
        for (_, _, img), (_, _, img2) in zip(a[0], x[0]):
            assert np.array_equal(img, img2)
        assert np.array_equal(_bits(x[1]), _bits(a[1])) and np.array_equal(x[2], a[2])
        assert x[4].paths == a[4].paths and x[4].rays == a[4].rays

    rgb, u32, n, stats = cs.render_progressive(s.camera, st, first_spp=1)  # no callback: the passes run back to back
    ref_rgb, _ = cs.render(s.camera, st)
    ref_u32, _ = cs.render_u32(s.camera, st)
    assert n == st.spp and np.array_equal(_bits(rgb), _bits(ref_rgb)) and np.array_equal(u32, ref_u32)

    # every output may be NULL: the call still runs every pass and fills the stats
    stats = pt.Stats()
    pg = pt.ProgressiveSettings(1, 0)
    rc = pt.core().ptc_render_progressive(cs._h, C.byref(s.camera), C.byref(st), C.byref(pg), pt.PREVIEW_FN(), None, None, None,
                                          None, C.byref(stats))
    assert rc == 0, pt.core().ptc_last_error()
    assert stats.paths == a[4].paths and stats.render_ms > 0
