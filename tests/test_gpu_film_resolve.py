"""Every render that returns an image resolves the scene's fixed-point film in one kernel (k_resolve_film).  Its images
must be, bit for bit, what the device-resident route gives: ptc_render_accumulate's fp32 film x the float32 1 / spp
for ptc_render, and ptc_resolve_device of that film for ptc_render_u32 — also for a sample sub-range, which still
divides by spp, and through ptc_multi_* on one device.  Cases: the Cornell box, the shipped teapot (C3s, shrunk) with
PTC_FLAG_NEE | PTC_FLAG_NEE_SKY, emitters beyond the fixed-point range (+inf in the film), and a 1920x1088 frame, whose
rgb image (25 MB) takes the pinned staging copy to the host.
"""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCENES = os.path.join(ROOT, "scenes")


def _case(pt, name):
    """-> (scene, render-settings keywords)"""
    if name == "cornell":
        s = pt.load_scene_from_json(os.path.join(SCENES, "cornell-box", "scene.json"))
        return s, dict(width=100, height=70, spp=8, max_depth=8, seed=3)
    if name == "teapot":
        s = pt.load_scene_from_json(os.path.join(SCENES, "teapot", "scene.json"), pt.LOAD_INFINITE_SPHERE_SKY | pt.LOAD_WO3_STRIDE16)
        return s, dict(width=128, height=72, spp=8, max_depth=16, seed=5, flags=pt.FLAG_NEE | pt.FLAG_NEE_SKY)
    if name == "full-hd":
        s = pt.load_scene_from_json(os.path.join(SCENES, "cornell-box", "scene.json"))
        return s, dict(width=1920, height=1088, spp=2, max_depth=3, seed=1)
    # test_gpu_render.py::test_film_nan_and_inf_survive_the_fixed_point_film: radiance beyond the film's range
    s = pt.Scene()
    m = s.add_material(pt.emissive((3e7 if name == "emitter-3e7" else float("inf"), 1.0, 0.0)))
    s.add_sphere((0, 0, 0), 1.0, m)
    s.set_camera((0, 0, 4), (0, 0, 0), (0, 1, 0), 30.0, 1.0)
    return s, dict(width=16, height=16, spp=8, max_depth=3)


def _film(cs, s, st):
    """ptc_render_accumulate into a zeroed device film -> (torch film, numpy [H, W, 3])"""
    torch = pytest.importorskip("torch")
    acc = torch.zeros(st.width * st.height * 3, dtype=torch.float32, device="cuda:0")
    cs.render_accumulate(s.camera, st, acc.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return acc, acc.cpu().numpy().reshape(st.height, st.width, 3)


def _resolve_device(pt, acc, n_px, scale):
    torch = pytest.importorskip("torch")
    out = torch.zeros(n_px, dtype=torch.int32, device="cuda:0")
    assert pt.core().ptc_resolve_device(acc.data_ptr(), n_px, float(scale), out.data_ptr(), torch.cuda.current_stream().cuda_stream) == 0
    torch.cuda.synchronize()
    return out.cpu().numpy().view(np.uint32)


@pytest.mark.parametrize("name", ["cornell", "teapot", "emitter-3e7", "emitter-inf", "full-hd"])
def test_images_are_the_accumulated_film_resolved(pt, name):
    s, base = _case(pt, name)
    cs = s.to_core().commit(0)
    m = cs.multi([0])
    ranges = [{}] if name == "full-hd" else [{}, dict(sample_begin=2, sample_end=5)]  # [2, 5) of spp 8: still x 1/8
    for extra in ranges:
        st = s.render_settings(**base, **extra)
        acc, film = _film(cs, s, st)
        scale = np.float32(1) / np.float32(st.spp)  # what the library computes, in float32
        rgb, a = cs.render(s.camera, st)
        assert np.array_equal(rgb, film * scale, equal_nan=True)
        packed, b = cs.render_u32(s.camera, st)
        assert np.array_equal(packed, _resolve_device(pt, acc, st.width * st.height, scale))
        assert a.paths == b.paths > 0 and a.rays == b.rays
        for shard in (pt.SHARD_SAMPLES, pt.SHARD_TILES):
            m_rgb, ms = m.render(s.camera, st, shard)
            assert np.array_equal(m_rgb, rgb, equal_nan=True) and ms.rays == a.rays
            m_packed, _ = m.render_u32(s.camera, st, shard)
            assert np.array_equal(m_packed, packed)
    if name.startswith("emitter"):
        assert np.isposinf(rgb[8, 8, 0]) and (packed[8 * 16 + 8] >> 16) == 255


def test_oversized_multi_render_is_refused_before_any_film_is_allocated(pt):
    torch = pytest.importorskip("torch")
    s, _ = _case(pt, "cornell")
    cs = s.to_core().commit(0)
    m = cs.multi([0])
    st = s.render_settings(width=32768, height=32768, spp=1, max_depth=1)  # 2^30 pixels, one over the limit
    torch.cuda.synchronize()
    free_before, _ = torch.cuda.mem_get_info(0)
    with pytest.raises(pt.PtcError) as e:
        m.render_u32(s.camera, st)  # a full-size host buffer (np.empty: no page is touched unless written)
    free_after, _ = torch.cuda.mem_get_info(0)
    assert e.value.code == pt.PTC_E_INVALID and "image too large" in str(e.value)
    # this image's film alone would take 32 GiB of the device; free memory is read device-wide, so other processes may
    # move it, but not by half the film within a call that returns at once
    assert free_before - free_after < (16 << 30)
