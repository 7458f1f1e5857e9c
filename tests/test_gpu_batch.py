"""Batch rendering (ptc_render_batch, ptc_render_batch_accumulate) on the B200.

Philox is keyed on (seed of the view, pixel within the view, sample) and the film sums are fixed-point, so view k of a
batch is, bit for bit, the single render of camera k with seed k.  Exactly (rgb compared as uint32 bit patterns, so NaN
and inf count):
  * every view equals render / render_u32 of its camera and seed, and the batch's paths and rays are the sums of the
    single renders — on the cases of test_gpu_progressive.py: the Cornell box, a shrunk semesterbild (mesh, depth 30),
    a shrunk teapot (C3s, NEE | NEE_SKY), a shrunk veach-mis (NEE), emitters beyond the fixed-point range, max_depth 0;
    five views each, moved by distinct offsets, one of them looking away from the scene;
  * edge shapes: one view, a 45 x 29 frame of seven views, no seeds, a sample sub-range;
  * jobs many times the pool (the host's drain bound), for a batch and for a single render;
  * the device route equals render_accumulate per view; repeated batches are identical.
"""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCENES = os.path.join(ROOT, "scenes")
CASES = ["cornell", "semesterbild", "teapot", "veach-mis", "emitter-3e7", "emitter-inf", "depth-0"]


def _case(pt, name):
    """-> (scene, render-settings keywords), as test_gpu_progressive.py's cases"""
    if name in ("cornell", "depth-0"):
        s = pt.load_scene_from_json(os.path.join(SCENES, "cornell-box", "scene.json"))
        return s, dict(width=64, height=48, spp=12, max_depth=0 if name == "depth-0" else 8, seed=3)
    if name == "semesterbild":
        return pt.load_scene_from_json(os.path.join(SCENES, "semesterbild.json")), dict(width=96, height=72, spp=10, max_depth=30, seed=7)
    if name == "teapot":
        s = pt.load_scene_from_json(os.path.join(SCENES, "teapot", "scene.json"), pt.LOAD_INFINITE_SPHERE_SKY | pt.LOAD_WO3_STRIDE16)
        return s, dict(width=128, height=72, spp=8, max_depth=16, seed=5, flags=pt.FLAG_NEE | pt.FLAG_NEE_SKY)
    if name == "veach-mis":
        s = pt.load_scene_from_json(os.path.join(SCENES, "veach-mis", "scene.json"))
        return s, dict(width=160, height=90, spp=16, max_depth=16, seed=11, flags=pt.FLAG_NEE)
    s = pt.Scene()
    m = s.add_material(pt.emissive((3e7 if name == "emitter-3e7" else float("inf"), 1.0, 0.0)))
    s.add_sphere((0, 0, 0), 1.0, m)
    s.set_camera((0, 0, 4), (0, 0, 0), (0, 1, 0), 30.0, 1.0)
    return s, dict(width=16, height=16, spp=8, max_depth=3)


def _moved(cam, right=0.0, up=0.0, look_up=False):
    """a copy of cam moved along its own right / up axes (scene units scaled by the distance from the origin); look_up:
    turned 90 degrees about its right axis and lifted far above, so that it sees nothing of the scene"""
    c = pt_camera_copy(cam)
    p, f, r, u = (np.array(x[:], np.float64) for x in (c.position, c.forward, c.right, c.true_up))
    scale = max(1.0, float(np.linalg.norm(p))) * 0.05
    p = p + r * right * scale + u * up * scale
    if look_up:
        p = p + u * 1e4
        f, u = u.copy(), -f
    for dst, src in ((c.position, p), (c.forward, f), (c.true_up, u)):
        for i in range(3):
            dst[i] = float(src[i])
    return c


def pt_camera_copy(cam):
    c = type(cam)()
    C.pointer(c)[0] = cam
    return c


def _views(cam, k=5):
    offsets = [(0.0, 0.0), (1.0, 0.0), (-1.0, 0.5), (0.0, -1.0), (2.0, 1.0), (-2.0, -1.5), (0.5, 2.0)]
    cams = [_moved(cam, *offsets[i]) for i in range(k - 1)]
    return cams + [_moved(cam, look_up=True)]


def _bits(rgb):
    return np.ascontiguousarray(rgb).view(np.uint32)


def _settings(s, base, **over):
    return s.render_settings(**dict(base, **over))


def _check_views(pt, cs, s, base, cams, seeds, rgb, u32, stats, **over):
    """every view of a batch against the single renders of its camera and seed"""
    paths = rays = 0
    for k, cam in enumerate(cams):
        st = _settings(s, base, seed=int(seeds[k]) if seeds is not None else base.get("seed", 0), **over)
        one, ost = cs.render(cam, st)
        one_u32, _ = cs.render_u32(cam, st)
        assert np.array_equal(_bits(rgb[k]), _bits(one)), f"view {k}: rgb"
        assert np.array_equal(u32[k], one_u32), f"view {k}: u32"
        paths += ost.paths
        rays += ost.rays
    assert stats.paths == paths and stats.rays == rays, (stats.paths, paths, stats.rays, rays)


@pytest.mark.parametrize("name", CASES)
def test_every_view_is_its_single_render(pt, name):
    s, base = _case(pt, name)
    cs = s.to_core().commit(0)
    cams = _views(s.camera)
    seeds = [base.get("seed", 0) + 1000 * k + 17 for k in range(len(cams))]
    rgb, u32, stats = cs.render_batch(cams, _settings(s, base), seeds)
    assert rgb.shape == (5, base["height"], base["width"], 3) and u32.shape == (5, base["height"] * base["width"])
    _check_views(pt, cs, s, base, cams, seeds, rgb, u32, stats)
    if base["max_depth"] > 0 and not name.startswith("emitter"):
        assert len({_bits(rgb[k]).tobytes() for k in range(5)}) == 5  # the views really differ


def test_one_view_is_ptc_render(pt):
    s, base = _case(pt, "cornell")
    cs = s.to_core().commit(0)
    rgb, u32, stats = cs.render_batch([s.camera], _settings(s, base), [base["seed"]])
    _check_views(pt, cs, s, base, [s.camera], [base["seed"]], rgb, u32, stats)


def test_odd_frame_of_seven_views(pt):
    s, base = _case(pt, "cornell")
    base = dict(base, width=45, height=29)
    cs = s.to_core().commit(0)
    cams = _views(s.camera, 7)
    seeds = [9 + 31 * k for k in range(7)]
    rgb, u32, stats = cs.render_batch(cams, _settings(s, base), seeds)
    _check_views(pt, cs, s, base, cams, seeds, rgb, u32, stats)


def test_no_seeds_gives_every_view_the_settings_seed(pt):
    s, base = _case(pt, "cornell")
    cs = s.to_core().commit(0)
    cams = [s.camera, _moved(s.camera, 1.0), s.camera]
    rgb, u32, stats = cs.render_batch(cams, _settings(s, base))
    assert np.array_equal(_bits(rgb[0]), _bits(rgb[2])) and np.array_equal(u32[0], u32[2])
    _check_views(pt, cs, s, base, cams, None, rgb, u32, stats)


def test_sample_range(pt):
    s, base = _case(pt, "veach-mis")
    base = dict(base, spp=8)
    cs = s.to_core().commit(0)
    cams = _views(s.camera, 3)
    seeds = [4, 5, 6]
    rgb, u32, stats = cs.render_batch(cams, _settings(s, base, sample_begin=2, sample_end=5), seeds)
    _check_views(pt, cs, s, base, cams, seeds, rgb, u32, stats, sample_begin=2, sample_end=5)


def test_batch_many_times_the_pool(pt):
    # a closed box: most paths live to max_depth, so the last paths reserved must still be traced to the end
    s, base = _case(pt, "cornell")
    base = dict(base, width=128, height=128, spp=16)
    cs = s.to_core().commit(0)
    cams = _views(s.camera, 8)[:7] + [_moved(s.camera, 0.3, 0.3)]
    seeds = [100 + k for k in range(8)]
    job = 8 * 16 * 1024 * 16
    rgb, u32, stats = cs.render_batch(cams, _settings(s, base, pool_paths=job // 16), seeds)
    assert cs.last_pool_slots() * 8 <= job, cs.last_pool_slots()
    _check_views(pt, cs, s, base, cams, seeds, rgb, u32, stats)


def test_single_render_many_times_the_pool(pt):
    s, base = _case(pt, "cornell")
    base = dict(base, width=256, height=256, spp=64)
    cs = s.to_core().commit(0)
    job = 64 * 1024 * 64
    small, sst = cs.render(s.camera, _settings(s, base, pool_paths=job // 16))
    assert cs.last_pool_slots() * 8 <= job, cs.last_pool_slots()
    full, fst = cs.render(s.camera, _settings(s, base))
    assert np.array_equal(_bits(small), _bits(full))
    assert sst.paths == fst.paths and sst.rays == fst.rays


def test_device_route_is_render_accumulate_per_view(pt):
    torch = pytest.importorskip("torch")
    s, base = _case(pt, "teapot")
    cs = s.to_core().commit(0)
    st = _settings(s, base)
    cams = _views(s.camera, 4)
    seeds = [21, 22, 23, 24]
    h, w = base["height"], base["width"]
    stream = torch.cuda.current_stream().cuda_stream
    acc = torch.zeros((4, h, w, 3), dtype=torch.float32, device="cuda:0")
    stats = cs.render_batch_accumulate(cams, st, acc.data_ptr(), stream, seeds)
    torch.cuda.synchronize()
    paths = 0
    for k in range(4):
        one = torch.zeros((h, w, 3), dtype=torch.float32, device="cuda:0")
        ost = cs.render_accumulate(cams[k], _settings(s, base, seed=seeds[k]), one.data_ptr(), stream)
        torch.cuda.synchronize()
        assert np.array_equal(_bits(acc[k].cpu().numpy()), _bits(one.cpu().numpy())), f"view {k}"
        paths += ost.paths
    assert stats.paths == paths


def test_repeated_batches_are_identical(pt):
    s, base = _case(pt, "semesterbild")
    cs = s.to_core().commit(0)
    cams = _views(s.camera)
    seeds = [1, 2, 3, 4, 5]
    a = cs.render_batch(cams, _settings(s, base), seeds)
    b = cs.render_batch(cams, _settings(s, base), seeds)
    assert np.array_equal(_bits(a[0]), _bits(b[0])) and np.array_equal(a[1], b[1])
    assert a[2].rays == b[2].rays
