"""Adaptive sampling (ptc_render_adaptive) on the B200.

Philox is keyed on the global (pixel, sample) and the film sums are fixed-point, so a pixel that received samples [0, n)
over several passes holds exactly the film of a uniform render at n spp.  Hence, on the Cornell box (PTC_FLAG_NEE), a
shrunk teapot (C3s, PTC_FLAG_NEE | PTC_FLAG_NEE_SKY) and a shrunk semesterbild (plain):
  * the count of every pixel is predicted exactly by the host build of the decision (tests/hostsim/adaptsim.cpp) fed
    with the films of uniform renders at every n of the schedule;
  * every pixel's rgb and packed value are those of the uniform render at its count, bit for bit;
  * threshold 0 is the uniform render at spp, +inf the uniform render at min_spp, and so is min_spp = spp;
  * pixels whose whole 3x3 neighbourhood sees only the constant background stop at min_spp;
  * on a half-background, half-lit scene adaptive beats uniform sampling of the same total paths, and stays unbiased;
  * deterministic and independent of the pool size.
"""
import os

import numpy as np
import pytest

from test_adaptive_host import np_needs_more, sim_step

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCENES = os.path.join(ROOT, "scenes")


def _case(pt, name):
    """-> (scene, render-settings keywords, min_spp)"""
    if name == "cornell":
        s = pt.load_scene_from_json(os.path.join(SCENES, "cornell-box", "scene.json"))
        return s, dict(width=64, height=64, spp=64, max_depth=8, seed=3, flags=pt.FLAG_NEE), 4
    if name == "teapot":
        s = pt.load_scene_from_json(os.path.join(SCENES, "teapot", "scene.json"), pt.LOAD_INFINITE_SPHERE_SKY | pt.LOAD_WO3_STRIDE16)
        return s, dict(width=128, height=72, spp=32, max_depth=16, seed=5, flags=pt.FLAG_NEE | pt.FLAG_NEE_SKY), 4
    s = pt.load_scene_from_json(os.path.join(SCENES, "semesterbild.json"))
    return s, dict(width=160, height=120, spp=64, max_depth=30, seed=7), 2


_committed = {}


def _commit(pt, name):
    if name not in _committed:
        s, base, min_spp = _case(pt, name)
        _committed[name] = (s, s.to_core().commit(0), base, min_spp)
    return _committed[name]


def _film(cs, s, base, n):
    """fp32 film sums of samples [0, n) (what k_film_to_accum leaves in a zeroed film), W*H x 3"""
    torch = pytest.importorskip("torch")
    acc = torch.zeros(base["width"] * base["height"] * 3, dtype=torch.float32, device="cuda:0")
    cs.render_accumulate(s.camera, s.render_settings(**dict(base, spp=n, sample_begin=0, sample_end=n)), acc.data_ptr(),
                         torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return acc.cpu().numpy().reshape(-1, 3)


def _schedule(min_spp, spp):
    ns = [min_spp // 2, min_spp]
    while ns[-1] < spp:
        ns.append(min(2 * ns[-1], spp))
    return ns


def _median_error_threshold(V, Vp, n, m):
    """a threshold in the middle of the first decision's errors, so that pixels both stop and go on"""
    with np.errstate(all="ignore"):
        I, A = V / np.float32(n), (V - Vp) / np.float32(n - m)
        e = np.abs(I - A).sum(1) / (np.float32(1e-4) + np.sqrt(I.sum(1)))
    return float(np.median(e[np.isfinite(e)]))


@pytest.mark.parametrize("name", ["cornell", "teapot", "semesterbild"])
def test_counts_predicted_and_pixels_are_uniform_renders(pt, name):
    s, cs, base, min_spp = _commit(pt, name)
    w, h, spp = base["width"], base["height"], base["spp"]
    ns = _schedule(min_spp, spp)
    films = {n: _film(cs, s, base, n) for n in ns}
    thr = _median_error_threshold(films[ns[1]], films[ns[0]], ns[1], ns[0])
    assert np_needs_more(films[ns[1]], films[ns[0]], ns[1], ns[0], thr).any()

    # the host build of the decision, fed with the uniform films
    needs = np.zeros(w * h, np.uint8)
    counts = np.full(w * h, spp, np.int32)
    active = np.arange(w * h, dtype=np.uint32)
    for k in range(1, len(ns) - 1):
        active = sim_step(w, h, films[ns[k]], films[ns[k - 1]], active, ns[k], ns[k - 1], thr, needs, counts)
        if len(active) == 0:
            break

    rgb, u32, got, st = cs.render_adaptive(s.camera, s.render_settings(**base), min_spp, thr)
    assert np.array_equal(got.reshape(-1), counts)
    assert st.paths == int(counts.sum())
    distinct = np.unique(counts)
    assert len(distinct) >= 2, distinct  # the threshold splits the frame
    for n in distinct:
        sel = got == n
        ref, _ = cs.render(s.camera, s.render_settings(**dict(base, spp=int(n))))
        ref_u32, _ = cs.render_u32(s.camera, s.render_settings(**dict(base, spp=int(n))))
        assert np.array_equal(rgb[sel], ref[sel]), n
        assert np.array_equal(u32.reshape(h, w)[sel], ref_u32.reshape(h, w)[sel]), n


@pytest.mark.parametrize("name", ["cornell", "teapot"])
def test_limits(pt, name):
    s, cs, base, min_spp = _commit(pt, name)
    st = s.render_settings(**base)
    spp = base["spp"]
    uni, _ = cs.render(s.camera, st)
    uni_u32, _ = cs.render_u32(s.camera, st)
    rgb, u32, cnt, stats = cs.render_adaptive(s.camera, st, min_spp, 0.0)
    assert np.all(cnt == spp) and stats.paths == spp * cnt.size
    assert np.array_equal(rgb, uni) and np.array_equal(u32, uni_u32)

    lo = s.render_settings(**dict(base, spp=min_spp))
    uni_lo, _ = cs.render(s.camera, lo)
    uni_lo_u32, _ = cs.render_u32(s.camera, lo)
    rgb, u32, cnt, stats = cs.render_adaptive(s.camera, st, min_spp, float("inf"))
    assert np.all(cnt == min_spp) and stats.paths == min_spp * cnt.size
    assert np.array_equal(rgb, uni_lo) and np.array_equal(u32, uni_lo_u32)

    rgb, u32, cnt, _ = cs.render_adaptive(s.camera, lo, min_spp, 0.5)  # min_spp = spp
    assert np.all(cnt == min_spp)
    assert np.array_equal(rgb, uni_lo) and np.array_equal(u32, uni_lo_u32)


def test_zero_variance_background_stops_at_min_spp(pt):
    s, cs, base, _ = _commit(pt, "semesterbild")
    w, h, spp, min_spp = base["width"], base["height"], base["spp"], 4
    st = s.render_settings(**base)
    bg = np.ones(w * h, bool)  # every sample's primary ray misses: the constant gray background, nothing else
    for k in range(spp):
        o, d = cs.primary_rays(s.camera, st, k)
        hits, _ = cs.intersect(o, d)
        bg &= hits["object"] < 0
    pad = np.zeros((h + 2, w + 2), bool)
    pad[1:-1, 1:-1] = bg.reshape(h, w)
    quiet = np.ones((h, w), bool)
    for dy in range(3):
        for dx in range(3):
            quiet &= pad[dy:dy + h, dx:dx + w]
    assert quiet.sum() > 100, quiet.sum()
    _, _, cnt, _ = cs.render_adaptive(s.camera, st, min_spp, 1e-3)
    assert np.all(cnt[quiet] == min_spp)
    assert cnt[~quiet].max() > min_spp


def _half_lit_scene(pt):
    """left: the constant gray background; right: a diffuse and a glossy (plastic) sphere under a small bright light"""
    s = pt.Scene()
    s.add_sphere((1.2, 0.0, -4.0), 1.5, s.add_material(pt.lambertian((0.7, 0.6, 0.5))))
    s.add_sphere((0.55, -0.75, -2.8), 0.4, s.add_material(pt.plastic((0.3, 0.4, 0.8))))
    s.add_sphere((0.4, 1.6, -2.5), 0.25, s.add_material(pt.emissive((30.0, 28.0, 24.0))))
    s.set_camera((0, 0, 0), (0, 0, -1), (0, 1, 0), 40.0, 1.0)
    s.set_settings(128, 128, 256, 8)
    return s


def _unbiased(img, ref):
    """the bounds of the PTC_FLAG_NEE tests: per-channel means within 1 %, 8x8 block means within 2 % (median)"""
    for c in range(3):
        assert abs(img[..., c].mean() - ref[..., c].mean()) <= 0.01 * ref[..., c].mean(), (c, img[..., c].mean(), ref[..., c].mean())
    h, w, _ = img.shape
    bi = img.reshape(h // 8, 8, w // 8, 8, 3).mean(axis=(1, 3))
    br = ref.reshape(h // 8, 8, w // 8, 8, 3).mean(axis=(1, 3))
    assert np.median(np.abs(bi - br) / (br + 1e-2)) < 0.02


def test_beats_uniform_at_equal_paths(pt):
    # With NEE, as adaptive sampling is meant to be used: without it a pixel whose first samples all missed the small
    # light looks converged and stops early, which darkens the lit region (DESIGN.md 5f).
    s = _half_lit_scene(pt)
    cs = s.to_core().commit(0)
    ref, _ = cs.render(s.camera, s.render_settings(spp=8192, seed=1))  # plain
    rgb, _, cnt, st = cs.render_adaptive(s.camera, s.render_settings(seed=2, flags=pt.FLAG_NEE), 16, 0.02)
    uni_spp = -(-int(st.paths) // cnt.size)  # uniform gets at least as many paths
    uni, ust = cs.render(s.camera, s.render_settings(spp=uni_spp, seed=2, flags=pt.FLAG_NEE))
    assert ust.paths >= st.paths
    relmse = lambda a: float(np.mean((a - ref) ** 2 / (ref ** 2 + 1e-2)))  # noqa: E731
    assert relmse(rgb) < relmse(uni), (relmse(rgb), relmse(uni), uni_spp, np.unique(cnt, return_counts=True))
    _unbiased(rgb, ref)


def test_deterministic_and_pool_invariant(pt):
    s, cs, base, min_spp = _commit(pt, "cornell")
    st = s.render_settings(**base)
    a = cs.render_adaptive(s.camera, st, min_spp, 0.05)
    b = cs.render_adaptive(s.camera, st, min_spp, 0.05)
    c = cs.render_adaptive(s.camera, s.render_settings(**dict(base, pool_paths=4096)), min_spp, 0.05)
    assert len(np.unique(a[2])) >= 2
    for x in (b, c):
        for k in range(3):
            assert np.array_equal(a[k], x[k]), k
        assert x[3].paths == a[3].paths and x[3].rays == a[3].rays


@pytest.mark.parametrize("min_spp", [64, 4])  # min_spp = spp: the last work queued is k_adapt_init, not a render pass
def test_stats_only_call_without_outputs(pt, min_spp):
    # every output may be NULL: the call still returns once its work (and the render_ms event) is done
    import ctypes as C
    s, cs, base, _ = _commit(pt, "cornell")
    st = s.render_settings(**base)
    *_, want = cs.render_adaptive(s.camera, st, min_spp, 0.05)
    stats = pt.Stats()
    ad = pt.Adaptive(min_spp, 0.05)
    rc = pt.core().ptc_render_adaptive(cs._h, C.byref(s.camera), C.byref(st), C.byref(ad), None, None, None, C.byref(stats))
    assert rc == 0, pt.core().ptc_last_error()
    assert stats.paths == want.paths and stats.render_ms > 0
