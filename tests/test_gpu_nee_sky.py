"""The HDR sky as a light in next-event estimation (PTC_FLAG_NEE_SKY) on the B200.  Like PTC_FLAG_NEE it must change
how fast a render converges, never what it converges to:

  * the device's sky_sample / sky_pdf are the host build's (tests/hostsim/skysim.cpp), on the teapot envmap and a random sky;
  * without an HDR sky (or with an all-zero one) the flag changes nothing, bit for bit; without PTC_FLAG_NEE it is refused;
  * furnace under a constant HDR sky: the sphere's mean is the plain render's (and exactly the sky for albedo-1 diffuse);
  * a "sun" sky with one analytic light as well: unbiased against a plain render of 16x the samples, and at equal spp
    less than half the error of PTC_FLAG_NEE alone;
  * the reference's teapot scene (C3s, shrunk) against the oracle, which renders it with the reference's own RNG;
  * deterministic, pool- and shard-invariant, and the same image through ptc_multi_render.
"""
import os

import numpy as np
import pytest

from bindings import RNG_CHACHA, OracleScene
from test_nee_sky_host import ENVMAP, SimSky, _random_sky

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCENES = os.path.join(ROOT, "scenes")


def relmse(a, b):
    return float(np.mean((a - b) ** 2 / (b ** 2 + 1e-2)))


def blocks(img, k=8):
    h, w, _ = img.shape
    return img[:h // k * k, :w // k * k].reshape(h // k, k, w // k, k, 3).mean(axis=(1, 3))


def assert_unbiased(img, ref, p99=0.15):
    """the bounds of the PTC_FLAG_NEE tests: per-channel means within 1 %, 8x8 block means within 2 % (median) / 15 % (p99)"""
    for c in range(3):
        assert abs(img[..., c].mean() - ref[..., c].mean()) <= 0.01 * ref[..., c].mean(), (c, img[..., c].mean(), ref[..., c].mean())
    bi, br = blocks(img), blocks(ref)
    rel = np.abs(bi - br) / (br + 1e-2)
    assert np.median(rel) < 0.02 and np.percentile(rel, 99) < p99, (np.median(rel), np.percentile(rel, 99))


def flags_sky(pt):
    return pt.FLAG_NEE | pt.FLAG_NEE_SKY


@pytest.mark.parametrize("which", ["envmap", "random32x16"])
def test_hooks_match_hostsim(pt, which):
    kw = dict(hdr_file=ENVMAP) if which == "envmap" else dict(sky=_random_sky(16, 32, 1))
    sim = SimSky(pt, **kw)
    cs = sim.scene.to_core().commit(0)
    n = 1 << 18
    u4 = np.random.default_rng(11).random((n, 4), dtype=np.float32)
    d_dev, p_dev, c_dev = cs.sky_sample(u4)
    d_sim, p_sim, c_sim = sim.sample(u4)
    # the pdf is table arithmetic only: bit for bit.  Directions go through sin / cos, whose CUDA and glibc versions
    # differ in the last bits (as in check_scatter_all_materials), so they agree to a few ulps, and the radiance and
    # pdf looked up along them agree except where such a direction sits on a cell border.
    assert np.array_equal(p_dev, p_sim)
    np.testing.assert_allclose(d_dev, d_sim, rtol=0, atol=2e-6)
    assert np.mean(np.all(c_dev == c_sim, axis=1)) >= 0.9999
    dirs = np.random.default_rng(12).normal(size=(n, 3)).astype(np.float32)
    assert np.mean(cs.sky_pdf(dirs) == sim.pdf(dirs)) >= 0.9999
    assert np.mean(cs.sky_pdf(d_sim) == sim.pdf(d_sim)) >= 0.9999


def test_hooks_need_a_sky_distribution(pt):
    for sky in (None, np.zeros((4, 8, 3), np.float32)):
        s = pt.Scene()
        s.add_sphere((0, 0, 0), 1.0, s.add_material(pt.lambertian((0.5, 0.5, 0.5))))
        if sky is not None:
            s.set_sky(sky)
        cs = s.to_core().commit(0)
        for call in (lambda: cs.sky_sample(np.zeros((4, 4), np.float32)), lambda: cs.sky_pdf(np.ones((4, 3), np.float32))):
            with pytest.raises(pt.PtcError) as e:
                call()
            assert e.value.code == pt.PTC_E_STATE


@pytest.mark.parametrize("name,w,h,depth", [("cornell-box/scene.json", 96, 96, 8), ("semesterbild.json", 160, 120, 30)])
def test_flag_changes_nothing_without_a_sky(pt, name, w, h, depth):
    s = pt.load_scene_from_json(os.path.join(SCENES, name))
    cs = s.to_core().commit(0)
    base = dict(width=w, height=h, spp=8, max_depth=depth, seed=5)
    a, sa = cs.render(s.camera, s.render_settings(flags=pt.FLAG_NEE, **base))
    b, sb = cs.render(s.camera, s.render_settings(flags=flags_sky(pt), **base))
    assert np.array_equal(a, b) and sa.rays == sb.rays
    with pytest.raises(pt.PtcError) as e:
        cs.render(s.camera, s.render_settings(flags=pt.FLAG_NEE_SKY, **base))
    assert e.value.code == pt.PTC_E_INVALID


def test_flag_changes_nothing_under_an_all_zero_sky(pt):
    s = pt.Scene()
    s.add_sphere((0, 0, 0), 1.0, s.add_material(pt.lambertian((0.7, 0.7, 0.7))))
    s.add_sphere((0, 3, 0), 0.5, s.add_material(pt.emissive((5, 5, 5))))
    s.set_sky(np.zeros((8, 16, 3), np.float32))
    s.set_camera((0, 1, 6), (0, 0.5, 0), (0, 1, 0), 40.0, 1.0)
    cs = s.to_core().commit(0)
    base = dict(width=64, height=64, spp=16, max_depth=8, seed=3)
    a, sa = cs.render(s.camera, s.render_settings(flags=pt.FLAG_NEE, **base))
    b, sb = cs.render(s.camera, s.render_settings(flags=flags_sky(pt), **base))
    assert np.array_equal(a, b) and sa.rays == sb.rays


@pytest.mark.parametrize("which", ["lambert", "checker", "plastic", "ggx", "beckmann"])
def test_furnace_under_constant_hdr_sky(pt, which):
    mats = {"lambert": pt.lambertian((1, 1, 1)), "checker": pt.checker((1, 1, 1), (1, 1, 1), 0.5), "plastic": pt.plastic((1, 1, 1), 1.5),
            "ggx": pt.rough_conductor((1, 1, 1), 0.3, "al", pt.DIST_GGX), "beckmann": pt.rough_conductor((1, 1, 1), 0.25, "cu", pt.DIST_BECKMANN)}
    s = pt.Scene()
    s.add_sphere((0, 0, 0), 1.0, s.add_material(mats[which]))
    s.set_sky(np.full((4, 8, 3), 0.5, np.float32))
    s.set_camera((0, 0, 4), (0, 0, 0), (0, 1, 0), 30.0, 1.0)
    cs = s.to_core().commit(0)
    w = h = 64
    base = dict(width=w, height=h, spp=1024, max_depth=64)
    plain, _ = cs.render(s.camera, s.render_settings(seed=1, **base))
    sky, _ = cs.render(s.camera, s.render_settings(seed=2, flags=flags_sky(pt), **base))
    yy, xx = np.mgrid[0:h, 0:w]
    on_sphere = ((xx - w / 2 + 0.5) ** 2 + (yy - h / 2 + 0.5) ** 2) < (0.8 * w / 2 * np.tan(np.arcsin(1 / 4)) / np.tan(np.radians(15))) ** 2
    gm, pm = sky[on_sphere].mean(), plain[on_sphere].mean()
    assert abs(gm - pm) <= 0.005 * pm, (which, gm, pm)
    if which in ("lambert", "checker"):
        assert abs(gm - 0.5) < 1e-3, gm  # KA5: energy conserving -> the sky itself


def _sun_scene(pt):
    sky = np.full((32, 64, 3), (0.25, 0.3, 0.4), np.float32)
    sky[8:10, 40:42] = (30.0, 28.0, 24.0)  # ~100x the rest: a "sun" 2 x 2 texels wide, above the horizon
    s = pt.Scene()
    floor = s.add_material(pt.lambertian((0.6, 0.6, 0.6)))
    s.add_quad(floor, scale=(40, 1, 40), rotation=(0, 0, 180), position=(0, 0, 0))
    s.add_sphere((-2.2, 1.0, 0.0), 1.0, s.add_material(pt.plastic((0.2, 0.5, 0.8), 1.5)))
    s.add_sphere((0.0, 1.0, 0.0), 1.0, s.add_material(pt.rough_conductor((1, 1, 1), 0.3, "au", pt.DIST_GGX)))
    s.add_sphere((2.2, 1.0, 0.0), 1.0, s.add_material(pt.lambertian((0.7, 0.3, 0.3))))
    s.add_sphere((1.0, 4.0, 2.0), 0.3, s.add_material(pt.emissive((40, 30, 20))))  # one analytic light as well
    s.set_sky(sky)
    s.set_camera((0, 3, 8), (0, 0.8, 0), (0, 1, 0), 40.0, 2.0)
    return s


def test_sun_sky_unbiased_and_converges_faster(pt):
    s = _sun_scene(pt)
    cs = s.to_core().commit(0)
    base = dict(width=128, height=64, max_depth=8)
    ref, _ = cs.render(s.camera, s.render_settings(spp=16384, seed=1, **base))  # plain, converged
    hi, _ = cs.render(s.camera, s.render_settings(spp=1024, seed=3, flags=flags_sky(pt), **base))
    assert_unbiased(hi, ref)
    nee, ns = cs.render(s.camera, s.render_settings(spp=64, seed=2, flags=pt.FLAG_NEE, **base))
    sky, ss = cs.render(s.camera, s.render_settings(spp=64, seed=2, flags=flags_sky(pt), **base))
    assert ss.paths == ns.paths
    e_nee, e_sky = relmse(nee, ref), relmse(sky, ref)
    assert e_sky < 0.5 * e_nee, (e_sky, e_nee)


def _teapot(pt):
    return pt.load_scene_from_json(os.path.join(SCENES, "teapot", "scene.json"), pt.LOAD_INFINITE_SPHERE_SKY | pt.LOAD_WO3_STRIDE16)


def test_c3s_against_the_oracle(pt):
    s = _teapot(pt)
    w, h, depth = 128, 72, 64
    ref, _ = OracleScene(s).render(s.camera, w, h, 4096, depth, rng_mode=RNG_CHACHA, seed=1)
    cs = s.to_core().commit(0)
    base = dict(width=w, height=h, max_depth=depth, spp=256, seed=2)
    sky, _ = cs.render(s.camera, s.render_settings(flags=flags_sky(pt), **base))
    assert_unbiased(sky, ref)
    nee, _ = cs.render(s.camera, s.render_settings(flags=pt.FLAG_NEE, **base))
    plain, _ = cs.render(s.camera, s.render_settings(**base))
    assert np.array_equal(nee, plain)  # no analytic emitter in this scene: NEE alone is the plain integrator
    assert relmse(sky, ref) < relmse(nee, ref), (relmse(sky, ref), relmse(nee, ref))


def test_deterministic_and_shard_invariant(pt):
    s = _sun_scene(pt)
    cs = s.to_core().commit(0)
    base = dict(width=100, height=70, spp=6, max_depth=8, seed=4, flags=flags_sky(pt))
    whole, st = cs.render(s.camera, s.render_settings(**base))
    again, _ = cs.render(s.camera, s.render_settings(**base))
    assert np.array_equal(again, whole)
    small, _ = cs.render(s.camera, s.render_settings(pool_paths=2048, **base))
    assert np.array_equal(small, whole)
    by_sample = sum(cs.render(s.camera, s.render_settings(sample_begin=b, sample_end=e, **base))[0] for b, e in [(0, 1), (1, 4), (4, 6)])
    assert np.allclose(by_sample, whole, rtol=1e-5, atol=1e-6)


def test_multi_gpu_matches_one_gpu(pt):
    if pt.device_count() < 2:
        pytest.skip("needs 2 or more GPUs")
    s = _teapot(pt)
    cs = s.to_core().commit(0)
    st = s.render_settings(width=128, height=72, spp=8, max_depth=16, seed=6, flags=flags_sky(pt))
    one, s1 = cs.render(s.camera, st)
    m = cs.multi(list(range(pt.device_count())))
    for shard in (pt.SHARD_SAMPLES, pt.SHARD_TILES):
        img, sm = m.render(s.camera, st, shard)
        assert np.array_equal(img, one) and sm.rays == s1.rays
