"""Emissive meshes and cubes in next-event estimation, lights chosen by power (PTC_FLAG_NEE_EMITTERS), on the B200.  Like
PTC_FLAG_NEE it must change how fast a render converges, never what it converges to:

  * alone the flag is refused; on a scene without emitters it changes nothing, and on the Cornell box (one quad light)
    NEE | EMITTERS is NEE, bit for bit;
  * the device's light_sample / light_pdf are the host build's (tests/hostsim/emsim.cpp); triangles are drawn with their
    live-area proportions, dead ones never; along a visible sampled direction light_pdf is light_sample's density;
  * one light, two shapes: a quad light and the same rectangle as a 2-triangle mesh converge to one image;
  * unbiased against a plain render of 16x the samples on a scaled, rotated text sign (dead triangles, the mesh t quirk),
    a concave emissive mesh, a rotated, non-uniformly scaled cube and a mixed scene (also under a "sun" sky); there, at
    equal spp, less than half PTC_FLAG_NEE's error;
  * the same image whichever builder made the tree; no pixel made non-finite by 3e7 or +inf emitters;
  * deterministic, pool- and shard-invariant, and every render entry point gives the same image.
"""
import os

import numpy as np
import pytest

from bindings import OracleScene
from test_nee_emitters_host import TEXT_OBJ, SimEmitters, _box_mesh, mixed_scene

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


def em(pt):
    return pt.FLAG_NEE | pt.FLAG_NEE_EMITTERS


def _room(pt, closed=False):
    """an open-fronted grey box, 2 x 2 x 2, with a diffuse sphere and a plastic cube; camera in front (closed: the box goes
    on behind the camera and is shut there, so the background lights nothing, and its walls are dark, so that direct light
    dominates)"""
    s = pt.Scene()
    k = 0.25 if closed else 1.0
    grey, red, green = (s.add_material(pt.lambertian(tuple(k * x for x in c))) for c in ((0.7, 0.7, 0.7), (0.7, 0.2, 0.2), (0.2, 0.7, 0.2)))
    s.add_quad(grey, scale=(2, 1, 2), position=(0, 0, 0))
    s.add_quad(grey, scale=(2, 1, 2), rotation=(180, 0, 0), position=(0, 2, 0))
    s.add_quad(grey, scale=(2, 1, 2), rotation=(90, 0, 0), position=(0, 1, -1))
    s.add_quad(red, scale=(2, 1, 2), rotation=(0, 0, 90), position=(-1, 1, 0))
    s.add_quad(green, scale=(2, 1, 2), rotation=(0, 0, 90), position=(1, 1, 0))
    if closed:
        s.add_quad(grey, scale=(2, 1, 3), position=(0, 0, 2.5))
        s.add_quad(grey, scale=(2, 1, 3), rotation=(180, 0, 0), position=(0, 2, 2.5))
        s.add_quad(grey, scale=(2, 1, 3), rotation=(0, 0, 90), position=(-1, 1, 2.5))
        s.add_quad(grey, scale=(2, 1, 3), rotation=(0, 0, 90), position=(1, 1, 2.5))
        s.add_quad(grey, scale=(2, 1, 2), rotation=(90, 0, 0), position=(0, 1, 4))
    s.add_sphere((-0.4, 0.35, -0.2), 0.35, s.add_material(pt.lambertian((0.8, 0.8, 0.8))))
    s.add_cube(s.add_material(pt.plastic((0.3, 0.4, 0.8), 1.5)), scale=(0.5, 0.7, 0.5), rotation=(0, 25, 0), position=(0.4, 0.35, 0.1))
    s.set_camera((0, 1, 3.6), (0, 1, 0), (0, 1, 0), 40.0, 1.5)
    return s


# the ceiling light, tilted 15 degrees: an axis-aligned rectangle as a mesh would lie under a flat node of the reference's
# BVH, where no ray can hit it
LIGHT = dict(scale=(0.6, 1, 0.4), rotation=(15, 0, 0), position=(0, 1.85, 0))


def _light_as_mesh(pt):
    o2w, _ = pt.transform(LIGHT["scale"], LIGHT["rotation"], LIGHT["position"])
    m = o2w.astype(np.float64).reshape(4, 4).T
    corners = np.array([[-0.5, 0, -0.5, 1], [0.5, 0, -0.5, 1], [0.5, 0, 0.5, 1], [-0.5, 0, 0.5, 1]]) @ m.T
    return corners[:, :3].astype(np.float32), np.array([[0, 1, 2], [0, 2, 3]], np.int32)


def _dome_mesh(n=8):
    """an open, gently curved panel: an n x n grid over [-0.5, 0.5]^2 bent up at the rim (y = 0.25 (x^2 + z^2)), so that
    no node of the reference's BVH over it is flat and nothing of it hides the rest from below"""
    g = np.linspace(-0.5, 0.5, n + 1, dtype=np.float32)
    x, z = np.meshgrid(g, g, indexing="ij")
    v = np.stack([x, 0.25 * (x * x + z * z), z], axis=-1).reshape(-1, 3)
    idx = []
    for i in range(n):
        for j in range(n):
            a, b, c, d = i * (n + 1) + j, (i + 1) * (n + 1) + j, (i + 1) * (n + 1) + j + 1, i * (n + 1) + j + 1
            idx += [[a, b, c], [a, c, d]]
    return v, np.array(idx, np.int32)


def _room_with(pt, kind, closed=False):
    s = _room(pt, closed)
    lm = s.add_material(pt.emissive((12.0, 11.0, 9.0)))
    if kind == "quad":
        s.add_quad(lm, **LIGHT)
    elif kind == "mesh":
        v, idx = _light_as_mesh(pt)
        s.add_mesh(v, idx, lm)
    elif kind == "text":  # the text mesh as a sign on the back wall (4,748 triangles, 1,982 dead), scaled and rotated
        s.add_obj(TEXT_OBJ, s.add_material(pt.emissive((6.0, 3.0, 1.5))), scale=(0.09, 0.14, 0.05), rotation=(8, -12, 4),
                  position=(0, 1.3, -0.85))
    elif kind == "concave":
        v, idx = _box_mesh()
        s.add_mesh(v, idx, s.add_material(pt.emissive((4.0, 4.0, 5.0))), scale=(0.4, 0.3, 0.4), rotation=(20, 30, 0), position=(0, 1.5, -0.3))
    elif kind == "cube":
        s.add_cube(s.add_material(pt.emissive((5.0, 4.0, 3.0))), scale=(0.15, 0.4, 0.25), rotation=(30, 45, 20), position=(0.3, 1.5, -0.4))
    elif kind == "mixed":  # a small bright sphere, a large dim emissive mesh (a curved ceiling panel) and a small quad
        s.add_sphere((-0.6, 1.7, 0.2), 0.08, s.add_material(pt.emissive((40.0, 38.0, 30.0))))
        v, idx = _dome_mesh()
        s.add_mesh(v, idx, s.add_material(pt.emissive((2.5, 2.5, 3.0))), scale=(1.0, 1.0, 0.8), rotation=(0, 20, 0), position=(0.2, 1.7, -0.3))
        s.add_quad(s.add_material(pt.emissive((3.0, 3.0, 3.0))), scale=(0.3, 1, 0.3), rotation=(100, 0, 0), position=(0.6, 0.9, -0.98))
    return s


def test_flag_alone_refused_and_changes_nothing_without_new_emitters(pt):
    s = pt.load_scene_from_json(os.path.join(SCENES, "cornell-box", "scene.json"))
    cs = s.to_core().commit(0)
    with pytest.raises(pt.PtcError) as e:
        cs.render(s.camera, s.render_settings(width=16, height=16, spp=1, flags=pt.FLAG_NEE_EMITTERS))
    assert e.value.code == pt.PTC_E_INVALID
    base = dict(width=96, height=96, spp=16, max_depth=8, seed=3)
    a, sa = cs.render(s.camera, s.render_settings(flags=pt.FLAG_NEE, **base))
    b, sb = cs.render(s.camera, s.render_settings(flags=em(pt), **base))
    assert np.array_equal(a, b) and sa.rays == sb.rays  # one quad light: selection by power is selection by count
    s = pt.load_scene_from_json(os.path.join(SCENES, "semesterbild.json"))
    cs = s.to_core().commit(0)
    base = dict(width=160, height=120, spp=4, max_depth=30, seed=5)
    a, sa = cs.render(s.camera, s.render_settings(**base))
    b, sb = cs.render(s.camera, s.render_settings(flags=em(pt), **base))
    assert np.array_equal(a, b) and sa.rays == sb.rays
    with pytest.raises(pt.PtcError) as e:  # no emitter this mode samples
        cs.light_sample(np.zeros((1, 3)), np.zeros((1, 4)))
    assert e.value.code == pt.PTC_E_STATE


def test_hooks_match_hostsim(pt):
    scene = mixed_scene(pt)
    sim = SimEmitters(scene)
    cs = scene.to_core().commit(0)
    n = 1 << 18
    u4 = np.random.default_rng(11).random((n, 4), dtype=np.float32)
    x = (np.random.default_rng(12).random((n, 3), dtype=np.float32) - 0.5) * np.float32(6.0)
    p_dev, pdf_dev, o_dev, t_dev = cs.light_sample(x, u4)
    p_sim, pdf_sim, _, o_sim, t_sim = sim.sample(x, u4)
    # the choices are table arithmetic and comparisons: equal; points and densities through sqrt: to a few ulps
    assert np.array_equal(o_dev, o_sim) and np.array_equal(t_dev, t_sim)
    np.testing.assert_allclose(p_dev, p_sim, rtol=0, atol=2e-5)
    assert np.isclose(pdf_dev, pdf_sim, rtol=2e-5, atol=0).mean() > 0.999
    np.testing.assert_allclose(pdf_dev, pdf_sim, rtol=1e-3, atol=0)  # (sphere points go through sincos: CUDA vs glibc)
    # light_pdf = the host's MIS density wherever the device's extend kernels and pt_prims.h find the same closest hit
    ok = o_dev >= 0
    d = p_dev[ok] - x[ok]
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    q_dev, q_sim = cs.light_pdf(x[ok], d), sim.pdf(x[ok], d)
    assert np.isclose(q_dev, q_sim, rtol=1e-4, atol=0).mean() > 0.999


def test_text_mesh_histogram_and_visible_densities(pt):
    s = pt.Scene()
    obj = s.add_obj(TEXT_OBJ, s.add_material(pt.emissive((4.0, 4.0, 4.0))), scale=(1.0, 0.5, 2.0), rotation=(10, 20, 30))
    cs = s.to_core().commit(0)
    n_tri = len(s.mesh(s.objects[obj].mesh))
    _, _, _, dead, _ = OracleScene(s).mesh_bvh_info(obj, n_tri)
    n = 1 << 20
    u4 = np.random.default_rng(21).random((n, 4), dtype=np.float32)
    x = np.tile(np.array([[0.5, 2.0, 30.0]], np.float32), (n, 1))
    pts, pdf, o, tri = cs.light_sample(x, u4)
    drawn = tri[tri >= 0]
    assert not dead[drawn].any()
    cdf, ent = SimEmitters(s).entries(0)
    p = np.diff(cdf.astype(np.float64))
    # the draws are u[3] against the CDF; rejections (edge-on from x) only thin them out
    counts = np.bincount(tri[tri >= 0], minlength=n_tri).astype(np.float64)
    live = p > 0
    expect = p * counts.sum()
    big = expect > 20
    z = (counts[big] - expect[big]) / np.sqrt(expect[big])
    assert np.abs(z).max() < 6.5 and abs(np.mean(z ** 2) - 1) < 0.25, (np.abs(z).max(), np.mean(z ** 2))
    assert counts[~live].sum() == 0
    # visible samples: the density light_pdf gives the sampled direction is light_sample's
    d = pts - x
    dist = np.linalg.norm(d, axis=1)
    d /= dist[:, None]
    m = o >= 0
    hits, _ = cs.intersect(x[m], d[m])
    vis = (hits["object"] == obj) & (np.linalg.norm(hits["position"] - pts[m], axis=1) < 1e-4 * dist[m])
    cos = np.abs(np.sum(hits["normal"] * d[m], axis=1))
    vis &= cos > 0.05
    assert vis.sum() > 20000
    q = cs.light_pdf(x[m][vis], d[m][vis])
    # (a point on a shared edge may be hit on the neighbouring triangle, whose stored normal the record then reports)
    agree = np.isclose(q, pdf[m][vis], rtol=1e-3, atol=0)
    assert agree.mean() > 0.99, agree.mean()


def test_same_light_two_shapes(pt):
    base = dict(width=96, height=64, max_depth=8)
    sq, sm = _room_with(pt, "quad"), _room_with(pt, "mesh")
    cq, cm = sq.to_core().commit(0), sm.to_core().commit(0)
    ref, _ = cq.render(sq.camera, sq.render_settings(spp=8192, seed=1, flags=pt.FLAG_NEE, **base))
    hi, _ = cm.render(sm.camera, sm.render_settings(spp=1024, seed=2, flags=em(pt), **base))
    assert_unbiased(hi, ref)
    mesh_em, _ = cm.render(sm.camera, sm.render_settings(spp=64, seed=3, flags=em(pt), **base))
    mesh_plain, _ = cm.render(sm.camera, sm.render_settings(spp=64, seed=3, **base))
    quad_nee, _ = cq.render(sq.camera, sq.render_settings(spp=64, seed=3, flags=pt.FLAG_NEE, **base))
    e_em, e_plain, e_quad = relmse(mesh_em, ref), relmse(mesh_plain, ref), relmse(quad_nee, ref)
    assert e_em < 0.5 * e_plain and e_em < 1.5 * e_quad, (e_em, e_plain, e_quad)


@pytest.mark.parametrize("kind", ["text", "concave", "cube", "mixed", "mixed-sky"])
def test_unbiased_against_plain(pt, kind):
    # (the mixed scene is closed, so that its emitters light it; under the sky it stays open)
    s = _room_with(pt, kind.replace("-sky", ""), closed=kind == "mixed")
    flags = em(pt)
    if kind == "mixed-sky":
        from test_gpu_nee_sky import _sun_scene  # the "sun" sky of the PTC_FLAG_NEE_SKY tests
        s.set_sky(_sun_scene(pt).sky)
        flags |= pt.FLAG_NEE_SKY
    cs = s.to_core().commit(0)
    base = dict(width=96, height=64, max_depth=8)
    ref, _ = cs.render(s.camera, s.render_settings(spp=16384, seed=1, **base))
    hi, _ = cs.render(s.camera, s.render_settings(spp=1024, seed=2, flags=flags, **base))
    assert_unbiased(hi, ref)
    if kind == "mixed":
        nee, _ = cs.render(s.camera, s.render_settings(spp=64, seed=3, flags=flags & ~pt.FLAG_NEE_EMITTERS, **base))
        emi, _ = cs.render(s.camera, s.render_settings(spp=64, seed=3, flags=flags, **base))
        assert relmse(emi, ref) < 0.5 * relmse(nee, ref), (relmse(emi, ref), relmse(nee, ref))


def test_same_image_from_every_builder(pt):
    s = _room_with(pt, "text")
    st = s.render_settings(width=96, height=64, spp=8, max_depth=8, seed=4, flags=em(pt))
    host, _ = s.to_core().commit(0).render_u32(s.camera, st)
    dev_sah, _ = s.to_core().commit(0, device_sah=True).render_u32(s.camera, st)
    fast, _ = s.to_core().commit(0, fast_build=True).render_u32(s.camera, st)
    assert np.array_equal(host, dev_sah) and np.array_equal(host, fast)


@pytest.mark.parametrize("value", [3e7, float("inf")])
def test_huge_emitters_make_no_finite_pixel_non_finite(pt, value):
    s = _room_with(pt, "concave")
    s.add_sphere((0.5, 1.6, 0.3), 0.1, s.add_material(pt.emissive((value, 1.0, 0.0))))
    cs = s.to_core().commit(0)
    base = dict(width=64, height=48, spp=16, max_depth=6, seed=5)
    nee, _ = cs.render(s.camera, s.render_settings(flags=pt.FLAG_NEE, **base))
    emi, _ = cs.render(s.camera, s.render_settings(flags=em(pt), **base))
    assert np.all(np.isfinite(emi[np.isfinite(nee)]))


def test_deterministic_and_every_entry_point(pt):
    s = _room_with(pt, "mixed")
    cs = s.to_core().commit(0)
    base = dict(width=100, height=70, spp=6, max_depth=8, seed=4, flags=em(pt))
    st = s.render_settings(**base)
    whole, stats = cs.render(s.camera, st)
    again, _ = cs.render(s.camera, st)
    assert np.array_equal(again, whole)
    small, _ = cs.render(s.camera, s.render_settings(pool_paths=2048, **base))
    assert np.array_equal(small, whole)
    by_sample = sum(cs.render(s.camera, s.render_settings(sample_begin=b, sample_end=e, **base))[0] for b, e in [(0, 1), (1, 4), (4, 6)])
    assert np.allclose(by_sample, whole, rtol=1e-5, atol=1e-6)
    u32, _ = cs.render_u32(s.camera, st)
    # a batch's views are the single renders
    cams = [s.camera, pt.camera_new((0.3, 1.1, 3.4), (0, 1, 0), (0, 1, 0), 40.0, 100 / 70)]
    rgb_b, u32_b, _ = cs.render_batch(cams, st, seeds=[4, 9])
    assert np.array_equal(rgb_b[0], whole) and np.array_equal(u32_b[0], u32)
    other, _ = cs.render(cams[1], s.render_settings(**dict(base, seed=9)))
    assert np.array_equal(rgb_b[1], other)
    # the final adaptive image at threshold 0 and the final progressive image are render_u32's
    _, u32_a, spp_a, _ = cs.render_adaptive(s.camera, st, 2, 0.0)
    assert (spp_a == 6).all() and np.array_equal(u32_a, u32)
    _, u32_p, n_p, _ = cs.render_progressive(s.camera, st, first_spp=1)
    assert n_p == 6 and np.array_equal(u32_p, u32)
    if pt.device_count() >= 2:
        m = cs.multi(list(range(pt.device_count())))
        for shard in (pt.SHARD_SAMPLES, pt.SHARD_TILES):
            img, sm = m.render(s.camera, st, shard)
            assert np.array_equal(img, whole) and sm.rays == stats.rays
