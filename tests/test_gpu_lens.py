"""Thin-lens depth of field (ptc_scene_set_lens) on the device.

  1. nothing changes without a lens: a handle with R = 0, or with a lens set and then reset, returns bit for bit the
     images of a handle that never had a lens, from every entry point;
  2. hook parity: ptc_primary_rays under a lens equals the host build of the model (hostsim) within a few ulp, and with
     R = 0 is the pinhole hook bit for bit;
  3. defocus follows the formula: the image of a small emitter at depth z is its pinhole image convolved with a disk of
     radius R |1/z - 1/F| (second moments), centred, with the same total;
  4. consistency under a lens: progressive previews, adaptive pixels, the denoiser's noisy image and batch views are the
     uniform / single renders with the same lens, bit for bit;
  5. NEE under a lens agrees with a plain render of much higher spp with the same lens (8x8 block means);
  6. determinism: repeated renders and different pool sizes give identical images.
"""
import ctypes as C
import os

import numpy as np
import pytest

from test_lens_host import _sim_rays, _within

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCENES = os.path.join(ROOT, "scenes")


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _case(pt, name):
    if name == "cornell":
        return pt.load_scene_from_json(os.path.join(SCENES, "cornell-box", "scene.json")), dict(width=48, height=40, spp=8, max_depth=8, seed=3)
    return pt.load_scene_from_json(os.path.join(SCENES, "semesterbild.json")), dict(width=96, height=72, spp=8, max_depth=30, seed=7)


def _moved(pt, cam, dz):
    c = pt.Camera()
    C.pointer(c)[0] = cam
    for i in range(3):
        c.position[i] += dz * c.forward[i] * 0.02
    return c


def _all_entry_points(pt, cs, s, base):
    """every single-camera entry point and the batch, as bit patterns"""
    torch = pytest.importorskip("torch")
    cam = s.camera
    st = s.render_settings(**base)
    out = {}
    out["render"] = _bits(cs.render(cam, st)[0])
    out["u32"] = cs.render_u32(cam, st)[0]
    acc = torch.zeros((base["height"], base["width"], 3), dtype=torch.float32, device="cuda:0")
    cs.render_accumulate(cam, st, acc.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    out["accumulate"] = _bits(acc.cpu().numpy())
    rgb, u32, spp, _ = cs.render_adaptive(cam, s.render_settings(**dict(base, spp=16)), 4, 0.05)
    out["adaptive"] = np.concatenate([_bits(rgb).ravel(), u32, spp.ravel().view(np.uint32)])
    previews = []
    rgb, u32, n, _ = cs.render_progressive(cam, st, 1, 0, lambda j, k, img: previews.append(img))
    out["progressive"] = np.concatenate([_bits(rgb).ravel(), u32] + previews)
    dn = cs.render_denoised(cam, st, feature_spp=2, iterations=3)
    out["denoised"] = np.concatenate([_bits(a).ravel() if a.dtype == np.float32 else a.ravel() for a in dn[:6]])
    cams = [cam, _moved(pt, cam, 1.0), _moved(pt, cam, -1.0)]
    rgb, u32, _ = cs.render_batch(cams, st, seeds=[1, 2, 3])
    out["batch"] = np.concatenate([_bits(rgb).ravel(), u32.ravel()])
    if pt.device_count() >= 2:
        m = cs.multi([0, 1])
        out["multi"] = np.concatenate([_bits(m.render(cam, st, pt.SHARD_SAMPLES)[0]).ravel(), m.render_u32(cam, st, pt.SHARD_TILES)[0]])
    return out


@pytest.mark.parametrize("name", ["cornell", "semesterbild"])
def test_nothing_changes_without_a_lens(pt, name):
    s, base = _case(pt, name)
    never = s.to_core().commit(0)
    zero = s.to_core().commit(0).set_lens(0.0, 3.0)
    reset = s.to_core().commit(0).set_lens(0.3, 3.0).set_lens()
    zero_batch = s.to_core().commit(0).set_lens([(0.0, 1.0), (0.0, 2.0), (0.0, 5.0)])
    want = _all_entry_points(pt, never, s, base)
    for label, cs in (("R = 0", zero), ("reset", reset)):
        got = _all_entry_points(pt, cs, s, base)
        assert got.keys() == want.keys()
        for k in want:
            assert np.array_equal(got[k], want[k]), (label, k)
    st = s.render_settings(**base)
    cams = [s.camera, _moved(pt, s.camera, 1.0), _moved(pt, s.camera, -1.0)]
    rgb, u32, _ = zero_batch.render_batch(cams, st, seeds=[1, 2, 3])
    assert np.array_equal(np.concatenate([_bits(rgb).ravel(), u32.ravel()]), want["batch"])
    # a mixed batch: the view with R = 0 is its pinhole render
    mixed = s.to_core().commit(0).set_lens([(0.2, 2.0), (0.0, 2.0), (0.1, 4.0)])
    rgb, u32, _ = mixed.render_batch(cams, st, seeds=[1, 2, 3])
    one = never.render(cams[1], s.render_settings(**dict(base, seed=2)))[0]
    assert np.array_equal(_bits(rgb[1]), _bits(one))
    assert not np.array_equal(_bits(rgb[0]), _bits(never.render(cams[0], s.render_settings(**dict(base, seed=1)))[0]))


def test_hook_parity(pt):
    s, base = _case(pt, "cornell")
    cs = s.to_core().commit(0)
    st = s.render_settings(width=53, height=31, seed=0xABCDEF12345)
    po, pd = cs.primary_rays(s.camera, st, 4)
    for R, F in ((0.0, 5.0), (0.1, 6.8), (0.5, 3.0)):
        cs.set_lens(R, F)
        o, d = cs.primary_rays(s.camera, st, 4)
        so, sd = _sim_rays(pt, s.camera, 53, 31, 0xABCDEF12345, 4, R, F)
        if R == 0:
            assert o.tobytes() == po.tobytes() and d.tobytes() == pd.tobytes()
        else:
            assert not np.array_equal(o, po)
        assert _within(o, so.astype(np.float64)).all() and _within(d, sd.astype(np.float64)).all(), (np.abs(o - so).max(), np.abs(d - sd).max())


def _defocus_scene(pt, z, rho):
    s = pt.Scene()
    s.add_sphere((0.0, 0.0, -z), rho, s.add_material(pt.emissive((1.0, 1.0, 1.0))))
    s.set_sky(np.zeros((1, 1, 3), np.float32))
    s.set_camera((0, 0, 0), (0, 0, -1), (0, 1, 0), 40.0, 1.0)
    return s


def _moments(img):
    lum = img.sum(axis=2).astype(np.float64)
    h, w = lum.shape
    y, x = np.mgrid[0:h, 0:w] + 0.5
    tot = lum.sum()
    cx, cy = (lum * x).sum() / tot, (lum * y).sum() / tot
    m2 = (lum * ((x - cx) ** 2 + (y - cy) ** 2)).sum() / tot
    return tot, cx, cy, m2


def test_defocus_follows_the_formula(pt):
    z, rho, F, R, W = 4.0, 0.06, 2.0, 0.23, 256
    assert R / z <= 0.06
    s = _defocus_scene(pt, z, rho)
    cs = s.to_core().commit(0)
    st = s.render_settings(width=W, height=W, spp=4096, max_depth=1, seed=11)
    hw = s.camera.half_width
    px = W / (2.0 * hw)
    a = rho / np.sqrt(z * z - rho * rho) * px
    pin_tot, pcx, pcy, pin_m2 = _moments(cs.render(s.camera, st)[0])
    assert pin_m2 == pytest.approx(a * a / 2 + 1 / 6, rel=0.03)
    cs.set_lens(R, F)
    b = R * abs(1 / z - 1 / F) * px
    assert 15 <= b <= 30
    tot, cx, cy, m2 = _moments(cs.render(s.camera, st)[0])
    assert abs(cx - W / 2) <= 0.05 and abs(cy - W / 2) <= 0.05, (cx, cy)
    assert m2 == pytest.approx(b * b / 2 + a * a / 2 + 1 / 6, rel=0.03), (m2, b, a)
    assert tot == pytest.approx(pin_tot, rel=0.01)
    # in focus: the pinhole image's spread
    cs.set_lens(R, z)
    tot, cx, cy, m2 = _moments(cs.render(s.camera, st)[0])
    assert m2 == pytest.approx(pin_m2, rel=0.03) and tot == pytest.approx(pin_tot, rel=0.01)


@pytest.mark.parametrize("name", ["cornell", "semesterbild"])
def test_consistency_under_a_lens(pt, name):
    s, base = _case(pt, name)
    cs = s.to_core().commit(0)
    lens = (0.15, 6.8) if name == "cornell" else (6.0, 310.0)
    cs.set_lens(*lens)
    cam = s.camera
    st = s.render_settings(**dict(base, spp=16))
    # progressive previews = render_u32 at their sample counts
    previews = []
    cs.render_progressive(cam, st, 1, 0, lambda j, k, img: previews.append((k, img)))
    assert [k for k, _ in previews] == [1, 2, 4, 8, 16]
    for k, img in previews:
        assert np.array_equal(img, cs.render_u32(cam, s.render_settings(**dict(base, spp=k)))[0]), k
    # adaptive: every pixel is the uniform render at its own count
    rgb, u32, spp, _ = cs.render_adaptive(cam, st, 2, 0.5 if name == "cornell" else 0.05)
    for n in np.unique(spp):
        uni, _ = cs.render(cam, s.render_settings(**dict(base, spp=int(n))))
        sel = spp == n
        assert np.array_equal(_bits(rgb[sel]), _bits(uni[sel])), n
    assert len(np.unique(spp)) > 1
    # the denoiser's noisy image is render()
    dn = cs.render_denoised(cam, st, feature_spp=2, iterations=3)
    assert np.array_equal(_bits(dn[2]), _bits(cs.render(cam, st)[0]))
    # batch: view k with lenses[k] is the single render with that lens and seed; and one lens for every view
    fs = [lens[1] * f for f in (0.5, 0.8, 1.0, 1.5, 3.0)]
    cams = [cam] * 5
    seeds = [4, 5, 6, 7, 8]
    bs = s.to_core().commit(0).set_lens([(lens[0], f) for f in fs])
    rgb, u32, _ = bs.render_batch(cams, s.render_settings(**base), seeds=seeds)
    for k in range(5):
        cs.set_lens(lens[0], fs[k])
        one, _ = cs.render(cam, s.render_settings(**dict(base, seed=seeds[k])))
        assert np.array_equal(_bits(rgb[k]), _bits(one)), k
        assert np.array_equal(u32[k], cs.render_u32(cam, s.render_settings(**dict(base, seed=seeds[k])))[0]), k
    assert not np.array_equal(_bits(rgb[0]), _bits(rgb[4]))
    bs.set_lens(*lens)
    cs.set_lens(*lens)
    moved = [cam, _moved(pt, cam, 1.0), _moved(pt, cam, -2.0)]
    rgb, u32, _ = bs.render_batch(moved, s.render_settings(**base), seeds=[9, 9, 10])
    for k in range(3):
        one, _ = cs.render(moved[k], s.render_settings(**dict(base, seed=[9, 9, 10][k])))
        assert np.array_equal(_bits(rgb[k]), _bits(one)), k


def _blocks(img, k=8):
    h, w, _ = img.shape
    return img[:h // k * k, :w // k * k].reshape(h // k, k, w // k, k, 3).mean(axis=(1, 3))


@pytest.mark.parametrize("flags", ["nee", "nee-emitters"])
def test_nee_under_a_lens_is_unbiased(pt, flags):
    s = pt.load_scene_from_json(os.path.join(SCENES, "veach-mis", "scene.json"))
    cs = s.to_core().commit(0)
    # focus on look_at, the plane of the light spheres; the plates nearer the camera blur by a few pixels
    cs.set_lens(0.3, 28.28)
    base = dict(width=160, height=90, max_depth=16)
    f = pt.FLAG_NEE | (pt.FLAG_NEE_EMITTERS if flags == "nee-emitters" else 0)
    ref, _ = cs.render(s.camera, s.render_settings(spp=8192, seed=1, **base))
    nee, _ = cs.render(s.camera, s.render_settings(spp=1024, seed=3, flags=f, **base))
    bn, br = _blocks(nee), _blocks(ref)
    rel = np.abs(bn - br) / (br + 1e-2)
    assert np.median(rel) < 0.02 and np.percentile(rel, 99) < 0.15, (np.median(rel), np.percentile(rel, 99))


def test_determinism_under_a_lens(pt):
    s, base = _case(pt, "semesterbild")
    cs = s.to_core().commit(0).set_lens(6.0, 310.0)
    st = s.render_settings(**base)
    a, _ = cs.render(s.camera, st)
    b, _ = cs.render(s.camera, st)
    c, _ = cs.render(s.camera, s.render_settings(**dict(base, pool_paths=20000)))
    d, _ = cs.render(s.camera, s.render_settings(**dict(base, flags=pt.FLAG_NEE)))
    e, _ = cs.render(s.camera, s.render_settings(**dict(base, flags=pt.FLAG_NEE, pool_paths=30000)))
    assert np.array_equal(_bits(a), _bits(b)) and np.array_equal(_bits(a), _bits(c))
    assert np.array_equal(_bits(d), _bits(e))
