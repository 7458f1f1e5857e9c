"""Motion blur (ptc_scene_set_object_motion / ptc_scene_set_camera_motion) on the device.

  1. zero motion is no motion: every D = 0 and every end camera equal to its start camera give, from every entry point,
     the images, launches, rays and iterations of a handle that never called the setters, bit for bit;
  2. the motion kernels equal the static kernels where nothing visible moves (a moving sphere and mesh sealed in a static
     opaque cube in the Cornell box), through tiles, pixel lists and batches, in every shade mode;
  3. ptc_intersect_at is pinned to ptc_intersect (itself bit-exact to the oracle) by transitivity: a common D is
     ptc_intersect on o - tau D with the position + tau D; distinct D equal the host build of the shifted scan;
  4. streak geometry: a moving emissive sphere keeps its image sum, and its second moment along D grows by delta^2 / 12;
  5. the renders are unbiased against the time integral (the mean of K static scenes at the midpoints of the shutter);
  6. translating the camera by c matches translating every object by -c;
  7. the exactness guarantees hold with motion on: determinism, pool size and tile shards, progressive previews, adaptive
     pixels, the denoiser's noisy image, batch views, multi-GPU, and the shutter times of the renders.
"""
import ctypes as C
import os

import numpy as np
import pytest

from test_motion_host import _F

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCENES = os.path.join(ROOT, "scenes")

TET_V = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]], np.float32) - 0.25
TET_I = np.array([[0, 2, 1], [0, 1, 3], [0, 3, 2], [1, 2, 3]], np.int32)


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _copy(pt, cam):
    return pt.Camera.from_buffer_copy(cam)


def _shifted(pt, cam, dx=0.0, dy=0.0, dz=0.0):
    c = _copy(pt, cam)
    c.position[0] += dx
    c.position[1] += dy
    c.position[2] += dz
    return c


def _sky_hdr():
    sky = np.full((16, 32, 3), 0.3, np.float32)
    sky[4:6, 10:12] = (40.0, 36.0, 30.0)  # a small bright "sun"
    return sky


def _stats_key(st):
    """What the render determines.  Not kernel_launches: the host enqueues iterations up to a few ahead of the device and
    stops when it sees the render's end in the progress word (ptcore.cu, render_accumulate), so the number of trailing
    empty launches depends on timing and differs from run to run of the very same kernels.  Which kernels ran is
    checked by name instead (_kernel_names)."""
    return (int(st.rays), int(st.iterations), int(st.paths))


def _kernel_names(torch, fn):
    """the names of the CUDA kernels `fn` launches (CUPTI through torch.profiler: every kernel of the process)"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}


# ---- 1. zero motion is no motion ---------------------------------------------------------------------------
def _entry_points(pt, cs, s, base, end_single=None, end_batch=None):
    """every entry point as bit patterns (+ the stats of the plain render); the camera motion set before the single
    calls and before the batch"""
    torch = pytest.importorskip("torch")
    cam = s.camera
    st = s.render_settings(**base)
    out = {}
    if end_single is not None:
        cs.set_camera_motion(end_single)
    img, stats = cs.render(cam, st)
    out["render"] = _bits(img)
    out["stats"] = np.array(_stats_key(stats), np.uint64).view(np.uint32)
    out["u32"] = cs.render_u32(cam, st)[0]
    acc = torch.zeros((base["height"], base["width"], 3), dtype=torch.float32, device="cuda:0")
    cs.render_accumulate(cam, st, acc.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    out["accumulate"] = _bits(acc.cpu().numpy())
    rgb, u32, spp, ast = cs.render_adaptive(cam, s.render_settings(**dict(base, spp=16)), 4, 0.05)
    out["adaptive"] = np.concatenate([_bits(rgb).ravel(), u32, spp.ravel().view(np.uint32),
                                      np.array(_stats_key(ast), np.uint64).view(np.uint32)])
    previews = []
    rgb, u32, n, _ = cs.render_progressive(cam, st, 1, 0, lambda j, k, im: previews.append(im))
    out["progressive"] = np.concatenate([_bits(rgb).ravel(), u32] + previews)
    dn = cs.render_denoised(cam, st, feature_spp=2, iterations=3)
    out["denoised"] = np.concatenate([_bits(a).ravel() if a.dtype == np.float32 else a.ravel() for a in dn[:6]])
    o, d = cs.primary_rays(cam, st, 1)
    out["primary_rays"] = np.concatenate([_bits(o).ravel(), _bits(d).ravel()])
    cams = [cam, _shifted(pt, cam, dx=0.1), _shifted(pt, cam, dz=-0.2)]
    if end_batch is not None:
        cs.set_camera_motion(end_batch(cams))
    rgb, u32, bst = cs.render_batch(cams, st, seeds=[1, 2, 3])
    out["batch"] = np.concatenate([_bits(rgb).ravel(), u32.ravel(), np.array(_stats_key(bst), np.uint64).view(np.uint32)])
    if pt.device_count() >= 2:
        if end_single is not None:
            cs.set_camera_motion(end_single)
        m = cs.multi([0, 1])
        out["multi"] = np.concatenate([_bits(m.render(cam, st, pt.SHARD_SAMPLES)[0]).ravel(), m.render_u32(cam, st, pt.SHARD_TILES)[0]])
    return out


@pytest.mark.parametrize("flags", [0, "nee"])
def test_zero_motion_is_no_motion(pt, flags):
    s = pt.load_scene_from_json(os.path.join(SCENES, "cornell-box", "scene.json"))
    base = dict(width=48, height=40, spp=8, max_depth=8, seed=3, flags=0 if flags == 0 else pt.FLAG_NEE)
    never = s.to_core().commit(0)
    zero = s.to_core().commit(0)
    n_obj = 8
    for k in range(n_obj):
        zero.set_object_motion(k, (0.3, 0.0, 0.0))  # set, then reset: static again
        zero.set_object_motion(k, (0.0, -0.0, 0.0))
    torch = pytest.importorskip("torch")
    outs = {}
    names_never = _kernel_names(torch, lambda: outs.update(want=_entry_points(pt, never, s, base)))
    names_zero = _kernel_names(torch, lambda: outs.update(
        got=_entry_points(pt, zero, s, base, end_single=s.camera, end_batch=lambda cams: cams)))
    want, got = outs["want"], outs["got"]
    assert set(got) == set(want)
    for k in want:
        assert np.array_equal(got[k], want[k]), k
    # the same kernels ran, and none of the motion twins
    assert any("k_extend_pre" in n for n in names_never) and any("k_shade" in n for n in names_never), sorted(names_never)
    assert names_zero == names_never, sorted(names_zero ^ names_never)
    assert not any("motion" in n or "k_ray_times" in n for n in names_zero)
    # (positive control: a moving object does run the twins, and the profiler sees them)
    zero.set_camera_motion()
    zero.set_object_motion(0, (0.0, 0.1, 0.0))
    moved = _kernel_names(torch, lambda: zero.render(s.camera, s.render_settings(**base)))
    assert any("k_shade_motion" in n for n in moved) and any("k_extend_pre_motion" in n for n in moved), sorted(moved)


# ---- 2. the motion kernels where nothing visible moves -----------------------------------------------------------
def _sealed_cornell(pt, sky):
    s = pt.load_scene_from_json(os.path.join(SCENES, "cornell-box", "scene.json"))
    grey = s.add_material(pt.lambertian((0.6, 0.6, 0.6)))
    red = s.add_material(pt.lambertian((0.8, 0.1, 0.1)))
    c = (0.45, 1.35, -0.5)
    mesh = s.add_mesh(TET_V, TET_I, red, scale=(0.08, 0.08, 0.08), position=c)      # listed before the cube: still parked
    sphere = s.add_sphere(c, 0.06, red)
    s.add_cube(grey, scale=(0.3, 0.3, 0.3), position=c)                             # half size 0.15: seals both
    if sky:
        s.set_sky(_sky_hdr())
    return s, mesh, sphere


@pytest.mark.parametrize("mode", ["plain", "nee", "nee_sky", "emitters", "emitters_sky"])
def test_motion_kernels_equal_static_kernels_where_nothing_visible_moves(pt, mode):
    flags = {"plain": 0, "nee": pt.FLAG_NEE, "nee_sky": pt.FLAG_NEE | pt.FLAG_NEE_SKY, "emitters": pt.FLAG_NEE | pt.FLAG_NEE_EMITTERS,
             "emitters_sky": pt.FLAG_NEE | pt.FLAG_NEE_SKY | pt.FLAG_NEE_EMITTERS}[mode]
    s, mesh, sphere = _sealed_cornell(pt, sky=mode.endswith("sky"))
    assert mesh == 8 and sphere == 9
    static = s.to_core().commit(0)
    moving = s.to_core().commit(0)
    moving.set_object_motion(mesh, (0.0, 0.04, 0.0)).set_object_motion(sphere, (0.05, 0.0, -0.03))
    cam = s.camera
    st = s.render_settings(width=64, height=48, spp=8, max_depth=10, seed=11, flags=flags)
    # tiles
    a, sa = static.render(cam, st)
    b, sb = moving.render(cam, st)
    assert _bits(a).tobytes() == _bits(b).tobytes() and sa.rays == sb.rays
    # pixel lists (the adaptive passes after the first two)
    ra = static.render_adaptive(cam, s.render_settings(width=64, height=48, spp=16, max_depth=10, seed=11, flags=flags), 2, 0.02)
    rb = moving.render_adaptive(cam, s.render_settings(width=64, height=48, spp=16, max_depth=10, seed=11, flags=flags), 2, 0.02)
    assert (ra[2] > 2).any()  # passes over pixel lists ran
    assert _bits(ra[0]).tobytes() == _bits(rb[0]).tobytes() and np.array_equal(ra[2], rb[2])
    # batches, the end camera of every view bitwise equal to its start camera
    cams = [cam, _shifted(pt, cam, dx=0.05)]
    ba = static.render_batch(cams, st, seeds=[5, 6])[0]
    moving.set_camera_motion([_copy(pt, c) for c in cams])
    bb = moving.render_batch(cams, st, seeds=[5, 6])[0]
    assert _bits(ba).tobytes() == _bits(bb).tobytes()
    # and a single render with an end camera bitwise equal to the start camera
    moving.set_camera_motion(_copy(pt, cam))
    assert _bits(moving.render(cam, st)[0]).tobytes() == _bits(a).tobytes()


# ---- 3. ptc_intersect_at -------------------------------------------------------------------------------------
def _rays_and_times(pt, s, n, seed):
    from parity_cases import rand_rays
    rng = np.random.default_rng(seed)
    o, d = rand_rays(rng, n, (0, 0, 0), 80.0)
    t = rng.random(n).astype(np.float32)
    t[:2] = (0.0, 1.0)
    return o, d, t


def test_intersect_at_common_displacement_is_intersect_on_the_shifted_ray(pt):
    from parity_cases import composite_scene
    s = composite_scene(pt)
    cs = s.to_core().commit(0)
    D = np.array([3.5, -2.25, 1.75], np.float32)
    n_obj = 6
    for k in range(n_obj):
        cs.set_object_motion(k, D)
    o, d, t = _rays_and_times(pt, s, 100_000, 1)
    got, _ = cs.intersect(o, d, times=t)
    ts = t[:, None]
    want, _ = cs.intersect((o - ts * D).astype(np.float32), d)
    hit = want["object"] >= 0
    want["position"][hit] = (want["position"][hit] + ts[hit] * D).astype(np.float32)
    assert hit.sum() > 20_000 and len(np.unique(want["object"][hit])) == n_obj
    assert got.tobytes() == want.tobytes()
    # times outside [0, 1] or not finite are refused
    for bad in (-1e-7, 1.0000001, np.nan, np.inf):
        tb = t.copy()
        tb[7] = bad
        with pytest.raises(pt.PtcError):
            cs.intersect(o, d, times=tb)


def test_intersect_at_distinct_displacements_equal_the_host_build(pt):
    from bindings import SimScene
    from parity_cases import composite_scene
    from test_motion_host import _sim_intersect_motion
    s = composite_scene(pt)
    cs = s.to_core().commit(0)
    disp = np.array([[4, 0, 0], [0, -6, 0], [0, 0, 0], [2, 2, -3], [-5, 1, 0], [0, 3, 0]], np.float32)
    for k, dk in enumerate(disp):
        cs.set_object_motion(k, dk)
    o, d, t = _rays_and_times(pt, s, 100_000, 2)
    got, _ = cs.intersect(o, d, times=t)
    sim = SimScene(s)
    want = _sim_intersect_motion(pt, sim.L, sim.h, disp, o, d, t)
    assert (want["object"] >= 0).sum() > 20_000
    assert got.tobytes() == want.tobytes()


# ---- 4. streak geometry ------------------------------------------------------------------------------------
def _glow(pt, center):
    s = pt.Scene()
    s.add_sphere(center, 0.15, s.add_material(pt.emissive((2.0, 2.0, 2.0))))
    s.set_sky(np.zeros((2, 4, 3), np.float32))
    s.set_camera((0, 0, 20), (0, 0, 0), (0, 1, 0), 8.0, 2.0)  # narrow: the sphere's image keeps its size across the frame
    s.set_settings(192, 96, 256, 2)
    return s


def _moments(img):
    w = img[..., 0].astype(np.float64)
    y, x = np.mgrid[0:w.shape[0], 0:w.shape[1]] + 0.5
    m = w.sum()
    cx, cy = (w * x).sum() / m, (w * y).sum() / m
    return m, cx, cy, (w * (x - cx) ** 2).sum() / m, (w * (y - cy) ** 2).sum() / m


def test_streak_second_moment(pt):
    D = np.array([1.5, 0.0, 0.0], np.float32)
    s0, s1 = _glow(pt, (-0.75, 0.0, 0.0)), _glow(pt, (0.75, 0.0, 0.0))
    st = s0.render_settings(seed=4)
    m0, cx0, _, vx0, vy0 = _moments(s0.to_core().commit(0).render(s0.camera, st)[0])
    m1, cx1, _, _, _ = _moments(s1.to_core().commit(0).render(s1.camera, st)[0])
    delta = cx1 - cx0  # pixels swept over the shutter
    assert 40 < delta < 80
    cs = s0.to_core().commit(0).set_object_motion(0, D)
    m, cx, _, vx, vy = _moments(cs.render(s0.camera, st)[0])
    assert abs(m / m0 - 1) < 0.01 and abs(m1 / m0 - 1) < 0.01
    assert abs(cx - (cx0 + cx1) / 2) < 0.5
    assert abs(vx / (vx0 + delta ** 2 / 12) - 1) < 0.03, (vx, vx0, delta)
    assert abs(vy / vy0 - 1) < 0.03, (vy, vy0)


# ---- 5. unbiased against the time integral -----------------------------------------------------------------
PANEL_V = np.array([[-0.3, 0, -0.2], [0.3, 0, -0.2], [0.3, 0, 0.2], [-0.3, 0, 0.2]], np.float32)
PANEL_I = np.array([[0, 2, 1], [0, 3, 2]], np.int32)
MOVING = [  # (kind, displacement over the shutter)
    ("sphere", (0.25, 0.0, 0.0)), ("quad", (0.0, 0.2, 0.0)), ("cube", (-0.2, 0.0, 0.1)), ("mesh", (0.0, -0.2, 0.15)),
    ("light_sphere", (0.3, 0.0, 0.0)), ("light_mesh", (-0.25, 0.0, 0.0)),
]


def _mover_scene(pt, tau, sky, scene_shift=(0.0, 0.0, 0.0)):
    """the scene at shutter time tau (objects placed by their parameters / the translation of object_to_world), every
    object also shifted by scene_shift"""
    s = pt.Scene()
    grey = s.add_material(pt.lambertian((0.6, 0.6, 0.6)))
    red = s.add_material(pt.lambertian((0.7, 0.2, 0.2)))
    blue = s.add_material(pt.lambertian((0.2, 0.3, 0.7)))
    lamp = s.add_material(pt.emissive((6.0, 5.5, 5.0)))
    panel = s.add_material(pt.emissive((3.0, 3.0, 4.0)))
    sh = np.array(scene_shift, np.float64)

    def at(p, k):
        return tuple(np.array(p, np.float64) + tau * np.array(MOVING[k][1], np.float64) + sh)
    s.add_sphere(at((-0.6, 0.0, 0.0), 0), 0.35, red)
    s.add_quad(blue, scale=(0.6, 1.0, 0.6), rotation=(90, 0, 0), position=at((0.5, 0.1, -0.4), 1))
    s.add_cube(grey, scale=(0.4, 0.4, 0.4), rotation=(0, 30, 0), position=at((0.5, -0.3, 0.4), 2))
    s.add_mesh(TET_V, TET_I, red, scale=(0.6, 0.6, 0.6), rotation=(10, 20, 0), position=at((-0.1, 0.35, 0.5), 3))
    s.add_sphere(at((0.0, 1.1, 0.2), 4), 0.15, lamp)
    s.add_mesh(PANEL_V, PANEL_I, panel, rotation=(180, 0, 0), position=at((-0.5, 1.0, -0.3), 5))
    s.add_plane(tuple(np.array((0.0, -0.6, 0.0)) + sh), (0, 1, 0), grey)
    if sky:
        from test_gpu_nee_sky import _sun_scene
        s.set_sky(_sun_scene(pt).sky)
    s.set_camera((0.0, 0.6, 3.2), (0.0, 0.0, 0.0), (0, 1, 0), 45.0, 1.0)
    s.set_settings(64, 64, 8, 6)
    return s


def _blocks(img):
    h, w = img.shape[:2]
    return img.reshape(h // 8, 8, w // 8, 8, 3).mean(axis=(1, 3))


def _flags(pt, name, sky):
    f = {"plain": 0, "nee": pt.FLAG_NEE, "emitters": pt.FLAG_NEE | pt.FLAG_NEE_EMITTERS}[name]
    return f | (pt.FLAG_NEE_SKY if sky and f else 0)


@pytest.mark.parametrize("sky", [False, True])
def test_motion_is_unbiased_against_the_time_integral(pt, sky):
    """The reference is the midpoint rule over K = 64 static scenes at tau_k = (k + 1/2) / K.  Every 8 x 8 block mean is a
    continuous function of tau; the objects move at most 0.3 units (about 8 px here) over the shutter, so a block mean
    changes by at most its full contrast over the shutter and is Lipschitz in tau with a constant of at most that
    contrast.  The midpoint rule's error is then at most 1 / (4K) of the contrast, under 0.4 % for K = 64, and in
    practice far less because the sweep is close to linear: below the 2 % bar.
    The noise bar is 4 sigma of the difference, each side's sigma from the spread of R = 32 independent estimates: R
    motion renders with their own seeds, and R averages over all K static scenes (one sample per pixel each, own seeds),
    so that the reference's spread holds Monte Carlo noise only, not the variation of the image over the shutter.  Each
    side has 2048 samples per pixel.  Every block has to pass."""
    K, R, spp = 64, 32, 64
    moving = _mover_scene(pt, 0.0, sky).to_core().commit(0)
    for k, (_, dk) in enumerate(MOVING):
        moving.set_object_motion(k, dk)
    statics = [_mover_scene(pt, (k + 0.5) / K, sky) for k in range(K)]
    committed = [x.to_core().commit(0) for x in statics]
    cam = statics[0].camera
    for name in ("plain", "nee", "emitters"):
        flags = _flags(pt, name, sky)
        runs = np.stack([_blocks(moving.render(cam, statics[0].render_settings(spp=spp, seed=100 + j, flags=flags))[0])
                         for j in range(R)])
        refs = np.stack([np.mean([_blocks(cs.render(cam, statics[0].render_settings(spp=spp // K, seed=10_000 + j * K + k,
                                                                                    flags=flags))[0])
                                  for k, cs in enumerate(committed)], axis=0)
                         for j in range(R)])
        ref, mean = refs.mean(axis=0), runs.mean(axis=0)
        sigma = np.sqrt(runs.var(axis=0, ddof=1) / R + refs.var(axis=0, ddof=1) / R)
        bar = np.maximum(0.02 * np.abs(ref), 4 * sigma)
        bad = (np.abs(mean - ref) > bar + 1e-6).any(axis=2)
        assert bad.sum() == 0, (name, sky, bad.sum(), float(np.abs(mean - ref).max()))


# ---- 6. camera translation == scene translation ----------------------------------------------------------------
@pytest.mark.parametrize("name", ["plain", "nee"])
def test_camera_translation_matches_scene_translation(pt, name):
    """A camera moving by tau c against every object moving by -tau c under a static camera.  Statistical only (8 x 8
    block means): the two renders cannot be bit-equal, because the bounces after the first start from hit positions
    rounded in different frames, and the sample points on moving lights differ by the same rounding."""
    c = np.array([0.4, 0.15, 0.0], np.float32)
    s = _mover_scene(pt, 0.0, False)
    cam = s.camera
    cam_moves = s.to_core().commit(0).set_camera_motion(_shifted(pt, cam, *c))
    scene_moves = s.to_core().commit(0)
    for k in range(7):
        scene_moves.set_object_motion(k, -c)
    flags = _flags(pt, name, False)
    n = 32  # independent renders per side, 32 spp each: sigma from 31 degrees of freedom per side; every block must pass
    a = np.stack([_blocks(cam_moves.render(cam, s.render_settings(spp=32, seed=200 + j, flags=flags))[0]) for j in range(n)])
    b = np.stack([_blocks(scene_moves.render(cam, s.render_settings(spp=32, seed=300 + j, flags=flags))[0]) for j in range(n)])
    sigma = np.sqrt(a.var(axis=0, ddof=1) / n + b.var(axis=0, ddof=1) / n)
    bar = np.maximum(0.02 * np.abs(b.mean(0)), 4 * sigma)
    bad = (np.abs(a.mean(0) - b.mean(0)) > bar + 1e-6).any(axis=2)
    assert bad.sum() == 0, (bad.sum(), float(np.abs(a.mean(0) - b.mean(0)).max()))
    # and the camera motion is visible at all
    static = s.to_core().commit(0).render(cam, s.render_settings(spp=64, seed=200, flags=flags))[0]
    assert np.abs(_blocks(static) - a.mean(0)).max() > 0.05


# ---- 7. the exactness guarantees with motion on ----------------------------------------------------------------
def _motion_handle(pt, sky=False):
    s = _mover_scene(pt, 0.0, sky)
    cs = s.to_core().commit(0)
    for k, (_, dk) in enumerate(MOVING):
        cs.set_object_motion(k, dk)
    end = _shifted(pt, s.camera, dx=0.2, dy=-0.1)
    end.forward[0] += 0.05
    cs.set_camera_motion(end)
    return s, cs, end


@pytest.mark.parametrize("name", ["plain", "emitters"])
def test_exactness_guarantees_hold_with_motion(pt, name):
    torch = pytest.importorskip("torch")
    s, cs, end = _motion_handle(pt, sky=name == "emitters")
    cam = s.camera
    flags = _flags(pt, name, name == "emitters")
    st = s.render_settings(spp=16, seed=9, flags=flags)
    img, stats = cs.render(cam, st)
    assert stats.rays > 0
    # determinism, and the motion is visible
    assert _bits(cs.render(cam, st)[0]).tobytes() == _bits(img).tobytes()
    plain = s.to_core().commit(0).render(cam, st)[0]
    assert not np.array_equal(plain, img)
    # pool size
    small = s.render_settings(spp=16, seed=9, flags=flags, pool_paths=1 << 16)
    assert _bits(cs.render(cam, small)[0]).tobytes() == _bits(img).tobytes()
    # tile shards, added into one fp32 film
    one = torch.zeros((64, 64, 3), dtype=torch.float32, device="cuda:0")
    cs.render_accumulate(cam, st, one.data_ptr(), torch.cuda.current_stream().cuda_stream)
    shards = torch.zeros((64, 64, 3), dtype=torch.float32, device="cuda:0")
    for rem in range(3):
        cs.render_accumulate(cam, s.render_settings(spp=16, seed=9, flags=flags, tile_mod=3, tile_rem=rem), shards.data_ptr(),
                             torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert _bits(one.cpu().numpy()).tobytes() == _bits(shards.cpu().numpy()).tobytes()
    # progressive preview j == the one-shot render at its sample count
    previews = []
    cs.render_progressive(cam, st, 2, 0, lambda j, n, im: previews.append((n, im)))
    assert [n for n, _ in previews] == [2, 4, 8, 16]
    for n, im in previews:
        assert np.array_equal(im, cs.render_u32(cam, s.render_settings(spp=n, seed=9, flags=flags))[0]), n
    # adaptive pixels == the uniform render at their own count
    rgb, _, spp, _ = cs.render_adaptive(cam, s.render_settings(spp=32, seed=9, flags=flags), 4, 0.05)
    counts = np.unique(spp)
    assert len(counts) >= 2
    for n in counts:
        u = cs.render(cam, s.render_settings(spp=int(n), seed=9, flags=flags))[0]
        assert _bits(rgb[spp == n]).tobytes() == _bits(u[spp == n]).tobytes(), n
    # the denoised call's noisy image == ptc_render
    noisy = cs.render_denoised(cam, st, feature_spp=2, iterations=2)[2]
    assert _bits(noisy).tobytes() == _bits(img).tobytes()
    # batch view k with cams[k], end_cams[k], seeds[k] == the single render
    cams = [cam, _shifted(pt, cam, dx=-0.3), _shifted(pt, cam, dz=0.4)]
    ends = [end, _shifted(pt, cams[1], dy=0.2), _copy(pt, cams[2])]
    cs.set_camera_motion(ends)
    rgb, _, _ = cs.render_batch(cams, st, seeds=[3, 4, 5])
    for k in range(3):
        cs.set_camera_motion(ends[k])
        single = cs.render(cams[k], s.render_settings(spp=16, seed=3 + k, flags=flags))[0]
        assert _bits(rgb[k]).tobytes() == _bits(single).tobytes(), k
    # one end camera for every view
    cs.set_camera_motion(end)
    rgb, _, _ = cs.render_batch(cams, st, seeds=[3, 4, 5])
    single = cs.render(cams[1], s.render_settings(spp=16, seed=4, flags=flags))[0]
    assert _bits(rgb[1]).tobytes() == _bits(single).tobytes()


@pytest.mark.skipif("__import__('ptload').load().device_count() < 2")
def test_multi_render_with_motion_equals_one_gpu(pt):
    s, cs, _ = _motion_handle(pt)
    st = s.render_settings(spp=8, seed=5, flags=pt.FLAG_NEE)
    one = cs.render_u32(s.camera, st)[0]
    m = cs.multi(list(range(min(pt.device_count(), 4))))
    for shard in (pt.SHARD_SAMPLES, pt.SHARD_TILES):
        assert np.array_equal(m.render_u32(s.camera, st, shard)[0], one)


def test_ray_times_and_primary_rays_are_the_renders_times(pt):
    from test_lens_host import _philox
    from bindings import sim_lib
    s, cs, end = _motion_handle(pt)
    st = s.render_settings(width=37, height=23, seed=0x1234_5678_9ABC)
    pixel = np.arange(37 * 23, dtype=np.uint64)
    for sample in (0, 7):
        tau = cs.ray_times(st, sample)
        r = _philox([pixel, np.full_like(pixel, sample), np.full_like(pixel, 0xFFFFFFFF), np.ones_like(pixel)],
                    st.seed & 0xFFFFFFFF, st.seed >> 32)
        want = ((r[0] >> np.uint64(8)).astype(np.float64) / 16777216.0).astype(np.float32)
        assert tau.tobytes() == want.tobytes()
        # ptc_primary_rays starts from the camera at those times, as the host build does
        o, d = cs.primary_rays(s.camera, st, sample)
        L = sim_lib()
        L.sim_primary_rays_motion.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_float, _F, _F, _F]
        n = 37 * 23
        ho, hd, ht = np.empty((n, 3), np.float32), np.empty((n, 3), np.float32), np.empty(n, np.float32)
        cam = s.camera
        L.sim_primary_rays_motion(C.addressof(cam), C.addressof(end), C.addressof(st), sample, 0.0, 1.0, ho.ctypes.data_as(_F),
                                  hd.ctypes.data_as(_F), ht.ctypes.data_as(_F))
        assert ht.tobytes() == tau.tobytes()
        assert np.allclose(o, ho, atol=2e-6) and np.allclose(d, hd, atol=2e-6)
