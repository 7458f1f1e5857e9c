"""PTC_COMMIT_DEVICE_SAH: the host builder's SAH tree and collapse (csrc/pt_build.cpp) built on the device
(csrc/pt_build_dev.cu, DevBuildMode::Sah).

  * the tree is the host builder's: same dead mask and DFS order, same wide-node count, depth and byte sizes, and — walked
    by the same rays — the same hit records and the same node / triangle test counts;
  * also where the centroids of a node coincide and the host splits the order its std::partition left;
  * images equal the default commit's bit for bit; two commits agree with each other;
  * the 2 M-triangle mesh of C5 commits faster than with the default commit.
"""
import os
import time

import numpy as np
import pytest

import parity_cases as pc
from bindings import OracleScene

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCENES = os.path.join(ROOT, "scenes")


def _mesh_scene(pt, kind):
    s = pt.Scene()
    m = s.add_material(pt.lambertian((0.5, 0.5, 0.5)))
    if kind == "text":      # 4,748 triangles, 1,982 of them under flat nodes
        s.add_obj(os.path.join(SCENES, "RayTracingText.obj"), m, rotation=(-30, 45, 0))
    elif kind == "teapot":  # 6,320 triangles, scaled: the t_world quirk is live
        s.add_obj(os.path.join(SCENES, "teapot", "teapot.obj"), m, scale=(30, 30, 30), rotation=(10, 20, 30), position=(1, 2, 3))
    elif kind == "tiny":    # 2 triangles: a root with one leaf
        s.add_mesh([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0.5]], [[0, 1, 2], [1, 3, 2]], m)
    elif kind == "flat":    # every triangle in one plane: all dead
        v = [[x, y, 0] for y in range(5) for x in range(5)]
        f = [[y * 5 + x, y * 5 + x + 1, (y + 1) * 5 + x] for y in range(4) for x in range(4)]
        s.add_mesh(v, f, m)
    elif kind == "synthetic":  # C5's generator at 300x300 cells (180,000 triangles)
        return pt.synthetic_scene(cells=300)
    s.set_camera((0, 40, 150), (0, 10, 0), (0, 1, 0), 50.0, 4 / 3)
    return s


def _soup_scene(pt, seed=11):
    # random triangles, plus groups of triangles that share their box centre: nodes whose centroids all coincide
    rng = np.random.default_rng(seed)
    s = pt.Scene()
    m = s.add_material(pt.lambertian((0.6, 0.5, 0.4)))
    v, f = [], []
    for _ in range(3000):
        c = rng.uniform(-20, 20, 3)
        for _k in range(3):
            v.append(c + rng.uniform(-1.5, 1.5, 3))
        f.append([len(v) - 3, len(v) - 2, len(v) - 1])
    for _ in range(60):
        c = rng.uniform(-20, 20, 3)
        h = rng.uniform(0.2, 1.0, 3)
        for k in range(int(rng.integers(4, 24))):  # corners of one box, picked differently: the same box centre
            sx, sy = (1, -1)[k & 1], (1, -1)[(k >> 1) & 1]
            v += [c + h * (-sx, -sy, -1), c + h * (sx, -sy, 1 if k & 4 else -1), c + h * (sx * 0.3, sy, 1)]
            f.append([len(v) - 3, len(v) - 2, len(v) - 1])
    s.add_mesh([list(map(float, p)) for p in v], f, m)
    s.set_camera((0, 10, 70), (0, 0, 0), (0, 1, 0), 50.0, 4 / 3)
    return s


def _commit(scene, monkeypatch, mode=None, **kw):
    if mode is None:
        monkeypatch.delenv("PTC_BUILD", raising=False)
    else:
        monkeypatch.setenv("PTC_BUILD", mode)
    t0 = time.perf_counter()
    cs = scene.to_core().commit(0, **kw)
    return cs, time.perf_counter() - t0


def _info_tuple(i):
    return (i.triangles, i.live_triangles, i.ref_nodes, i.ref_leaves, i.ref_depth, i.wide_nodes, i.wide_depth, i.node_bytes, i.triangle_bytes)


def _counters(st):
    return st.nodes_visited, st.tris_tested, st.mesh_rays


def _assert_same_tree(pt, s, sah, host, o, d, oracle=True):
    si, sdead, sorder = sah.mesh_info(0)
    hi, hdead, horder = host.mesh_info(0)
    assert (sdead == hdead).all() and (sorder == horder).all()
    assert _info_tuple(si) == _info_tuple(hi)
    got, gs = sah.intersect(o, d)
    ref, hs = host.intersect(o, d)
    assert got.tobytes() == ref.tobytes()
    assert _counters(gs) == _counters(hs)  # same nodes entered, same triangles tested: the same tree
    if oracle:
        pc.assert_hits_identical(pt, got, OracleScene(s).intersect(pt, o, d))
    return si, gs


@pytest.mark.parametrize("kind", ["text", "teapot", "tiny", "flat", "synthetic"])
def test_device_sah_tree_equals_host_tree(pt, kind, monkeypatch):
    monkeypatch.setenv("PTC_STEAL", "0")
    s = _mesh_scene(pt, kind)
    sah, _ = _commit(s, monkeypatch, device_sah=True)
    host, _ = _commit(s, monkeypatch, "host")
    rng = np.random.default_rng(5)
    o, d = pc.rand_rays(rng, 100000, (0, 10, 0), 60.0)
    si, _ = _assert_same_tree(pt, s, sah, host, o, d)
    if kind == "flat":
        assert si.live_triangles == 0
    # the environment switch selects the same builder
    env, _ = _commit(s, monkeypatch, "device-sah")
    assert _info_tuple(env.mesh_info(0)[0]) == _info_tuple(si)


def test_device_sah_coincident_centroids(pt, monkeypatch):
    monkeypatch.setenv("PTC_STEAL", "0")
    s = _soup_scene(pt)
    sah, _ = _commit(s, monkeypatch, device_sah=True)
    dflt, _ = _commit(s, monkeypatch)
    host, _ = _commit(s, monkeypatch, "host")
    rng = np.random.default_rng(8)
    o, d = pc.rand_rays(rng, 100000, (0, 0, 0), 40.0)
    # the host splits such nodes at count / 2 of its partition's order, which the device restates: still the same tree
    _assert_same_tree(pt, s, sah, host, o, d)
    got, _ = sah.intersect(o, d)
    assert got.tobytes() == dflt.intersect(o, d)[0].tobytes()
    st = s.render_settings(width=160, height=120, spp=4, max_depth=8, seed=2)
    a, sa = sah.render(s.camera, st)
    b, sb = dflt.render(s.camera, st)
    assert sa.rays == sb.rays and np.array_equal(a, b)


@pytest.mark.parametrize("cfg", ["C2", "C3", "C3s", "C5"])
def test_device_sah_renders_equal_default(pt, cfg, monkeypatch):
    from raytracer_rust_b200 import workloads
    _, s = workloads.workload(cfg, cells=300) if cfg == "C5" else workloads.workload(cfg)
    sah, _ = _commit(s, monkeypatch, device_sah=True)
    dflt, _ = _commit(s, monkeypatch)
    for flags in (0, pt.FLAG_NEE):
        st = s.render_settings(width=192, height=108, spp=4, max_depth=12, seed=9, flags=flags)
        a, sa = sah.render(s.camera, st)
        b, sb = dflt.render(s.camera, st)
        assert sa.rays == sb.rays and sa.paths == sb.paths and np.array_equal(a, b)  # fixed-point film


def test_device_sah_is_deterministic(pt, monkeypatch):
    monkeypatch.setenv("PTC_STEAL", "0")
    s = _mesh_scene(pt, "synthetic")
    a, _ = _commit(s, monkeypatch, device_sah=True)
    b, _ = _commit(s, monkeypatch, device_sah=True)
    ai, adead, aorder = a.mesh_info(0)
    bi, bdead, border = b.mesh_info(0)
    assert _info_tuple(ai) == _info_tuple(bi) and (adead == bdead).all() and (aorder == border).all()
    o, d = pc.rand_rays(np.random.default_rng(3), 50000, (0, 10, 0), 60.0)
    ra, sa = a.intersect(o, d)
    rb, sb = b.intersect(o, d)
    assert ra.tobytes() == rb.tobytes() and _counters(sa) == _counters(sb)


def test_device_sah_flag_conflict(pt):
    cs = _mesh_scene(pt, "tiny").to_core()
    with pytest.raises(pt.PtcError) as e:
        cs.commit(0, fast_build=True, device_sah=True)
    assert e.value.code == pt.PTC_E_INVALID
    cs.commit(0, device_sah=True)  # the handle is still usable


@pytest.mark.skipif("__import__('ptload').load().device_count() < 2")
def test_device_sah_multi_replica(pt, monkeypatch):
    s = _mesh_scene(pt, "synthetic")
    cs, _ = _commit(s, monkeypatch, device_sah=True)
    st = s.render_settings(width=160, height=90, spp=4, max_depth=8, seed=4)
    whole, ws = cs.render(s.camera, st)
    img, ms = cs.multi([0, 1]).render(s.camera, st, pt.SHARD_SAMPLES)
    assert ms.rays == ws.rays and np.array_equal(img, whole)


def test_device_sah_full_size_c5(pt, monkeypatch, capfd):
    # BASELINE config C5's mesh: 1000x1000 cells = 2,000,000 triangles
    monkeypatch.setenv("PTC_STEAL", "0")
    monkeypatch.setenv("PTC_BUILD_TIMING", "1")
    s = pt.synthetic_scene(cells=1000)
    warm = pt.synthetic_scene(cells=64)
    _commit(warm, monkeypatch, device_sah=True)  # CUDA context, CUB temporaries, kernel load
    _commit(warm, monkeypatch)
    capfd.readouterr()
    sah, t_sah = _commit(s, monkeypatch, device_sah=True)
    sah_log = capfd.readouterr().err
    dflt, t_dflt = _commit(s, monkeypatch)
    dflt_log = capfd.readouterr().err
    host, _ = _commit(s, monkeypatch, "host")
    capfd.readouterr()
    st = s.render_settings(width=480, height=270, spp=1, max_depth=1, seed=3)
    o, d = sah.primary_rays(s.camera, st, 0)
    si, gs = _assert_same_tree(pt, s, sah, host, o, d, oracle=False)
    ref, _ = dflt.intersect(o, d)
    assert ref.tobytes() == sah.intersect(o, d)[0].tobytes()
    with capfd.disabled():
        print(f"\n[C5 commit] device SAH {t_sah * 1e3:.0f} ms, default (hybrid) {t_dflt * 1e3:.0f} ms; {si.wide_nodes} wide nodes, "
              f"{gs.nodes_visited / max(1, gs.mesh_rays):.2f} node steps / mesh ray")
        print("device SAH phases:\n" + "".join(l + "\n" for l in sah_log.splitlines() if "pt_build" in l or "commit" in l))
        print("default phases:\n" + "".join(l + "\n" for l in dflt_log.splitlines() if "pt_build" in l or "commit" in l))
    assert t_sah < t_dflt
