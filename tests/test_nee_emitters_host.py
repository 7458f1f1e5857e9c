"""Emissive meshes and cubes in next-event estimation (PTC_FLAG_NEE_EMITTERS), checked on the host through
tests/hostsim/emsim.cpp: the g++ build of the very table-building, emitter_sample and emitter_mis_pdf code the shade
stage runs.

  * tables: the selection CDF is max(r, g, b) x area over the emitters of finite positive power, in object order, against
    a float64 restatement; a mesh's entry CDF is by world area over its live triangles in original order (rotated and
    non-uniformly scaled), a cube's by the areas of its six faces; the text mesh's dead triangles have probability 0;
  * the sampler puts its points on the triangle or face it reports, and draws the triangles with the tables'
    probabilities;
  * for meshes with geometric normals the estimator's divisor, the sampler's MIS density and the density a BSDF ray
    along the sampled direction is given agree.
"""
import ctypes as C
import os
import re

import numpy as np
import pytest

from bindings import OracleScene, _feed, sim_lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TEXT_OBJ = os.path.join(ROOT, "scenes", "RayTracingText.obj")
_F = C.POINTER(C.c_float)


def _lib():
    L = sim_lib()
    L.em_sim_scene_create.restype = C.c_void_p
    L.em_sim_scene_destroy.argtypes = [C.c_void_p]
    L.em_sim_scene_destroy.restype = None
    L.em_sim_scene_add_material.argtypes = [C.c_void_p, C.c_void_p]
    L.em_sim_scene_add_sphere.argtypes = [C.c_void_p, _F, C.c_float, C.c_int]
    L.em_sim_scene_add_plane.argtypes = [C.c_void_p, _F, _F, C.c_int]
    L.em_sim_scene_add_quad.argtypes = [C.c_void_p, _F, _F, _F, _F, C.c_float, C.c_float, C.c_float, C.c_int]
    L.em_sim_scene_add_cube.argtypes = [C.c_void_p, _F, _F, C.c_int]
    L.em_sim_scene_add_mesh.argtypes = [C.c_void_p, _F, C.c_int64, _F, _F, C.c_int]
    L.em_sim_scene_set_sky_hdr.argtypes = [C.c_void_p, _F, C.c_int32, C.c_int32]
    L.em_sim_commit.argtypes = [C.c_void_p]
    L.em_sim_lights.argtypes = [C.c_void_p, C.c_void_p, _F, _F]
    L.em_sim_lights.restype = C.c_int32
    L.em_sim_entries.argtypes = [C.c_void_p, C.c_int32, _F, _F]
    L.em_sim_entries.restype = C.c_int64
    L.em_sim_light_ids.argtypes = [C.c_void_p, C.c_void_p]
    L.em_sim_light_ids.restype = None
    L.em_sim_sample.argtypes = [C.c_void_p, _F, _F, C.c_int64, _F, _F, _F, C.c_void_p, C.c_void_p]
    L.em_sim_pdf.argtypes = [C.c_void_p, _F, _F, C.c_int64, _F]
    return L


def _fp(a):
    return a.ctypes.data_as(_F)


class SimEmitters:
    """The host build of a package `Scene`'s PTC_FLAG_NEE_EMITTERS tables and sampler."""

    def __init__(self, scene):
        self.scene = scene
        self.L = _lib()
        self.h = self.L.em_sim_scene_create()
        _feed(self.L, "em_sim_", self.h, scene)
        assert self.L.em_sim_commit(self.h) == 0

    def __del__(self):
        try:
            self.L.em_sim_scene_destroy(self.h)
        except Exception:
            pass

    def lights(self):
        n = self.L.em_sim_lights(self.h, None, None, None)
        toc, area, cdf = np.zeros((max(n, 1), 3), np.int32), np.zeros(max(n, 1), np.float32), np.zeros(n + 1, np.float32)
        self.L.em_sim_lights(self.h, toc.ctypes.data, _fp(area), _fp(cdf))
        return toc[:n], area[:n], cdf

    def entries(self, k):
        n = self.L.em_sim_entries(self.h, k, None, None)
        cdf, ent = np.zeros(n + 1, np.float32), np.zeros((n, 12), np.float32)
        assert self.L.em_sim_entries(self.h, k, _fp(cdf), _fp(ent)) == n
        return cdf, ent.reshape(n, 3, 4)

    def light_ids(self):
        ids = np.zeros(len(self.scene.objects), np.int32)
        self.L.em_sim_light_ids(self.h, ids.ctypes.data)
        return ids

    def sample(self, x, u4):
        x, u = np.ascontiguousarray(x, np.float32), np.ascontiguousarray(u4, np.float32)
        n = len(u)
        p, pdf, pmis = np.zeros((n, 3), np.float32), np.zeros(n, np.float32), np.zeros(n, np.float32)
        obj, tri = np.zeros(n, np.int32), np.zeros(n, np.int32)
        rc = self.L.em_sim_sample(self.h, _fp(x), _fp(u), n, _fp(p), _fp(pdf), _fp(pmis), obj.ctypes.data, tri.ctypes.data)
        assert rc == 0, rc
        return p, pdf, pmis, obj, tri

    def pdf(self, o, d):
        o, d = np.ascontiguousarray(o, np.float32), np.ascontiguousarray(d, np.float32)
        out = np.zeros(len(o), np.float32)
        assert self.L.em_sim_pdf(self.h, _fp(o), _fp(d), len(o), _fp(out)) == 0
        return out


def _box_mesh():
    """a closed, concave 'L'-shaped prism: 12 triangles of a box plus a notch, geometric normals"""
    v = np.array([[0, 0, 0], [2, 0, 0], [2, 1, 0], [1, 1, 0], [1, 2, 0], [0, 2, 0],
                  [0, 0, 1], [2, 0, 1], [2, 1, 1], [1, 1, 1], [1, 2, 1], [0, 2, 1]], np.float32) - 0.75
    idx = [[0, 2, 1], [0, 3, 2], [0, 5, 3], [3, 5, 4],  # bottom
           [6, 7, 8], [6, 8, 9], [6, 9, 11], [9, 10, 11]]  # top
    for a in range(6):  # sides
        b = (a + 1) % 6
        idx += [[a, b, b + 6], [a, b + 6, a + 6]]
    return v, np.array(idx, np.int32)


def mixed_scene(pt, extra=()):
    s = pt.Scene()
    grey = s.add_material(pt.lambertian((0.5, 0.5, 0.5)))
    s.add_plane((0, -2, 0), (0, 1, 0), s.add_material(pt.emissive((1.0, 1.0, 1.0))))  # planes are never sampled
    s.add_sphere((0, 3, 0), 0.25, s.add_material(pt.emissive((20.0, 10.0, 5.0))))
    s.add_sphere((3, 0, 0), 0.5, s.add_material(pt.emissive((0.0, 0.0, 0.0))))  # no radiance
    s.add_quad(s.add_material(pt.emissive((2.0, 2.0, 2.0))), scale=(1.5, 1, 0.5), rotation=(90, 0, 0), position=(0, 2.5, -2))
    s.add_cube(s.add_material(pt.emissive((0.5, 3.0, 1.0))), scale=(0.5, 1.0, 2.0), rotation=(20, 35, 10), position=(-2, 0, 0))
    v, idx = _box_mesh()
    s.add_mesh(v, idx, s.add_material(pt.emissive((0.3, 0.2, 0.1))), scale=(1.0, 2.0, 0.5), rotation=(30, 45, 60), position=(2, 0, 1))
    s.add_sphere((0, -1, 2), 0.4, grey)
    for e in extra:
        e(s)
    return s


def _world_tris(pt, scene, obj):
    o = scene.objects[obj]
    t = scene.mesh(o.mesh).astype(np.float64)
    o2w = np.asarray(o.o2w, np.float64).reshape(4, 4).T  # column-major
    pts = np.concatenate([t[:, 0:9].reshape(-1, 3, 3), np.ones((len(t), 3, 1))], axis=2) @ o2w.T
    return pts[..., :3]


def _cube_faces(scene, obj):
    o2w = np.asarray(scene.objects[obj].o2w, np.float64).reshape(4, 4).T
    a = o2w[:3, :3]
    areas = []
    for ax in range(3):
        u, v = a[:, (ax + 1) % 3], a[:, (ax + 2) % 3]
        areas += [np.linalg.norm(np.cross(u, v))] * 2
    return np.array(areas)


def test_tables_match_float64(pt):
    scene = mixed_scene(pt)
    sim = SimEmitters(scene)
    toc, area, cdf = sim.lights()
    objs = scene.objects
    # sampled: the emissive sphere, quad, cube and mesh with radiance, in object order; not the plane, not the black sphere
    assert list(toc[:, 1]) == [1, 3, 4, 5]
    assert list(toc[:, 0]) == [pt.OBJ_SPHERE, pt.OBJ_QUAD, pt.OBJ_CUBE, pt.OBJ_MESH]
    ids = sim.light_ids()
    assert list(ids) == [0, 1, 0, 2, 3, 4, 0]
    # areas in float64
    mats = scene.materials
    r_sph = objs[1].radius
    q = objs[3]
    a_quad = np.linalg.norm(np.cross(np.asarray(q.edge0, np.float64), np.asarray(q.edge1, np.float64)))
    a_cube = _cube_faces(scene, 4)
    w = _world_tris(pt, scene, 5)
    _, _, _, dead, _ = OracleScene(scene).mesh_bvh_info(5, len(w))
    a_tri = 0.5 * np.linalg.norm(np.cross(w[:, 1] - w[:, 0], w[:, 2] - w[:, 0]), axis=1) * (dead == 0)
    want_area = np.array([4 * np.pi * r_sph ** 2, a_quad, a_cube.sum(), a_tri.sum()])
    np.testing.assert_allclose(area, want_area, rtol=2e-6)
    rad = np.array([max(mats[objs[k].material].albedo) for k in (1, 3, 4, 5)], np.float64)
    pw = rad * want_area
    want_cdf = np.concatenate([[0.0], np.cumsum(pw) / pw.sum()])
    np.testing.assert_allclose(cdf, want_cdf, rtol=0, atol=2e-7)
    assert cdf[0] == 0.0 and cdf[-1] == 1.0 and np.all(np.diff(cdf) > 0)
    # the cube: six faces by area (non-uniform scale, no shear)
    ccdf, cent = sim.entries(2)
    np.testing.assert_allclose(np.diff(ccdf), a_cube / a_cube.sum(), rtol=0, atol=2e-7)
    # the mesh: its triangles in original order, by world area (rotated, non-uniformly scaled)
    mcdf, ment = sim.entries(3)
    assert len(mcdf) == len(a_tri) + 1
    np.testing.assert_allclose(np.diff(mcdf), a_tri / a_tri.sum(), rtol=0, atol=2e-7)
    np.testing.assert_allclose(ment[:, 0, :3], w[:, 0], rtol=0, atol=1e-5)
    np.testing.assert_allclose(ment[:, 1, :3], w[:, 1] - w[:, 0], rtol=0, atol=1e-5)
    np.testing.assert_allclose(ment[:, 2, :3], w[:, 2] - w[:, 0], rtol=0, atol=1e-5)
    # the record normal is the geometric one (the package derives a mesh's normals from its vertices), up to sign
    ng = np.cross(w[:, 1] - w[:, 0], w[:, 2] - w[:, 0])
    ng /= np.linalg.norm(ng, axis=1, keepdims=True)
    nrec = ment[:, :, 3]
    np.testing.assert_allclose(np.abs(np.sum(ng * nrec, axis=1)), 1.0, atol=1e-5)


def test_non_finite_and_huge_emitters(pt):
    def add(s):
        s.add_sphere((5, 5, 5), 0.5, s.add_material(pt.emissive((float("inf"), 1.0, 1.0))))
        s.add_sphere((-5, 5, 5), 0.5, s.add_material(pt.emissive((3e7, 3e7, 3e7))))
        s.add_sphere((-5, -5, 5), 0.5, s.add_material(pt.emissive((float("nan"), 1.0, 1.0))))
        s.add_sphere((5, -5, 5), 0.5, s.add_material(pt.emissive((1.0, float("nan"), 1.0))))
        s.add_cube(s.add_material(pt.emissive((1.0, 1.0, float("nan")))), position=(5, -5, -5))
        s.add_sphere((-5, -5, -5), 0.5, s.add_material(pt.emissive((1.0, 1.0, float("-inf")))))
    scene = mixed_scene(pt, [add])
    sim = SimEmitters(scene)
    toc, area, cdf = sim.lights()
    assert list(toc[:, 1]) == [1, 3, 4, 5, 8]  # the 3e7 sphere; no emitter with a non-finite channel
    assert np.all(np.isfinite(cdf)) and cdf[-1] == 1.0 and np.all(np.diff(cdf) >= 0)
    assert cdf[-1] - cdf[-2] > 0.99  # the 3e7 sphere dominates, with a finite weight
    assert list(sim.light_ids()[7:]) == [0, 5, 0, 0, 0, 0]


def test_cap_of_63_lights(pt):
    s = pt.Scene()
    m = s.add_material(pt.emissive((1.0, 1.0, 1.0)))
    for i in range(70):
        s.add_cube(m, scale=(0.1, 0.1, 0.1), position=(i, 0, 0))
    sim = SimEmitters(s)
    toc, _, cdf = sim.lights()
    assert len(toc) == 63 and list(toc[:, 1]) == list(range(63))
    ids = sim.light_ids()
    assert list(ids[:63]) == list(range(1, 64)) and not ids[63:].any()
    np.testing.assert_allclose(np.diff(cdf), 1 / 63, atol=1e-6)


def test_text_mesh_dead_triangles_have_probability_zero(pt):
    s = pt.Scene()
    obj = s.add_obj(TEXT_OBJ, s.add_material(pt.emissive((4.0, 4.0, 4.0))), scale=(1.0, 0.5, 2.0), rotation=(10, 20, 30))
    sim = SimEmitters(s)
    n = len(s.mesh(s.objects[obj].mesh))
    assert n == 4748
    _, _, _, dead, _ = OracleScene(s).mesh_bvh_info(obj, n)
    assert int(dead.sum()) == 1982
    cdf, _ = sim.entries(0)
    p = np.diff(cdf.astype(np.float64))
    assert np.all(p[dead.astype(bool)] == 0.0)
    w = _world_tris(pt, s, obj)
    a = 0.5 * np.linalg.norm(np.cross(w[:, 1] - w[:, 0], w[:, 2] - w[:, 0]), axis=1) * (dead == 0)
    np.testing.assert_allclose(p, a / a.sum(), rtol=0, atol=2e-7)
    # and the sampler never draws one
    u4 = np.random.default_rng(3).random((1 << 16, 4), dtype=np.float32)
    x = np.tile(np.array([[0.0, 0.0, 30.0]], np.float32), (len(u4), 1))
    _, _, _, o, tri = sim.sample(x, u4)
    drawn = tri[tri >= 0]
    assert len(drawn) > 0.9 * len(u4) and not dead[drawn].any()


def test_points_on_the_chosen_entry_and_histogram(pt):
    scene = mixed_scene(pt)
    sim = SimEmitters(scene)
    n = 1 << 18
    u4 = np.random.default_rng(5).random((n, 4), dtype=np.float32)
    x = np.tile(np.array([[0.2, -1.5, 4.0]], np.float32), (n, 1))
    p, pdf, pmis, obj, tri = sim.sample(x, u4)
    ok = obj >= 0
    assert ok.mean() > 0.95
    # mesh samples: on the reported triangle
    mcdf, ment = sim.entries(3)
    m = obj == 5
    t = tri[m]
    v0, e1, e2 = ment[t, 0, :3].astype(np.float64), ment[t, 1, :3].astype(np.float64), ment[t, 2, :3].astype(np.float64)
    rel = p[m] - v0
    g = np.stack([e1, e2], axis=2)
    st, *_ = zip(*[np.linalg.lstsq(g[i], rel[i], rcond=None) for i in range(min(len(t), 4000))])
    st = np.array(st)
    resid = np.linalg.norm(np.einsum("nij,nj->ni", g[:len(st)], st) - rel[:len(st)], axis=1)
    assert resid.max() < 1e-4
    assert st.min() > -1e-4 and st.sum(axis=1).max() < 1 + 1e-4
    # the triangles with the tables' probabilities (chi-square over the mesh's 28 triangles)
    counts = np.bincount(t, minlength=len(mcdf) - 1).astype(np.float64)
    expect = np.diff(mcdf.astype(np.float64)) * counts.sum()
    chi2 = np.sum((counts - expect) ** 2 / np.maximum(expect, 1))
    assert chi2 < 80, chi2
    # cube samples: on a face of the unit cube in object space
    c = obj == 4
    w2o = np.asarray(scene.objects[4].w2o, np.float64).reshape(4, 4).T
    po = (np.concatenate([p[c], np.ones((c.sum(), 1))], axis=1) @ w2o.T)[:, :3]
    assert np.abs(np.abs(po).max(axis=1) - 0.5).max() < 1e-4 and np.abs(po).max() < 0.5 + 1e-4
    # emitter choice by power
    toc, _, cdf = sim.lights()
    frac = np.array([(obj == o).sum() for o in toc[:, 1]]) / ok.sum()
    np.testing.assert_allclose(frac, np.diff(cdf), atol=0.01)


def test_divisor_and_mis_density_agree(pt):
    """geometric normals: the estimator's divisor, the MIS density of the light sample and the density a BSDF ray along the
    sampled direction is given (scene_hit over the same object table) are one density"""
    scene = mixed_scene(pt)
    sim = SimEmitters(scene)
    n = 1 << 15
    u4 = np.random.default_rng(9).random((n, 4), dtype=np.float32)
    x = np.tile(np.array([[0.2, -1.5, 4.0]], np.float32), (n, 1))
    p, pdf, pmis, obj, tri = sim.sample(x, u4)
    ok = obj >= 0
    np.testing.assert_allclose(pdf[ok], pmis[ok], rtol=2e-3)
    d = p[ok] - x[ok]
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    # the BSDF side: the closest hit along the direction; where it is the sampled point (not occluded) the densities agree
    back = sim.pdf(x[ok], d)
    hits = OracleScene(scene).intersect(pt, x[ok], d)
    dist = np.linalg.norm(p[ok] - x[ok], axis=1)
    # (meshes and cubes, away from grazing angles, where a point a hair off the sampled one changes the cosine a lot)
    cos = np.abs(np.sum(hits["normal"] * d, axis=1))
    vis = (hits["object"] == obj[ok]) & (np.linalg.norm(hits["position"] - p[ok], axis=1) < 1e-4 * dist) & (cos > 0.05)
    vis &= (obj[ok] == 4) | (obj[ok] == 5)
    assert vis.sum() > 2000
    # (a point on a cube's edge may be hit on the neighbouring face, whose normal the record then reports)
    agree = np.isclose(back[vis], pmis[ok][vis], rtol=2e-3, atol=0)
    assert agree.mean() > 0.999, agree.mean()


def test_flag_and_hooks_declared(pt):
    assert pt.FLAG_NEE_EMITTERS == 16
    hdr = open(os.path.join(ROOT, "include", "ptcore.h")).read()
    assert re.search(r"\bPTC_FLAG_NEE_EMITTERS\s*=\s*16\b", hdr)
    assert re.search(r"\bptc_light_sample\s*\(", hdr) and re.search(r"\bptc_light_pdf\s*\(", hdr)
    rs = open(os.path.join(ROOT, "rust", "ptcore-sys", "src", "lib.rs")).read()
    assert re.search(r"pub const PTC_FLAG_NEE_EMITTERS: i32 = 16;", rs)
    assert re.search(r"\bptc_light_sample\b", rs) and re.search(r"\bptc_light_pdf\b", rs)
