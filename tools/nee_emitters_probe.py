#!/usr/bin/env python3
"""What PTC_FLAG_NEE_EMITTERS buys, and what it costs at commit.
  * an emissive-mesh scene at 1280x720 (a closed room lit by the text mesh as a sign and a 2-triangle mesh light panel):
    error against a converged plain render at equal spp, and the render time, of plain, PTC_FLAG_NEE and
    PTC_FLAG_NEE | PTC_FLAG_NEE_EMITTERS (PTC_FLAG_NEE samples no mesh: it is the plain integrator there);
  * the mixed scene of tests/test_gpu_nee_emitters.py at 1280x720 (a closed, dark room lit by a small bright sphere, a
    large dim curved mesh panel and a small quad): plain, PTC_FLAG_NEE and PTC_FLAG_NEE | PTC_FLAG_NEE_EMITTERS;
  * veach-mis (C4): PTC_FLAG_NEE against PTC_FLAG_NEE | PTC_FLAG_NEE_EMITTERS, same emitters, only the selection differs;
  * commit time of C5's 2 M-triangle height field as a lone mesh, Lambertian against emissive (the emitter tables);
One JSON line per measurement, then one with the GPU's name and power limit."""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ptload  # noqa: E402

pt = ptload.load()
from raytracer_rust_b200 import workloads  # noqa: E402

TEXT_OBJ = os.path.join(ROOT, "scenes", "RayTracingText.obj")
NEE, EM = pt.FLAG_NEE, pt.FLAG_NEE | pt.FLAG_NEE_EMITTERS


def relmse(a, b):
    return float(np.mean((a - b) ** 2 / (b ** 2 + 1e-2)))


def sign_room():
    s = pt.Scene()
    grey, red, green = (s.add_material(pt.lambertian(c)) for c in ((0.7, 0.7, 0.7), (0.7, 0.2, 0.2), (0.2, 0.7, 0.2)))
    s.add_quad(grey, scale=(2, 1, 2), position=(0, 0, 0))
    s.add_quad(grey, scale=(2, 1, 2), rotation=(180, 0, 0), position=(0, 2, 0))
    s.add_quad(grey, scale=(2, 1, 2), rotation=(90, 0, 0), position=(0, 1, -1))
    s.add_quad(grey, scale=(2, 1, 5), rotation=(90, 0, 0), position=(0, 1, 4))  # closes the room behind the camera
    s.add_quad(red, scale=(2, 1, 5), rotation=(0, 0, 90), position=(-1, 1, 1.5))
    s.add_quad(green, scale=(2, 1, 5), rotation=(0, 0, 90), position=(1, 1, 1.5))
    s.add_sphere((-0.4, 0.35, -0.2), 0.35, s.add_material(pt.lambertian((0.8, 0.8, 0.8))))
    s.add_cube(s.add_material(pt.plastic((0.3, 0.4, 0.8), 1.5)), scale=(0.5, 0.7, 0.5), rotation=(0, 25, 0), position=(0.4, 0.35, 0.1))
    s.add_obj(TEXT_OBJ, s.add_material(pt.emissive((6.0, 3.0, 1.5))), scale=(0.09, 0.14, 0.05), rotation=(8, -12, 4), position=(0, 1.3, -0.85))
    o2w, _ = pt.transform((0.6, 1, 0.4), (15, 0, 0), (0, 1.85, 0))
    m = o2w.astype(np.float64).reshape(4, 4).T
    v = (np.array([[-0.5, 0, -0.5, 1], [0.5, 0, -0.5, 1], [0.5, 0, 0.5, 1], [-0.5, 0, 0.5, 1]]) @ m.T)[:, :3].astype(np.float32)
    s.add_mesh(v, np.array([[0, 1, 2], [0, 2, 3]], np.int32), s.add_material(pt.emissive((12.0, 11.0, 9.0))))
    s.set_camera((0, 1, 3.6), (0, 1, 0), (0, 1, 0), 40.0, 16 / 9)
    return s


def mixed_room():
    """the closed, dark room of the mixed scene: walls of albedo 0.25 x (0.7 grey, red, green), so direct light dominates"""
    s = pt.Scene()
    grey, red, green = (s.add_material(pt.lambertian(tuple(0.25 * x for x in c))) for c in ((0.7, 0.7, 0.7), (0.7, 0.2, 0.2), (0.2, 0.7, 0.2)))
    for m, kw in ((grey, dict(scale=(2, 1, 2), position=(0, 0, 0))), (grey, dict(scale=(2, 1, 2), rotation=(180, 0, 0), position=(0, 2, 0))),
                  (grey, dict(scale=(2, 1, 2), rotation=(90, 0, 0), position=(0, 1, -1))),
                  (red, dict(scale=(2, 1, 2), rotation=(0, 0, 90), position=(-1, 1, 0))),
                  (green, dict(scale=(2, 1, 2), rotation=(0, 0, 90), position=(1, 1, 0))),
                  (grey, dict(scale=(2, 1, 3), position=(0, 0, 2.5))), (grey, dict(scale=(2, 1, 3), rotation=(180, 0, 0), position=(0, 2, 2.5))),
                  (grey, dict(scale=(2, 1, 3), rotation=(0, 0, 90), position=(-1, 1, 2.5))),
                  (grey, dict(scale=(2, 1, 3), rotation=(0, 0, 90), position=(1, 1, 2.5))),
                  (grey, dict(scale=(2, 1, 2), rotation=(90, 0, 0), position=(0, 1, 4)))):
        s.add_quad(m, **kw)
    s.add_sphere((-0.4, 0.35, -0.2), 0.35, s.add_material(pt.lambertian((0.8, 0.8, 0.8))))
    s.add_cube(s.add_material(pt.plastic((0.3, 0.4, 0.8), 1.5)), scale=(0.5, 0.7, 0.5), rotation=(0, 25, 0), position=(0.4, 0.35, 0.1))
    s.add_sphere((-0.6, 1.7, 0.2), 0.08, s.add_material(pt.emissive((40.0, 38.0, 30.0))))
    n = 8
    g = np.linspace(-0.5, 0.5, n + 1, dtype=np.float32)
    x, z = np.meshgrid(g, g, indexing="ij")
    v = np.stack([x, 0.25 * (x * x + z * z), z], axis=-1).reshape(-1, 3)
    idx = []
    for i in range(n):
        for j in range(n):
            a, b, c, d = i * (n + 1) + j, (i + 1) * (n + 1) + j, (i + 1) * (n + 1) + j + 1, i * (n + 1) + j + 1
            idx += [[a, b, c], [a, c, d]]
    s.add_mesh(v, np.array(idx, np.int32), s.add_material(pt.emissive((2.5, 2.5, 3.0))), scale=(1.0, 1.0, 0.8), rotation=(0, 20, 0),
               position=(0.2, 1.7, -0.3))
    s.add_quad(s.add_material(pt.emissive((3.0, 3.0, 3.0))), scale=(0.3, 1, 0.3), rotation=(100, 0, 0), position=(0.6, 0.9, -0.98))
    s.set_camera((0, 1, 3.6), (0, 1, 0), (0, 1, 0), 40.0, 16 / 9)
    return s


def compare(label, s, st_kw, spp, ref_spp, ref_flags, integrators):
    cs = s.to_core().commit(0)
    ref, _ = cs.render(s.camera, s.render_settings(spp=ref_spp, seed=1, flags=ref_flags, **st_kw))
    row = {"config": label, "spp": spp, "reference": f"flags {ref_flags} at {ref_spp} spp"}
    for name, flags in integrators:
        cs.render(s.camera, s.render_settings(spp=spp, seed=2, flags=flags, **st_kw))  # warm-up
        img, st = cs.render(s.camera, s.render_settings(spp=spp, seed=2, flags=flags, **st_kw))
        row[name] = {"relmse": relmse(img, ref), "render_ms": st.render_ms, "rays": st.rays}
    base = integrators[0][0]
    for name, _ in integrators[1:]:
        err = row[base]["relmse"] / row[name]["relmse"]
        tim = row[name]["render_ms"] / row[base]["render_ms"]
        row[f"error_ratio_{base}_over_{name}"] = err
        row[f"time_ratio_{name}_over_{base}"] = tim
        row[f"efficiency_gain_{name}_over_{base}"] = err / tim
    print(json.dumps(row), flush=True)


compare("sign room 1280x720 depth 8 (text mesh sign, 4,748 triangles, 1,982 dead, + 2-triangle mesh light panel)", sign_room(),
        dict(width=1280, height=720, max_depth=8), 64, 4096, 0, (("plain", 0), ("nee", NEE), ("nee_emitters", EM)))
compare("mixed room 1280x720 depth 8 (sphere r 0.08, 128-triangle curved mesh panel, small quad; dark closed room)", mixed_room(),
        dict(width=1280, height=720, max_depth=8), 64, 4096, 0, (("plain", 0), ("nee", NEE), ("nee_emitters", EM)))
label, c4 = workloads.workload("C4")
compare(label, c4, {}, 64, 8192, NEE, (("nee", NEE), ("nee_emitters", EM)))

# commit time: C5's height field alone, Lambertian vs emissive (the emitter tables are built only for emissive meshes)
_, c5 = workloads.workload("C5")
mesh_obj = [o for o in c5.objects if o.type == pt.OBJ_MESH][0]
tris = c5.mesh(mesh_obj.mesh)
verts = np.ascontiguousarray(tris[:, 0:9].reshape(-1, 3))
idx = np.arange(len(verts), dtype=np.int32).reshape(-1, 3)
row = {"measurement": f"commit ms of C5's height field ({len(tris)} triangles) as a lone mesh, 3 commits each, alternated"}
for k in range(3):
    for name, mat in (("lambert", pt.lambertian((0.5, 0.5, 0.5))), ("emissive", pt.emissive((1.0, 1.0, 1.0)))):
        s = pt.Scene()
        s.add_mesh(verts, idx, s.add_material(mat))
        core = s.to_core()
        t0 = time.perf_counter()
        core.commit(0)
        row.setdefault(name + "_commit_ms", []).append((time.perf_counter() - t0) * 1e3)
        del core
print(json.dumps(row), flush=True)
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
print(json.dumps({"gpu": gpu.strip().splitlines()[0] if gpu.strip() else "unknown"}), flush=True)
