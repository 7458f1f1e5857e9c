#!/usr/bin/env python3
"""What a thin lens (ptc_scene_set_lens) costs.
  * C2 (semesterbild, 800x600, 256 spp, depth 30) at native settings: pinhole against a lens focused at half the depth
    of the text mesh, with the aperture that blurs the text mesh over a disk of about 10 px (R |1/z - 1/F| x W / (2
    half_width) = 10); 1 warm-up each, then 3 renders each, alternated;
  * a 64-view focus pull on C2's camera at 400x300, 64 spp, as one ptc_render_batch: one lens per view, F from half to
    twice the text mesh's depth, against the same batch without a lens;
One JSON line per measurement, then one with the GPU's name and power limit."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ptload  # noqa: E402

pt = ptload.load()
from raytracer_rust_b200 import workloads  # noqa: E402

label, s = workloads.workload("C2")
cs = s.to_core().commit(0)
cam = s.camera
pos = np.array(cam.position[:], np.float64)
fwd = np.array(cam.forward[:], np.float64)
fwd /= np.linalg.norm(fwd)
mesh = [o for o in s.objects if o.type == pt.OBJ_MESH][0]
tris = s.mesh(mesh.mesh)
o2w = np.array(mesh.o2w[:], np.float64).reshape(4, 4).T
v = tris[:, 0:9].reshape(-1, 3).astype(np.float64)
centre = (np.c_[v, np.ones(len(v))] @ o2w.T)[:, :3].mean(axis=0)
z = float((centre - pos) @ fwd)  # depth of the text mesh along the view axis
st = s.render_settings()
px = st.width / (2.0 * cam.half_width)
F = 0.5 * z
R = 10.0 / (px * abs(1.0 / z - 1.0 / F))

row = {"config": label, "text_mesh_depth": z, "lens": {"aperture_radius": R, "focus_distance": F, "blur_px_at_text": 10.0}}
for k in range(4):
    for name, lens in (("pinhole", None), ("lens", (R, F))):
        cs.set_lens(*lens) if lens else cs.set_lens()
        _, stats = cs.render(cam, st)
        if k > 0:
            row.setdefault(name + "_render_ms", []).append(stats.render_ms)
            row[name + "_rays"] = stats.rays
row["time_ratio_lens_over_pinhole"] = float(np.median(row["lens_render_ms"]) / np.median(row["pinhole_render_ms"]))
print(json.dumps(row), flush=True)

bst = s.render_settings(width=400, height=300, spp=64)
fs = np.geomspace(0.5 * z, 2.0 * z, 64)
R2 = 5.0 / ((bst.width / (2.0 * cam.half_width)) * abs(1.0 / z - 1.0 / (0.5 * z)))
row = {"measurement": "64-view focus pull, C2's camera at 400x300, 64 spp, depth 30, one ptc_render_batch",
       "aperture_radius": R2, "focus_distance": [float(fs[0]), float(fs[-1])]}
for k in range(3):
    for name, lenses in (("pinhole", []), ("lens", [(R2, float(f)) for f in fs])):
        cs.set_lens(lenses)
        _, _, stats = cs.render_batch([cam] * 64, bst)
        if k > 0:
            row.setdefault(name + "_render_ms", []).append(stats.render_ms)
row["time_ratio_lens_over_pinhole"] = float(np.median(row["lens_render_ms"]) / np.median(row["pinhole_render_ms"]))
print(json.dumps(row), flush=True)
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
print(json.dumps({"gpu": gpu.strip().splitlines()[0] if gpu.strip() else "unknown"}), flush=True)
