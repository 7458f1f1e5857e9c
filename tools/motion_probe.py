#!/usr/bin/env python3
"""What motion blur (ptc_scene_set_object_motion / ptc_scene_set_camera_motion) costs.
  * C2 (semesterbild, 800x600, 256 spp, depth 30) at native settings:
      - static against the text mesh displaced by 1e-3 units over the shutter: the pure overhead of the motion kernels
        (the tau array read and written per ray, the per-object displacement test), the image all but unchanged;
      - the text mesh moving about 20 px across the frame;
      - a camera pan: the end camera's forward turned by about 20 px at the image centre;
  * C4 (veach-mis) at 1280x720, 128 spp, depth 16, under PTC_FLAG_NEE: static against its emissive spheres moving by
    about one radius;
  * a 64-view batch on C2's camera at 400x300, 64 spp, every view with its own end camera (a pan of 0 to 20 px), against
    the same batch without motion.
Each pair: one warm-up each, then 3 renders each (the batch: 2), alternated; medians.  Every JSON line carries the GPU's name and
power limit.  `--out FILE` also writes the lines to FILE (profiles/r3_motion_probe.jsonl holds a run's)."""
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

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
GPU = gpu.strip().splitlines()[0] if gpu.strip() else "unknown"
rows = []


def emit(row):
    row["gpu"] = GPU
    rows.append(row)
    print(json.dumps(row), flush=True)


def alternate(row, variants, render, reps=3):
    """variants: (name, setup) pairs; setup() prepares the handle.  One warm-up each, then `reps` rounds alternated."""
    for k in range(reps + 1):
        for name, setup in variants:
            setup()
            stats = render()
            if k > 0:
                row.setdefault(name + "_render_ms", []).append(stats.render_ms)
                row[name + "_rays"] = stats.rays
    for name, _ in variants:
        row[name + "_median_ms"] = float(np.median(row[name + "_render_ms"]))
    base = variants[0][0]
    for name, _ in variants[1:]:
        row[f"time_ratio_{name}_over_{base}"] = row[name + "_median_ms"] / row[base + "_median_ms"]
    return row


def unit(v):
    v = np.asarray(v, np.float64)
    return v / np.linalg.norm(v)


# ---- C2
label, s = workloads.workload("C2")
cs = s.to_core().commit(0)
cam = s.camera
st = s.render_settings()
pos, fwd, rgt = np.array(cam.position[:], np.float64), unit(cam.forward[:]), unit(cam.right[:])
mesh_k = [k for k, o in enumerate(s.objects) if o.type == pt.OBJ_MESH][0]
mesh = s.objects[mesh_k]
tris = s.mesh(mesh.mesh)
o2w = np.array(mesh.o2w[:], np.float64).reshape(4, 4).T
v = tris[:, 0:9].reshape(-1, 3).astype(np.float64)
centre = (np.c_[v, np.ones(len(v))] @ o2w.T)[:, :3].mean(axis=0)
z = float((centre - pos) @ fwd)  # depth of the text mesh along the view axis
px_per_ndc = st.width / (2.0 * cam.half_width)  # pixels per unit of lateral offset / depth (unit forward)
d20 = 20.0 / px_per_ndc * z  # world units that move a point at the text mesh's depth by 20 px
D20 = (rgt * d20).astype(np.float32)

pan = pt.Camera.from_buffer_copy(cam)
nf = np.array(cam.forward[:], np.float64) + np.linalg.norm(cam.forward[:]) * (20.0 / px_per_ndc) * rgt
for i in range(3):
    pan.forward[i] = float(nf[i])


def static():
    cs.set_object_motion(mesh_k, (0.0, 0.0, 0.0))
    cs.set_camera_motion()


def tiny():
    cs.set_camera_motion()
    cs.set_object_motion(mesh_k, (1e-3, 0.0, 0.0))


def moving():
    cs.set_camera_motion()
    cs.set_object_motion(mesh_k, D20)


def panning():
    cs.set_object_motion(mesh_k, (0.0, 0.0, 0.0))
    cs.set_camera_motion(pan)


render = lambda: cs.render(cam, st)[1]  # noqa: E731
emit(alternate({"config": label, "measurement": "C2 native: static vs the text mesh displaced by 1e-3 units"},
               [("static", static), ("tiny_motion", tiny)], render))
emit(alternate({"config": label, "measurement": "C2 native: the text mesh moving ~20 px, and a ~20 px camera pan",
                "text_mesh_depth": z, "displacement": [float(x) for x in D20]},
               [("static", static), ("mesh_20px", moving), ("pan_20px", panning)], render))

# ---- a 64-view batch with per-view end cameras
bst = s.render_settings(width=400, height=300, spp=64)
ends = []
for k in range(64):
    e = pt.Camera.from_buffer_copy(cam)
    f = np.array(cam.forward[:], np.float64) + np.linalg.norm(cam.forward[:]) * (20.0 * k / 63 / (bst.width / (2.0 * cam.half_width))) * rgt
    for i in range(3):
        e.forward[i] = float(f[i])
    ends.append(e)
static()
emit(alternate({"measurement": "64-view batch, C2's camera at 400x300, 64 spp, depth 30, one ptc_render_batch; per-view end "
                               "cameras panning 0 to 20 px"},
               [("static", lambda: cs.set_camera_motion()), ("per_view_end_cameras", lambda: cs.set_camera_motion(ends))],
               lambda: cs.render_batch([cam] * 64, bst)[2], reps=2))

# ---- C4 under PTC_FLAG_NEE, its emissive spheres moving
label4, s4 = workloads.workload("C4")
cs4 = s4.to_core().commit(0)
st4 = s4.render_settings(spp=128, flags=pt.FLAG_NEE)
spheres = [k for k, o in enumerate(s4.objects) if o.type == pt.OBJ_SPHERE]
radii = [float(s4.objects[k].radius) for k in spheres]


def c4_static():
    for k in spheres:
        cs4.set_object_motion(k, (0.0, 0.0, 0.0))


def c4_moving():
    for k, r in zip(spheres, radii):
        cs4.set_object_motion(k, (r, 0.0, 0.0))


emit(alternate({"config": label4 + " (here 128 spp)", "measurement": "C4 under PTC_FLAG_NEE: static vs its emissive spheres "
                "moving by one radius", "spheres": spheres, "radii": radii},
               [("static", c4_static), ("lights_moving", c4_moving)], lambda: cs4.render(s4.camera, st4)[1]))

if "--out" in sys.argv:  # e.g. --out profiles/r3_motion_probe.jsonl
    out = sys.argv[sys.argv.index("--out") + 1]
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        for r in rows:
            f.write(json.dumps(r) + "\n")
