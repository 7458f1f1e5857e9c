#!/usr/bin/env python3
"""Commit time and traversal quality of the mesh builders on one B200: host (SAH + DP collapse), device (reference tree
as the wide tree), device-sah (the host's SAH tree built on the device) and hybrid (the default commit), for C5
(2 M triangles), C3 (teapot) and C2's text mesh.  PTC_BUILD_TIMING=1 prints the builders' own step times on stderr.  One
JSON line per (config, builder) plus one naming the GPU and its power limit.

  python tools/build_probe.py [config ...] [--modes host,device,device-sah,hybrid]"""
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ptload  # noqa: E402

pt = ptload.load()
from raytracer_rust_b200 import workloads  # noqa: E402

os.environ["PTC_BUILD_TIMING"] = "1"
args = sys.argv[1:]
modes = ("host", "device", "device")
if "--modes" in args:
    i = args.index("--modes")
    modes = tuple(args[i + 1].split(","))
    del args[i:i + 2]
import torch  # noqa: E402
import subprocess  # noqa: E402
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
print(json.dumps({"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi}), flush=True)
pt.synthetic_scene(cells=32).to_core().commit(0)  # context + module load outside the timings
for cfg in args or ["C5", "C3", "C2"]:
    label, scene = workloads.workload(cfg)
    w, h, spp, depth = scene.settings
    for mode in modes:
        if mode == "hybrid":
            os.environ.pop("PTC_BUILD", None)
        else:
            os.environ["PTC_BUILD"] = mode
        t0 = time.perf_counter()
        cs = scene.to_core().commit(0)
        commit_s = time.perf_counter() - t0
        st = scene.render_settings(spp=max(1, min(spp, 32)), seed=0, pool_paths=3 << 22)
        best = None
        for _ in range(4):
            _, s = cs.render_u32(scene.camera, st)
            if best is None or s.render_ms < best.render_ms:
                best = s
        st.flags = pt.FLAG_COUNTERS
        os.environ["PTC_STEAL"] = "0"
        _, c = cs.render_u32(scene.camera, scene.render_settings(spp=2, seed=0, flags=pt.FLAG_COUNTERS))
        os.environ.pop("PTC_STEAL")
        mesh_obj = [i for i, o in enumerate(scene.objects) if o.type == pt.OBJ_MESH][0]
        info = cs.mesh_info(mesh_obj)[0]
        print(json.dumps({"config": cfg, "builder": mode, "commit_s": commit_s, "wide_nodes": info.wide_nodes, "wide_depth": info.wide_depth,
                          "render_ms": best.render_ms, "mpaths_s": best.paths / best.render_ms / 1e3, "spp": st.spp,
                          "nodes_per_mesh_ray": c.nodes_visited / max(1, c.mesh_rays), "tris_per_mesh_ray": c.tris_tested / max(1, c.mesh_rays)}), flush=True)
