#!/usr/bin/env python3
"""What adaptive sampling (ptc_render_adaptive) costs and buys, at native frames (raytracer_rust_b200.workloads).

overhead: threshold 0 (every pixel to spp, the uniform image bit for bit) against ptc_render at the same spp, for C2,
  C3s (NEE | NEE_SKY), C4 (NEE) and C5; medians of 3 alternated renders, the number of passes, and where the time goes:
  a second pair of runs with PTC_FLAG_TIMING splits the adaptive render into the passes' extend + shade launches and
  the rest (decision kernels, compaction, count read-back, per-pass set-up and resolve).
quality: relMSE against a high-spp uniform render, for uniform sampling at `base_spp` and for adaptive renders with a
  few thresholds, each next to a uniform render of about the same time (spp scaled by the measured time per sample);
  sum of paths and the histogram of counts.
bias: the mean of adaptive images with and without NEE on the half-lit scene of tests/test_gpu_adaptive.py.
One JSON line per measurement, each with the GPU's name and power limit."""
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

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
GPU = smi.strip().splitlines()[0] if smi.strip() else "unknown"
NEE, NEE_SKY = pt.FLAG_NEE, pt.FLAG_NEE | pt.FLAG_NEE_SKY


def emit(row):
    row["gpu"] = GPU
    print(json.dumps(row), flush=True)


def relmse(a, b):
    return float(np.mean((a - b) ** 2 / (b ** 2 + 1e-2)))


def passes(counts, min_spp, spp):
    n, k = min_spp, 2
    top = int(counts.max())
    while n < top:
        n = min(2 * n, spp)
        k += 1
    return k


def overhead(cfg, flags, min_spp):
    label, s = workloads.workload(cfg)
    cs = s.to_core().commit(0)
    st = s.render_settings(seed=2, flags=flags)
    cs.render(s.camera, st)
    cs.render_adaptive(s.camera, st, min_spp, 0.0)  # warm-up of both
    uni, ada = [], []
    for _ in range(3):
        uni.append(cs.render(s.camera, st)[1].render_ms)
        _, _, cnt, a = cs.render_adaptive(s.camera, st, min_spp, 0.0)
        ada.append(a.render_ms)
    stt = s.render_settings(seed=2, flags=flags | pt.FLAG_TIMING)
    ut = cs.render(s.camera, stt)[1]
    _, _, cnt, at = cs.render_adaptive(s.camera, stt, min_spp, 0.0)
    um, am = float(np.median(uni)), float(np.median(ada))
    emit({"measurement": "overhead: threshold 0 against the uniform render at the same spp", "config": label, "flags": flags,
          "spp": st.spp, "min_spp": min_spp, "passes": passes(cnt, min_spp, st.spp),
          "uniform_render_ms": uni, "adaptive_render_ms": ada, "uniform_median_ms": um, "adaptive_median_ms": am,
          "overhead_ms": am - um, "overhead_pct": 100.0 * (am - um) / um,
          "timing_runs": {"uniform": {"render_ms": ut.render_ms, "extend_ms": ut.extend_ms, "shade_ms": ut.shade_ms, "iterations": ut.iterations},
                          "adaptive": {"render_ms": at.render_ms, "extend_ms": at.extend_ms, "shade_ms": at.shade_ms, "iterations": at.iterations,
                                       "outside_extend_and_shade_ms": at.render_ms - at.extend_ms - at.shade_ms}}})
    del cs


def quality(cfg, flags, base_spp, ref_spp, min_spp, max_spp, thresholds):
    label, s = workloads.workload(cfg)
    cs = s.to_core().commit(0)
    ref, _ = cs.render(s.camera, s.render_settings(spp=ref_spp, seed=1, flags=flags))
    cs.render(s.camera, s.render_settings(spp=base_spp, seed=2, flags=flags))
    img, ust = cs.render(s.camera, s.render_settings(spp=base_spp, seed=2, flags=flags))
    ms_per_spp = ust.render_ms / base_spp
    rows = {"uniform": {"spp": base_spp, "relmse": relmse(img, ref), "render_ms": ust.render_ms, "paths": ust.paths}}
    for thr in thresholds:
        st = s.render_settings(spp=max_spp, seed=2, flags=flags)
        cs.render_adaptive(s.camera, st, min_spp, thr)
        rgb, _, cnt, ast = cs.render_adaptive(s.camera, st, min_spp, thr)
        eq_spp = max(1, int(round(ast.render_ms / ms_per_spp)))
        uimg, eq = cs.render(s.camera, s.render_settings(spp=eq_spp, seed=2, flags=flags))
        vals, num = np.unique(cnt, return_counts=True)
        e_a, e_u = relmse(rgb, ref), relmse(uimg, ref)
        rows[f"adaptive_thr_{thr}"] = {
            "threshold": thr, "min_spp": min_spp, "max_spp": max_spp, "relmse": e_a, "render_ms": ast.render_ms, "paths": ast.paths,
            "mean_spp": ast.paths / cnt.size, "passes": passes(cnt, min_spp, max_spp),
            "count_histogram": {int(v): int(k) for v, k in zip(vals, num)},
            "equal_time_uniform": {"spp": eq_spp, "relmse": e_u, "render_ms": eq.render_ms, "paths": eq.paths},
            "error_ratio_uniform_over_adaptive": e_u / e_a, "adaptive_wins": bool(e_a < e_u)}
    emit({"measurement": "equal-time quality", "config": label, "flags": flags, "reference": f"uniform render at {ref_spp} spp",
          **rows})
    del cs


def half_lit_scene():
    """tests/test_gpu_adaptive.py's scene: left the constant gray background, right a diffuse and a plastic sphere under
    a small bright light"""
    s = pt.Scene()
    s.add_sphere((1.2, 0.0, -4.0), 1.5, s.add_material(pt.lambertian((0.7, 0.6, 0.5))))
    s.add_sphere((0.55, -0.75, -2.8), 0.4, s.add_material(pt.plastic((0.3, 0.4, 0.8))))
    s.add_sphere((0.4, 1.6, -2.5), 0.25, s.add_material(pt.emissive((30.0, 28.0, 24.0))))
    s.set_camera((0, 0, 0), (0, 0, -1), (0, 1, 0), 40.0, 1.0)
    s.set_settings(128, 128, 256, 8)
    return s


def bias():
    """early stopping with and without NEE: mean of the image against the plain 8192-spp render, adaptive and uniform at
    equal paths, over 4 seeds"""
    s = half_lit_scene()
    cs = s.to_core().commit(0)
    ref, _ = cs.render(s.camera, s.render_settings(spp=8192, seed=1))
    for flags in (0, NEE):
        for min_spp in (8, 16):
            ada, uni = [], []
            for seed in range(2, 6):
                rgb, _, cnt, st = cs.render_adaptive(s.camera, s.render_settings(seed=seed, flags=flags), min_spp, 0.02)
                u, _ = cs.render(s.camera, s.render_settings(spp=-(-int(st.paths) // cnt.size), seed=seed, flags=flags))
                ada.append(float(rgb.mean() / ref.mean() - 1.0))
                uni.append(float(u.mean() / ref.mean() - 1.0))
            emit({"measurement": "mean of the image relative to the plain 8192-spp render (half-lit test scene 128x128, depth 8, "
                                 "spp 256, threshold 0.02), adaptive and uniform at equal paths, seeds 2-5",
                  "flags": flags, "min_spp": min_spp, "adaptive_rel_mean_error": ada, "uniform_rel_mean_error": uni})


only = sys.argv[1:]
if not only or "overhead" in only:
    for cfg, flags, min_spp in (("C2", 0, 16), ("C3s", NEE_SKY, 16), ("C4", NEE, 16), ("C5", 0, 16)):
        overhead(cfg, flags, min_spp)
if not only or "quality" in only:
    for cfg, flags, ref_spp in (("C1", NEE, 16384), ("C4", NEE, 8192), ("C3s", NEE_SKY, 8192), ("C2", 0, 4096)):
        quality(cfg, flags, 64, ref_spp, 16, 512, (0.01, 0.03, 0.1))
if not only or "bias" in only:
    bias()
