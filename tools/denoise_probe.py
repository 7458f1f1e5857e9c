#!/usr/bin/env python3
"""What denoised rendering (ptc_render_denoised) costs and gains, at native frames (raytracer_rust_b200.workloads).

Cost, for C1, C2, C3s, C4 and C5 at native spp and flags 0, feature_spp 4, 5 levels; medians of 3 alternated runs:
  * render_ms of ptc_render and of ptc_render_denoised (device events; the latter from the first pass to the end of the
    filter);
  * from one run under torch.profiler, the device-time windows of the feature pass (the first k_primary_rays to
    k_feature_mean) and of the filter (k_denoise_prepare to k_denoise_finish, 5 levels of k_atrous);
  * the rest: the split render's extra wavefront drain plus the snapshot, resolve and variance kernels
    (denoised - plain - feature - filter).
Quality, for C1 (NEE), C2, C3s (NEE | NEE_SKY) and C4 (NEE) at native resolution against a 4096-spp render of the same
integrator (another seed): relMSE (as tests/test_gpu_nee.py computes it) of the noisy and the denoised image at 4, 16 and
64 spp; a sweep of the filter parameters at 16 spp (ptc_denoise_image on the same inputs); and an equal-time row, the
denoised render at 16 spp against a plain render whose spp takes the same render_ms.
One JSON line per row, each with the GPU's name and power limit, printed and appended to the output file.

  python tools/denoise_probe.py [out.jsonl] [configs...]     (default: profiles/r3_denoise_probe.jsonl C1 C2 C3s C4 C5)
"""
import itertools
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
QUALITY_FLAGS = {"C1": pt.FLAG_NEE, "C2": 0, "C3s": pt.FLAG_NEE | pt.FLAG_NEE_SKY, "C4": pt.FLAG_NEE}
FEATURE_SPP, ITERATIONS = 4, 5


def relmse(a, b):  # tests/test_gpu_nee.py
    return float(np.mean((a - b) ** 2 / (b ** 2 + 1e-2)))


def kernel_windows(cs, s, st):
    """device-time windows (ms) of the feature pass and the filter in one profiled ptc_render_denoised"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        cs.render_denoised(s.camera, st, feature_spp=FEATURE_SPP, iterations=ITERATIONS)
        torch.cuda.synchronize()
    ks = [(e.name, e.time_range.start, e.time_range.end) for e in prof.events() if e.device_type.name == "CUDA"]

    def window(first, last):
        a = min(t0 for n, t0, _ in ks if first in n)
        b = max(t1 for n, _, t1 in ks if last in n)
        return (b - a) / 1e3

    return window("k_primary_rays", "k_feature_mean"), window("k_denoise_prepare", "k_denoise_finish"), \
        sum(1 for n, _, _ in ks if "k_atrous" in n)


def cost(cfg):
    label, s = workloads.workload(cfg)
    cs = s.to_core().commit(0)
    st = s.render_settings(seed=2)
    cs.render_u32(s.camera, st)
    cs.render_denoised(s.camera, st, feature_spp=FEATURE_SPP)  # warm-up of both
    plain, dn = [], []
    for _ in range(3):
        plain.append(cs.render(s.camera, st)[1].render_ms)
        dn.append(cs.render_denoised(s.camera, st, feature_spp=FEATURE_SPP, iterations=ITERATIONS)[6].render_ms)
    row = {"probe": "cost", "config": cfg, "workload": label, "width": st.width, "height": st.height, "spp": st.spp,
           "feature_spp": FEATURE_SPP, "iterations": ITERATIONS, "render_ms": float(np.median(plain)),
           "denoised_render_ms": float(np.median(dn)), "render_ms_runs": plain, "denoised_render_ms_runs": dn}
    try:
        feat, filt, n_atrous = kernel_windows(cs, s, st)
        row.update(feature_pass_ms=feat, filter_ms=filt, atrous_launches=n_atrous,
                   split_render_and_tail_ms=row["denoised_render_ms"] - row["render_ms"] - feat - filt)
    except Exception as e:  # the cost rows stand without the profile
        row.update(feature_pass_ms="not measured", filter_ms="not measured", profile_error=repr(e))
    return row


def quality(cfg):
    label, s = workloads.workload(cfg)
    cs = s.to_core().commit(0)
    flags = QUALITY_FLAGS[cfg]
    ref, _ = cs.render(s.camera, s.render_settings(spp=4096, seed=99, flags=flags))
    rows = []
    for spp in (4, 16, 64):
        st = s.render_settings(spp=spp, seed=2, flags=flags)
        rgb, _, noisy, albedo, normal, var, stats = cs.render_denoised(s.camera, st, feature_spp=min(spp, FEATURE_SPP))
        e_n, e_d = relmse(noisy, ref), relmse(rgb, ref)
        rows.append({"probe": "quality", "config": cfg, "flags": flags, "spp": spp, "reference_spp": 4096, "relmse_noisy": e_n,
                     "relmse_denoised": e_d, "ratio": e_d / e_n, "mean_denoised": float(rgb.mean()),
                     "mean_reference": float(ref.mean()), "denoised_render_ms": stats.render_ms})
        if spp == 16:
            sweep = []
            for k, sl, sn, sa in itertools.product((3, 5, 7), (1.0, 4.0, 16.0), (0.1, 0.5), (0.1, 0.5)):
                out = cs.denoise_image(noisy, var, albedo, normal, k, sl, sn, sa)
                sweep.append({"iterations": k, "sigma_luminance": sl, "sigma_normal": sn, "sigma_albedo": sa,
                              "relmse": relmse(out, ref), "ratio": relmse(out, ref) / e_n})
            rows.append({"probe": "sweep", "config": cfg, "flags": flags, "spp": 16, "relmse_noisy": e_n,
                         "best": min(sweep, key=lambda r: r["relmse"]), "rows": sweep})
            # equal time: a plain render whose spp takes what the denoised 16-spp render took
            t_dn = np.median([cs.render_denoised(s.camera, st, feature_spp=FEATURE_SPP)[6].render_ms for _ in range(3)])
            t_16 = np.median([cs.render(s.camera, st)[1].render_ms for _ in range(3)])
            m = max(16, int(round(16 * t_dn / t_16)))
            stm = s.render_settings(spp=m, seed=2, flags=flags)
            img, _ = cs.render(s.camera, stm)
            t_m = np.median([cs.render(s.camera, stm)[1].render_ms for _ in range(3)])
            rows.append({"probe": "equal_time", "config": cfg, "flags": flags, "denoised_spp": 16, "denoised_render_ms": float(t_dn),
                         "relmse_denoised": e_d, "plain_spp": m, "plain_render_ms": float(t_m), "relmse_plain": relmse(img, ref)})
    return rows


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_denoise_probe.jsonl")
    cfgs = sys.argv[2:] or ["C1", "C2", "C3s", "C4", "C5"]
    rows = [cost(c) for c in cfgs]
    for c in cfgs:
        if c in QUALITY_FLAGS:
            rows += quality(c)
    with open(out, "a") as f:
        for r in rows:
            r["gpu"] = GPU
            line = json.dumps(r)
            print(line if r["probe"] != "sweep" else json.dumps({k: v for k, v in r.items() if k != "rows"}))
            f.write(line + "\n")


if __name__ == "__main__":
    main()
