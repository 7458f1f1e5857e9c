#!/usr/bin/env python3
"""What next-event estimation buys: error against a converged render at equal spp, and the render time, of each integrator.
  veach-mis (BASELINE config C4, native 1280x720, depth 16) and the Cornell box: plain vs PTC_FLAG_NEE;
  the reference's teapot under its HDR envmap (C3s, native 1280x720, depth 64): plain vs PTC_FLAG_NEE vs
  PTC_FLAG_NEE | PTC_FLAG_NEE_SKY.
One JSON line per scene, then one with the GPU's name and power limit."""
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


def relmse(a, b):
    return float(np.mean((a - b) ** 2 / (b ** 2 + 1e-2)))


NEE, NEE_SKY = pt.FLAG_NEE, pt.FLAG_NEE | pt.FLAG_NEE_SKY
# config, spp, reference: (spp, flags, name), second reference (spp, flags), integrators compared
RUNS = (("C4", 64, (8192, NEE, "NEE"), (8192, 0), (("plain", 0), ("nee", NEE))),
        ("C1", 64, (16384, NEE, "NEE"), (16384, 0), (("plain", 0), ("nee", NEE))),
        ("C3s", 64, (8192, 0, "plain"), (4096, NEE_SKY), (("plain", 0), ("nee", NEE), ("nee_sky", NEE_SKY))))
only = sys.argv[1:]
for cfg, spp, (ref_spp, ref_flags, ref_name), (ref2_spp, ref2_flags), integrators in RUNS:
    if only and cfg not in only:
        continue
    label, s = workloads.workload(cfg)
    cs = s.to_core().commit(0)
    ref, _ = cs.render(s.camera, s.render_settings(spp=ref_spp, seed=1, flags=ref_flags))
    ref2, _ = cs.render(s.camera, s.render_settings(spp=ref2_spp, seed=9, flags=ref2_flags))
    row = {"config": label, "spp": spp, "reference": f"{ref_name} render at {ref_spp} spp",
           "relmse_between_references": relmse(ref2, ref), "second_reference_flags": ref2_flags}
    for name, flags in integrators:
        cs.render(s.camera, s.render_settings(spp=spp, seed=2, flags=flags))
        img, st = cs.render(s.camera, s.render_settings(spp=spp, seed=2, flags=flags))
        row[name] = {"relmse": relmse(img, ref), "render_ms": st.render_ms, "rays": st.rays, "mpaths_s": st.paths / st.render_ms / 1e3}
    for name, _ in integrators[1:]:
        err, tim = row["plain"]["relmse"] / row[name]["relmse"], row[name]["render_ms"] / row["plain"]["render_ms"]
        suffix = "" if name == "nee" else "_" + name
        row["error_ratio_plain_over_" + name] = err
        row["time_ratio_" + name + "_over_plain"] = tim
        row["efficiency_gain" + suffix] = err / tim
    print(json.dumps(row), flush=True)
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
print(json.dumps({"gpu": gpu.strip().splitlines()[0] if gpu.strip() else "unknown"}), flush=True)
