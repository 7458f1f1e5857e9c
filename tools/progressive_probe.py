#!/usr/bin/env python3
"""What progressive rendering (ptc_render_progressive) costs, at native frames (raytracer_rust_b200.workloads).

For C2, C3s, C4 and C5 (default flags), medians of 3 alternated runs of
  * the one-shot render_u32,
  * progressive renders with first_spp 1 and 16 (samples doubling every pass, a callback that only takes the image),
  * a progressive render with first_spp 1 that stops at pass 2;
recording host wall time of the call, render_ms, passes, the time from the call to each preview, the cost per extra
pass ((progressive - one-shot) render_ms / (passes - 1)) and the stop latency (callback's return -> the call's return).
One JSON line per configuration, each with the GPU's name and power limit, printed and appended to the output file.

  python tools/progressive_probe.py [out.jsonl] [configs...]     (default: profiles/r3_progressive_probe.jsonl C2 C3s C4 C5)
"""
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

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
GPU = smi.strip().splitlines()[0] if smi.strip() else "unknown"


def one_shot(cs, s, st):
    t0 = time.perf_counter()
    _, stats = cs.render_u32(s.camera, st)
    return {"wall_ms": (time.perf_counter() - t0) * 1e3, "render_ms": stats.render_ms}


def progressive(cs, s, st, first_spp, stop_at=None):
    at = []
    t0 = time.perf_counter()

    def cb(k, n, img):
        at.append(((time.perf_counter() - t0) * 1e3, n))
        if k == stop_at:
            at.append(time.perf_counter())
            return 1
        return 0

    _, _, n, stats = cs.render_progressive(s.camera, st, first_spp=first_spp, on_preview=cb)
    t1 = time.perf_counter()
    row = {"wall_ms": (t1 - t0) * 1e3, "render_ms": stats.render_ms, "samples": n, "paths": stats.paths}
    if stop_at is not None:
        row["stop_latency_ms"] = (t1 - at.pop()) * 1e3
    row["passes"] = len(at)
    row["preview_at_ms"] = [round(t, 3) for t, _ in at]
    row["preview_samples"] = [m for _, m in at]
    return row


def med(rows, key):
    return float(np.median([r[key] for r in rows]))


def probe(cfg):
    label, s = workloads.workload(cfg)
    cs = s.to_core().commit(0)
    st = s.render_settings(seed=2)
    one_shot(cs, s, st)
    progressive(cs, s, st, 1)  # warm-up of both
    runs = {"one_shot": [], "first_1": [], "first_16": [], "stop_at_pass_2": []}
    for _ in range(3):
        runs["one_shot"].append(one_shot(cs, s, st))
        runs["first_1"].append(progressive(cs, s, st, 1))
        runs["first_16"].append(progressive(cs, s, st, 16))
        runs["stop_at_pass_2"].append(progressive(cs, s, st, 1, stop_at=2))
    one = med(runs["one_shot"], "render_ms")
    summary = {"one_shot_render_ms": one, "one_shot_wall_ms": med(runs["one_shot"], "wall_ms")}
    for key in ("first_1", "first_16"):
        passes = runs[key][0]["passes"]
        r = med(runs[key], "render_ms")
        summary[key] = {"passes": passes, "render_ms": r, "wall_ms": med(runs[key], "wall_ms"),
                        "overhead_ms": r - one, "overhead_pct": 100.0 * (r - one) / one,
                        "per_extra_pass_ms": (r - one) / (passes - 1) if passes > 1 else None,
                        "first_preview_ms": float(np.median([x["preview_at_ms"][0] for x in runs[key]]))}
    summary["stop_at_pass_2"] = {"stop_latency_ms": med(runs["stop_at_pass_2"], "stop_latency_ms"),
                                 "wall_ms": med(runs["stop_at_pass_2"], "wall_ms")}
    row = {"measurement": "progressive rendering against the one-shot render_u32, medians of 3 alternated runs", "config": label,
           "spp": st.spp, "summary": summary, "runs": runs, "gpu": GPU}
    del cs
    return row


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_progressive_probe.jsonl")
    cfgs = sys.argv[2:] or ["C2", "C3s", "C4", "C5"]
    for cfg in cfgs:
        row = probe(cfg)
        print(json.dumps(row), flush=True)
        with open(out, "a") as f:
            f.write(json.dumps(row) + "\n")


if __name__ == "__main__":
    main()
