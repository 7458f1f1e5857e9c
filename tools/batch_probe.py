#!/usr/bin/env python3
"""What batch rendering (ptc_render_batch) buys over a loop of single renders, and that default renders did not change.

  * Batch against loop: one ptc_render_batch of K views (packed images to the host) against K ptc_render_u32 calls with
    the same cameras, seeds and outputs; medians of alternated runs after one warm-up of each route; ms per view and
    Mpaths/s of both, host wall clock around each call (both return after a stream synchronise).  Cases: C1 Cornell box
    256x256x16 depth 8, K in {1, 4, 16, 64}; semesterbild 200x150x16 depth 30, K in {1, 16, 64}; C3s teapot 320x180x16
    depth 16 with NEE | NEE_SKY, K in {1, 16}.  The views orbit the scene's camera position by a few degrees each.
  * With --parent DIR (a built tree of the parent commit): stats.kernel_launches of render_u32 at the native settings of
    C1-C5 in both builds, and `bench.py --gpus 1 --config C1 / C2` of both builds alternated, --rounds times each.

One JSON line per measurement, the first with the GPU's name and power limit, printed and appended to the output file.

  python tools/batch_probe.py [--out profiles/r3_batch_probe.jsonl] [--parent DIR] [--runs 5] [--rounds 3]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# kernel_launches of render_u32 at the native settings of C1-C5, in the tree this runs in (argv[1])
LAUNCHES = r"""
import json, sys
sys.path.insert(0, sys.argv[1])
import ptload
pt = ptload.load()
from raytracer_rust_b200 import workloads
out = {}
for name in ("C1", "C2", "C3s", "C4", "C5"):
    _, s = workloads.workload(name)
    w, h, spp, depth = s.settings
    cs = s.to_core().commit(0)
    st = s.render_settings(seed=0)
    _, a = cs.render_u32(s.camera, st)
    _, b = cs.render_u32(s.camera, st)
    out[name] = {"kernel_launches": [a.kernel_launches, b.kernel_launches], "iterations": a.iterations, "paths": a.paths,
                 "rays": a.rays, "pool_slots": cs.last_pool_slots(), "job_paths": ((w + 31) // 32) * ((h + 31) // 32) * 1024 * spp}
    del cs
print(json.dumps(out))
"""


def gpu_name():
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout
    return smi.strip().splitlines()[0] if smi.strip() else "unknown"


def orbit(pt, cam, k, n, degrees=3.0):
    """the camera turned about the vertical axis through the point it looks at 10 units ahead, by (k - n/2) * degrees"""
    p, f = np.array(cam.position[:], np.float64), np.array(cam.forward[:], np.float64)
    centre = p + 10.0 * f
    a = np.radians((k - n / 2) * degrees)
    rot = np.array([[np.cos(a), 0, np.sin(a)], [0, 1, 0], [-np.sin(a), 0, np.cos(a)]])
    c = pt.Camera()
    C.pointer(c)[0] = cam
    for dst, v in ((c.position, centre + rot @ (p - centre)), (c.forward, rot @ f), (c.right, rot @ np.array(cam.right[:])),
                   (c.true_up, rot @ np.array(cam.true_up[:]))):
        for i in range(3):
            dst[i] = float(v[i])
    return c


def batch_vs_loop(pt, label, scene, st, ks, runs, gpu, out):
    core = pt.core()
    cs = scene.to_core().commit(0)
    n_px = st.width * st.height
    for k in ks:
        cams = [orbit(pt, scene.camera, i, k) for i in range(k)]
        seeds = np.arange(1, k + 1, dtype=np.uint64)
        arr = (pt.Camera * k)(*cams)
        batch_u32 = np.empty(k * n_px, np.uint32)
        loop_u32 = np.empty((k, n_px), np.uint32)
        sts = []
        for i in range(k):
            s = pt.RenderSettings()
            C.pointer(s)[0] = st
            s.seed = int(seeds[i])
            sts.append(s)

        def batch():
            stats = pt.Stats()
            t0 = time.perf_counter()
            pt._ck(core.ptc_render_batch(cs._h, arr, k, seeds.ctypes.data, C.byref(st), None, batch_u32.ctypes.data, C.byref(stats)))
            return (time.perf_counter() - t0) * 1e3, stats.paths, stats.kernel_launches, stats.render_ms

        def loop():
            paths = launches = 0
            render_ms = 0.0
            t0 = time.perf_counter()
            for i in range(k):
                stats = pt.Stats()
                pt._ck(core.ptc_render_u32(cs._h, C.byref(cams[i]), C.byref(sts[i]), loop_u32[i].ctypes.data, C.byref(stats)))
                paths += stats.paths
                launches += stats.kernel_launches
                render_ms += stats.render_ms
            return (time.perf_counter() - t0) * 1e3, paths, launches, render_ms

        batch(), loop()  # warm-up
        tb, tl = [], []
        for _ in range(runs):
            tb.append(batch())
            tl.append(loop())
        assert np.array_equal(batch_u32.reshape(k, n_px), loop_u32), "batch and loop images differ"
        mb, ml = statistics.median(t[0] for t in tb), statistics.median(t[0] for t in tl)
        paths = tb[0][1]
        row = {"probe": "batch_vs_loop", "gpu": gpu, "case": label, "frame": [st.width, st.height], "spp": st.spp,
               "max_depth": st.max_depth, "flags": st.flags, "views": k, "runs": runs, "paths": paths,
               "batch_ms": round(mb, 3), "loop_ms": round(ml, 3), "batch_ms_range": [round(min(t[0] for t in tb), 3), round(max(t[0] for t in tb), 3)],
               "loop_ms_range": [round(min(t[0] for t in tl), 3), round(max(t[0] for t in tl), 3)],
               "batch_ms_per_view": round(mb / k, 4), "loop_ms_per_view": round(ml / k, 4),
               "batch_mpaths_s": round(paths / mb / 1e3, 1), "loop_mpaths_s": round(paths / ml / 1e3, 1), "speedup": round(ml / mb, 3),
               "batch_launches": tb[0][2], "loop_launches": tl[0][2],
               "batch_render_ms": round(statistics.median(t[3] for t in tb), 3), "loop_render_ms_sum": round(statistics.median(t[3] for t in tl), 3),
               "images_equal": True}
        print(json.dumps(row), flush=True)
        out.write(json.dumps(row) + "\n")
        out.flush()
    del cs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_batch_probe.jsonl"))
    ap.add_argument("--parent", help="a built tree of the parent commit, for the launch counts and the bench.py comparison")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()
    import ptload
    pt = ptload.load()
    from raytracer_rust_b200 import workloads
    gpu = gpu_name()
    with open(args.out, "a") as out:
        head = {"probe": "gpu", "gpu": gpu, "note": "name, power limit (nvidia-smi)"}
        print(json.dumps(head), flush=True)
        out.write(json.dumps(head) + "\n")

        _, c1 = workloads.workload("C1")
        batch_vs_loop(pt, "C1 cornell-box", c1, c1.render_settings(seed=0), [1, 4, 16, 64], args.runs, gpu, out)
        _, c2 = workloads.workload("C2")
        batch_vs_loop(pt, "semesterbild 200x150", c2, c2.render_settings(width=200, height=150, spp=16, max_depth=30, seed=0),
                      [1, 16, 64], args.runs, gpu, out)
        _, c3 = workloads.workload("C3s")
        batch_vs_loop(pt, "C3s teapot 320x180", c3, c3.render_settings(width=320, height=180, spp=16, max_depth=16, seed=0,
                                                                        flags=pt.FLAG_NEE | pt.FLAG_NEE_SKY), [1, 16], args.runs, gpu, out)
        if not args.parent:
            return 0
        trees = {"parent": os.path.abspath(args.parent), "new": ROOT}
        launches = {}
        for tag, tree in trees.items():
            r = subprocess.run([sys.executable, "-c", LAUNCHES, tree], capture_output=True, text=True, cwd=tree)
            if r.returncode:
                raise SystemExit(f"{tag}: {r.stderr[-2000:]}")
            launches[tag] = json.loads(r.stdout.strip().splitlines()[-1])
        row = {"probe": "kernel_launches", "gpu": gpu, "api": "render_u32 at native settings, seed 0, twice", **launches,
               "equal": {n: launches["parent"][n]["kernel_launches"] == launches["new"][n]["kernel_launches"] for n in launches["new"]}}
        print(json.dumps(row), flush=True)
        out.write(json.dumps(row) + "\n")
        for cfg in ("C1", "C2"):
            for rnd in range(args.rounds):
                for tag, tree in trees.items():
                    r = subprocess.run([sys.executable, os.path.join(tree, "bench.py"), "--gpus", "1", "--steps", "8", "--warmup", "2",
                                        "--no-cpu-baseline", "--config", cfg], capture_output=True, text=True, cwd=tree)
                    if r.returncode:
                        raise SystemExit(f"bench {tag} {cfg}: {r.stderr[-2000:]}")
                    line = json.loads(r.stdout.strip().splitlines()[-1])
                    row = {"probe": "bench", "gpu": gpu, "config": cfg, "round": rnd, "build": tag, "value": line.get("value"),
                           "unit": line.get("unit"), "ms_per_step": line.get("ms_per_step"), "kernel_launches": line.get("kernel_launches")}
                    print(json.dumps(row), flush=True)
                    out.write(json.dumps(row) + "\n")
                    out.flush()
    return 0


if __name__ == "__main__":
    sys.exit(main())
