#!/usr/bin/env python3
"""Commit time of the 2 M-triangle mesh (config C5) on one B200, five times in a row: `device` (everything on the GPU,
PTC_COMMIT_FAST_BUILD), `device-sah` (everything on the GPU, the host builder's SAH tree: PTC_COMMIT_DEVICE_SAH), `host`, or
`hybrid` (the default of ptc_scene_commit: reference-BVH restatement on the device, SAH + collapse on the host).
PTC_BUILD_TIMING prints the builders' phase times on stderr.

  python tools/commit_probe.py [device|device-sah|host|hybrid]"""
import os, sys, time
sys.path.insert(0, os.getcwd())
import ptload
pt = ptload.load()
os.environ["PTC_BUILD_TIMING"] = "1"
mode = sys.argv[1] if len(sys.argv) > 1 else "device"  # device | device-sah | host | hybrid (the default of ptc_scene_commit)
if mode != "hybrid":
    os.environ["PTC_BUILD"] = mode
pt.synthetic_scene(cells=64).to_core().commit(0)
s = pt.synthetic_scene(cells=1000)
for i in range(5):
    t0 = time.perf_counter(); c = s.to_core(); t1 = time.perf_counter(); c.commit(0); t2 = time.perf_counter()
    print(f"run {i}: to_core {1e3*(t1-t0):.0f} ms, commit {1e3*(t2-t1):.0f} ms", flush=True)
    t0 = time.perf_counter(); del c; print(f"   destroy {1e3*(time.perf_counter()-t0):.0f} ms", flush=True)
