#!/usr/bin/env python3
"""Progressive preview through the C ABI (SURVEY.md 8f-4, second half: what would replace the reference's minifb window,
src/main.rs:60-75, which only shows the finished frame).  `ptc_render_progressive` renders the frame in passes of
first_spp, then doubling samples, and calls back on this thread after each pass with the packed image of all samples so
far, while the device renders the next pass.  Here the callback saves one PNG per preview.  Philox is keyed on the global
(pixel, sample) and the film is a fixed-point sum, so each preview is the one-shot render at its sample count bit for
bit; the script checks that for the last one.

  python tools/progressive_preview.py [scene.json] [spp] [first_spp] [out_dir]
"""
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ptload  # noqa: E402

pt = ptload.load()


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "scenes", "cornell-box", "scene.json")
    spp = int(sys.argv[2]) if len(sys.argv) > 2 else 64
    first = int(sys.argv[3]) if len(sys.argv) > 3 else 1
    out_dir = sys.argv[4] if len(sys.argv) > 4 else os.path.join(ROOT, "gpurun_out")
    os.makedirs(out_dir, exist_ok=True)
    scene = pt.load_scene_from_json(path)
    w, h, _, _ = scene.settings
    w, h = min(w, 512), min(h, 512)
    cs = scene.to_core().commit(0)
    st = scene.render_settings(width=w, height=h, spp=spp, seed=0)
    t0 = time.perf_counter()
    last = {}

    def show(k, n, img):
        pt.save_image(os.path.join(out_dir, f"preview_{k:02d}.png"), img, w, h)
        print(f"pass {k}: {n} spp so far, preview at {(time.perf_counter() - t0) * 1e3:.2f} ms")
        last["n"], last["img"] = n, img
        return 0

    _, u32, n, stats = cs.render_progressive(scene.camera, st, first_spp=first, on_preview=show)
    print(f"{n} spp in {stats.render_ms:.2f} ms of device time, {(time.perf_counter() - t0) * 1e3:.2f} ms in all")
    once, _ = cs.render_u32(scene.camera, st)
    assert last["n"] == n == spp and np.array_equal(last["img"], once) and np.array_equal(u32, once)
    print(f"the last preview is the one-shot render of {spp} spp, bit for bit")


if __name__ == "__main__":
    main()
