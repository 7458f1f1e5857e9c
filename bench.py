#!/usr/bin/env python3
"""bench.py — the headline benchmark: BASELINE.json's metric (Mpaths/s, with Mrays/s beside it) on config C2,
`semesterbild.json` at its native 800x600 / 256 spp / 30 bounces, on N B200s of one node.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config C1|C2|C3|C3s|C4|C5] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...

A "step" is one full render of the frame (render_scene, src/renderer.rs:67-123 of the reference, timed like the
reference times it: renderer.rs:82,109 — scene load, BVH build and PNG encode are outside) at the configuration's
NATIVE resolution / spp / bounce limit (raytracer-rust_b200/workloads.py); `--config` selects another BASELINE.json
configuration than the default C2.

  value  device-resident: scene resident in HBM, film accumulated in HBM (ptc_render_accumulate) and, for N > 1, one
         NCCL reduce of the fp32 film to rank 0 + the film resolve, all inside the timed region.
  e2e    the reference-facing call with HOST buffers: `render_scene` returning its Vec<u32>.  N = 1: ptc_render_u32.
         N > 1: the in-process route ptc_multi_render_u32 (one host thread per GPU, one ncclReduce, the packed image copied
         to the host), driven by rank 0 alone while the other ranks wait on the rendezvous store (no kernel of theirs
         runs); `e2e_ranks` keeps the torch.distributed route + device->host copy of the packed image.

N > 1 is STRONG scaling: the FIXED native job, its sample range split N ways (Philox is keyed on the global sample
index, so the reduced film is the same image); value = the job's paths / max-over-ranks time.  The weak-scaling number of
round 1 (every rank renders the whole frame at the config's spp, an N*spp job) rides along as `weak`.

`--impl reference` times the CPU restatement of the reference (oracle/, the reference's own ChaCha stream, all host
threads) on a bounded sample of the same frame.  The Rust reference itself cannot be built in this image (no
cargo/rustc; see DESIGN.md).  That arm loads libpthost (scene description) and liboracle only — not the CUDA library.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

DEFAULT_POOL = 0  # the library's default: the whole job in flight at once if it fits a quarter of the free memory, else 48 Mi slots
DUMP_PIXELS = 1 << 20  # --dump-outputs: frames up to 1 Mi pixels (C1-C4) whole, 32 MiB at most; larger ones (C5) as a sample of this many


def metric_name(cfg, w, h, spp, depth):
    names = {"C1": "cornell-box", "C2": "semesterbild", "C3": "teapot", "C3s": "teapot-shipped", "C4": "veach-mis", "C5": "synthetic-2M"}
    return f"Mpaths/s ({names[cfg]} {w}x{h}x{spp}spp, depth {depth})"


def load_json(name):
    p = os.path.join(ROOT, "profiles", name)
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except ValueError:
            return None
    return None


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d.get("sm_max_mhz", 1965.0)), "MEASURED_PEAKS.json"
    return 6650.0, 1965.0, "B200_PROFILING.md fallback"


def l2_peak():
    """Measured L2 read bandwidth of a resident set (tools/micro/l2_bw.cu, committed as profiles/r2_l2_bw.json):
    the best coalesced figure over the sets that fit the L2."""
    d = load_json("r2_l2_bw.json")
    if not d:
        return None, "unmeasured"
    fit = [r["gb_per_s"] for r in d["coalesced_read"] if r["set_mib"] * (1 << 20) <= 0.5 * d["l2_bytes"]]
    return (max(fit) if fit else None), "profiles/r2_l2_bw.json (tools/micro/l2_bw.cu, resident-set read, ld.global.cg)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled while the timed region runs (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_render_sample(scene, seconds):
    """The oracle (C++ restatement of the reference's renderer, ChaCha12 per-row stream, all host threads) on a bounded
    sample of the frame: the native resolution and depth at as many spp as fit `seconds` of CPU work.
    -> (OracleScene, spp to run)"""
    from bindings import OracleScene, RNG_CHACHA
    w, h, spp, depth = scene.settings
    orc = OracleScene(scene)
    _, st = orc.render(scene.camera, w, h, 1, depth, rng_mode=RNG_CHACHA)  # calibration: one sample per pixel
    n = int(max(1, round(seconds / max(st.seconds, 1e-3))))  # may exceed the config's spp for a small frame (C1)
    return orc, n


def run_reference(args):
    """CPU arm: the oracle on all host threads.  Only libpthost (scene description) and liboracle are loaded."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import ptload
    pt = ptload.load()
    from raytracer_rust_b200 import workloads
    from bindings import RNG_CHACHA
    label, scene = workloads.workload(args.config)
    w, h, spp, depth = scene.settings
    cores = os.cpu_count() or 1
    # a step is a bounded sample: ~6 s of CPU work, less when many steps are asked for (the whole run stays within minutes)
    orc, spp_step = cpu_render_sample(scene, min(6.0, 150.0 / max(1, args.steps + args.warmup)))
    for _ in range(args.warmup):
        orc.render(scene.camera, w, h, spp_step, depth, rng_mode=RNG_CHACHA)
    paths = rays = 0
    secs = 0.0
    for _ in range(args.steps):
        _, st = orc.render(scene.camera, w, h, spp_step, depth, rng_mode=RNG_CHACHA)
        paths += st.paths
        rays += st.rays
        secs += st.seconds
    value = paths / secs / 1e6
    sample = (f"{w}x{h} at {spp_step} spp per step (of {spp}), depth {depth}, {secs / args.steps:.1f} s of CPU work per step; "
              "Mpaths/s does not depend on spp")
    line = {
        "impl": "reference", "metric": metric_name(args.config, w, h, spp, depth), "value": value, "unit": "Mpaths/s",
        "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": secs / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong" if args.gpus > 1 else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "mrays_per_s": rays / secs / 1e6,
        "config": {"workload": label, "sample": sample},
        "cpu_baseline": {"value": value, "unit": "Mpaths/s", "cores": cores, "kind": "port", "sample": sample,
                         "note": "C++ restatement of the reference CPU path (oracle/), row-parallel like rayon, ChaCha12 per-row "
                                 "RNG; `cargo run --release` is impossible here (no Rust toolchain)"},
        "e2e": {"value": value, "unit": "Mpaths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "loaded_cuda_library": "raytracer_rust_b200" in sys.modules and sys.modules["raytracer_rust_b200"]._core is not None,
    }
    print(json.dumps(line), flush=True)
    return 0


def cpu_baseline(scene):
    from bindings import RNG_CHACHA
    w, h, spp, depth = scene.settings
    orc, n = cpu_render_sample(scene, 12.0)
    _, st = orc.render(scene.camera, w, h, n, depth, rng_mode=RNG_CHACHA)
    return {"value": st.paths / st.seconds / 1e6, "unit": "Mpaths/s", "cores": os.cpu_count() or 1, "kind": "port",
            "mrays_per_s": st.rays / st.seconds / 1e6,
            "sample": f"{w}x{h} at {n} spp (of {spp}), depth {depth}, {st.seconds:.1f} s of CPU work; C++ restatement of the reference "
                      "(oracle/), row-parallel, ChaCha12 per-row RNG as the reference"}


def dump_outputs(out_dir, film, packed, w, h, counts):
    """What the timed path hands its caller in its last step, as DIR/<name>.npy:
      film   [H, W, 3] float32  the radiance sum ptc_render_accumulate leaves in the device film (reduced over ranks)
      image  [H, W, 3] float32  the 0x00RRGGBB pixels of ptc_resolve_device as channel levels 0-255
      stats  [2]       float64  paths and rays of the step, summed over ranks
    A frame of more than DUMP_PIXELS pixels keeps a fixed, seeded sample of them: film and image are [DUMP_PIXELS, 3]
    and pixel_index (float64) holds their row-major indices into the frame."""
    import numpy as np
    u = packed.reshape(-1).view(np.uint32)
    arrays = {"film": film.reshape(h * w, 3).astype(np.float32),
              "image": np.stack([(u >> 16) & 255, (u >> 8) & 255, u & 255], -1).astype(np.float32)}
    if h * w > DUMP_PIXELS:
        idx = np.sort(np.random.default_rng(0).choice(h * w, DUMP_PIXELS, replace=False))
        arrays = {k: v[idx] for k, v in arrays.items()}
        arrays["pixel_index"] = idx.astype(np.float64)
    else:
        arrays = {k: v.reshape(h, w, 3) for k, v in arrays.items()}
    arrays["stats"] = np.asarray(counts, np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="C2", choices=["C1", "C2", "C3", "C3s", "C4", "C5"])
    ap.add_argument("--pool", type=int, default=DEFAULT_POOL, help="path-pool slots")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-weak", action="store_true", help="N > 1: skip the extra weak-scaling measurement")
    ap.add_argument("--no-inprocess", action="store_true", help="N > 1: skip the in-process ptc_multi_* measurement on rank 0")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the film, image and path / ray counts of the last timed step "
                                                          "as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        # the reference arm sizes its sample by a CPU timing, so its output is not the same from run to run
        ap.error("--dump-outputs applies to --impl b200")
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import ptload
    pt = ptload.load()
    from raytracer_rust_b200 import workloads

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available() or pt.device_count() < 1:
        raise SystemExit("bench.py needs a CUDA device: the path tracer has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        # NCCL prints its version banner on stdout at communicator creation; stdout carries exactly one JSON line,
        # so park fd 1 on stderr until the communicator exists
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.all_reduce(torch.zeros(1, device=dev))
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)

    label, scene = workloads.workload(args.config)
    w, h, spp, depth = scene.settings
    t_commit = time.perf_counter()
    cs = scene.to_core().commit(local)
    commit_s = time.perf_counter() - t_commit
    cam = scene.camera
    stream = torch.cuda.current_stream()
    accum = torch.zeros(h * w * 3, dtype=torch.float32, device=dev)
    out_u32 = torch.zeros(h * w, dtype=torch.int32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    from raytracer_rust_b200.dist import sample_range

    def settings(mode, flags=0):
        if mode == "strong":  # the fixed native job, this rank's share of its sample range
            b, e = sample_range(spp, rank, world)
            return scene.render_settings(spp=spp, sample_begin=b, sample_end=e, seed=0, pool_paths=args.pool, flags=flags), e > b
        return scene.render_settings(spp=spp * world, sample_begin=rank * spp, sample_end=(rank + 1) * spp, seed=0,
                                     pool_paths=args.pool, flags=flags), True

    def step_device(mode="strong", flags=0):
        accum.zero_()
        st, busy = settings(mode, flags)
        stats = cs.render_accumulate(cam, st, accum.data_ptr(), stream.cuda_stream) if busy else pt.Stats()
        if world > 1:
            dist.reduce(accum, dst=0, op=dist.ReduceOp.SUM)
        if rank == 0:
            pt._ck(pt.core().ptc_resolve_device(accum.data_ptr(), h * w, 1.0 / st.spp, out_u32.data_ptr(), stream.cuda_stream))
        return stats

    def step_e2e():
        # the reference-facing call: host buffers in and out
        if world == 1:
            _, st = cs.render_u32(cam, settings("strong")[0])  # render_scene -> Vec<u32>, resolved on the device
            return st
        st = step_device()
        if rank == 0:
            out_u32.cpu()
        return st

    def timed(fn, n, wall_clock=False):
        tot_ms, stats = 0.0, []
        for _ in range(n):
            flush.fill_(1)  # evict L2 between timed iterations (untimed)
            torch.cuda.synchronize()
            if dist:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record(stream)
            stats.append(fn())
            e1.record(stream)
            torch.cuda.synchronize()
            wall = (time.perf_counter() - t0) * 1e3
            # the wavefront loop synchronises its stream before returning, so wall and event time agree; calls that use
            # the library's internal streams (ptc_render_u32, ptc_multi_*) are only visible to the wall clock
            tot_ms += max(e0.elapsed_time(e1), wall if wall_clock else 0.0)
        t = torch.tensor([tot_ms], dtype=torch.float64, device=dev)
        if dist:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), stats

    def summed(stats, *names):
        cnt = torch.tensor([float(sum(getattr(s, n) for s in stats)) for n in names], dtype=torch.float64, device=dev)
        if dist:
            dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        return [float(x) for x in cnt.tolist()]

    for _ in range(max(args.warmup, 3)):
        step_device()
    torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # `value`: the production path, exactly K steps.  Then K more steps of the same work with PTC_FLAG_TIMING, which
    # brackets every stage launch with CUDA events on the launching stream (a few per cent slower): these give the
    # per-kernel share and the roofline's launch durations.  Clocks are sampled across both.
    ms_total, vstats = timed(lambda: step_device("strong", 0), args.steps)
    if args.dump_outputs:
        last = summed(vstats[-1:], "paths", "rays")  # a collective: every rank takes part
        if rank == 0:
            dump_outputs(args.dump_outputs, accum.cpu().numpy(), out_u32.cpu().numpy(), w, h, last)
    _, stats = timed(lambda: step_device("strong", pt.FLAG_TIMING), args.steps)
    clocks = sampler.stop() if rank == 0 else None

    paths_all, rays_all = summed(vstats, "paths", "rays")
    rays_rank = sum(s.rays for s in stats)
    value = paths_all / ms_total / 1e3
    launches = sum(s.kernel_launches for s in vstats) + args.steps * 2  # + memset + resolve

    weak = None
    if world > 1 and not args.no_weak:
        step_device("weak")
        ms_weak, wstats = timed(lambda: step_device("weak", 0), args.steps)
        wp, wr = summed(wstats, "paths", "rays")
        weak = {"value": wp / ms_weak / 1e3, "unit": "Mpaths/s", "ms_per_step": ms_weak / args.steps, "spp_total": spp * world,
                "mrays_per_s": wr / ms_weak / 1e3, "note": "every rank renders the whole frame at the config's spp (round 1's definition)"}

    for _ in range(2):
        step_e2e()
    ms_e2e, e2e_stats = timed(step_e2e, args.steps, wall_clock=True)
    (e2e_paths,) = summed(e2e_stats, "paths")
    e2e_ranks_value = e2e_paths / ms_e2e / 1e3
    d2h = h * w * 4 + 64 * (1 + spp // 8)  # the packed image + the control-block snapshots the host polls
    h2d = 256                               # control block + launch parameters (the scene is resident)
    e2e = {"value": e2e_ranks_value, "unit": "Mpaths/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "ms_per_step": ms_e2e / args.steps, "api": "ptc_render_u32 (host Vec<u32> out)"}
    e2e_ranks = None
    if world > 1:
        # in-process route of the C ABI, rank 0 alone; the other ranks wait on the rendezvous store (CPU side), so none of
        # their kernels shares the GPUs with the measurement
        e2e_ranks = dict(e2e, api="ptc_render_accumulate per rank + dist.reduce + ptc_resolve_device + D2H copy of the packed image")
        e2e = None
        if not args.no_inprocess:
            torch.cuda.synchronize()
            store = torch.distributed.distributed_c10d._get_default_store()
            if rank == 0:
                try:
                    m = cs.multi(list(range(world)))
                    st = scene.render_settings(spp=spp, seed=0, pool_paths=args.pool)
                    for _ in range(2):
                        m.render_u32(cam, st, pt.SHARD_SAMPLES)
                    tot, mst = 0.0, None
                    for _ in range(args.steps):
                        t0 = time.perf_counter()
                        _, mst = m.render_u32(cam, st, pt.SHARD_SAMPLES)
                        tot += (time.perf_counter() - t0) * 1e3
                    e2e = {"value": mst.paths * args.steps / tot / 1e3, "unit": "Mpaths/s", "h2d_bytes_per_step": h2d * world,
                           "d2h_bytes_per_step": h * w * 4 + 64 * world * (1 + spp // 8), "ms_per_step": tot / args.steps,
                           "api": "ptc_multi_render_u32 (in-process: one host thread per GPU, one ncclReduce, host Vec<u32> out), "
                                  "host wall clock, rank 0 only", "film_reduce_bytes": h * w * (24 + 8),
                           "film_reduce_note": "fixed-point film: 3 x int64 sums + one 64-bit flag word per pixel"}
                    del m
                except Exception as ex:  # noqa: BLE001 — report, do not lose the whole line
                    e2e = dict(e2e_ranks, inprocess_error=str(ex))
                store.set("inprocess_done", "1")
            else:
                import datetime
                try:
                    store.wait(["inprocess_done"], datetime.timedelta(seconds=300))
                except Exception:  # noqa: BLE001 — rank 0 is reporting the problem; do not add a second one
                    pass
        if e2e is None:
            e2e = e2e_ranks

    line = None
    if rank == 0:
        line = build_line(args, pt, torch, scene, cs, label, local, world, value, ms_total, paths_all, rays_all, rays_rank, stats, launches,
                          clocks, e2e, e2e_ranks, weak, commit_s)
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline(scene)
        print(json.dumps(line), flush=True)
    if dist:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def build_line(args, pt, torch, scene, cs, label, local, world, value, ms_total, paths_all, rays_all, rays_rank, stats, launches, clocks, e2e,
               e2e_ranks, weak, commit_s):
    w, h, spp, depth = scene.settings
    cam = scene.camera
    ext_ms = sum(s.extend_ms for s in stats)
    ext_launches = sum(s.extend_launches for s in stats)
    shade_ms = sum(s.shade_ms for s in stats)
    render_ms = sum(s.render_ms for s in stats)
    # instrumented build of the same kernels, outside the timed region: wide nodes popped / triangles tested per ray
    # (work stealing off for this one render: a thief walks subtrees its donor might have culled later, which is not
    # algorithmic work, and a frame this small is all kernel tail)
    os.environ["PTC_STEAL"] = "0"
    c = cs.render(cam, scene.render_settings(width=min(w, 1280), height=min(h, 720), spp=4, seed=0, flags=pt.FLAG_COUNTERS))[1]
    os.environ.pop("PTC_STEAL", None)
    nodes_per_ray, tris_per_ray = c.nodes_visited / c.rays, c.tris_tested / c.rays
    objs = scene.objects
    cost = {pt.OBJ_SPHERE: 25, pt.OBJ_PLANE: 14, pt.OBJ_QUAD: 35, pt.OBJ_CUBE: 80, pt.OBJ_MESH: 64}
    analytic_instr = sum(cost[o.type] for o in objs)
    mesh_objs = [i for i, o in enumerate(objs) if o.type == pt.OBJ_MESH]
    node_bytes = 80.0
    bvh_bytes = 0
    for i in mesh_objs:
        info = cs.mesh_info(i)[0]
        bvh_bytes += info.node_bytes + info.triangle_bytes
        if info.wide_nodes:
            node_bytes = info.node_bytes / info.wide_nodes
    bytes_per_ray = 32 + 16 + node_bytes * nodes_per_ray + 48.0 * tris_per_ray      # SURVEY.md §8(d)
    instr_per_ray = analytic_instr + 170.0 * nodes_per_ray + 45.0 * tris_per_ray
    hbm_peak, sm_max_mhz, peak_kind = peaks()
    l2_gbs, l2_src = l2_peak()
    rays_per_launch = rays_rank / max(1, ext_launches)
    ext_s = ext_ms / 1e3
    ext_rays_s = rays_rank / ext_s if ext_s > 0 else 0.0
    sm_mhz = (clocks or {}).get("sm_mhz") or sm_max_mhz
    props = torch.cuda.get_device_properties(local)
    sms = props.multi_processor_count
    l2_bytes = getattr(props, "L2_cache_size", 126 << 20)
    fp32_peak = sms * 128 * sm_mhz * 1e6 / 1e12  # T instr/s at the clock sampled under load
    hbm = {"bound": "hbm", "achieved": bytes_per_ray * ext_rays_s / 1e9, "peak": hbm_peak, "unit": "GB/s", "peak_source": peak_kind}
    hbm["frac"] = hbm["achieved"] / hbm_peak
    fp32 = {"bound": "fp32_issue", "achieved": instr_per_ray * ext_rays_s / 1e12, "peak": fp32_peak, "unit": "Tinstr/s",
            "peak_source": f"{sms} SMs x 128 lanes x {sm_mhz:.0f} MHz sampled under load"}
    fp32["frac"] = fp32["achieved"] / fp32_peak
    l2 = None
    if l2_gbs:
        l2 = {"bound": "l2", "achieved": bytes_per_ray * ext_rays_s / 1e9, "peak": l2_gbs, "unit": "GB/s", "peak_source": l2_src}
        l2["frac"] = l2["achieved"] / l2_gbs
    traffic = load_json("r2_extend_traffic.json") or load_json("r1_extend_traffic.json")
    traffic_cfg = (traffic or {}).get(args.config) if traffic and args.config in (traffic or {}) else (traffic if args.config == "C2" else None)
    dram_per_ray = float(traffic_cfg["dram_bytes_per_ray"]) if traffic_cfg and "dram_bytes_per_ray" in traffic_cfg else None
    # Which bound binds (SURVEY.md 8d): no mesh (C1/C4) -> the wavefront's path-state traffic over HBM; BVH + triangles
    # resident in L1/L2 (C2/C3) -> whichever of FP32 issue and L2 bandwidth gives the lower ray-rate ceiling, i.e. the
    # larger fraction; a working set that straddles the L2 (C5) -> L2 if the committed ncu capture shows > 80 % L2 hit rate
    # on the traversal's fetches, else HBM.
    if not mesh_objs:
        seg_bytes = 150.0
        it_s = (ext_ms + shade_ms) / 1e3
        binding = {"bound": "hbm", "achieved": seg_bytes * rays_rank / it_s / 1e9 if it_s > 0 else 0.0, "peak": hbm_peak, "unit": "GB/s",
                   "peak_source": peak_kind, "kernel": "wavefront iteration = k_extend_pre + k_shade (analytic scene: no BVH stage)",
                   "algorithmic_bytes_per_ray": seg_bytes,
                   "why": "analytic primitives only: ~150 B of path state per ray segment over HBM binds (SURVEY.md 8d)"}
        binding["frac"] = binding["achieved"] / hbm_peak
        rays_per_launch_b, avg_ms = rays_per_launch, (ext_ms + shade_ms) / max(1, ext_launches)
        alg_bytes_launch = seg_bytes * rays_per_launch
    else:
        kernel = "extend stage = k_extend_pre + k_traverse + k_extend_post (one logical kernel, timed together)"
        if bvh_bytes < 0.25 * l2_bytes:
            cands = [fp32] + ([l2] if l2 else [])
            binding = dict(max(cands, key=lambda r: r["frac"]))
            binding["why"] = (f"BVH + triangles = {bvh_bytes / 1e6:.2f} MB, L1/L2-resident: min(FP32 issue, L2 bandwidth) binds "
                              "(SURVEY.md 8d); the larger of the two fractions is reported")
        else:
            hit = (traffic_cfg or {}).get("l2_hit_rate")
            use_l2 = l2 is not None and hit is not None and hit > 0.8
            binding = dict(l2 if use_l2 else hbm)
            binding["why"] = (f"BVH + triangles = {bvh_bytes / 1e6:.0f} MB against a {l2_bytes / 1e6:.0f} MB L2; ncu L2 hit rate of the "
                              f"traversal fetches = {hit}: bound = {'L2' if use_l2 else 'HBM'} bandwidth (SURVEY.md 8d)")
        binding["kernel"] = kernel
        rays_per_launch_b, avg_ms = rays_per_launch, ext_ms / max(1, ext_launches)
        alg_bytes_launch = bytes_per_ray * rays_per_launch
    binding.update({
        "traffic": dram_per_ray * rays_per_launch if dram_per_ray else None,
        "traffic_note": "DRAM bytes per launch of the stage: dram__bytes_read.sum + dram__bytes_write.sum per ray of the committed ncu "
                        "capture (profiles/) x rays per launch",
        "algorithmic_bytes_per_launch": alg_bytes_launch, "algorithmic_instr_per_ray": instr_per_ray,
        "algorithmic_bytes_per_ray_extend": bytes_per_ray, "nodes_per_ray": nodes_per_ray, "tris_per_ray": tris_per_ray,
        "node_bytes": node_bytes, "rays_per_launch": rays_per_launch_b, "avg_launch_ms": avg_ms,
        "extend_grays_per_s": ext_rays_s / 1e9,
        "note": "algorithmic bytes = 32 B ray + 16 B hit + node bytes per wide node popped + 48 B per triangle tested; algorithmic instr = "
                "sum of analytic primitive costs + 64 per mesh instance + 170 per node + 45 per triangle, FMA = 1 (SURVEY.md 8d)"})
    line = {
        "metric": metric_name(args.config, w, h, spp, depth), "value": value, "unit": "Mpaths/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3),
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong" if world > 1 else "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": label, "parallelism": f"sample range split x{world} (fixed job)" if world > 1 else "single GPU",
                   "spp_total": spp, "l2": "256 MiB flush write between timed steps", "pool_paths": cs.last_pool_slots(),
                   "pool_policy": "library default" if args.pool == 0 else "--pool",
                   "rng": "Philox4x32-10 keyed (pixel, sample, bounce)", "commit_s": commit_s},
        "mrays_per_s": rays_all / ms_total / 1e3, "rays_per_path": rays_all / paths_all,
        "e2e": e2e,
        "gpu_launches": int(launches),
        "clocks": clocks,
        "kernel_share": {"k_extend_pre": sum(s.pre_ms for s in stats) / render_ms,
                         "k_traverse": sum(s.traverse_ms for s in stats) / render_ms,
                         "k_extend_post": sum(s.post_ms for s in stats) / render_ms,
                         "k_shade (incl. path regeneration)": shade_ms / render_ms,
                         "launch gaps": max(0.0, 1.0 - (ext_ms + shade_ms) / render_ms)},
        "roofline": binding,
        "roofline_all": {"hbm": hbm, "fp32_issue": fp32, "l2": l2},
    }
    if e2e_ranks:
        line["e2e_ranks"] = e2e_ranks
    if weak:
        line["weak"] = weak
    return line


if __name__ == "__main__":
    sys.exit(main())
