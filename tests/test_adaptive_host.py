"""Adaptive sampling (ptc_render_adaptive) without a device.

  * the decision: one step of the g++ build of pt_adaptive.h (tests/hostsim/adaptsim.cpp: decision, 3x3 dilation over
    the active set, stable compaction) equals a numpy restatement bit for bit — random film sums, zeros, NaN / +-inf
    channels, frame borders and corners, frames one pixel wide or high, thresholds 0 and +inf;
  * the schedule: min_spp/2, min_spp, then doubling up to spp;
  * the ABI: ptc_adaptive has the same layout in C and in ctypes, the Rust crate declares it and the function;
  * the wrapper passes its arguments, and bad arguments are refused before the scene's state is looked at.
"""
import ctypes as C
import os
import re
import subprocess
import zlib

import numpy as np
import pytest

from bindings import sim_lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_F = C.POINTER(C.c_float)
_vp = C.c_void_p


def _lib():
    L = sim_lib()
    L.adapt_sim_next_end.argtypes = [C.c_int32, C.c_int32]
    L.adapt_sim_next_end.restype = C.c_int32
    L.adapt_sim_step.argtypes = [C.c_int32, C.c_int32, _F, _F, _vp, C.c_int64, C.c_int32, C.c_int32, C.c_float, _vp, _vp, _vp]
    L.adapt_sim_step.restype = C.c_int64
    return L


def sim_step(w, h, V, Vp, active, n, m, threshold, needs, counts):
    """The host build of one decision; updates needs / counts in place, returns the next active list."""
    V, Vp = np.ascontiguousarray(V, np.float32), np.ascontiguousarray(Vp, np.float32)
    active = np.ascontiguousarray(active, np.uint32)
    nxt = np.zeros(max(len(active), 1), np.uint32)
    k = _lib().adapt_sim_step(w, h, V.ctypes.data_as(_F), Vp.ctypes.data_as(_F), active.ctypes.data, len(active), n, m,
                              threshold, needs.ctypes.data, counts.ctypes.data, nxt.ctypes.data)
    return nxt[:k].copy()


def np_needs_more(v, vp, n, m, threshold):
    """pt_adaptive.h adapt_needs_more in numpy float32, operation for operation (v, vp: k x 3)."""
    v, vp = v.astype(np.float32), vp.astype(np.float32)
    fn, fd = np.float32(n), np.float32(n - m)
    with np.errstate(all="ignore"):
        I = v / fn
        A = (v - vp) / fd
        d = np.abs(I - A)
        num = ((np.float32(0) + d[:, 0]) + d[:, 1]) + d[:, 2]
        lum = ((np.float32(0) + I[:, 0]) + I[:, 1]) + I[:, 2]
        e = num / (np.float32(1e-4) + np.sqrt(lum))
        return np.isfinite(v).all(axis=1) & (e >= np.float32(threshold))


def np_step(w, h, V, Vp, active, n, m, threshold, needs, counts):
    """numpy restatement of one decision: needs of the active pixels, keep = 3x3 dilation restricted to the active set,
    the pixels that leave get their count and a cleared needs byte, the rest stays in ascending order."""
    V, Vp = V.reshape(-1, 3), Vp.reshape(-1, 3)
    active = np.asarray(active, np.int64)
    needs[active] = np_needs_more(V[active], Vp[active], n, m, threshold)
    pad = np.zeros((h + 2, w + 2), np.uint8)
    pad[1:-1, 1:-1] = needs.reshape(h, w)
    dil = np.zeros((h, w), np.uint8)
    for dy in range(3):
        for dx in range(3):
            dil |= pad[dy:dy + h, dx:dx + w]
    keep = dil.reshape(-1)[active] != 0
    leave = active[~keep]
    needs[leave] = 0
    counts[leave] = n
    return active[keep].astype(np.uint32)


def _films(rng, w, h, kind):
    n_px = w * h
    V = rng.uniform(0.0, 4.0, (n_px, 3)).astype(np.float32)
    Vp = (V * rng.uniform(0.3, 0.7, (n_px, 3))).astype(np.float32)
    if kind == "zeros":
        V[rng.random(n_px) < 0.5] = 0.0
        Vp[rng.random(n_px) < 0.5] = 0.0
    elif kind == "nonfinite":
        for val in (np.nan, np.inf, -np.inf):
            idx = rng.choice(n_px, max(1, n_px // 8))
            V[idx, rng.integers(0, 3, len(idx))] = val
            idx = rng.choice(n_px, max(1, n_px // 8))
            Vp[idx, rng.integers(0, 3, len(idx))] = val
    elif kind == "flat":  # zero variance: I == A exactly
        V[:] = np.float32(2.0)
        Vp[:] = np.float32(1.0)
    return V, Vp


def _threshold(rng, V, Vp, n, m, which):
    if which == "zero":
        return 0.0
    if which == "inf":
        return float("inf")
    # a threshold among the pixels' own errors, so that both decisions occur
    with np.errstate(all="ignore"):
        I, A = V / np.float32(n), (V - Vp) / np.float32(n - m)
        e = np.abs(I - A).sum(1) / (np.float32(1e-4) + np.sqrt(I.sum(1)))
    e = e[np.isfinite(e)]
    return float(np.quantile(e, 0.6)) if len(e) else 1.0


@pytest.mark.parametrize("w, h", [(17, 13), (1, 9), (9, 1), (1, 1), (2, 2), (32, 5)])
@pytest.mark.parametrize("kind", ["random", "zeros", "nonfinite", "flat"])
@pytest.mark.parametrize("which", ["quantile", "zero", "inf"])
def test_decision_matches_numpy(w, h, kind, which):
    rng = np.random.default_rng(zlib.crc32(repr((w, h, kind, which)).encode()))
    n_px = w * h
    needs_sim, needs_np = np.zeros(n_px, np.uint8), np.zeros(n_px, np.uint8)
    counts_sim, counts_np = np.full(n_px, 64, np.int32), np.full(n_px, 64, np.int32)
    active = np.arange(n_px, dtype=np.uint32)
    n, m = 4, 2
    for _ in range(4):  # a whole schedule: the active set shrinks, the needs map carries over
        if len(active) == 0:
            break
        V, Vp = _films(rng, w, h, kind)
        thr = _threshold(rng, V, Vp, n, m, which)
        a = sim_step(w, h, V, Vp, active, n, m, thr, needs_sim, counts_sim)
        b = np_step(w, h, V, Vp, active, n, m, thr, needs_np, counts_np)
        assert np.array_equal(a, b), (n, thr)
        assert np.array_equal(needs_sim, needs_np)
        assert np.array_equal(counts_sim, counts_np)
        assert np.all(np.diff(a.astype(np.int64)) > 0)  # ascending
        assert set(a.tolist()) <= set(active.tolist())  # pixels that left never return
        active, m, n = a, n, 2 * n
    # (a non-finite Vp under a finite V gives e = inf; on the device flags are sticky, so Vp non-finite implies V non-finite)
    if which == "inf" and kind != "nonfinite":
        assert np.all(counts_sim == 4)  # everybody stops at the first decision
    if which == "zero" and kind in ("random", "zeros", "flat"):
        assert len(active) == n_px  # nobody stops early


def test_borders_and_corners():
    # one pixel needing more keeps exactly its 3x3 neighbourhood, clipped at the frame
    w, h = 6, 5
    for px in [0, w - 1, (h - 1) * w, w * h - 1, 2 * w + 3, 3]:
        V = np.zeros((w * h, 3), np.float32)
        Vp = np.zeros((w * h, 3), np.float32)
        V[px] = (4.0, 4.0, 4.0)  # at n = 4, m = 2: I = 1, A = 0.5, e > 0 here only
        Vp[px] = (3.0, 3.0, 3.0)
        for impl in (sim_step, np_step):
            needs = np.zeros(w * h, np.uint8)
            counts = np.full(w * h, 16, np.int32)
            nxt = impl(w, h, V, Vp, np.arange(w * h, dtype=np.uint32), 4, 2, 1e-3, needs, counts)
            y, x = divmod(px, w)
            want = sorted(yy * w + xx for yy in range(max(0, y - 1), min(h, y + 2)) for xx in range(max(0, x - 1), min(w, x + 2)))
            assert nxt.tolist() == want, (impl.__name__, px)
            assert np.all(counts[want] == 16) and np.all(np.delete(counts, want) == 4)


def test_nonfinite_never_needs_more():
    w, h = 3, 3
    V = np.full((9, 3), 1.0, np.float32)
    Vp = np.zeros((9, 3), np.float32)  # huge error everywhere
    V[4, 1] = np.nan
    needs = np.zeros(9, np.uint8)
    counts = np.zeros(9, np.int32)
    sim_step(w, h, V, Vp, np.arange(9, dtype=np.uint32), 4, 2, 0.0, needs, counts)
    assert needs[4] == 0 and needs.sum() == 8


@pytest.mark.parametrize("min_spp, spp", [(2, 2), (2, 3), (2, 64), (4, 100), (6, 7), (8, 1 << 20), (16, 2147483647)])
def test_schedule(min_spp, spp):
    L = _lib()
    n, got = min_spp, [min_spp // 2, min_spp]
    while n < spp:
        n = L.adapt_sim_next_end(n, spp)
        got.append(n)
    want = [min_spp // 2, min_spp]
    while want[-1] < spp:
        want.append(min(2 * want[-1], spp))
    assert got == want


def test_adaptive_struct_layout(pt, tmp_path):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "ptcore.h"\nint main(){printf("%zu %zu %zu\\n",'
                   "sizeof(ptc_adaptive),offsetof(ptc_adaptive,min_spp),offsetof(ptc_adaptive,threshold));return 0;}\n")
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    assert got == [C.sizeof(pt.Adaptive), pt.Adaptive.min_spp.offset, pt.Adaptive.threshold.offset] == [8, 0, 4]


def test_rust_crate_declares_it():
    src = open(os.path.join(ROOT, "rust", "ptcore-sys", "src", "lib.rs")).read()
    assert re.search(r"pub struct ptc_adaptive \{\s*pub min_spp: i32,\s*pub threshold: f32,\s*\}", src)
    assert re.search(r"pub fn ptc_render_adaptive\(s: \*mut ptc_scene, cam: \*const ptc_camera, st: \*const ptc_render_settings, "
                     r"ad: \*const ptc_adaptive,\s*out_rgb: \*mut f32, out_u32: \*mut u32, out_spp: \*mut i32, stats: \*mut ptc_stats\) -> c_int;", src)


def _scene(pt):
    s = pt.Scene()
    s.add_sphere((0, 0, -1), 0.5, s.add_material(pt.lambertian((0.5, 0.5, 0.5))))
    s.set_camera((0, 0, 0), (0, 0, -1), (0, 1, 0), 60.0, 1.0)
    s.set_settings(8, 6, 16, 4)
    return s


def test_wrapper_passes_arguments(pt, monkeypatch):
    s = _scene(pt)
    st = s.render_settings()
    seen = []

    def fake(h, cam, settings, ad, rgb, u32, spp, stats):
        a = ad._obj
        seen.append((settings._obj.width, settings._obj.height, settings._obj.spp, a.min_spp, a.threshold,
                     bool(rgb), bool(u32), bool(spp)))
        return 0

    monkeypatch.setattr(pt.core(), "ptc_render_adaptive", fake)
    rgb, u32, spp, stats = s.to_core().render_adaptive(s.camera, st, 4, 0.25)
    assert seen == [(8, 6, 16, 4, 0.25, True, True, True)]
    assert rgb.shape == (6, 8, 3) and rgb.dtype == np.float32
    assert u32.shape == (48,) and u32.dtype == np.uint32
    assert spp.shape == (6, 8) and spp.dtype == np.int32
    assert isinstance(stats, pt.Stats)


@pytest.mark.parametrize("min_spp, threshold, over", [
    (3, 0.1, {}), (0, 0.1, {}), (-2, 0.1, {}), (18, 0.1, {}),              # odd, 0, negative, > spp
    (4, float("nan"), {}), (4, -0.5, {}), (4, -float("inf"), {}),         # NaN or negative threshold
    (4, 0.1, {"sample_begin": 0, "sample_end": 8}), (4, 0.1, {"sample_begin": 2, "sample_end": 8}),
    (4, 0.1, {"tile_mod": 2, "tile_rem": 1}), (4, 0.1, {"flags": 8}),     # sample range, tile_mod, NEE_SKY without NEE
])
def test_bad_arguments_are_refused_without_a_device(pt, min_spp, threshold, over):
    s = _scene(pt)
    cs = s.to_core()  # not committed: the arguments are checked first
    with pytest.raises(pt.PtcError) as e:
        cs.render_adaptive(s.camera, s.render_settings(**over), min_spp, threshold)
    assert e.value.code == pt.PTC_E_INVALID


@pytest.mark.parametrize("min_spp, threshold", [(2, 0.0), (4, 0.1), (16, float("inf"))])
def test_uncommitted_scene_is_a_state_error(pt, min_spp, threshold):
    s = _scene(pt)
    with pytest.raises(pt.PtcError) as e:
        s.to_core().render_adaptive(s.camera, s.render_settings(), min_spp, threshold)
    assert e.value.code == pt.PTC_E_STATE
