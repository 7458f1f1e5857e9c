"""The HDR sky as a light (PTC_FLAG_NEE_SKY), checked on the host through tests/hostsim/skysim.cpp: the g++ build of the
very sky_sample / sky_pdf / table-building code the shade stage runs.

  * tables: the cell probabilities are max-channel x solid angle over the cells of the reference's lookup, normalised;
    the last texel column and row (reached by the lookup on a null set only) have probability 0; an all-zero sky has
    no distribution;
  * sky_pdf integrates to 1 over the sphere;
  * sky_sample returns the pdf sky_pdf gives its direction and the radiance the lookup gives it, and its directions
    fall into the cells with the tables' probabilities.
Each check runs on the teapot scene's envmap (1024 x 512), a random 32 x 16 sky and skies one texel wide or high.
"""
import ctypes as C
import os
import re

import numpy as np
import pytest

from bindings import sim_lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENVMAP = os.path.join(ROOT, "scenes", "teapot", "textures", "envmap.hdr")
_F = C.POINTER(C.c_float)


def _lib():
    L = sim_lib()
    L.sky_sim_create.argtypes = [_F, C.c_int32, C.c_int32]
    L.sky_sim_create.restype = C.c_void_p
    L.sky_sim_destroy.argtypes = [C.c_void_p]
    L.sky_sim_destroy.restype = None
    L.sky_sim_dist.argtypes = [C.c_void_p, _F]
    L.sky_sim_dist.restype = C.c_int64
    L.sky_sim_sample.argtypes = [C.c_void_p, _F, C.c_int64, _F, _F, _F]
    L.sky_sim_pdf.argtypes = [C.c_void_p, _F, C.c_int64, _F]
    return L


def _fp(a):
    return a.ctypes.data_as(_F)


class SimSky:
    """A scene (pt.Scene, for the device) with this sky, and the host build of its sky light."""

    def __init__(self, pt, sky=None, hdr_file=None):
        s = pt.Scene()
        s.add_sphere((0, -1000, 0), 1.0, s.add_material(pt.lambertian((0.5, 0.5, 0.5))))
        if hdr_file:
            s.set_sky_hdr_file(hdr_file)
        else:
            s.set_sky(np.asarray(sky, np.float32))
        self.scene = s
        self.sky = np.ascontiguousarray(s.sky, np.float32)
        self.L = _lib()
        self.h = self.L.sky_sim_create(_fp(self.sky), self.sky.shape[1], self.sky.shape[0])
        assert self.h

    def __del__(self):
        try:
            self.L.sky_sim_destroy(self.h)
        except Exception:
            pass

    def tables(self):
        n = self.L.sky_sim_dist(self.h, None)
        if n == 0:
            return None
        d = np.zeros(n, np.float32)
        assert self.L.sky_sim_dist(self.h, _fp(d)) == n
        h, w = self.sky.shape[:2]
        wc, hc = max(w - 1, 1), max(h - 1, 1)
        return dict(marg=d[:hc + 1], cos=d[hc + 1:2 * hc + 2], inv_sa=d[2 * hc + 2:3 * hc + 2],
                    cond=d[3 * hc + 2:].reshape(hc, wc + 1), wc=wc, hc=hc)

    def sample(self, u4):
        u = np.ascontiguousarray(u4, np.float32)
        n = len(u)
        d, pdf, rgb = np.zeros((n, 3), np.float32), np.zeros(n, np.float32), np.zeros((n, 3), np.float32)
        assert self.L.sky_sim_sample(self.h, _fp(u), n, _fp(d), _fp(pdf), _fp(rgb)) == 0
        return d, pdf, rgb

    def pdf(self, dirs):
        d = np.ascontiguousarray(dirs, np.float32)
        out = np.zeros(len(d), np.float32)
        assert self.L.sky_sim_pdf(self.h, _fp(d), len(d), _fp(out)) == 0
        return out


def reference_probabilities(sky):
    """float64 build: P(cell) = max(r, g, b) x solid angle over the Wc x Hc cells, normalised (and the row / column split)."""
    h, w = sky.shape[:2]
    wc, hc = max(w - 1, 1), max(h - 1, 1)
    cb = np.cos(np.pi * np.arange(hc + 1, dtype=np.float64) / hc)
    sa = 2.0 * np.pi / wc * (cb[:-1] - cb[1:])
    with np.errstate(invalid="ignore", over="ignore"):
        wgt = sky[:hc, :wc].astype(np.float64).max(axis=2) * sa[:, None]
    wgt[~np.isfinite(wgt) | (wgt < 0)] = 0.0
    p = wgt / wgt.sum()
    prow = p.sum(axis=1)
    pcond = np.divide(p, prow[:, None], out=np.zeros_like(p), where=prow[:, None] > 0)
    return p, prow, pcond, sa


def stored_probabilities(t):
    """P(cell) as the device computes it: differences of the stored float CDF entries, multiplied in float32."""
    return np.diff(t["marg"])[:, None] * np.diff(t["cond"], axis=1)


def lookup_cells(sky_shape, dirs):
    """The reference's texel lookup (renderer.rs:40-54) in float64, clamped to the cells."""
    h, w = sky_shape[:2]
    d = dirs.astype(np.float64)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    u = (np.arctan2(d[:, 2], d[:, 0]) + np.pi) / (2 * np.pi)
    v = np.arccos(np.clip(d[:, 1], -1, 1)) / np.pi
    x = np.clip(np.floor(u * (w - 1)), 0, max(w - 2, 0)).astype(np.int64)
    y = np.clip(np.floor(v * (h - 1)), 0, max(h - 2, 0)).astype(np.int64)
    return x, y


def _random_sky(h, w, seed):
    rng = np.random.default_rng(seed)
    sky = rng.exponential(1.0, size=(h, w, 3)).astype(np.float32)
    sky[rng.random((h, w)) < 0.1] = 0.0  # some black texels
    sky[h // 3, w // 2] = (40.0, 35.0, 30.0)  # a hot spot
    return sky


SKIES = {
    "envmap": dict(hdr_file=ENVMAP),
    "random32x16": dict(sky=_random_sky(16, 32, 1)),
    "w1": dict(sky=_random_sky(16, 1, 2)),
    "h1": dict(sky=_random_sky(1, 32, 3)),
}


@pytest.fixture(scope="module", params=sorted(SKIES))
def sky(pt, request):
    return SimSky(pt, **SKIES[request.param])


def test_tables(sky):
    t = sky.tables()
    assert t is not None
    p, prow, pcond, sa = reference_probabilities(sky.sky)
    ps = stored_probabilities(t).astype(np.float64)
    assert ps.shape == p.shape == (t["hc"], t["wc"])  # Wc x Hc cells: the last texel column / row have no cell
    assert abs(ps.sum() - 1.0) < 1e-6
    assert t["marg"][0] == 0 and t["marg"][-1] == 1 and np.all(t["cond"][:, 0] == 0) and np.all(t["cond"][:, -1] == 1)
    assert np.all(np.diff(t["marg"]) >= 0) and np.all(np.diff(t["cond"], axis=1) >= 0)
    # 1e-5 relative, plus what rounding each CDF entry to float can move a difference of two of them by (<= 2^-23 of 1)
    tol = 1e-5 * p + 1.2e-7 * (prow[:, None] + pcond)
    assert np.all(np.abs(ps - p) <= tol), float(np.max(np.abs(ps - p) - tol))
    np.testing.assert_allclose(t["inv_sa"], (1.0 / sa).astype(np.float32), rtol=1e-6)


def test_last_column_and_row_have_probability_zero(sky):
    h, w = sky.sky.shape[:2]
    dirs = []
    if w > 1:
        dirs.append((-1.0, 0.0, 0.0))  # atan2(+0, -1) = pi: u = 1, the last column
    if h > 1:
        dirs.append((0.0, -1.0, 0.0))  # acos(-1) = pi: v = 1, the last row
    if dirs:
        assert np.all(sky.pdf(np.array(dirs, np.float32)) == 0.0)


def test_pdf_integrates_to_one(sky):
    # 2 M stratified directions, uniform over the sphere: y = cos(theta) and phi on a jittered 2048 x 1024 grid
    rng = np.random.default_rng(5)
    ny, nphi = 1024, 2048
    iy, iphi = np.meshgrid(np.arange(ny), np.arange(nphi), indexing="ij")
    y = 1.0 - 2.0 * (iy + rng.random(iy.shape)) / ny
    phi = 2.0 * np.pi * (iphi + rng.random(iphi.shape)) / nphi
    s = np.sqrt(np.maximum(0.0, 1.0 - y * y))
    dirs = np.stack([s * np.cos(phi), y, s * np.sin(phi)], axis=-1).reshape(-1, 3).astype(np.float32)
    assert abs(4.0 * np.pi * sky.pdf(dirs).astype(np.float64).mean() - 1.0) < 5e-3


def test_sample_matches_pdf_lookup_and_probabilities(sky):
    n = 1 << 20
    u4 = np.random.default_rng(7).random((n, 4), dtype=np.float32)
    d, pdf, rgb = sky.sample(u4)
    t = sky.tables()
    assert np.all(np.isfinite(d)) and np.all(pdf > 0)
    np.testing.assert_allclose(np.linalg.norm(d.astype(np.float64), axis=1), 1.0, atol=1e-5)
    # the pdf returned with a direction is the pdf of that direction (cell borders aside)
    assert np.mean(sky.pdf(d) == pdf) >= 0.9999
    # the radiance returned is the lookup's: the texel of the cell the sampler chose (same search as the device)
    yc = np.searchsorted(t["marg"][1:], u4[:, 0], side="right")
    xc = _row_search(t["cond"], yc, u4[:, 1])
    assert np.all(xc < t["wc"]) and np.all(yc < t["hc"])
    assert np.mean(np.all(rgb == sky.sky[yc, xc], axis=1)) >= 0.9999
    # the directions land in the cells with the tables' probabilities: cells (found by an independent float64 lookup)
    # merged in row-major order into bins expecting >= 1000 samples each, every bin within 5 sigma
    x, y = lookup_cells(sky.sky.shape, d)
    counts = np.bincount(y * t["wc"] + x, minlength=t["wc"] * t["hc"]).astype(np.float64)
    expect = stored_probabilities(t).astype(np.float64).ravel() * n
    edges = np.searchsorted(np.cumsum(expect), np.arange(1000.0, n, 1000.0))
    starts = np.unique(np.r_[0, edges[edges < len(expect)]])
    got_b, exp_b = np.add.reduceat(counts, starts), np.add.reduceat(expect, starts)
    keep = exp_b > 0
    z = (got_b[keep] - exp_b[keep]) / np.sqrt(exp_b[keep])
    assert np.max(np.abs(z)) < 5.0, float(np.max(np.abs(z)))


def _row_search(cond, rows, u):
    """first column x with cond[row, x + 1] > u, per sample"""
    out = np.empty(len(rows), np.int64)
    order = np.argsort(rows, kind="stable")
    r_sorted = rows[order]
    starts = np.searchsorted(r_sorted, np.arange(cond.shape[0] + 1))
    for r in range(cond.shape[0]):
        idx = order[starts[r]:starts[r + 1]]
        out[idx] = np.searchsorted(cond[r, 1:], u[idx], side="right")
    return out


def test_zero_sky_has_no_distribution(pt):
    s = SimSky(pt, sky=np.zeros((8, 16, 3), np.float32))
    assert s.tables() is None
    u = np.zeros((1, 4), np.float32)
    out = np.zeros((1, 3), np.float32)
    assert s.L.sky_sim_sample(s.h, _fp(u), 1, _fp(out), _fp(np.zeros(1, np.float32)), _fp(out)) == -4


def test_flag_constant_everywhere(pt):
    assert pt.FLAG_NEE_SKY == 8 and pt.FLAG_NEE == 4
    hdr = open(os.path.join(ROOT, "include", "ptcore.h")).read()
    assert re.search(r"\bPTC_FLAG_NEE_SKY\s*=\s*8\b", hdr)
    rs = open(os.path.join(ROOT, "rust", "ptcore-sys", "src", "lib.rs")).read()
    assert re.search(r"pub const PTC_FLAG_NEE_SKY: i32 = 8;", rs)
    assert re.search(r"\bptc_sky_sample\b", rs) and re.search(r"\bptc_sky_pdf\b", rs)
