"""The expected results of RG_OPT_SUPERSAMPLE_EDGES (include/raingun_b200.h), built from the CPU oracle alone.

The frame is a pure function of two oracle frames: where(mask(R, T), reduce(oracle f32 at n w x n h), oracle n = 1),
with R the oracle's RGBA8 frame at n = 1.  The counters follow from the oracle's per-pixel ray counts
(edge_oracle_counts.cpp, which includes the oracle's source verbatim and is compiled here into a temporary directory)."""
from __future__ import annotations

import ctypes
import os
import subprocess
import tempfile

import numpy as np

from raingun_b200.scene import SceneDesc

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="rg_edge_oracle_"), "libedge_oracle.so")
        # the oracle's own flags (oracle/Makefile): one IEEE rounding per operation, as the reference
        subprocess.run(["g++", "-O3", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-pthread", "-shared",
                        "-o", out, os.path.join(_HERE, "edge_oracle_counts.cpp")], check=True)
        L = ctypes.CDLL(out)
        L.rgo_render_rows_counts.restype = ctypes.c_int
        L.rgo_render_rows_counts.argtypes = [ctypes.POINTER(SceneDesc), ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32,
                                             ctypes.c_uint32, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        _lib = L
    return _lib


def render_counts(scene, w, h, y0=0, y1=None):
    """(RGBA8 (rows, w, 4), f32 (rows, w, 3), counts (rows, w, 7)) of rows [y0, y1): the oracle's pixels, and per pixel its
    primary, shadow, reflection and transmission rays and its three error counts."""
    y1 = h if y1 is None else y1
    rows = y1 - y0
    rgba = np.zeros((rows, w, 4), np.uint8)
    f32 = np.zeros((rows, w, 3), np.float32)
    counts = np.zeros((rows, w, 7), np.uint64)
    desc, keep = scene.to_desc()
    rc = lib().rgo_render_rows_counts(ctypes.byref(desc), w, h, y0, y1, os.cpu_count() or 1, rgba.ctypes.data, f32.ctypes.data,
                                      counts.ctypes.data)
    del keep
    if rc != 0:
        raise RuntimeError(f"oracle render failed: {rc}")
    return rgba, f32, counts


def mask(img, t):
    """Refined pixels of an RGBA8 frame: some in-image 8-neighbour differs by more than t in r, g or b (alpha ignored)."""
    a = img[..., :3].astype(np.int16)
    h, w = a.shape[:2]
    m = np.zeros((h, w), bool)
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            if dx == 0 and dy == 0:
                continue
            ys, yd = slice(max(0, -dy), h - max(0, dy)), slice(max(0, dy), h - max(0, -dy))
            xs, xd = slice(max(0, -dx), w - max(0, dx)), slice(max(0, dx), w - max(0, -dx))
            m[ys, xs] |= (np.abs(a[ys, xs] - a[yd, xd]) > t).any(axis=2)
    return m


def reduce(samples, n):
    """(n h, n w, 3) float32 samples -> (h, w, 3) float32 averages, summed in the contract's order."""
    h, w = samples.shape[0] // n, samples.shape[1] // n
    s = np.zeros((h, w, 3), np.float32)
    for j in range(n):
        for i in range(n):
            s = s + samples[j::n, i::n]
    return s / np.float32(n * n)


def quantise(oracle, avg):
    """Color::rgba of every pixel (the oracle's quantiser, once per distinct value)."""
    u, inv = np.unique(avg, return_inverse=True)
    q = np.array([oracle.quantise(float(v)) for v in u], np.uint8)[inv.reshape(-1)].reshape(avg.shape)
    return np.concatenate([q, np.full(avg.shape[:2] + (1,), 255, np.uint8)], axis=2)


class Expected:
    """Everything a test compares against for one (scene, w, h, n): the n = 1 frame and its per-pixel counts, the full
    n x n frame and its per-pixel counts (summed over each pixel's samples)."""

    def __init__(self, oracle, scene, w, h, n):
        self.w, self.h, self.n = w, h, n
        self.ref, self.ref32, self.counts1 = render_counts(scene, w, h)
        _, samples, cs = render_counts(scene, n * w, n * h)
        self.full32 = reduce(samples, n)
        self.full = quantise(oracle, self.full32)
        self.counts_n = cs.reshape(h, n, w, n, 7).sum(axis=(1, 3))

    def frame(self, t):
        """(RGBA8, f32, mask) of the adaptive frame at threshold t."""
        m = mask(self.ref, t)
        return (np.where(m[..., None], self.full, self.ref), np.where(m[..., None], self.full32, self.ref32), m)

    def counters(self, t, rows):
        """rays_primary, shadow, reflection, transmission and the three error counts of a call that requests `rows`
        (image rows in call order, duplicates included): R' = those rows and their in-image neighbours, once each,
        at n = 1, plus the n x n samples of every refined requested pixel."""
        m = mask(self.ref, t)
        rows = np.asarray(rows, np.int64)
        halo = np.unique(np.concatenate([rows - 1, rows, rows + 1]))
        halo = halo[(halo >= 0) & (halo < self.h)]
        total = self.counts1[halo].sum(axis=(0, 1))
        total = total + (self.counts_n[rows] * m[rows][..., None]).sum(axis=(0, 1))
        return tuple(int(v) for v in total)


def counters(st):
    return (st.rays_primary, st.rays_shadow, st.rays_reflection, st.rays_transmission,
            st.err_nan_distance, st.err_transmission_none, st.err_aabb_normal)
