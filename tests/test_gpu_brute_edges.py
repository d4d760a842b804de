"""The brute-force trace kernels (rg_trace.cuh) at the edges where they can go wrong, against the CPU oracle.

launch_trace (rg_wavefront.cu) picks a kernel per queue from the queue's capacity and the sphere count:
    k_trace_brute_resident   capacity >= sm_count * 2048 and the cull records fit in one CTA's shared memory
                             (R = 3 below 4096 spheres, R = 4 from 4096 on; tiles of 32 R rays per warp);
    k_trace_brute R = 4      capacity >= sm_count * 4096 (tiles of R * 256 rays per block),
                  R = 2      capacity >= sm_count * 2048,
                  R = 1      below;
and RG_BRUTE_VARIANT, RG_RESIDENT_VARIANT and RG_BRUTE_RESIDENT=0 select the other instantiations.  The cull
decision for a (ray, sphere) pair is the same bits in every form, so every kernel must queue the same exact tests:
equal `exact_tests` across kernels shows that no survivor was lost or duplicated.

Every case checks pixels byte for byte, the four ray counts and the three error counters; RG_OPT_VERIFY_CULL=2
additionally re-traces every queued ray on the device with the verbatim FP64 scan (cull_unsound == 0).  Scenes are
built as SceneData arrays (per-body dicts are too slow at millions of bodies): a plane and a box (the non-sphere
prologue), two spherical lights (light-major shadow queues, the ANY kernels) and reflective and refractive spheres
(secondary levels), all within the ~60-unit extents the FP32 cull is made for."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:   # (also run as a script: the variant subprocesses)
    sys.path.insert(0, ROOT)

import raingun_b200 as rg  # noqa: E402
from raingun_b200.scene import (BODY_AABB, BODY_PLANE, BODY_SPHERE, LIGHT_SPHERICAL, SURFACE_DIFFUSE, SURFACE_REFLECTING,
                                SURFACE_REFRACTIVE, SceneData)  # noqa: E402

pytestmark = pytest.mark.gpu

# Mirrors of rg_trace.cuh / rg_wavefront.cu, used to aim frame sizes and sphere counts at the kernel switches.
K_CHUNK = 1024                   # kChunkSpheres
K_RESIDENT_SMEM_MAX = 232448 - 1024   # kResidentSmemMax


def resident_smem_bytes(n_records, R, warps):   # resident_smem_bytes() in rg_trace.cuh
    per_warp = 32 * R * (8 + 4 + 1) + 64 * 4
    return (n_records + 4) * 16 + warps * ((per_warp + 15) & ~15) + 16


def largest_resident_count():   # brute_resident_fits() in rg_wavefront.cu: records padded to 4, R = 4, 20 warps
    n = 4
    while resident_smem_bytes(n + 4, 4, 20) <= K_RESIDENT_SMEM_MAX:
        n += 4
    return n


def sm_count():
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------ scenes
def make_scene(centres, radii, seed=0, depth=4, colours=None, surfaces=None, lights=((-6.0, 14.0, -5.0), (12.0, 9.0, -14.0))):
    """Plane + box + the given spheres (sphere k is body k + 2); materials drawn from `seed`:
    40 % reflective, 30 % refractive, 30 % diffuse unless `surfaces` says otherwise."""
    rng = np.random.default_rng(seed)
    n = len(radii)
    m = n + 2
    sd = SceneData()
    sd.fov = 90.0
    sd.default_color = np.array([0.4, 0.5, 1.0], np.float32)
    sd.max_recursion_depth = depth
    sd.body_kind = np.full(m, BODY_SPHERE, np.uint8)
    sd.body_kind[:2] = (BODY_PLANE, BODY_AABB)
    sd.body_geom = np.zeros((m, 8), np.float64)
    sd.body_geom[0, :6] = (0.0, -2.0, -5.0, 0.0, -1.0, 0.0)
    sd.body_geom[1, :6] = (-3.5, -2.0, -9.0, -1.5, 0.5, -7.0)
    if n:
        sd.body_geom[2:, 0:3] = centres
        sd.body_geom[2:, 3] = radii
    sd.coloration_kind = np.zeros(m, np.uint8)
    sd.color = rng.uniform(0.05, 1.0, (m, 3)).astype(np.float32) if colours is None else np.concatenate(
        [np.full((2, 3), 0.6, np.float32), np.asarray(colours, np.float32)])
    sd.texture_id = np.full(m, -1, np.int32)
    sd.texture_offset = np.zeros((m, 2), np.float32)
    sd.albedo = rng.uniform(0.2, 0.9, m).astype(np.float32)
    if surfaces is None:
        u = rng.uniform(0.0, 1.0, m)
        surfaces = np.where(u < 0.4, SURFACE_REFLECTING, np.where(u < 0.7, SURFACE_REFRACTIVE, SURFACE_DIFFUSE))[2:]
    sd.surface_kind = np.concatenate([[SURFACE_DIFFUSE, SURFACE_REFLECTING], surfaces]).astype(np.uint8)
    sd.surface_param = np.zeros((m, 2), np.float32)
    refl, refr = sd.surface_kind == SURFACE_REFLECTING, sd.surface_kind == SURFACE_REFRACTIVE
    sd.surface_param[refl, 0] = rng.uniform(0.2, 0.9, int(refl.sum()))
    sd.surface_param[refr, 0] = rng.uniform(1.1, 1.8, int(refr.sum()))
    sd.surface_param[refr, 1] = rng.uniform(0.7, 1.0, int(refr.sum()))
    nl = len(lights)
    sd.light_kind = np.full(nl, LIGHT_SPHERICAL, np.uint8)
    sd.light_vec = np.array(lights, np.float64).reshape(nl, 3)
    sd.light_color = np.array([[1.0, 0.9, 0.8], [0.8, 0.9, 1.0], [1.0, 1.0, 1.0]][:nl], np.float32)
    sd.light_intensity = np.full(nl, 6000.0, np.float32)
    return sd


def cloud(n, seed):
    """n visible spheres in front of the camera."""
    rng = np.random.default_rng(1000 + seed)
    c = np.stack([rng.uniform(-12, 12, n), rng.uniform(-1.5, 10, n), rng.uniform(-30, -5, n)], axis=1)
    return c, rng.uniform(0.1, 0.45, n)


def cloud_scene(n, seed=None, depth=4):
    seed = n if seed is None else seed
    c, r = cloud(n, seed)
    return make_scene(c, r, seed=seed, depth=depth)


# ------------------------------------------------------------------ rendering and comparing
def render(data, w, h, accel=rg.ACCEL_BRUTE, verify=0, batch_pixels=0):
    with rg.Scene(data) as sc:
        sc.set_pipeline(rg.PIPELINE_WAVEFRONT)
        sc.set_accel(accel)
        if verify:
            sc.set_option(rg._native.OPT_VERIFY_CULL, verify)
        if batch_pixels:
            sc.set_option(rg._native.OPT_BATCH_PIXELS, batch_pixels)
        img = sc.render_image(w, h)
        return img, sc.last_stats


def counts(st):
    return (st.rays_primary, st.rays_shadow, st.rays_reflection, st.rays_transmission,
            st.err_nan_distance, st.err_transmission_none, st.err_aabb_normal)


def assert_same(img, st, ref, ost, label):
    bad = int((img != ref).any(axis=2).sum())
    assert bad == 0, f"{label}: {bad} pixels differ"
    assert counts(st) == counts(ost), f"{label}: counts {counts(st)} vs {counts(ost)}"


def check_frame(oracle, data, w, h, label, bands=None, batch_pixels=0):
    """The brute-force frame against the oracle (whole frame, or row `bands` with the ray and error counts taken
    from the grid tracer's frame, itself byte-compared), plainly and under RG_OPT_VERIFY_CULL=2.  Returns the
    exact-test count of the plain render."""
    img, st = render(data, w, h, batch_pixels=batch_pixels)
    if bands is None:
        ref, ost, _ = oracle.render(data, w, h)
        assert_same(img, st, ref, ost, label)
    else:
        gimg, gst = render(data, w, h, accel=rg.ACCEL_GRID, batch_pixels=batch_pixels)
        assert_same(img, st, gimg, gst, f"{label} vs grid")
        for y0, y1 in bands:
            ref, _, _ = oracle.render_rows(data, w, h, y0, y1)
            assert np.array_equal(img[y0:y1], ref), f"{label}: rows [{y0},{y1}) differ from the oracle"
    vimg, vst = render(data, w, h, verify=2, batch_pixels=batch_pixels)
    assert vst.cull_unsound == 0, f"{label}: {vst.cull_unsound} rays differ from the verbatim scan"
    assert_same(vimg, vst, img, st, f"{label} VERIFY_CULL=2")
    assert vst.exact_tests == st.exact_tests, label
    return st.exact_tests


# ------------------------------------------------------------------ 1. sphere indices >= 2^22
def big_index_scene():
    """2^22 + 4096 spheres.  The last 4096 are visible; filler k < 4096 sits at the centre of visible sphere
    2^22 + k with half its radius and another colour (a sphere index that lost its top bits would test the filler
    instead: wrong hits, not only misses); the other fillers are specks on a lattice behind the camera."""
    nv, nf = 4096, 1 << 22
    vc, vr = cloud(nv, 22)
    c = np.empty((nf + nv, 3))
    r = np.empty(nf + nv)
    c[nf:], r[nf:] = vc, vr
    c[:nv], r[:nv] = vc, 0.5 * vr
    side = 162
    k = np.arange(nf - nv)
    c[nv:nf, 0] = -20.0 + 0.25 * (k % side)
    c[nv:nf, 1] = 0.25 * ((k // side) % side)
    c[nv:nf, 2] = 5.0 + 0.25 * (k // (side * side))
    r[nv:nf] = 1e-3
    rng = np.random.default_rng(5)
    colours = rng.uniform(0.05, 1.0, (nf + nv, 3)).astype(np.float32)
    colours[:nv] = (0.0, 1.0, 0.0)
    surfaces = np.full(nf + nv, SURFACE_DIFFUSE, np.uint8)
    u = rng.uniform(0.0, 1.0, nv)
    surfaces[nf:] = np.where(u < 0.4, SURFACE_REFLECTING, np.where(u < 0.7, SURFACE_REFRACTIVE, SURFACE_DIFFUSE))
    return make_scene(c, r, seed=22, depth=3, colours=colours, surfaces=surfaces)


def test_sphere_indices_above_2_pow_22(oracle):
    data = big_index_scene()
    S = sm_count()
    w, h = 1280, 720
    assert w * h >= S * 4096   # level 0 runs the streaming R = 4 kernel
    img, st = render(data, w, h)
    gimg, gst = render(data, w, h, accel=rg.ACCEL_GRID)
    assert_same(img, st, gimg, gst, "1280x720 vs grid")
    ref, _, _ = oracle.render_rows(data, w, h, 300, 301)   # (~1e10 body tests per row at this size)
    assert np.array_equal(img[300:301], ref), "1280x720 row 300"
    w, h = 320, 180
    assert 2 * w * h < S * 2048   # the level-0 path and shadow queues run the R = 1 kernel
    img, st = render(data, w, h, verify=2)
    assert st.cull_unsound == 0
    ref, _, _ = oracle.render_rows(data, w, h, 75, 76)
    assert np.array_equal(img[75:76], ref), "320x180 row 75"


# ------------------------------------------------------------------ 2. sphere-count edges
@pytest.mark.parametrize("n", [0, 1, 2, 3, 5, K_CHUNK - 1, K_CHUNK, K_CHUNK + 1, 2 * K_CHUNK + 1])
def test_streaming_sphere_counts(oracle, n):
    """Chunk boundaries of the double-buffered stream (candidates carried across chunks) and the kCullPad padding."""
    check_frame(oracle, cloud_scene(n), 192, 108, f"{n} spheres")


def test_resident_sphere_counts(oracle):
    """Both resident variants, the 4096 switch between them, and the largest count that is resident and the one
    after it (the streaming R = 2 kernel).  The frame's level-0 queue is exactly sm_count * 2048 rays."""
    S = sm_count()
    w, h = 1024, 2 * S
    top = largest_resident_count()
    assert top == 12056
    for n in (1, 5, 4095, 4096, top, top + 1):
        bands = None if n <= 5 else ((h // 2, h // 2 + 1), (h - 40, h - 39))
        check_frame(oracle, cloud_scene(n), w, h, f"{n} spheres, {w}x{h}", bands=bands)


# ------------------------------------------------------------------ 3. queue-size edges
def test_queue_sizes_around_tiles_and_thresholds(oracle):
    """Level-0 queues of one tile, one ray less and one more (batches of one row of that width), and queues just
    under and just over each capacity threshold of launch_trace, on a scene too large for the resident kernel
    (streaming R = 1 / 2 / 4) and one that fits (streaming R = 1 below sm_count * 2048, resident from there)."""
    S = sm_count()
    big = cloud_scene(largest_resident_count() + 44, seed=3)
    small = cloud_scene(3000, seed=4)
    for wd in (255, 256, 257):    # R = 1 tile: 256 rays
        check_frame(oracle, big, wd, 4, f"streaming queue of {wd} rays", batch_pixels=wd)
    for wd in (95, 96, 97, 127, 128, 129):   # resident tiles are 96 / 128 rays; a queue this small streams (R = 1)
        check_frame(oracle, small, wd, 4, f"queue of {wd} rays", batch_pixels=wd)
    # (width, rows per batch): level-0 queue = width * rows.  T2 = S * 2048, T4 = S * 4096.
    for scene, label, sizes in ((big, "streaming", ((1023, 2 * S), (1024, 2 * S), (1025, 2 * S), (1023, 4 * S),
                                                    (1024, 4 * S), (1024 + 1, 4 * S))),
                                (small, "resident", ((1023, 2 * S), (1024, 2 * S), (1025, 2 * S)))):
        for wd, rows in sizes:
            h = rows + 2      # two batches: a full one and a short tail
            bands = ((rows // 2, rows // 2 + 1), (h - 1, h))
            check_frame(oracle, scene, wd, h, f"{label} queue of {wd}x{rows} rays", bands=bands, batch_pixels=wd * rows)


# ------------------------------------------------------------------ 4. every kernel variant, one process each
VARIANTS = ([("default", {})] + [(f"brute{v}", {"RG_BRUTE_VARIANT": str(v)}) for v in range(1, 10)]
            + [(f"resident{v}", {"RG_RESIDENT_VARIANT": str(v)}) for v in range(1, 7)]
            + [("no-resident", {"RG_BRUTE_RESIDENT": "0"})])
VARIANT_FRAME = (1280, 720)


def variant_scenes():
    return {"streaming": cloud_scene(13000, seed=7), "resident": cloud_scene(5000, seed=8)}


def _variant_child(out):
    """Runs in a subprocess (the variant switches are read once per process): renders both scenes plainly and
    under RG_OPT_VERIFY_CULL=2 and writes the frames and the counters to `out`."""
    w, h = VARIANT_FRAME
    res = {}
    for name, data in variant_scenes().items():
        for verify in (0, 2):
            img, st = render(data, w, h, verify=verify)
            res[f"{name}-{verify}-img"] = img
            res[f"{name}-{verify}-stats"] = np.array(counts(st) + (st.exact_tests, st.cull_unsound), np.uint64)
    np.savez(out, **res)


def test_every_variant_renders_the_same_frame(oracle, tmp_path):
    assert VARIANT_FRAME[0] * VARIANT_FRAME[1] >= sm_count() * 4096   # level 0 reaches the RG_BRUTE_VARIANT switch
    got = {}
    for label, env in VARIANTS:
        out = tmp_path / f"{label}.npz"
        r = subprocess.run([sys.executable, os.path.abspath(__file__), str(out)], cwd=ROOT, env={**os.environ, **env},
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, f"{label}: {r.stderr[-2000:]}"
        got[label] = dict(np.load(out))
    base = got["default"]
    for label, res in got.items():
        for key, val in res.items():
            assert np.array_equal(val, base[key]), f"{label}: {key} differs from the default kernels"
    w, h = VARIANT_FRAME
    for name, data in variant_scenes().items():
        assert base[f"{name}-2-stats"][-1] == 0, name
        assert np.array_equal(base[f"{name}-0-img"], base[f"{name}-2-img"]), name
        assert np.array_equal(base[f"{name}-0-stats"][:-1], base[f"{name}-2-stats"][:-1]), name
        for y0, y1 in ((200, 201), (500, 501)):
            ref, _, _ = oracle.render_rows(data, w, h, y0, y1)
            assert np.array_equal(base[f"{name}-0-img"][y0:y1], ref), f"{name}: rows [{y0},{y1})"
        gimg, gst = render(data, w, h, accel=rg.ACCEL_GRID)
        assert np.array_equal(base[f"{name}-0-img"], gimg), name
        assert tuple(int(x) for x in base[f"{name}-0-stats"][:7]) == counts(gst), name


# ------------------------------------------------------------------ 5. many occluders per shadow ray
def test_shadow_rays_with_several_occluders_and_hits_beyond_the_light(oracle):
    """Shadow rays from the floor towards two lights pass through a slab of spheres below the lights (several
    candidates of one ray in one drain: the ANY kernels' shared `occluded` write) and would go on to hit spheres
    above the lights, beyond the light distance (the tmax comparison in drain)."""
    rng = np.random.default_rng(9)
    lights = ((-2.0, 6.0, -10.0), (3.0, 6.5, -12.0))
    below = np.stack([rng.uniform(-6, 6, 300), rng.uniform(2.0, 4.5, 300), rng.uniform(-16, -6, 300)], axis=1)
    above = np.stack([rng.uniform(-6, 6, 300), rng.uniform(7.5, 12.0, 300), rng.uniform(-16, -6, 300)], axis=1)
    c = np.concatenate([below, above])
    r = np.concatenate([rng.uniform(0.2, 0.5, 300), rng.uniform(0.5, 1.2, 300)])
    data = make_scene(c, r, seed=9, depth=3, lights=lights)
    check_frame(oracle, data, 160, 90, "occluder slab")


if __name__ == "__main__":
    _variant_child(sys.argv[1])
