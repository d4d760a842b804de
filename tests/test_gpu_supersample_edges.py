"""RG_OPT_SUPERSAMPLE_EDGES: n x n samples only for pixels on an edge of the reference frame (include/raingun_b200.h,
DESIGN.md section 4.6).  The expected frame is built from the CPU oracle alone (tests/edge_oracle.py):
where(mask(R, T), reduce(oracle f32 at n w x n h), oracle n = 1), and the expected counters from the oracle's per-pixel
ray counts: the requested rows and their neighbours at n = 1, plus the samples of the refined requested pixels.  Every
comparison is exact: RGBA8 bytes, f32 bits, counters."""
import importlib.util
import os

import numpy as np
import pytest

import raingun_b200 as rg
from raingun_b200 import _native
from raingun_b200.examples import example_scene
from raingun_b200.scene import scene_from_dict
from raingun_b200.synth import make_light_scene, make_scene

pytestmark = pytest.mark.gpu

_spec = importlib.util.spec_from_file_location("edge_oracle", os.path.join(os.path.dirname(os.path.abspath(__file__)), "edge_oracle.py"))
eo = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(eo)
counters = eo.counters

W, H = 96, 54
PIPES = [("grid", rg.PIPELINE_WAVEFRONT, rg.ACCEL_GRID), ("brute", rg.PIPELINE_WAVEFRONT, rg.ACCEL_BRUTE),
         ("mega", rg.PIPELINE_MEGAKERNEL, rg.ACCEL_BRUTE)]
ROWS = np.array([H - 1, 0, 5, 6, 7, 40, 33, 6, 41], np.uint32)   # unordered, adjacent rows, a duplicate, first and last row


def _glass_scene():
    glass = lambda r: {"Sphere": {"center": [0.0, 0.0, 0.0], "radius": r, "material": {
        "coloration": {"Color": "#e0f0ff"}, "albedo": 0.5, "surface": {"Refractive": {"index": 1.3, "transparency": 0.95}}}}}
    diffuse = {"Sphere": {"center": [0.3, -0.2, -0.5], "radius": 0.2, "material": {
        "coloration": {"Color": "#ff8040"}, "albedo": 0.7, "surface": "Diffuse"}}}
    lights = [{"Spherical": {"position": [0.2, 0.6, 0.1], "color": "#ffffff", "intensity": 3.0}},
              {"Directional": {"direction": {"x": 0.3, "y": -1.0, "z": -0.5}, "color": "#ffe0c0", "intensity": 0.7}}]
    return scene_from_dict({"maxRecursionDepth": 5, "lights": lights,
                            "bodies": [diffuse, glass(1.0), glass(2.0), glass(4.0), glass(8.0), glass(16.0)]})


_scenes = {}


def scene(name):
    if name not in _scenes:
        if name == "C4":
            _scenes[name] = make_scene("C4", spheres=400, depth=8)[0]
        elif name == "L33":
            _scenes[name] = make_light_scene(33, spheres=300, depth=5)[0]
        elif name == "glass":
            _scenes[name] = _glass_scene()
        else:
            _scenes[name] = example_scene(name)
    return _scenes[name]


_expected = {}


def expected(oracle, name, n, w=W, h=H):
    key = (name, n, w, h)
    if key not in _expected:
        _expected[key] = eo.Expected(oracle, scene(name), w, h, n)
    return _expected[key]


def _open(data, pipeline, accel, n=None, t=None, **kw):
    sc = rg.Scene(data, **kw)
    sc.set_pipeline(pipeline)
    sc.set_accel(accel)
    if n is not None:
        sc.set_supersample(n)
    if t is not None:
        sc.set_supersample_edges(t)
    return sc


def _check_frame(sc, ex, t, label):
    ref, ref32, m = ex.frame(t)
    want = ex.counters(t, np.arange(ex.h))
    img = sc.render_image(ex.w, ex.h)
    bad = int((img != ref).any(axis=2).sum())
    assert bad == 0, f"{label}: {bad} pixels differ ({int(m.sum())} refined)"
    assert counters(sc.last_stats) == want, (label, counters(sc.last_stats), want)
    st = sc.last_stats
    f32 = sc.render_rows_f32(ex.w, ex.h)
    assert np.array_equal(f32.view(np.uint32), ref32.view(np.uint32)), label
    assert counters(sc.last_stats) == want, label
    return st


@pytest.mark.parametrize("pipe", PIPES, ids=[p[0] for p in PIPES])
@pytest.mark.parametrize("t", [0, 16])
@pytest.mark.parametrize("n", [2, 3])
@pytest.mark.parametrize("name", ["test1", "test2", "C4"])
def test_matches_oracle(oracle, name, n, t, pipe):
    ex = expected(oracle, name, n)
    assert ex.frame(t)[2].any(), "the case must refine some pixels"
    with _open(scene(name), pipe[1], pipe[2], n, t) as sc:
        for it in range(2):
            st = _check_frame(sc, ex, t, f"{name} n={n} T={t} {pipe[0]} frame {it}")
            assert st.pipeline_used == pipe[1]


@pytest.mark.parametrize("pipe", PIPES, ids=[p[0] for p in PIPES])
def test_threshold_255_is_the_n1_frame(oracle, pipe):
    ex = expected(oracle, "C4", 2)
    with _open(scene("C4"), pipe[1], pipe[2], 2, 255) as sc:
        img = sc.render_image(W, H)
        assert np.array_equal(img, ex.ref)
        assert counters(sc.last_stats) == tuple(int(v) for v in ex.counts1.sum(axis=(0, 1)))
        assert np.array_equal(sc.render_rows_f32(W, H).view(np.uint32), ex.ref32.view(np.uint32))
        assert counters(sc.last_stats) == tuple(int(v) for v in ex.counts1.sum(axis=(0, 1)))


@pytest.mark.parametrize("pipe", PIPES, ids=[p[0] for p in PIPES])
def test_n1_ignores_the_option(pipe):
    """With n = 1 the option changes nothing: the same bytes, f32 bits, counters, launches, batches and graph replays
    as a handle that never set it, over three rounds.  (One warm-up round first: each handle adopts whatever device
    context an earlier scene parked, and its staging buffers, part of the graph keys, may grow on first use.)"""
    data = scene("C4")
    with _open(data, pipe[1], pipe[2]) as a, _open(data, pipe[1], pipe[2], 1, 0) as b:
        for sc in (a, b):
            sc.render_image(W, H)
            sc.render_rows_f32(W, H)
        for it in range(3):
            got = []
            for sc in (a, b):
                img = sc.render_image(W, H)
                si = sc.last_stats
                f32 = sc.render_rows_f32(W, H)
                got.append((img, f32, si, sc.last_stats))
            (ia, fa, sia, sfa), (ib, fb, sib, sfb) = got
            assert np.array_equal(ia, ib) and np.array_equal(fa.view(np.uint32), fb.view(np.uint32)), it
            for x, y in ((sia, sib), (sfa, sfb)):
                assert counters(x) == counters(y), it
                assert (x.gpu_launches, x.batches, x.graph_replays, x.accel_used, x.pipeline_used) == \
                       (y.gpu_launches, y.batches, y.graph_replays, y.accel_used, y.pipeline_used), it


def _refined_rows(m):
    return [y for y in range(m.shape[0]) if m[y].any()]


@pytest.mark.parametrize("pipeline", [rg.PIPELINE_WAVEFRONT, rg.PIPELINE_MEGAKERNEL], ids=["wavefront", "mega"])
def test_every_entry_point(oracle, pipeline):
    import torch

    n, t = 2, 16
    ex = expected(oracle, "C4", n)
    ref, ref32, m = ex.frame(t)
    stream = torch.cuda.current_stream().cuda_stream
    with _open(scene("C4"), pipeline, rg.ACCEL_AUTO, n, t) as sc:
        # a row range whose first and last rows have refined pixels, so the halo rows decide them
        rr = [y for y in _refined_rows(m) if 3 <= y <= H - 4]
        y0, y1 = rr[0], rr[-1] + 1
        assert y0 > 0 and y1 < H
        band = sc.render_rows(W, H, y0, y1)
        assert np.array_equal(band, ref[y0:y1])
        assert counters(sc.last_stats) == ex.counters(t, np.arange(y0, y1))
        assert np.array_equal(sc.render_rows_f32(W, H, y0, y1).view(np.uint32), ref32[y0:y1].view(np.uint32))

        # both streaming renders, bands that do not divide H: every band has its own halo
        bands = [np.arange(b, min(b + 37, H)) for b in range(0, H, 37)]
        want = tuple(map(sum, zip(*[ex.counters(t, b) for b in bands])))
        got = np.zeros_like(ref)
        assert sc.streaming_render(W, H, lambda yb, rows: got.__setitem__(slice(yb, yb + rows.shape[0]), rows) or True,
                                   band_rows=37) is True
        assert np.array_equal(got, ref)
        assert counters(sc.last_stats) == want
        got32 = np.zeros_like(ref32)
        assert sc.streaming_render_f32(W, H, lambda yb, rows: got32.__setitem__(slice(yb, yb + rows.shape[0]), rows) or True,
                                       band_rows=37) is True
        assert np.array_equal(got32.view(np.uint32), ref32.view(np.uint32))
        assert counters(sc.last_stats) == want

        want_list = ex.counters(t, ROWS)
        out = torch.zeros(H * W * 4, dtype=torch.uint8, device="cuda")
        sc.render_rowlist_device(W, H, ROWS, out.data_ptr(), stream)
        torch.cuda.synchronize()
        assert np.array_equal(out[:ROWS.size * W * 4].cpu().numpy().reshape(ROWS.size, W, 4), ref[ROWS])
        assert counters(sc.last_stats) == want_list
        if pipeline == rg.PIPELINE_WAVEFRONT:
            out.zero_()
            sc.render_rowlist_scatter(W, H, ROWS, out.data_ptr(), stream)
            torch.cuda.synchronize()
            frame = out.cpu().numpy().reshape(H, W, 4)
            assert np.array_equal(frame[ROWS], ref[ROWS])
            assert not frame[np.setdiff1d(np.arange(H), ROWS)].any()   # nothing outside the listed rows
            assert counters(sc.last_stats) == want_list
        frame = np.zeros((H, W, 4), np.uint8)
        sc.render_rowlist_host(W, H, ROWS, frame.ctypes.data)
        assert np.array_equal(frame[ROWS], ref[ROWS])
        assert not frame[np.setdiff1d(np.arange(H), ROWS)].any()
        assert counters(sc.last_stats) == want_list

        out.zero_()
        sc.render_rows_device(W, H, 3, 50, out.data_ptr(), stream)
        torch.cuda.synchronize()
        assert np.array_equal(out[:47 * W * 4].cpu().numpy().reshape(47, W, 4), ref[3:50])
        assert counters(sc.last_stats) == ex.counters(t, np.arange(3, 50))

        # the f32 twins
        o32 = torch.zeros(H * W * 3, dtype=torch.float32, device="cuda")
        sc.render_rows_f32_device(W, H, 3, 50, o32.data_ptr(), stream)
        torch.cuda.synchronize()
        assert np.array_equal(o32[:47 * W * 3].cpu().numpy().reshape(47, W, 3).view(np.uint32), ref32[3:50].view(np.uint32))
        sc.render_rowlist_f32_device(W, H, ROWS, o32.data_ptr(), stream)
        torch.cuda.synchronize()
        assert np.array_equal(o32[:ROWS.size * W * 3].cpu().numpy().reshape(ROWS.size, W, 3).view(np.uint32),
                              ref32[ROWS].view(np.uint32))
        assert counters(sc.last_stats) == want_list
        if pipeline == rg.PIPELINE_WAVEFRONT:
            o32.zero_()
            sc.render_rowlist_f32_scatter(W, H, ROWS, o32.data_ptr(), stream)
            torch.cuda.synchronize()
            frame32 = o32.cpu().numpy().reshape(H, W, 3)
            assert np.array_equal(frame32[ROWS].view(np.uint32), ref32[ROWS].view(np.uint32))
            assert not frame32[np.setdiff1d(np.arange(H), ROWS)].any()
        frame32 = np.zeros((H, W, 3), np.float32)
        sc.render_rowlist_f32_host(W, H, ROWS, frame32.ctypes.data)
        assert np.array_equal(frame32[ROWS].view(np.uint32), ref32[ROWS].view(np.uint32))
        assert counters(sc.last_stats) == want_list


def test_multi_device(oracle):
    """The RGBA8 entry points on multi-device handles: the single-device frame whatever the tile height and schedule."""
    ex = expected(oracle, "C4", 2)
    ref = ex.frame(16)[0]
    for kw in (dict(devices=[0, 0]), dict(device=rg.DEVICE_ALL)):
        for tile in (1, 3, 5):
            with _open(scene("C4"), rg.PIPELINE_AUTO, rg.ACCEL_AUTO, 2, 16, **kw) as sc:
                sc.set_option(_native.OPT_TILE_ROWS, tile)
                for it in range(2):
                    assert np.array_equal(sc.render_image(W, H), ref), (kw, tile, it)
                assert np.array_equal(sc.render_rows(W, H, 13, 41), ref[13:41]), (kw, tile)
                got = np.zeros_like(ref)
                assert sc.streaming_render(W, H, lambda yb, rows: got.__setitem__(slice(yb, yb + rows.shape[0]), rows) or True,
                                           band_rows=37) is True
                assert np.array_equal(got, ref), (kw, tile)


@pytest.mark.parametrize("pipeline", [rg.PIPELINE_WAVEFRONT, rg.PIPELINE_MEGAKERNEL], ids=["wavefront", "mega"])
def test_several_batches_per_phase(oracle, pipeline):
    """A small RG_OPT_BATCH_PIXELS: the reference pass runs in several row batches, the refined pixels in several
    batches (megakernel: sample bands) of whole pixels."""
    n, t = 3, 0
    ex = expected(oracle, "C4", n)
    m = ex.frame(t)[2]
    bp = 5 * W + 17
    with _open(scene("C4"), pipeline, rg.ACCEL_GRID, n, t) as sc:
        sc.set_option(_native.OPT_BATCH_PIXELS, bp)
        for it in range(2):
            st = _check_frame(sc, ex, t, f"batches frame {it}")
            ref_batches = -(-H // (bp // W))
            list_batches = -(-int(m.sum()) // (bp // (n * n)))
            if pipeline == rg.PIPELINE_WAVEFRONT:
                assert st.batches == ref_batches + list_batches, (st.batches, ref_batches, list_batches)
            else:
                assert st.gpu_launches == 1 + 3 + 2 * list_batches, st.gpu_launches
        assert np.array_equal(sc.render_rows(W, H, 11, 29), ex.frame(t)[0][11:29])


def test_queue_overflow(oracle):
    """Nested glass shells: a level of the refined samples outgrows its queue, and the batch (its resolve included)
    is repeated with grown queues."""
    n, t, w, h = 2, 0, 80, 45
    ex = expected(oracle, "glass", n, w, h)
    assert int(ex.counts_n[..., 2:4].sum()) > 8 * n * n * w * h
    with _open(scene("glass"), rg.PIPELINE_WAVEFRONT, rg.ACCEL_AUTO, n, t) as sc:
        for it in range(3):
            _check_frame(sc, ex, t, f"overflow frame {it}")


def test_many_lights(oracle):
    ex = expected(oracle, "L33", 2)
    for pipe in PIPES:
        with _open(scene("L33"), pipe[1], pipe[2], 2, 8) as sc:
            _check_frame(sc, ex, 8, f"L33 {pipe[0]}")


def test_graphs_with_alternating_modes(oracle):
    """Adaptive frames interleaved with n = 1 and full n = 2 frames on one wavefront grid handle: each result is right,
    and from the third round on the adaptive frame's batches (reference pass and refined pixels) are all replays."""
    t = 16
    ex = expected(oracle, "C4", 2)
    ref, ref32, _ = ex.frame(t)
    want = ex.counters(t, np.arange(H))
    with _open(scene("C4"), rg.PIPELINE_WAVEFRONT, rg.ACCEL_GRID) as sc:
        for it in range(3):
            sc.set_supersample(1)
            assert np.array_equal(sc.render_image(W, H), ex.ref), it
            sc.set_supersample(2)
            sc.set_supersample_edges(None)
            assert np.array_equal(sc.render_image(W, H), ex.full), it
            sc.set_supersample_edges(t)
            assert np.array_equal(sc.render_image(W, H), ref), it
            st = sc.last_stats
            assert counters(st) == want, it
            assert np.array_equal(sc.render_rows_f32(W, H).view(np.uint32), ref32.view(np.uint32)), it
            if it == 2:
                assert st.batches == 2 and st.graph_replays == 2, (st.batches, st.graph_replays)
                assert sc.last_stats.batches == 2 and sc.last_stats.graph_replays == 2
            sc.set_supersample_edges(None)


def test_full_c4_against_own_frames():
    """C4 with all 10,000 spheres at 640x360, n = 2, T = 8, on the grid: the same handle's own n = 1 and full n = 2
    frames, combined through the mask (GPU self-consistency, no oracle)."""
    w, h, n, t = 640, 360, 2, 8
    with _open(make_scene("C4")[0], rg.PIPELINE_WAVEFRONT, rg.ACCEL_GRID) as sc:
        r = sc.render_image(w, h)
        r32 = sc.render_rows_f32(w, h)
        sc.set_supersample(n)
        full = sc.render_image(w, h)
        full32 = sc.render_rows_f32(w, h)
        sc.set_supersample_edges(t)
        m = eo.mask(r, t)
        assert 0 < m.mean() < 1
        img = sc.render_image(w, h)
        assert np.array_equal(img, np.where(m[..., None], full, r))
        assert sc.last_stats.rays_primary == w * h + n * n * int(m.sum())
        f32 = sc.render_rows_f32(w, h)
        assert np.array_equal(f32.view(np.uint32), np.where(m[..., None], full32, r32).view(np.uint32))


def test_validation():
    for kw in (dict(), dict(devices=[0, 0])):
        with rg.Scene(scene("test1"), **kw) as sc:
            for bad in (-2, 256, 1000):
                with pytest.raises(rg.RaingunError) as e:
                    sc.set_supersample_edges(bad)
                assert e.value.code == _native.E_INVALID
            for ok in (None, 0, 255, 16):
                sc.set_supersample_edges(ok)
            sc.set_supersample(2)
            lib = _native.lib()
            assert lib.rg_render_rows(sc._h, 40000, 30000, 0, 30000, None, None) == _native.E_TOO_LARGE
            with pytest.raises(rg.RaingunError) as e:
                sc.render_image(60, 80)
            assert e.value.code == _native.E_PORTRAIT
