"""RG_OPT_SUPERSAMPLE: n x n primary rays per pixel, averaged on the GPU.  A (w x h) frame is the reference's render
at (n w x n h) reduced n x n (include/raingun_b200.h): per channel, in float32, s = 0, then s + sample(n x + i, n y + j)
for j, then i, in 0..n, then s / (n n).  The reference of every test below is the oracle's f32 render at n x the size,
reduced by `reduce` in exactly that order; the RGBA8 reference quantises that with the oracle's Color::rgba.  Every
result must equal it bit for bit, and the ray and error counters must be the oracle's at n x the size."""
import numpy as np
import pytest

import raingun_b200 as rg
from raingun_b200 import _native
from raingun_b200.examples import example_scene
from raingun_b200.scene import scene_from_dict
from raingun_b200.synth import make_light_scene, make_scene

pytestmark = pytest.mark.gpu

W, H = 96, 54
PIPES = [("grid", rg.PIPELINE_WAVEFRONT, rg.ACCEL_GRID), ("brute", rg.PIPELINE_WAVEFRONT, rg.ACCEL_BRUTE),
         ("mega", rg.PIPELINE_MEGAKERNEL, rg.ACCEL_BRUTE)]
ROWS = np.array([H - 1, 0, 5, 6, 7, 40, 33], np.uint32)   # unordered, with the first and the last row


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


def _counters(st):
    return (st.rays_primary, st.rays_shadow, st.rays_reflection, st.rays_transmission,
            st.err_nan_distance, st.err_transmission_none, st.err_aabb_normal)


_cache = {}


def reference(oracle, name, data, n, w=W, h=H):
    """(RGBA8, f32, oracle stats at n x the size) of the n x n supersampled (w x h) frame."""
    key = (name, n, w, h)
    if key not in _cache:
        _, ost, samples = oracle.render(data, n * w, n * h, want_f32=True)
        avg = reduce(samples, n)
        _cache[key] = (quantise(oracle, avg), avg, ost)
    return _cache[key]


_scenes = {}


def scene(name):
    if name not in _scenes:
        if name == "C4":
            _scenes[name] = make_scene("C4", spheres=400, depth=8)[0]
        elif name == "L33":
            _scenes[name] = make_light_scene(33, spheres=300, depth=5)[0]
        else:
            _scenes[name] = example_scene(name)
    return _scenes[name]


def _open(data, pipeline, accel, n=None):
    sc = rg.Scene(data)
    sc.set_pipeline(pipeline)
    sc.set_accel(accel)
    if n is not None:
        sc.set_supersample(n)
    return sc


def _assert_frame(sc, ref, ref32, ost, n, label, w=W, h=H):
    img = sc.render_image(w, h)
    st = sc.last_stats
    bad = int((img != ref).any(axis=2).sum())
    assert bad == 0, f"{label}: {bad} pixels differ from the reduced oracle render"
    assert _counters(st) == _counters(ost), (label, _counters(st), _counters(ost))
    assert st.rays_primary == n * n * w * h, label
    f32 = sc.render_rows_f32(w, h)
    assert f32.shape == (h, w, 3)
    assert np.array_equal(f32.view(np.uint32), ref32.view(np.uint32)), label
    assert _counters(sc.last_stats) == _counters(ost), label
    return st


@pytest.mark.parametrize("pipe", PIPES, ids=[p[0] for p in PIPES])
def test_supersample_one_is_todays_frame(pipe):
    """set_supersample(1) against a handle that never set it: the same bytes, f32 bits, counters, launches, batches
    and graph replays over three rounds."""
    _, pipeline, accel = pipe
    data = scene("C4")
    with _open(data, pipeline, accel) as a, _open(data, pipeline, accel, 1) as b:
        for it in range(3):
            got = []
            for sc in (a, b):
                img = sc.render_image(W, H)
                si = sc.last_stats
                f32 = sc.render_rows_f32(W, H)
                sf = sc.last_stats
                got.append((img, f32, si, sf))
            (ia, fa, sia, sfa), (ib, fb, sib, sfb) = got
            assert np.array_equal(ia, ib), it
            assert np.array_equal(fa.view(np.uint32), fb.view(np.uint32)), it
            for x, y in ((sia, sib), (sfa, sfb)):
                assert _counters(x) == _counters(y), it
                assert (x.gpu_launches, x.batches, x.graph_replays, x.accel_used, x.pipeline_used) == \
                       (y.gpu_launches, y.batches, y.graph_replays, y.accel_used, y.pipeline_used), it


@pytest.mark.parametrize("pipe", PIPES, ids=[p[0] for p in PIPES])
@pytest.mark.parametrize("name", ["C4", "test1"])
@pytest.mark.parametrize("n", [2, 3])
def test_matches_reduced_oracle(oracle, n, name, pipe):
    _, pipeline, accel = pipe
    data = scene(name)
    ref, ref32, ost = reference(oracle, name, data, n)
    with _open(data, pipeline, accel, n) as sc:
        for it in range(2):
            st = _assert_frame(sc, ref, ref32, ost, n, f"{name} n={n} {pipe[0]} frame {it}")
            assert st.pipeline_used == pipeline


@pytest.mark.parametrize("pipeline", [rg.PIPELINE_WAVEFRONT, rg.PIPELINE_MEGAKERNEL], ids=["wavefront", "mega"])
def test_every_entry_point(oracle, pipeline):
    """One n = 2 handle: a row range, both streaming renders, the three row-list entry points (no scatter on the
    megakernel, which refuses it) and the device-output entry point."""
    import torch

    data = scene("C4")
    ref, ref32, ost = reference(oracle, "C4", data, 2)
    stream = torch.cuda.current_stream().cuda_stream
    with _open(data, pipeline, rg.ACCEL_AUTO, 2) as sc:
        band = sc.render_rows(W, H, 7, 38)
        assert band.shape == (31, W, 4)
        assert np.array_equal(band, ref[7:38])
        assert sc.last_stats.rays_primary == 4 * 31 * W

        got = np.zeros_like(ref)
        assert sc.streaming_render(W, H, lambda y0, rows: got.__setitem__(slice(y0, y0 + rows.shape[0]), rows) or True,
                                   band_rows=37) is True
        assert np.array_equal(got, ref)
        assert _counters(sc.last_stats) == _counters(ost)
        got32 = np.zeros_like(ref32)
        assert sc.streaming_render_f32(W, H, lambda y0, rows: got32.__setitem__(slice(y0, y0 + rows.shape[0]), rows) or True,
                                       band_rows=37) is True
        assert np.array_equal(got32.view(np.uint32), ref32.view(np.uint32))
        assert _counters(sc.last_stats) == _counters(ost)

        out = torch.zeros(H * W * 4, dtype=torch.uint8, device="cuda")
        sc.render_rowlist_device(W, H, ROWS, out.data_ptr(), stream)
        torch.cuda.synchronize()
        assert np.array_equal(out[:ROWS.size * W * 4].cpu().numpy().reshape(ROWS.size, W, 4), ref[ROWS])
        assert sc.last_stats.rays_primary == 4 * ROWS.size * W
        if pipeline == rg.PIPELINE_WAVEFRONT:
            out.zero_()
            sc.render_rowlist_scatter(W, H, ROWS, out.data_ptr(), stream)
            torch.cuda.synchronize()
            frame = out.cpu().numpy().reshape(H, W, 4)
            assert np.array_equal(frame[ROWS], ref[ROWS])
            others = np.setdiff1d(np.arange(H), ROWS)
            assert not frame[others].any()   # nothing outside the listed rows
        frame = np.zeros((H, W, 4), np.uint8)
        sc.render_rowlist_host(W, H, ROWS, frame.ctypes.data)
        assert np.array_equal(frame[ROWS], ref[ROWS])

        out.zero_()
        sc.render_rows_device(W, H, 3, 50, out.data_ptr(), stream)
        torch.cuda.synchronize()
        assert np.array_equal(out[:47 * W * 4].cpu().numpy().reshape(47, W, 4), ref[3:50])


@pytest.mark.parametrize("pipeline", [rg.PIPELINE_WAVEFRONT, rg.PIPELINE_MEGAKERNEL], ids=["wavefront", "mega"])
@pytest.mark.parametrize("rows_per_batch,extra", [(5, 17), (1, -1)], ids=["five_rows", "below_one_row"])
def test_several_batches_per_frame(oracle, pipeline, rows_per_batch, extra):
    """RG_OPT_BATCH_PIXELS that is not a multiple of n W: batches (and the megakernel's sample bands) of whole output
    rows, several per frame.  One sample short of an output row still makes batches of one output row (n sample rows)."""
    data = scene("C4")
    n = 3
    ref, ref32, ost = reference(oracle, "C4", data, n)
    n_batches = (H + rows_per_batch - 1) // rows_per_batch
    with _open(data, pipeline, rg.ACCEL_GRID, n) as sc:
        sc.set_option(_native.OPT_BATCH_PIXELS, n * n * W * rows_per_batch + extra)
        for it in range(2):
            st = _assert_frame(sc, ref, ref32, ost, n, f"batches frame {it}")
            if pipeline == rg.PIPELINE_WAVEFRONT:
                assert st.batches == n_batches, st.batches
            else:
                assert st.gpu_launches == 2 * n_batches, st.gpu_launches
        assert np.array_equal(sc.render_rows(W, H, 11, 29), ref[11:29])


def test_queue_overflow(oracle):
    """Nested glass shells double the rays at every level, so a level of the sample image outgrows its queue: the
    frame is repeated with grown queues and must still be the reference's."""
    glass = lambda r: {"Sphere": {"center": [0.0, 0.0, 0.0], "radius": r, "material": {
        "coloration": {"Color": "#e0f0ff"}, "albedo": 0.5, "surface": {"Refractive": {"index": 1.3, "transparency": 0.95}}}}}
    diffuse = {"Sphere": {"center": [0.3, -0.2, -0.5], "radius": 0.2, "material": {
        "coloration": {"Color": "#ff8040"}, "albedo": 0.7, "surface": "Diffuse"}}}
    lights = [{"Spherical": {"position": [0.2, 0.6, 0.1], "color": "#ffffff", "intensity": 3.0}},
              {"Directional": {"direction": {"x": 0.3, "y": -1.0, "z": -0.5}, "color": "#ffe0c0", "intensity": 0.7}}]
    doc = {"maxRecursionDepth": 5, "lights": lights,
           "bodies": [diffuse, glass(1.0), glass(2.0), glass(4.0), glass(8.0), glass(16.0)]}
    data = scene_from_dict(doc)
    w, h, n = 80, 45, 2
    ref, ref32, ost = reference(oracle, "glass", data, n, w, h)
    # A scene's queues start at 2x the batch's pixels per level (level_growth = 2, DESIGN 4.3), so levels 1-4 of this
    # depth-5 tree hold at most 8x the samples before they grow: more secondary rays than that means some level
    # overflowed in the first frame, and the frame was repeated with grown queues.
    assert ost.rays_reflection + ost.rays_transmission > 8 * n * n * w * h
    with _open(data, rg.PIPELINE_WAVEFRONT, rg.ACCEL_AUTO, n) as sc:
        for it in range(3):
            _assert_frame(sc, ref, ref32, ost, n, f"overflow frame {it}", w, h)


def test_larger_frame_equals_reduced_n1_frame(oracle):
    """C4 with its 10,000 spheres at 640x360, n = 2 on the grid, against the same handle's own 1280x720 f32 frame."""
    data = make_scene("C4")[0]
    w, h = 640, 360
    with _open(data, rg.PIPELINE_WAVEFRONT, rg.ACCEL_GRID) as sc:
        samples = sc.render_rows_f32(2 * w, 2 * h)
        big = sc.last_stats
        avg = reduce(samples, 2)
        sc.set_supersample(2)
        f32 = sc.render_rows_f32(w, h)
        assert np.array_equal(f32.view(np.uint32), avg.view(np.uint32))
        assert _counters(sc.last_stats) == _counters(big)
        img = sc.render_image(w, h)
        assert np.array_equal(img, quantise(oracle, avg))


def test_many_lights(oracle):
    """33 lights: the wavefront shades them in two light chunks; the megakernel reads every light from the arena."""
    data = scene("L33")
    ref, ref32, ost = reference(oracle, "L33", data, 2)
    for pipe in PIPES:
        with _open(data, pipe[1], pipe[2], 2) as sc:
            _assert_frame(sc, ref, ref32, ost, 2, f"L33 {pipe[0]}")


def test_multi_device(oracle):
    """Two lanes on device 0, and every device: the option reaches each lane, and the frame is the single-device one
    whatever the tile height.  devices_used is what the same handle reports at n = 1."""
    data = scene("C4")
    ref, _, ost = reference(oracle, "C4", data, 2)
    layouts = [dict(devices=[0, 0]), dict(device=rg.DEVICE_ALL)]
    for kw in layouts:
        for tile in (1, 3, 5):
            with rg.Scene(data, **kw) as sc:
                sc.set_option(_native.OPT_TILE_ROWS, tile)
                sc.render_image(W, H)
                used = sc.last_stats.devices_used
                sc.set_supersample(2)
                for it in range(2):
                    img = sc.render_image(W, H)
                    assert np.array_equal(img, ref), (kw, tile, it)
                    assert _counters(sc.last_stats) == _counters(ost), (kw, tile, it)
                    assert sc.last_stats.devices_used == used, (kw, tile, it)
                assert np.array_equal(sc.render_rows(W, H, 13, 41), ref[13:41])


def test_graphs_with_alternating_factors(oracle):
    """n = 1 and n = 2 frames, f32 and row-list scatters interleaved on one wavefront grid handle: each call's result
    is right, and from the third round on every call is a replay of its own graph."""
    import torch

    data = scene("C4")
    ref1, _, ref1_32 = oracle.render(data, W, H, want_f32=True)
    ref2, ref2_32, _ = reference(oracle, "C4", data, 2)
    out = torch.zeros(H * W * 4, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    with _open(data, rg.PIPELINE_WAVEFRONT, rg.ACCEL_GRID) as sc:
        for it in range(3):
            replays = {}
            for n, ref, ref32 in ((1, ref1, ref1_32), (2, ref2, ref2_32)):
                sc.set_supersample(n)
                assert np.array_equal(sc.render_image(W, H), ref), (it, n)
                replays[f"image{n}"] = sc.last_stats.graph_replays
                assert np.array_equal(sc.render_rows_f32(W, H).view(np.uint32), ref32.view(np.uint32)), (it, n)
                replays[f"f32_{n}"] = sc.last_stats.graph_replays
                out.zero_()
                sc.render_rowlist_scatter(W, H, ROWS, out.data_ptr(), stream)
                torch.cuda.synchronize()
                replays[f"scatter{n}"] = sc.last_stats.graph_replays
                assert np.array_equal(out.cpu().numpy().reshape(H, W, 4)[ROWS], ref[ROWS]), (it, n)
            if it == 2:
                assert all(v == 1 for v in replays.values()), replays


def test_validation(oracle):
    data = scene("test1")
    lib = _native.lib()
    for kw in (dict(), dict(devices=[0, 0])):
        with rg.Scene(data, **kw) as sc:
            for bad in (0, 9, -1):
                with pytest.raises(rg.RaingunError) as e:
                    sc.set_supersample(bad)
                assert e.value.code == _native.E_INVALID
                assert "14" in str(e.value)
            sc.set_supersample(8)
            sc.set_supersample(2)
            # 40000 x 30000 fits u32; its 80000 x 60000 samples do not.  Refused before anything is allocated.
            assert lib.rg_render_rows(sc._h, 40000, 30000, 0, 30000, None, None) == _native.E_TOO_LARGE
            assert b"overflow" in lib.rg_last_error()
            with pytest.raises(rg.RaingunError) as e:
                sc.render_rows(40000, 30000, 0, 1)
            assert e.value.code == _native.E_TOO_LARGE
            with pytest.raises(rg.RaingunError) as e:
                sc.render_image(60, 80)
            assert e.value.code == _native.E_PORTRAIT
