"""Scenes with more than RG_MAX_LIGHTS lights.  The wavefront loop shades them in chunks of 32 lights, carrying each
lit hit's partial sum from chunk to chunk in light order; the megakernel walks every light.  Every result must be the
oracle's: RGBA8 bytes, f32 bits, ray and error counters.  32 lights is the boundary (one full chunk), 33 leaves a
one-light last chunk, 100 makes four chunks."""
import numpy as np
import pytest

import raingun_b200 as rg
from raingun_b200.scene import scene_from_dict
from raingun_b200.synth import make_light_scene

pytestmark = pytest.mark.gpu

W, H = 256, 144
LIGHTS = [32, 33, 64, 100]


def _counters(st):
    return (st.rays_primary, st.rays_shadow, st.rays_reflection, st.rays_transmission,
            st.err_nan_distance, st.err_transmission_none, st.err_aabb_normal)


def _assert_same(img, ref, st, ost, label):
    bad = int((img != ref).any(axis=2).sum())
    assert bad == 0, f"{label}: {bad} pixels differ from the oracle"
    assert _counters(st) == _counters(ost), (label, _counters(st), _counters(ost))


_cache = {}


def _scene(oracle, lights, spheres):
    """(data, RGBA8, stats, f32) of the many-light scene, rendered once by the oracle."""
    key = (lights, spheres)
    if key not in _cache:
        data, _ = make_light_scene(lights, spheres=spheres, depth=5)
        ref, ost, ref32 = oracle.render(data, W, H, want_f32=True)
        assert ost.rays_shadow > 0
        _cache[key] = (data, ref, ost, ref32)
    return _cache[key]


@pytest.mark.parametrize("lights", LIGHTS)
def test_wavefront_grid_matches_oracle(oracle, lights):
    """Grid tracer, overlap and origin hints on and off, the f32 output, and three frames on one handle (the third
    a graph replay)."""
    data, ref, ost, ref32 = _scene(oracle, lights, 300)
    for overlap in (2, 1):
        for hints in (1, 0):
            with rg.Scene(data) as sc:
                sc.set_pipeline(rg.PIPELINE_WAVEFRONT)
                sc.set_accel(rg.ACCEL_GRID)
                sc.set_option(rg._native.OPT_OVERLAP, overlap)
                sc.set_option(rg._native.OPT_ORIGIN_HINTS, hints)
                label = f"L={lights} grid overlap={overlap} hints={hints}"
                for it in range(3):
                    img = sc.render_image(W, H)
                    _assert_same(img, ref, sc.last_stats, ost, f"{label} frame {it}")
                    assert sc.last_stats.accel_used == rg.ACCEL_GRID
                    if it == 2:
                        assert sc.last_stats.graph_replays == 1, label
                f32 = sc.render_rows_f32(W, H)
                assert np.array_equal(f32.view(np.uint32), ref32.view(np.uint32)), label


@pytest.mark.parametrize("lights", LIGHTS)
def test_wavefront_brute_force_matches_oracle(oracle, lights):
    data, ref, ost, ref32 = _scene(oracle, lights, 300)
    with rg.Scene(data) as sc:
        sc.set_pipeline(rg.PIPELINE_WAVEFRONT)
        sc.set_accel(rg.ACCEL_BRUTE)
        for it in range(3):
            img = sc.render_image(W, H)
            _assert_same(img, ref, sc.last_stats, ost, f"L={lights} brute frame {it}")
            assert sc.last_stats.accel_used == rg.ACCEL_BRUTE
        f32 = sc.render_rows_f32(W, H)
        assert np.array_equal(f32.view(np.uint32), ref32.view(np.uint32))


@pytest.mark.parametrize("lights", LIGHTS)
def test_megakernel_matches_oracle(oracle, lights):
    """AUTO picks the megakernel for a scene of at most 24 bodies; forced, it renders the 301-body scene too."""
    data, ref, ost, ref32 = _scene(oracle, lights, 20)
    with rg.Scene(data) as sc:
        img = sc.render_image(W, H)
        assert sc.last_stats.pipeline_used == rg.PIPELINE_MEGAKERNEL
        _assert_same(img, ref, sc.last_stats, ost, f"L={lights} mega auto")
        f32 = sc.render_rows_f32(W, H)
        assert np.array_equal(f32.view(np.uint32), ref32.view(np.uint32))
    data, ref, ost, _ = _scene(oracle, lights, 300)
    with rg.Scene(data) as sc:
        sc.set_pipeline(rg.PIPELINE_MEGAKERNEL)
        img = sc.render_image(W, H)
        assert sc.last_stats.pipeline_used == rg.PIPELINE_MEGAKERNEL
        _assert_same(img, ref, sc.last_stats, ost, f"L={lights} mega forced")


@pytest.mark.parametrize("lights", [33, 100])
def test_verify_cull_every_chunk(oracle, lights):
    """RG_OPT_VERIFY_CULL=2 re-traces every chunk's shadow queue with the reference scan."""
    data, ref, ost, _ = _scene(oracle, lights, 300)
    for accel in (rg.ACCEL_GRID, rg.ACCEL_BRUTE):
        with rg.Scene(data) as sc:
            sc.set_pipeline(rg.PIPELINE_WAVEFRONT)
            sc.set_accel(accel)
            sc.set_option(rg._native.OPT_VERIFY_CULL, 2)
            img = sc.render_image(W, H)
            _assert_same(img, ref, sc.last_stats, ost, f"L={lights} verify accel={accel}")
            assert sc.last_stats.cull_unsound == 0


@pytest.mark.parametrize("lights", [33, 100])
def test_batches_bands_and_row_lists(oracle, lights):
    """Several batches per frame, streamed bands (RGBA8 and f32), a scattered row list and a host row list."""
    import torch

    data, ref, ost, ref32 = _scene(oracle, lights, 300)
    with rg.Scene(data) as sc:
        sc.set_pipeline(rg.PIPELINE_WAVEFRONT)
        sc.set_option(rg._native.OPT_BATCH_PIXELS, W * 20)
        for it in range(2):
            img = sc.render_image(W, H)
            _assert_same(img, ref, sc.last_stats, ost, f"L={lights} batches frame {it}")
            assert sc.last_stats.batches > 1
        got = np.zeros_like(ref)
        assert sc.streaming_render(W, H, lambda y0, rows: got.__setitem__(slice(y0, y0 + rows.shape[0]), rows) or True,
                                   band_rows=17) is True
        assert np.array_equal(got, ref)
        assert _counters(sc.last_stats) == _counters(ost)
        got32 = np.zeros_like(ref32)
        assert sc.streaming_render_f32(W, H, lambda y0, rows: got32.__setitem__(slice(y0, y0 + rows.shape[0]), rows) or True,
                                       band_rows=23) is True
        assert np.array_equal(got32.view(np.uint32), ref32.view(np.uint32))
        rows = np.array([H - 1, 0, 5, 6, 7, 40, 99], np.uint32)
        out = torch.zeros(H * W * 4, dtype=torch.uint8, device="cuda")
        sc.render_rowlist_scatter(W, H, rows, out.data_ptr(), torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        assert np.array_equal(out.cpu().numpy().reshape(H, W, 4)[rows], ref[rows])
        frame = np.zeros((H, W, 4), np.uint8)
        sc.render_rowlist_host(W, H, rows, frame.ctypes.data)
        assert np.array_equal(frame[rows], ref[rows])
        band = sc.render_rows(W, H, 13, 101)
        assert np.array_equal(band, ref[13:101])


@pytest.mark.parametrize("lights", [33, 100])
def test_multi_device_scene(oracle, lights):
    """Every lane's scene is built by the same upload: two lanes on device 0, and all devices where there are several."""
    data, ref, ost, _ = _scene(oracle, lights, 300)
    ndev = rg.device_count()
    layouts = [[0, 0]] + ([list(range(ndev))] if ndev > 1 else [])
    for devices in layouts:
        with rg.Scene(data, devices=devices) as sc:
            sc.set_pipeline(rg.PIPELINE_WAVEFRONT)
            for it in range(2):
                img = sc.render_image(W, H)
                _assert_same(img, ref, sc.last_stats, ost, f"L={lights} devices={devices} frame {it}")
            band = sc.render_rows(W, H, 13, 101)
            assert np.array_equal(band, ref[13:101])


def test_queue_overflow_with_forty_lights(oracle):
    """Nested glass shells around the camera double the rays at every level, so a level outgrows its queue: the frame
    is repeated with grown queues (and grown light-chunk buffers) and must still be the oracle's."""
    glass = lambda r: {"Sphere": {"center": [0.0, 0.0, 0.0], "radius": r, "material": {
        "coloration": {"Color": "#e0f0ff"}, "albedo": 0.5, "surface": {"Refractive": {"index": 1.3, "transparency": 0.95}}}}}
    diffuse = {"Sphere": {"center": [0.3, -0.2, -0.5], "radius": 0.2, "material": {
        "coloration": {"Color": "#ff8040"}, "albedo": 0.7, "surface": "Diffuse"}}}
    lights = []
    for i in range(40):
        c = "#%02x%02x%02x" % (40 + 5 * i, 255 - 4 * i, 90 + 3 * i)
        if i % 2 == 0:
            lights.append({"Spherical": {"position": [0.05 * (i - 20), 0.6 - 0.02 * i, 0.1], "color": c,
                                         "intensity": 2.0 + 0.25 * i}})
        else:
            lights.append({"Directional": {"direction": {"x": 0.1 * (i - 20), "y": -1.0, "z": -0.5}, "color": c,
                                           "intensity": 0.05 * i}})
    doc = {"maxRecursionDepth": 5, "lights": lights,
           "bodies": [diffuse, glass(1.0), glass(2.0), glass(4.0), glass(8.0), glass(16.0)]}
    data = scene_from_dict(doc)
    w, h = 160, 90
    ref, ost, _ = oracle.render(data, w, h)
    assert ost.rays_reflection + ost.rays_transmission > 6 * w * h   # the tree really doubles
    assert ost.rays_shadow > 0
    with rg.Scene(data) as sc:
        sc.set_pipeline(rg.PIPELINE_WAVEFRONT)
        for it in range(3):
            img = sc.render_image(w, h)
            _assert_same(img, ref, sc.last_stats, ost, f"overflow frame {it}")
            if it >= 1:
                assert sc.last_stats.graph_replays == 1, (it, sc.last_stats.graph_replays)
