"""GPU parity tests proper: the CUDA path (through the C ABI) against the CPU oracle on the same
inputs.  Bar: every byte equal.  The only tolerated exception would be a texel flip caused by
the <=2 ulp difference between CUDA's and glibc's atan2/acos before their narrowing to f32
(probability ~1e-8 per textured hit); none has been observed, so the tests demand equality."""
import os

import numpy as np
import pytest

import raingun_b200 as rg
from raingun_b200.examples import bundled_texture_loader, example_golden, example_scene
from raingun_b200.synth import make_scene

pytestmark = pytest.mark.gpu

MODES = [
    ("mega", rg.PIPELINE_MEGAKERNEL, rg.ACCEL_BRUTE),
    ("wavefront-brute", rg.PIPELINE_WAVEFRONT, rg.ACCEL_BRUTE),
    ("wavefront-grid", rg.PIPELINE_WAVEFRONT, rg.ACCEL_GRID),
]


# The brute-force tracer twice: RG_OPT_VERIFY_CULL=1 runs its debug loop, which re-tests every culled pair exactly
# (cull soundness); =2 runs the shipped FFMA2 loop and then re-traces every queued ray with the verbatim FP64 scan.
CULL_MODES = MODES[:2] + [("wavefront-brute-shipped", rg.PIPELINE_WAVEFRONT, rg.ACCEL_BRUTE)] + MODES[2:]
VERIFY = {"wavefront-brute": 1, "wavefront-brute-shipped": 2}


def _render(data, w, h, pipeline, accel, verify=0):
    with rg.Scene(data) as sc:
        sc.set_pipeline(pipeline)
        sc.set_accel(accel)
        if verify:
            sc.set_option(rg._native.OPT_VERIFY_CULL, int(verify))
        img = sc.render_image(w, h)
        return img, sc.last_stats


def _assert_same(img, ref, st, ost, label):
    diff = np.abs(img.astype(np.int32) - ref.astype(np.int32)).max(axis=2)
    assert int((diff > 0).sum()) == 0, f"{label}: {(diff > 0).sum()} pixels differ (max {diff.max()})"
    assert (st.rays_primary, st.rays_shadow, st.rays_reflection, st.rays_transmission) == (
        ost.rays_primary, ost.rays_shadow, ost.rays_reflection, ost.rays_transmission), label
    assert (st.err_nan_distance, st.err_transmission_none, st.err_aabb_normal) == (
        ost.err_nan_distance, ost.err_transmission_none, ost.err_aabb_normal), label


@pytest.mark.parametrize("mode", MODES, ids=[m[0] for m in MODES])
@pytest.mark.parametrize("name", ["test1", "test2", "test3"])
def test_examples_match_oracle(oracle, name, mode):
    """configs[0..1]: the shipped scenes at their native 800x600."""
    data = example_scene(name)
    ref, ost, _ = oracle.render(data, 800, 600)
    img, st = _render(data, 800, 600, mode[1], mode[2])
    _assert_same(img, ref, st, ost, f"{name}/{mode[0]}")


@pytest.mark.parametrize("name", ["test1", "test2", "test3"])
def test_examples_match_reference_png(name):
    """The device path against the reference's own committed renders: every byte equal, for every
    pipeline (the native JPEG decoder restates jpeg-decoder 0.1.11, so textured pixels match too)."""
    gold = example_golden(name)
    for label, pipeline, accel in MODES:
        img, _ = _render(example_scene(name), 800, 600, pipeline, accel)
        diff = np.abs(img.astype(np.int32) - gold.astype(np.int32)).max(axis=2)
        assert int((diff > 0).sum()) == 0, f"{name}/{label}: {(diff > 0).sum()} pixels differ from the reference PNG"


SYNTH = [("C3", 300, 4, 320, 180), ("C4", 400, 8, 256, 144), ("C5", 500, 6, 192, 108)]


@pytest.mark.parametrize("mode", CULL_MODES, ids=[m[0] for m in CULL_MODES])
@pytest.mark.parametrize("cfg", SYNTH, ids=[c[0] for c in SYNTH])
def test_synthetic_match_oracle(oracle, cfg, mode):
    """configs[2..4] shrunk (same generator stream, fewer spheres / pixels) so the CPU oracle
    finishes in seconds."""
    name, spheres, depth, w, h = cfg
    data, _ = make_scene(name, spheres=spheres, depth=depth, texture_loader=bundled_texture_loader)
    ref, ost, _ = oracle.render(data, w, h)
    img, st = _render(data, w, h, mode[1], mode[2], verify=VERIFY.get(mode[0], 0))
    _assert_same(img, ref, st, ost, f"{name}/{mode[0]}")
    assert st.cull_unsound == 0


def test_row_split_equals_full_frame():
    data, _ = make_scene("C4", spheres=300, depth=6)
    with rg.Scene(data) as sc:
        full = sc.render_image(320, 180)
        parts = [sc.render_rows(320, 180, a, b) for a, b in ((0, 1), (1, 77), (77, 77), (77, 180))]
    assert np.array_equal(np.concatenate(parts, axis=0), full)


def test_small_batches_equal_one_batch():
    data, _ = make_scene("C4", spheres=300, depth=6)
    with rg.Scene(data) as sc:
        full = sc.render_image(320, 180)
        sc.set_option(rg._native.OPT_BATCH_PIXELS, 320 * 7)
        tiled = sc.render_image(320, 180)
        assert sc.last_stats.batches == (180 + 6) // 7
    assert np.array_equal(tiled, full)


def test_host_free_loop_and_graph_replay_agree(oracle):
    """The level loop without host involvement (device-sized launches) and its CUDA-graph replay (the second
    identical frame is a replay) produce the oracle's bytes and ray counts, on a grid scene and on a brute-force
    one, for a full frame, a row band and a scattered row list.  RG_OPT_HOST_FREE is obsolete: setting it
    changes nothing."""
    import torch

    for name, data, w, h in (("C4-small", make_scene("C4", spheres=400, depth=8)[0], 256, 144),
                             ("test1", example_scene("test1"), 200, 150)):
        ref, ost, _ = oracle.render(data, w, h)
        with rg.Scene(data) as sc:
            sc.set_pipeline(rg.PIPELINE_WAVEFRONT)   # (the default would pick the megakernel for test1's handful of bodies)
            for it in range(4):
                img = sc.render_image(w, h)
                st = sc.last_stats
                _assert_same(img, ref, st, ost, f"{name}/host-free frame {it}")
                assert st.host_free == 1
                assert st.graph_replays == (1 if it >= 1 else 0), (name, it, st.graph_replays)
            band = sc.render_rows(w, h, 17, 90)
            assert np.array_equal(band, ref[17:90])
            rows = np.array([h - 1, 0, 5, 6, 7, 40], np.uint32)
            out = torch.empty(rows.size * w * 4, dtype=torch.uint8, device="cuda")
            for _ in range(3):   # eager, capture, replay
                sc.render_rowlist_device(w, h, rows, out.data_ptr(), torch.cuda.current_stream().cuda_stream)
                assert np.array_equal(out.cpu().numpy().reshape(rows.size, w, 4), ref[rows])
            sc.set_option(rg._native.OPT_GRAPH, 1)
            img = sc.render_image(w, h)
            assert sc.last_stats.graph_replays == 0 and sc.last_stats.host_free == 1
            assert np.array_equal(img, ref)
            sc.set_option(rg._native.OPT_HOST_FREE, 1)
            img = sc.render_image(w, h)
            _assert_same(img, ref, sc.last_stats, ost, f"{name}/OPT_HOST_FREE=1")
            assert sc.last_stats.host_free == 1


def test_host_free_queue_overflow_grows_the_queues(oracle):
    """Device-sized queues start at 2x the pixels per level.  Nested glass spheres around the camera
    double the rays at every level (reflection stays inside, transmission meets the next shell), so
    level 2 outgrows its queue: the device flags it, the library doubles the scene's queue growth and
    repeats the frame until it fits, and keeps the larger queues for this scene.  The image must still be
    the oracle's, every frame runs the host-free loop, and from the second frame on it is a graph replay."""
    from raingun_b200.scene import scene_from_dict

    glass = lambda r: {"Sphere": {"center": [0.0, 0.0, 0.0], "radius": r, "material": {
        "coloration": {"Color": "#e0f0ff"}, "albedo": 0.5, "surface": {"Refractive": {"index": 1.3, "transparency": 0.95}}}}}
    doc = {"maxRecursionDepth": 5, "lights": [{"Spherical": {"position": [0.5, 0.5, 0.5], "color": "#ffffff", "intensity": 50.0}}],
           "bodies": [glass(1.0), glass(2.0), glass(4.0), glass(8.0), glass(16.0)]}
    data = scene_from_dict(doc)
    w, h = 160, 90
    ref, ost, _ = oracle.render(data, w, h)
    assert ost.rays_reflection + ost.rays_transmission > 6 * w * h   # the tree really doubles
    with rg.Scene(data) as sc:
        sc.set_pipeline(rg.PIPELINE_WAVEFRONT)   # (the default would pick the megakernel for five bodies)
        for it in range(3):
            img = sc.render_image(w, h)
            _assert_same(img, ref, sc.last_stats, ost, f"overflow frame {it}")
            assert sc.last_stats.host_free == 1
            if it >= 1:
                assert sc.last_stats.graph_replays == 1, (it, sc.last_stats.graph_replays)


def test_multi_device_scene_renders_the_single_device_frame(oracle):
    """Multi-GPU inside the library (rg_scene_create_multi / RG_DEVICE_ALL; rayon's par_iter, rendering.rs:27-35):
    one thread per device, row tiles owned statically or claimed from the atomic tile counter, every device
    copying its rows into the caller's buffer.  On a one-GPU box the same machinery runs as several lanes
    of device 0; with more GPUs it spans them.  Bytes and ray counts must equal the single-device render."""
    ndev = rg.device_count()
    layouts = [[0, 0, 0]] + ([list(range(ndev))] if ndev > 1 else [])
    for name, data, w, h in (("C4-small", make_scene("C4", spheres=400, depth=6)[0], 256, 147),
                             ("test3", example_scene("test3"), 200, 150)):
        ref, ost, _ = oracle.render(data, w, h)
        for devices in layouts:
            with rg.Scene(data, devices=devices) as sc:
                assert sc.device_count == len(devices)
                for schedule, tile_rows in ((1, 8), (2, 8), (2, 3), (0, 16)):
                    sc.set_option(rg._native.OPT_SCHEDULE, schedule)
                    sc.set_option(rg._native.OPT_TILE_ROWS, tile_rows)
                    img = sc.render_image(w, h)
                    _assert_same(img, ref, sc.last_stats, ost, f"{name}/{devices}/schedule {schedule}/tiles {tile_rows}")
                    assert 1 <= sc.last_stats.devices_used <= len(devices)
                band = sc.render_rows(w, h, 13, 101)
                assert np.array_equal(band, ref[13:101])
                got = np.zeros_like(ref)
                assert sc.streaming_render(w, h, lambda y0, rows: got.__setitem__(slice(y0, y0 + rows.shape[0]), rows) or True,
                                           band_rows=40) is True
                assert np.array_equal(got, ref)
                import torch
                with pytest.raises(rg.RaingunError) as e:   # device-pointer entry points need one device
                    sc.render_rows_device(w, h, 0, h, torch.empty(w * h * 4, dtype=torch.uint8, device="cuda").data_ptr(), 0)
                assert e.value.code == rg._native.E_INVALID
    with rg.Scene(example_scene("test2"), device=rg.DEVICE_ALL) as sc:   # every visible GPU
        assert sc.device_count == ndev
        ref, _, _ = oracle.render(example_scene("test2"), 160, 120)
        assert np.array_equal(sc.render_image(160, 120), ref)


def test_concurrent_render_on_one_handle_is_refused():
    """The reference's &Scene is Sync; a device scene owns its scratch queues, so a second render on a busy
    handle returns RG_E_BUSY instead of racing (one handle per thread is the supported way)."""
    import threading

    data, _ = make_scene("C3", spheres=600, depth=4)
    w, h = 1920, 1080
    with rg.Scene(data) as sc:
        ref = sc.render_image(w, h)
        results = []

        def work():
            try:
                results.append(("ok", sc.render_image(w, h)))
            except rg.RaingunError as e:
                results.append(("err", e.code))

        for _ in range(6):
            ts = [threading.Thread(target=work) for _ in range(3)]
            for t in ts:
                t.start()
            for t in ts:
                t.join()
        assert all(kind == "ok" and np.array_equal(val, ref) or kind == "err" and val == rg._native.E_BUSY for kind, val in results)
        assert any(kind == "ok" for kind, _ in results)
        assert np.array_equal(sc.render_image(w, h), ref)   # the handle is usable afterwards


def test_depth_limit_like_draft(oracle):
    """src/main.rs:74-75,119-123: --draft lowers max_recursion_depth to 4; depth 0 still traces
    the primary ray (rendering.rs:71-78) and returns default_color for every child."""
    data = example_scene("test1")
    for limit in (0, 1, 4):
        ref, ost, _ = oracle.render(data, 200, 150, max_depth=limit)
        with rg.Scene(data) as sc:
            sc.set_max_depth_limit(limit)
            img = sc.render_image(200, 150)
            _assert_same(img, ref, sc.last_stats, ost, f"depth {limit}")


def test_streaming_render_bands_and_cancel():
    data = example_scene("test2")
    with rg.Scene(data) as sc:
        full = sc.render_image(160, 120)
        got = np.zeros_like(full)
        seen = []

        def on_rows(y0, rows):
            got[y0:y0 + rows.shape[0]] = rows
            seen.append((y0, rows.shape[0]))
            return True

        assert sc.streaming_render(160, 120, on_rows, band_rows=50) is True
        assert seen == [(0, 50), (50, 50), (100, 20)]
        assert np.array_equal(got, full)
        calls = []
        assert sc.streaming_render(160, 120, lambda y0, rows: calls.append(y0) or False, band_rows=40) is False
        assert calls == [0]     # cancelled after the first band (closed channel, rendering.rs:53-54,67)


def test_unquantised_f32_colours_match_oracle_bit_for_bit(oracle):
    """RenderedPixel.color is an f32 Color (rendering.rs:18-22,59-65): rg_render_rows_f32 / rg_render_stream_f32 deliver
    the colour before Color::rgba narrows it.  Every float must carry the oracle's bits, in every pipeline."""
    for name, data, w, h in (("test1", example_scene("test1"), 200, 150),
                             ("C4-small", make_scene("C4", spheres=300, depth=6)[0], 192, 108)):
        _, _, ref = oracle.render(data, w, h, want_f32=True)
        for label, pipeline, accel in MODES:
            with rg.Scene(data) as sc:
                sc.set_pipeline(pipeline)
                sc.set_accel(accel)
                got = sc.render_rows_f32(w, h)
                assert np.array_equal(got.view(np.uint32), ref.view(np.uint32)), f"{name}/{label}"
                band = sc.render_rows_f32(w, h, 11, 60)
                assert np.array_equal(band.view(np.uint32), ref[11:60].view(np.uint32)), f"{name}/{label} band"
                acc = np.zeros_like(ref)
                assert sc.streaming_render_f32(w, h, lambda y0, rows: acc.__setitem__(slice(y0, y0 + rows.shape[0]), rows) or True,
                                               band_rows=37) is True
                assert np.array_equal(acc.view(np.uint32), ref.view(np.uint32)), f"{name}/{label} stream"
                calls = []
                assert sc.streaming_render_f32(w, h, lambda y0, rows: calls.append(y0) or False, band_rows=50) is False
                assert calls == [0]
                rgba = sc.render_image(w, h)   # the quantised entry point still works on the same handle
                assert (rgba[..., 3] == 255).all()


def test_scatter_rows_odd_width(oracle):
    """rg_render_rowlist_scatter with a width that is not a multiple of 4 (scalar store path) and rows in
    arbitrary order, into a SharedFrame (the buffer other ranks would map through CUDA IPC)."""
    import torch

    data = example_scene("test2")
    w, h = 202, 150
    ref, _, _ = oracle.render(data, w, h)
    rows = np.array([149, 0, 7, 8, 9, 77, 3], np.uint32)
    shared = rg.SharedFrame.create(0, w * h * 4)
    try:
        view = torch.as_tensor(shared, device="cuda:0").view(h, w, 4)
        view.zero_()
        torch.cuda.synchronize()
        with rg.Scene(data) as sc:
            sc.render_rowlist_scatter(w, h, rows, shared.ptr, 0)
        got = view.cpu().numpy()
    finally:
        shared.close()
    assert np.array_equal(got[rows], ref[rows])
    assert not got[np.setdiff1d(np.arange(h), rows)].any()


def test_error_codes():
    data = example_scene("test2")
    with rg.Scene(data) as sc:
        with pytest.raises(rg.RaingunError) as e:
            sc.render_image(100, 200)          # ray.rs:42 assert!(width >= height)
        assert e.value.code == rg._native.E_PORTRAIT
        with pytest.raises(rg.RaingunError) as e:
            sc.render_rows(100, 50, 10, 60)
        assert e.value.code == rg._native.E_INVALID
    deep = data.with_max_depth_limit(None)
    deep.max_recursion_depth = 1000
    with pytest.raises(rg.RaingunError) as e:
        rg.Scene(deep)
    assert e.value.code == rg._native.E_DEPTH


def test_non_unit_directions_and_unnormalised_normals(oracle):
    """Reflections off un-normalised plane/disk normals (bodies.rs:151-153) leave |d| != 1; the
    reference never renormalises, so sphere tests see non-unit rays.  Culling must step aside."""
    import copy
    from raingun_b200.scene import scene_from_dict
    from raingun_b200.synth import SPECS, make_scene_doc

    doc = make_scene_doc(SPECS["C4"], spheres=200, depth=5)
    doc = copy.deepcopy(doc)
    doc["bodies"][0]["Plane"]["normal"] = [0.0, -1.7, 0.3]
    doc["bodies"][0]["Plane"]["material"]["surface"] = {"Reflecting": {"reflectivity": 0.6}}
    data = scene_from_dict(doc)
    ref, ost, _ = oracle.render(data, 240, 135)
    for mode in CULL_MODES:
        img, st = _render(data, 240, 135, mode[1], mode[2], verify=VERIFY.get(mode[0], 0))
        _assert_same(img, ref, st, ost, mode[0])
        assert st.cull_unsound == 0


@pytest.mark.gpu
def test_cli_binary_reproduces_the_reference_pngs(tmp_path):
    """The whole drop-in, natively: `raingun examples/test1.yml` run from a directory laid out like the
    reference checkout (C++ YAML loader + JPEG decoder -> CUDA render -> PNG encoder) must produce
    the reference's committed PNG bit for bit; --preview takes the streaming entry point."""
    import subprocess

    from raingun_b200 import host
    from raingun_b200.examples import _bundle, example_golden

    if not os.path.exists(host.CLI_PATH):
        pytest.fail("raingun CLI is not built (python -c 'import __graft_entry__ as g; g.build()')")
    for key, blob in _bundle().items():
        kind, rel = key.split("/", 1)
        if kind == "golden":
            continue
        path = tmp_path / ("examples/" + rel if kind == "scene" else rel)
        path.parent.mkdir(parents=True, exist_ok=True)
        path.write_bytes(blob)
    for name, extra in (("test1", []), ("test2", []), ("test3", ["--preview"])):
        r = subprocess.run([host.CLI_PATH, f"examples/{name}.yml"] + extra, cwd=tmp_path, capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert f"examples/{name}.yml\t→\texamples/{name}.png\t(" in r.stdout and "render" in r.stdout
        img = host.open_image(str(tmp_path / f"examples/{name}.png"))
        assert img.shape == (600, 800, 4)
        assert np.array_equal(img, example_golden(name)), name
    # --draft lowers the depth to 4 (main.rs:74-75,119-123), -w/-h/-o are honoured
    r = subprocess.run([host.CLI_PATH, "--draft", "-w", "320", "-h", "240", "-o", "d.png", "examples/test1.yml"],
                       cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    with rg.Scene(example_scene("test1").with_max_depth_limit(4)) as sc:
        want = sc.render_image(320, 240)
    assert np.array_equal(host.open_image(str(tmp_path / "d.png")), want)


# ------------------------------------------------------------------ BASELINE.json's full sizes
def _full_frame(name):
    data, spec = make_scene(name, texture_loader=bundled_texture_loader)
    with rg.Scene(data) as sc:
        img = sc.render_image(spec.width, spec.height)
        st = sc.last_stats
    return data, spec, img, st


@pytest.mark.parametrize("name,bands,rays", [
    ("C3", ((0, 2), (1079, 1083), (2158, 2160)), 26532915),
    ("C4", ((300, 301), (1079, 1082), (2000, 2001)), 111009057),
])
def test_full_size_frames_match_oracle_on_row_bands(oracle, name, bands, rays):
    """configs[2..3] at their full 3840x2160: the oracle cannot render the whole frame in test time
    (~5 min on 16 cores for C4) but pixels are independent (rendering.rs:27-35), so full-resolution
    row bands are an exact check of the full-size frame.  The ray total pins the whole frame."""
    data, spec, img, st = _full_frame(name)
    assert st.rays == rays
    assert (st.err_nan_distance, st.err_transmission_none, st.err_aabb_normal) == (0, 0, 0)
    assert (img[..., 3] == 255).all()
    for y0, y1 in bands:
        ref, _, _ = oracle.render_rows(data, spec.width, spec.height, y0, y1)
        assert np.array_equal(img[y0:y1], ref), f"{name} rows [{y0},{y1})"


def test_full_size_c4_every_strategy_renders_the_same_frame():
    """Size-independent property at the headline configuration: exact culling (grid), the reference's
    all-pairs scan (brute force), the one- and two-stream schedules and a row-list split all produce
    the same 8.3 M pixels and the same ray counts."""
    data, spec = make_scene("C4")
    w, h = spec.width, spec.height
    frames, counts = {}, {}
    for label, accel, overlap in (("grid", rg.ACCEL_GRID, 0), ("grid-1stream", rg.ACCEL_GRID, 1),
                                  ("brute", rg.ACCEL_BRUTE, 0), ("brute-2stream", rg.ACCEL_BRUTE, 2)):
        with rg.Scene(data) as sc:
            sc.set_accel(accel)
            sc.set_option(rg._native.OPT_OVERLAP, overlap)
            frames[label] = sc.render_image(w, h)
            s = sc.last_stats
            counts[label] = (s.rays_primary, s.rays_shadow, s.rays_reflection, s.rays_transmission)
    for label in frames:
        assert np.array_equal(frames[label], frames["grid"]), label
        assert counts[label] == counts["grid"], label
    import torch
    rows = np.concatenate([np.arange(y, min(h, y + 8), dtype=np.uint32) for y in range(8, h, 24)])   # every third 8-row tile
    out = torch.empty(rows.size * w * 4, dtype=torch.uint8, device="cuda")
    with rg.Scene(data) as sc:
        sc.render_rowlist_device(w, h, rows, out.data_ptr(), torch.cuda.current_stream().cuda_stream)
    assert np.array_equal(out.cpu().numpy().reshape(rows.size, w, 4), frames["grid"][rows])
    # the gather-fused form: the same rows stored at their own place in a full frame (two batches)
    frame = torch.zeros((h, w, 4), dtype=torch.uint8, device="cuda")
    with rg.Scene(data) as sc:
        sc.set_option(rg._native.OPT_BATCH_PIXELS, w * 400)
        sc.render_rowlist_scatter(w, h, rows, frame.data_ptr(), torch.cuda.current_stream().cuda_stream)
        assert sc.last_stats.batches == 2
    got = frame.cpu().numpy()
    assert np.array_equal(got[rows], frames["grid"][rows])
    rest = np.setdiff1d(np.arange(h), rows)
    assert not got[rest].any()


def test_origin_hints_change_no_pixel_and_spare_the_exact_tests():
    """RG_OPT_ORIGIN_HINTS (rg_trace.cuh): k_shade tests every ray it emits against the sphere the ray starts on and
    the grid tracer skips that sphere.  Same frame, same ray counts, same error counters with the hints on and
    off and against the verbatim scan (RG_OPT_VERIFY_CULL=2 re-traces every queued ray without hints on the
    device); far fewer exact tests with them.  C4 (glass, mirrors, diffuse: rays that leave, enter and graze
    their own sphere) and the all-diffuse C3."""
    for name, w, h in (("C4", 1280, 720), ("C3", 960, 540)):
        data, _ = make_scene(name)
        got = {}
        for hints in (1, 0):
            with rg.Scene(data) as sc:
                sc.set_accel(rg.ACCEL_GRID)
                sc.set_option(rg._native.OPT_ORIGIN_HINTS, hints)
                sc.set_option(rg._native.OPT_VERIFY_CULL, 2)     # (eager host-free loop + the verbatim re-trace)
                img = sc.render_image(w, h)
                assert sc.last_stats.cull_unsound == 0, (name, hints)
                sc.set_option(rg._native.OPT_VERIFY_CULL, 0)
                for _ in range(3):                               # host-free loop, then its captured graph
                    assert np.array_equal(sc.render_image(w, h), img)
                got[hints] = (img, sc.last_stats)
        _assert_same(got[1][0], got[0][0], got[1][1], got[0][1], f"{name} hints on vs off")
        assert got[1][1].exact_tests < 0.85 * got[0][1].exact_tests, (name, got[1][1].exact_tests, got[0][1].exact_tests)


def test_resident_brute_kernel_cull_is_sound_at_scale():
    """The shared-memory-resident brute-force kernel (queues of >= 300 k rays, scenes of <= ~11,000
    spheres) with RG_OPT_VERIFY_CULL=1: every pair the FP32 cull rejects is re-tested exactly on the
    device and must miss; and with RG_OPT_VERIFY_CULL=2: the shipped loop's result for every ray must
    equal the verbatim scan's.  Both images must equal the grid tracer's."""
    data, _ = make_scene("C3")
    w, h = 1920, 1080
    ref, rst = _render(data, w, h, rg.PIPELINE_WAVEFRONT, rg.ACCEL_GRID)
    for verify in (1, 2):
        img, st = _render(data, w, h, rg.PIPELINE_WAVEFRONT, rg.ACCEL_BRUTE, verify=verify)
        assert st.cull_unsound == 0 and st.rays_primary == w * h, verify
        assert np.array_equal(img, ref) and st.rays == rst.rays, verify


def test_full_size_c5_row_matches_oracle(oracle):
    """configs[4]: 7680x4320, 100,000 spheres, 4 spherical lights, textured, depth 8 (two wavefront
    batches).  One full-resolution row through the oracle (~1.7e10 body tests) pins it."""
    data, spec, img, st = _full_frame("C5")
    assert st.rays == 673163668 and st.batches == 2
    y = 2600
    ref, _, _ = oracle.render_rows(data, spec.width, spec.height, y, y + 1)
    assert np.array_equal(img[y:y + 1], ref)


def test_c5_all_100k_spheres_grid_equals_verbatim_scan():
    """configs[4] with ALL 100,000 spheres (a grid near its 256-cells-per-axis cap, chained cell records, textured
    spheres, 4 spherical lights) on a whole 480x270 frame: the grid tracer's image and ray counts equal the
    megakernel's (the reference recursion with every body tested in FP64, itself oracle-checked above), and
    RG_OPT_VERIFY_CULL=2 — every traced ray re-traced on the device with the verbatim scan — finds no difference."""
    data, _ = make_scene("C5", texture_loader=bundled_texture_loader)
    w, h = 480, 270
    mega, mst = _render(data, w, h, rg.PIPELINE_MEGAKERNEL, rg.ACCEL_BRUTE)
    grid, gst = _render(data, w, h, rg.PIPELINE_WAVEFRONT, rg.ACCEL_GRID)
    assert np.array_equal(grid, mega)
    assert (gst.rays_primary, gst.rays_shadow, gst.rays_reflection, gst.rays_transmission) == (
        mst.rays_primary, mst.rays_shadow, mst.rays_reflection, mst.rays_transmission)
    with rg.Scene(data) as sc:
        sc.set_pipeline(rg.PIPELINE_WAVEFRONT)
        sc.set_accel(rg.ACCEL_GRID)
        sc.set_option(rg._native.OPT_VERIFY_CULL, 2)
        img = sc.render_image(w, h)
        assert sc.last_stats.cull_unsound == 0
    assert np.array_equal(img, mega)


def test_peer_store_gather_across_two_devices():
    """The fused gather on real hardware: a scene on GPU 1 stores its rows straight into a frame that lives on
    GPU 0 (rg_render_rowlist_scatter over NVLink peer access), GPU 0 renders the rest; the assembled frame must
    equal the one-GPU frame byte for byte.  Needs two GPUs (skipped on a one-GPU box)."""
    import torch

    if rg.device_count() < 2:
        pytest.skip("needs two GPUs")
    if not torch.cuda.can_device_access_peer(1, 0):
        pytest.skip("no peer access between GPU 1 and GPU 0")
    data, _ = make_scene("C4", spheres=2000, depth=8)
    w, h = 1280, 720
    with rg.Scene(data, device=0) as sc:
        sc.set_pipeline(rg.PIPELINE_WAVEFRONT)
        ref = sc.render_image(w, h)
    frame = torch.zeros((h, w, 4), dtype=torch.uint8, device="cuda:0")
    rg._native.check(rg._native.lib().rg_device_enable_peer(1, 0))   # kernels on GPU 1 may store into GPU 0's memory
    tiles = [np.arange(y, min(h, y + 8), dtype=np.uint32) for y in range(0, h, 8)]
    rows0 = np.concatenate(tiles[0::2])
    rows1 = np.concatenate(tiles[1::2])
    with rg.Scene(data, device=0) as s0, rg.Scene(data, device=1) as s1:
        for s_ in (s0, s1):
            s_.set_pipeline(rg.PIPELINE_WAVEFRONT)
        with torch.cuda.device(1):
            s1.render_rowlist_scatter(w, h, rows1, frame.data_ptr(), torch.cuda.current_stream(1).cuda_stream)
        with torch.cuda.device(0):
            s0.render_rowlist_scatter(w, h, rows0, frame.data_ptr(), torch.cuda.current_stream(0).cuda_stream)
    torch.cuda.synchronize(1)
    torch.cuda.synchronize(0)
    assert np.array_equal(frame.cpu().numpy(), ref)


def test_degenerate_scenes(oracle):
    """Edge cases of the level loop: no lights (no shadow side at all), no bodies (every pixel is
    default_color after one traced primary ray, rendering.rs:71-78), a single level."""
    import copy
    from raingun_b200.scene import scene_from_dict
    from raingun_b200.synth import SPECS, make_scene_doc

    base = make_scene_doc(SPECS["C4"], spheres=150, depth=5)
    no_lights = copy.deepcopy(base)
    no_lights["lights"] = []
    no_bodies = copy.deepcopy(base)
    no_bodies["bodies"] = []
    one_level = copy.deepcopy(base)
    one_level["maxRecursionDepth"] = 1
    for label, doc in (("no lights", no_lights), ("no bodies", no_bodies), ("one level", one_level)):
        data = scene_from_dict(doc)
        ref, ost, _ = oracle.render(data, 160, 90)
        for mode in MODES:
            img, st = _render(data, 160, 90, mode[1], mode[2])
            _assert_same(img, ref, st, ost, f"{label}/{mode[0]}")
    data = scene_from_dict(no_bodies)
    img, st = _render(data, 160, 90, rg.PIPELINE_WAVEFRONT, rg.ACCEL_AUTO)
    assert st.rays == 160 * 90 and (img[..., :3] == np.array([0x66, 0x7f, 0xff], np.uint8)).all()


# ------------------------------------------------------------------ adversarial geometry
def _mat(rng, kind=None, tex=None):
    kind = kind or rng.choice(["Diffuse", "Reflecting", "Refractive"], p=[0.4, 0.3, 0.3])
    surface = "Diffuse"
    if kind == "Reflecting":
        surface = {"Reflecting": {"reflectivity": float(np.round(rng.uniform(0.1, 1.0), 3))}}
    elif kind == "Refractive":
        surface = {"Refractive": {"index": float(np.round(rng.uniform(1.0, 2.4), 3)),
                                  "transparency": float(np.round(rng.uniform(0.0, 1.0), 3))}}
    col = {"Color": "#%06x" % int(rng.integers(0, 1 << 24))}
    if tex is not None:
        col = {"Texture": {"image": tex, "x_offset": float(np.round(rng.uniform(-2, 2), 3)),
                           "y_offset": float(np.round(rng.uniform(-2, 2), 3))}}
    return {"coloration": col, "albedo": float(np.round(rng.uniform(0.05, 1.0), 3)), "surface": surface}


def _sphere(rng, c, r, **kw):
    return {"Sphere": {"center": [float(x) for x in c], "radius": float(r), "material": _mat(rng, **kw)}}


def _adversarial_scenes():
    from raingun_b200.synth import CLAY, EARTH

    out = []
    sun = {"Directional": {"direction": [0.0, -1.0, 0.0], "color": "#ffffff", "intensity": 5.0}}   # axis-parallel shadow rays
    bulb = lambda p, i=3000.0: {"Spherical": {"position": [float(x) for x in p], "color": "#ffeedd", "intensity": i}}
    ground = lambda rng, **kw: {"Plane": {"origin": [0.0, -2.0, 0.0], "normal": [0.0, -1.0, 0.0], "material": _mat(rng, **kw)}}

    rng = np.random.default_rng(11)   # A: the camera sits inside a big refractive sphere
    bodies = [ground(rng, kind="Diffuse"), _sphere(rng, (0, 0, -1), 6.0, kind="Refractive")]
    bodies += [_sphere(rng, rng.uniform((-4, -1.5, -9), (4, 4, -2)), rng.uniform(0.1, 0.6)) for _ in range(40)]
    out.append(("camera-inside-glass", {"maxRecursionDepth": 6, "lights": [sun, bulb((2, 3, -3))], "bodies": bodies}))

    rng = np.random.default_rng(12)   # B: integer lattice, radii that touch cell walls, axis-parallel light
    bodies = [ground(rng, kind="Reflecting")]
    bodies += [_sphere(rng, (x, y, z), 0.5) for x in range(-3, 4) for y in range(-1, 3) for z in range(-10, -3)]
    out.append(("lattice", {"maxRecursionDepth": 5, "fov": 70.0, "lights": [sun, bulb((0, 6, -6))], "bodies": bodies}))

    rng = np.random.default_rng(13)   # C: dense overlapping cluster, one huge ("loose") sphere, specks
    bodies = [_sphere(rng, (0, -60, -20), 55.0, kind="Diffuse")]
    bodies += [_sphere(rng, rng.normal((0, 0, -8), 1.2), rng.uniform(0.2, 1.0)) for _ in range(120)]
    bodies += [_sphere(rng, rng.uniform((-3, -2, -7), (3, 3, -3)), rng.uniform(1e-3, 2e-2)) for _ in range(150)]
    out.append(("cluster+loose+specks", {"maxRecursionDepth": 7, "lights": [bulb((0, 8, -4)), bulb((-6, 1, -2), 800.0)],
                                        "bodies": bodies}))

    rng = np.random.default_rng(14)   # D: disks, boxes and textures among enough spheres to enable the grid
    bodies = [ground(rng, tex=CLAY),
              {"Disk": {"origin": [1.5, 0.5, -6.0], "normal": [0.3, -0.2, -1.0], "radius": 1.8, "material": _mat(rng, kind="Reflecting")}},
              {"Disk": {"origin": [-2.0, 1.0, -5.0], "normal": [0.0, 0.0, -2.5], "radius": 1.0, "material": _mat(rng, tex=EARTH)}},
              {"AABB": {"bounds": [[-3.5, -2.0, -9.0], [-1.5, 0.5, -7.0]], "material": _mat(rng, kind="Diffuse")}},
              {"AABB": {"bounds": [[1.0, -2.0, -4.5], [2.0, -1.0, -3.5]], "material": _mat(rng, kind="Reflecting")}}]
    bodies += [_sphere(rng, rng.uniform((-5, -1.5, -12), (5, 5, -3)), rng.uniform(0.15, 0.7),
                       tex=(EARTH if i % 3 == 0 else None)) for i in range(90)]
    out.append(("mixed-kinds+textures", {"maxRecursionDepth": 6, "defaultColor": "#203040",
                                         "lights": [sun, bulb((3, 5, -2)), bulb((-4, 2, -10), 1500.0)], "bodies": bodies}))

    rng = np.random.default_rng(15)   # E: far-away geometry (FP32 grid coordinates would fail) and horizon hits
    bodies = [ground(rng, kind="Reflecting")]
    bodies += [_sphere(rng, rng.uniform((-400, 0, -3000), (400, 600, -800)), rng.uniform(20, 90)) for _ in range(80)]
    out.append(("far-field", {"maxRecursionDepth": 5, "fov": 40.0,
                              "lights": [{"Directional": {"direction": [0.3, -1.0, -0.2], "color": "#ffffff", "intensity": 4.0}},
                                         bulb((0, 900, -1500), 4e7)], "bodies": bodies}))

    rng = np.random.default_rng(16)   # F: lights inside bodies / at a centre / with zero intensity; 12 spheres (grid only if forced)
    bodies = [ground(rng, kind="Diffuse")] + [_sphere(rng, rng.uniform((-3, -1, -8), (3, 3, -3)), rng.uniform(0.4, 1.2)) for _ in range(12)]
    c0 = bodies[1]["Sphere"]["center"]
    out.append(("odd-lights", {"maxRecursionDepth": 4, "lights": [bulb(c0, 500.0), bulb((0, 1, -5), 0.0), sun], "bodies": bodies}))

    rng = np.random.default_rng(17)   # G: degenerate parameters the reference accepts without complaint
    bodies = [ground(rng, kind="Diffuse"),
              _sphere(rng, (0, 0, 0), 0.75, kind="Refractive"),          # centred on the camera: h = 0
              _sphere(rng, (1, 0, -4), 0.0), _sphere(rng, (-1, 0.5, -4), -0.6, kind="Reflecting"),   # zero / negative radius
              {"Plane": {"origin": [0, 0, -9], "normal": [0.0, 0.0, 0.0], "material": _mat(rng)}},     # den = 0: never hit
              {"Disk": {"origin": [0, 1, -5], "normal": [0, 0, -1], "radius": 0.0, "material": _mat(rng)}},
              {"AABB": {"bounds": [[1.0, 1.0, -5.0], [-1.0, -1.0, -7.0]], "material": _mat(rng, kind="Diffuse")}},   # min > max
              {"AABB": {"bounds": [[2.0, -2.0, -6.0], [2.0, 0.0, -4.0]], "material": _mat(rng, kind="Diffuse")}}]    # zero thickness
    bodies += [_sphere(rng, rng.uniform((-4, -1.5, -10), (4, 4, -2)), rng.uniform(-0.5, 0.9)) for _ in range(30)]
    out.append(("degenerate-parameters", {"maxRecursionDepth": 6, "fov": 150.0, "lights": [sun, bulb((0, 0, 0), 200.0)],
                                          "bodies": bodies}))
    return out


@pytest.mark.parametrize("case", _adversarial_scenes(), ids=lambda c: c[0])
def test_adversarial_geometry_matches_oracle(oracle, case):
    """Scenes built to stress what the synthetic configs do not: origins inside spheres, rays parallel
    to grid axes and through cell corners, a sphere too large for the grid, specks, every body kind,
    far-away coordinates, lights inside geometry.  Every pipeline, byte for byte, equal ray counts and
    equal panic counters (NaN distances, failed transmissions, undecidable box normals)."""
    from raingun_b200.scene import scene_from_dict

    name, doc = case
    data = scene_from_dict(doc, bundled_texture_loader)
    w, h = 224, 126
    ref, ost, _ = oracle.render(data, w, h)
    for mode in CULL_MODES:
        img, st = _render(data, w, h, mode[1], mode[2], verify=VERIFY.get(mode[0], 0))
        _assert_same(img, ref, st, ost, f"{name}/{mode[0]}")
        assert st.cull_unsound == 0


def test_reference_panic_conditions_are_counted_not_raised(oracle):
    """Where the reference would panic, the library counts and carries on (include/raingun_b200.h):
    a hit point no face of a far-away box is within 1e-8 of -> `assert!(false)` bodies.rs:324; a sphere
    with an infinite centre -> NaN distance -> `partial_cmp().unwrap()` scene.rs:38.  Oracle and device
    must agree on the counts and on every pixel."""
    from raingun_b200.scene import scene_from_dict

    mat = lambda s="Diffuse": {"coloration": {"Color": "#c0c0c0"}, "albedo": 0.5, "surface": s}
    doc = {"maxRecursionDepth": 4,
           "lights": [{"Directional": {"direction": [0.2, -1.0, -0.3], "color": "#ffffff", "intensity": 5.0}}],
           "bodies": [
               {"Plane": {"origin": [0.0, -2.0, 0.0], "normal": [0.0, -1.0, 0.0], "material": mat({"Reflecting": {"reflectivity": 0.5}})}},
               {"AABB": {"bounds": [[1.0e9, -1.0e8, -1.0e10 + 0.3], [2.0e9 + 0.7, 1.0e8, -3.3e9 - 0.1]], "material": mat()}},
               {"Sphere": {"center": [-2.5, 0.0, -5.0], "radius": 1.0, "material": mat({"Refractive": {"index": 1.5, "transparency": 0.9}})}}]}
    far_box = scene_from_dict(doc)
    doc["bodies"].append({"Sphere": {"center": [float("inf"), 0.0, -5.0], "radius": 1.0, "material": mat()}})
    nan_sphere = scene_from_dict(doc)
    w, h = 224, 126
    for label, data, want_nan, want_aabb in (("far box", far_box, False, True), ("infinite sphere", nan_sphere, True, True)):
        ref, ost, _ = oracle.render(data, w, h)
        assert (ost.err_nan_distance > 0) == want_nan and (ost.err_aabb_normal > 0) == want_aabb
        for mode in MODES:
            img, st = _render(data, w, h, mode[1], mode[2])
            _assert_same(img, ref, st, ost, f"{label}/{mode[0]}")
