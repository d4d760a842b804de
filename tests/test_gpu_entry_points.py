"""The render entry points share one path per concern: the output kind (RGBA8 rows, RGBA8 rows scattered into a
full frame, unquantised f32 RGB) is an argument of the render, not state of the handle; the host-buffer and
streaming entry points go through one rows-to-host function and one band loop; every merge of per-part stats sums
the same counters.  These tests pin what no other test does: the kinds interleaved on one handle with CUDA graphs,
the stats of the streaming renders, and the trace stats of a multi-device scene."""
import numpy as np
import pytest

import raingun_b200 as rg
from raingun_b200.synth import make_scene

pytestmark = pytest.mark.gpu

W, H = 256, 144


@pytest.fixture(scope="module")
def grid_scene(oracle):
    data, _ = make_scene("C4", spheres=400, depth=8)
    ref, ost, ref32 = oracle.render(data, W, H, want_f32=True)
    return data, ref, ost, ref32


def _counters(st):
    return (st.rays_primary, st.rays_shadow, st.rays_reflection, st.rays_transmission,
            st.err_nan_distance, st.err_transmission_none, st.err_aabb_normal)


def test_output_kinds_interleaved_on_one_handle_replay_their_own_graphs(grid_scene):
    """Every output kind, three rounds, interleaved on one wavefront grid handle: each result must be the oracle's.
    The f32 and RGBA frames share the staging buffer and the scatter and compact row lists share the output
    tensor and the row list, so a graph key that missed the output kind would replay the wrong last kernel.  The
    first f32 call grows the staging buffer, which changes the RGBA key once; from the third round on every call
    is a graph replay."""
    import torch

    data, ref, _, ref32 = grid_scene
    rows = np.array([H - 1, 0, 5, 6, 7, 40, 99], np.uint32)
    out = torch.zeros(H * W * 4, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    with rg.Scene(data) as sc:
        sc.set_pipeline(rg.PIPELINE_WAVEFRONT)
        sc.set_accel(rg.ACCEL_GRID)
        for it in range(3):
            replays = {}
            img = sc.render_image(W, H)
            replays["image"] = sc.last_stats.graph_replays
            assert np.array_equal(img, ref), it
            f32 = sc.render_rows_f32(W, H)
            replays["f32"] = sc.last_stats.graph_replays
            assert np.array_equal(f32.view(np.uint32), ref32.view(np.uint32)), it
            out.zero_()
            sc.render_rowlist_scatter(W, H, rows, out.data_ptr(), stream)
            replays["scatter"] = sc.last_stats.graph_replays
            assert np.array_equal(out.cpu().numpy().reshape(H, W, 4)[rows], ref[rows]), it
            sc.render_rowlist_device(W, H, rows, out.data_ptr(), stream)
            replays["device"] = sc.last_stats.graph_replays
            assert np.array_equal(out[:rows.size * W * 4].cpu().numpy().reshape(rows.size, W, 4), ref[rows]), it
            if it == 2:
                assert replays == {"image": 1, "f32": 1, "scatter": 1, "device": 1}, replays


def test_streaming_stats_equal_one_call(grid_scene):
    """A streamed frame reports the ray and error counters of one call over the whole frame, and its wall time."""
    data, ref, ost, ref32 = grid_scene
    with rg.Scene(data) as sc:
        sc.render_rows(W, H, 0, H)
        one = sc.last_stats
        got = np.zeros_like(ref)
        assert sc.streaming_render(W, H, lambda y0, rows: got.__setitem__(slice(y0, y0 + rows.shape[0]), rows) or True,
                                   band_rows=37) is True
        assert np.array_equal(got, ref)
        assert _counters(sc.last_stats) == _counters(one) == _counters(ost)
        assert sc.last_stats.ms_wall > 0

        sc.render_rows_f32(W, H)
        one = sc.last_stats
        got32 = np.zeros_like(ref32)
        assert sc.streaming_render_f32(W, H, lambda y0, rows: got32.__setitem__(slice(y0, y0 + rows.shape[0]), rows) or True,
                                       band_rows=37) is True
        assert np.array_equal(got32.view(np.uint32), ref32.view(np.uint32))
        assert _counters(sc.last_stats) == _counters(one) == _counters(ost)
        assert sc.last_stats.ms_wall > 0


def test_multi_device_trace_stats_sum_the_devices(grid_scene):
    """RG_OPT_TRACE_STATS on a scene that spans two lanes: the grid counters are the sums over the lanes.  Each ray
    visits the same cells wherever it is traced, so the cells visited equal those of the single-device frame."""
    data, ref, _, _ = grid_scene
    with rg.Scene(data) as sc:
        sc.set_accel(rg.ACCEL_GRID)
        sc.set_option(rg._native.OPT_TRACE_STATS, 1)
        assert np.array_equal(sc.render_image(W, H), ref)
        single = sc.last_stats
    assert single.grid_cells > 0
    with rg.Scene(data, devices=[0, 0]) as sc:
        sc.set_accel(rg.ACCEL_GRID)
        sc.set_option(rg._native.OPT_TRACE_STATS, 1)
        assert np.array_equal(sc.render_image(W, H), ref)
        st = sc.last_stats
    assert st.devices_used == 2
    assert st.grid_cells == single.grid_cells
    assert st.grid_lane_slots > 0


def test_f32_entry_points_refuse_a_multi_device_scene(grid_scene):
    data = grid_scene[0]
    with rg.Scene(data, devices=[0, 0]) as sc:
        with pytest.raises(rg.RaingunError) as e:
            sc.render_rows_f32(W, H)
        assert e.value.code == rg._native.E_INVALID
        with pytest.raises(rg.RaingunError) as e:
            sc.streaming_render_f32(W, H, lambda y0, rows: True)
        assert e.value.code == rg._native.E_INVALID
