"""RG_OPT_LIGHT_GRIDS: shadow rays of a scene's first lights scan one list of a per-light grid instead of walking the
3-D grid (rg_light_grid.h, DESIGN.md section 4.2).  With the option on and off every scene must render the same
RGBA8 bytes and f32 bits, with the same per-type ray counts and error counters; the verbatim re-trace of every queued
ray (RG_OPT_VERIFY_CULL=2) must find no difference; and the light grids must spare exact tests."""
import numpy as np
import pytest

import raingun_b200 as rg
from raingun_b200.examples import bundled_texture_loader, example_scene
from raingun_b200.scene import scene_from_dict
from raingun_b200.synth import make_box_scene, make_light_scene, make_scene

pytestmark = pytest.mark.gpu

W, H = 320, 180


def _counters(st):
    return (st.rays_primary, st.rays_shadow, st.rays_reflection, st.rays_transmission,
            st.err_nan_distance, st.err_transmission_none, st.err_aabb_normal)


def _render(data, w, h, light_grids, verify=0, y0=0, y1=None):
    y1 = h if y1 is None else y1
    with rg.Scene(data) as sc:
        sc.set_pipeline(rg.PIPELINE_WAVEFRONT)
        sc.set_accel(rg.ACCEL_GRID)
        sc.set_option(rg._native.OPT_LIGHT_GRIDS, light_grids)
        if verify:
            sc.set_option(rg._native.OPT_VERIFY_CULL, verify)
        img = sc.render_rows(w, h, y0, y1)
        st = sc.last_stats
        f32 = sc.render_rows_f32(w, h, y0, y1) if not verify else None
    return img, f32, st


def _assert_on_off_equal(data, label, w=W, h=H):
    on = _render(data, w, h, 1)
    off = _render(data, w, h, 0)
    assert on[0].tobytes() == off[0].tobytes(), f"{label}: RGBA8 differs"
    assert on[1].tobytes() == off[1].tobytes(), f"{label}: f32 differs"
    assert _counters(on[2]) == _counters(off[2]), (label, _counters(on[2]), _counters(off[2]))
    return on[2], off[2]


def _scenes():
    out = [(n, lambda n=n: example_scene(n)) for n in ("test1", "test2", "test3")]
    out += [(f"{n}-small", lambda n=n: make_scene(n, spheres=s, depth=5, texture_loader=bundled_texture_loader)[0])
            for n, s in (("C3", 600), ("C4", 2000), ("C5", 3000))]
    out += [("B4-small", lambda: make_box_scene("B4", bodies=1500, depth=5, texture_loader=bundled_texture_loader)[0])]
    out += [(f"L{n}", lambda n=n: make_light_scene(n, spheres=300, depth=5)[0]) for n in (33, 64)]
    return out


@pytest.mark.parametrize("case", _scenes(), ids=lambda c: c[0])
def test_light_grids_on_and_off_render_the_same(case):
    name, make = case
    _assert_on_off_equal(make(), name)


def _adversarial():
    from test_gpu_parity import _adversarial_scenes

    return _adversarial_scenes()


@pytest.mark.parametrize("case", _adversarial(), ids=lambda c: c[0])
def test_light_grids_on_adversarial_scenes(case):
    name, doc = case
    _assert_on_off_equal(scene_from_dict(doc, bundled_texture_loader), name, 224, 126)


def test_full_c4_and_c5_band_verbatim_retrace_and_shorter_shadow_scans():
    """A full C4 frame and a band of C5 rows re-traced ray by ray with the verbatim FP64 scan: no difference.  With the
    light grids on, the any-hit launches fetch and cull far fewer records (RG_OPT_TRACE_STATS=2 counts those launches
    only).  (Exact tests per frame are not always fewer: measured on C4, 177.8 M with the light grids and 177.3 M
    without; on C5, 1,313 M and 1,336 M.)"""
    for name, y0, y1 in (("C4", None, None), ("C5", 2000, 2064)):
        data, spec = make_scene(name, texture_loader=bundled_texture_loader)
        w, h = spec.width, spec.height
        got = {}
        for lg in (1, 0):
            img, _, st = _render(data, w, h, lg, verify=2, y0=y0 or 0, y1=y1)
            assert st.cull_unsound == 0, (name, lg)
            got[lg] = (img, st)
        assert got[1][0].tobytes() == got[0][0].tobytes(), name
        assert _counters(got[1][1]) == _counters(got[0][1]), name
        scans = {}
        for lg in (1, 0):
            with rg.Scene(data) as sc:
                sc.set_accel(rg.ACCEL_GRID)
                sc.set_option(rg._native.OPT_LIGHT_GRIDS, lg)
                sc.set_option(rg._native.OPT_TRACE_STATS, 2)
                sc.render_rows(w, h, y0 or 0, y1 or h)
                scans[lg] = (sc.last_stats.grid_fetches, sc.last_stats.grid_culls)
        assert scans[1][0] < 0.5 * scans[0][0] and scans[1][1] < 0.5 * scans[0][1], (name, scans)
