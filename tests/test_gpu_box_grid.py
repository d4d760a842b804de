"""Boxes and disks in the grid (RG_ACCEL_GRID / AUTO bin them through enclosing spheres): every frame byte-equal
to the CPU oracle, with the same ray counts and panic counters, for every pipeline."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import raingun_b200 as rg
from raingun_b200.scene import scene_from_dict
from raingun_b200.synth import make_box_scene

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODES = [
    ("mega", rg.PIPELINE_MEGAKERNEL, rg.ACCEL_BRUTE),
    ("wavefront-brute", rg.PIPELINE_WAVEFRONT, rg.ACCEL_BRUTE),
    ("wavefront-grid", rg.PIPELINE_WAVEFRONT, rg.ACCEL_GRID),
]


def _render(data, w, h, pipeline, accel, verify=0):
    with rg.Scene(data) as sc:
        sc.set_pipeline(pipeline)
        sc.set_accel(accel)
        if verify:
            sc.set_option(rg._native.OPT_VERIFY_CULL, verify)
        img = sc.render_image(w, h)
        return img, sc.last_stats


def _assert_same(img, ref, st, ost, label):
    diff = np.abs(img.astype(np.int32) - ref.astype(np.int32)).max(axis=2)
    assert int((diff > 0).sum()) == 0, f"{label}: {(diff > 0).sum()} pixels differ (max {diff.max()})"
    assert (st.rays_primary, st.rays_shadow, st.rays_reflection, st.rays_transmission) == (
        ost.rays_primary, ost.rays_shadow, ost.rays_reflection, ost.rays_transmission), label
    assert (st.err_nan_distance, st.err_transmission_none, st.err_aabb_normal) == (
        ost.err_nan_distance, ost.err_transmission_none, ost.err_aabb_normal), label


def _check_all_modes(oracle, data, w, h, label):
    ref, ost, _ = oracle.render(data, w, h)
    stats = {}
    for name, pipeline, accel in MODES:
        img, st = _render(data, w, h, pipeline, accel)
        _assert_same(img, ref, st, ost, f"{label}/{name}")
        stats[name] = st
    assert stats["wavefront-grid"].accel_used == rg.ACCEL_GRID, label
    img, st = _render(data, w, h, rg.PIPELINE_WAVEFRONT, rg.ACCEL_GRID, verify=2)   # every queued ray re-traced verbatim
    _assert_same(img, ref, st, ost, f"{label}/grid+verify")
    assert st.cull_unsound == 0, label
    return ref, stats


def test_b4_small_grid_matches_oracle_with_a_fraction_of_the_exact_tests(oracle):
    data, _ = make_box_scene(bodies=800, depth=8)
    _, stats = _check_all_modes(oracle, data, 256, 144, "B4-800")
    grid, brute = stats["wavefront-grid"].exact_tests, stats["wavefront-brute"].exact_tests
    assert grid < 0.05 * brute, (grid, brute)
    img, st = _render(data, 256, 144, rg.PIPELINE_AUTO, rg.ACCEL_AUTO)   # the default picks the grid for 800 boxes / disks
    assert st.accel_used == rg.ACCEL_GRID


_MAT = {"coloration": {"Color": "#d0c0b0"}, "albedo": 0.6, "surface": "Diffuse"}


def _doc(bodies, lights, depth=4):
    return {"fov": 90.0, "defaultColor": "#667fff", "maxRecursionDepth": depth, "lights": lights, "bodies": bodies}


def _sun(x, y, z, intensity=5.0):
    return {"Directional": {"direction": {"x": x, "y": y, "z": z}, "color": "#ffffff", "intensity": intensity}}


def _box(lo, hi, mat=None):
    return {"AABB": {"bounds": [list(map(float, lo)), list(map(float, hi))], "material": mat or _MAT}}


def _ground(y=-2.0):
    return {"Plane": {"origin": [0.0, y, -5.0], "normal": [0.0, -1.0, 0.0], "material": _MAT}}


def _filler():   # enough binnable bodies, away from the frame's centre column, for the grid to be built
    return [_box((3 + 2 * i, 6, -30), (4 + 2 * i, 7, -29)) for i in range(10)]


FACE_CASES = {
    # the centre column of an odd-width frame (primary d.x = +0, ground hits at x = 0) and a box face on x = 0
    "lo-face/sun-0": ([_box((0, 3, -40), (1, 4, -39))], [_sun(0.0, -1.0, 0.0)]),      # shadow d.x = -0
    "hi-face/sun-0": ([_box((-1, 3, -40), (0, 4, -39))], [_sun(0.0, -1.0, 0.0)]),
    "lo-face/sun+0": ([_box((0, 3, -40), (1, 4, -39))], [_sun(-0.0, -1.0, 0.0)]),     # shadow d.x = +0
    "lo-face/sun-subnormal": ([_box((0, 3, -40), (1, 4, -39))], [_sun(-5e-324, -1.0, 0.0)]),   # 1.0 / d.x = inf
    "hi-face/sun+subnormal": ([_box((-1, 3, -40), (0, 4, -39))], [_sun(4e-320, -1.0, 0.0)]),
}


@pytest.mark.parametrize("case", sorted(FACE_CASES))
def test_origin_on_a_face_plane_matches_oracle(oracle, case):
    boxes, lights = FACE_CASES[case]
    data = scene_from_dict(_doc([_ground()] + boxes + _filler(), lights))
    _check_all_modes(oracle, data, 225, 126, case)


def _lattice(x0, z0, step, size):
    out = []
    for i in range(6):
        for j in range(6):
            lo = (x0 + step * i, -2, z0 - step * j)
            out.append(_box(lo, (lo[0] + size, -2 + size + (size // 2) * ((i + j) % 3), lo[2] + size)))
    return out


@pytest.mark.parametrize("shift", ["near", "thousands"])
def test_integer_lattice_under_an_axis_parallel_sun_matches_oracle(oracle, shift):
    """Boxes on integer coordinates standing on the ground, under suns along -y and -x: secondary rays start
    on face planes with zero direction components.  Shifted to coordinates of 1024 and more, hp + n * 1e-13
    rounds back onto the face (half an ulp there is 1.14e-13)."""
    boxes = _lattice(-6, -8, 3, 2) if shift == "near" else _lattice(1024, -1024, 96, 64)
    refl = {"coloration": {"Color": "#ffffff"}, "albedo": 0.5, "surface": {"Reflecting": {"reflectivity": 0.5}}}
    for k in range(0, len(boxes), 5):
        boxes[k]["AABB"]["material"] = refl
    data = scene_from_dict(_doc([_ground()] + boxes, [_sun(0.0, -1.0, 0.0), _sun(-1.0, 0.0, 0.0, 2.0)], depth=5))
    _check_all_modes(oracle, data, 225, 127, f"lattice-{shift}")


def _mixed_doc(seed):
    rng = np.random.default_rng(seed)

    def mat():
        kind = rng.choice(["Diffuse", "Reflecting", "Refractive"])
        surface = "Diffuse"
        if kind == "Reflecting":
            surface = {"Reflecting": {"reflectivity": float(np.round(rng.uniform(0.2, 0.9), 3))}}
        elif kind == "Refractive":
            surface = {"Refractive": {"index": float(np.round(rng.uniform(1.1, 1.8), 3)),
                                      "transparency": float(np.round(rng.uniform(0.5, 1.0), 3))}}
        return {"coloration": {"Color": "#%06x" % int(rng.integers(0, 1 << 24))},
                "albedo": float(np.round(rng.uniform(0.2, 0.9), 3)), "surface": surface}

    def r3(a, b):
        return [float(v) for v in np.round(rng.uniform(a, b, 3), 3)]

    bodies = [_ground()]
    for _ in range(40):
        bodies.append({"Sphere": {"center": [*r3(-6, 6)[:2], float(np.round(rng.uniform(-20, -5), 3))],
                                  "radius": float(np.round(rng.uniform(0.2, 0.8), 3)), "material": mat()}})
    for _ in range(40):
        c = r3(-6, 6)
        c[2] = float(np.round(rng.uniform(-20, -5), 3))
        h = r3(0.1, 0.7)
        bodies.append(_box([c[k] - h[k] for k in range(3)], [c[k] + h[k] for k in range(3)], mat()))
    for _ in range(30):
        n = r3(-3, 3)                                  # non-unit normals
        c = r3(-6, 6)
        c[2] = float(np.round(rng.uniform(-20, -5), 3))
        bodies.append({"Disk": {"origin": c, "normal": n, "radius": float(np.round(rng.uniform(0.2, 1.0), 3)),
                                "material": mat()}})
    bodies += [
        _box((1, 0, -12), (2, 1, -11), mat()), _box((2, 0, -12), (3, 1, -11), mat()),       # touching
        _box((2.5, 0.5, -11.5), (3.5, 1.5, -10.5), mat()),                                   # overlapping
        _box((-3, 0, -9), (-3, 1, -8), mat()), _box((-4, 2, -9), (-3, 2, -8), mat()),       # zero thickness
        _box((4, 1, -9), (3, 0, -10), mat()), _box((-2, 3, -7), (-3, 2, -6), mat()),        # inverted
        {"Disk": {"origin": [0.0, 1.0, -10.0], "normal": [0.0, 0.0, 0.0], "radius": 1.0, "material": mat()}},
        {"Disk": {"origin": [0.5, 1.5, -9.0], "normal": [0.0, 0.0, -1.0], "radius": 0.0, "material": mat()}},
        _box((-60, -2.5, -80), (60, -1.9, -3), mat()),                                       # too large for the grid
    ]
    glass = {"coloration": {"Color": "#ffffff"}, "albedo": 0.5,
             "surface": {"Refractive": {"index": 1.33, "transparency": 0.9}}}
    bodies += [_box((-1, -1, -1), (1, 1, 1), glass), _box((-2.5, -1.5, -3), (2.5, 2.5, 2), glass)]   # around the camera
    lights = [_sun(0.3, -1.0, -0.6), {"Spherical": {"position": [4.0, 8.0, -6.0], "color": "#ffeedd",
                                                    "intensity": 3000.0}}]
    return _doc(bodies, lights, depth=6)


@pytest.mark.parametrize("seed", [1, 2])
def test_mixed_spheres_boxes_disks_match_oracle(oracle, seed):
    data = scene_from_dict(_mixed_doc(seed))
    _check_all_modes(oracle, data, 240, 135, f"mixed-{seed}")


_HOST_BUILD = r"""
import json, sys
sys.path.insert(0, sys.argv[1])
import raingun_b200 as rg
from raingun_b200.synth import make_box_scene
data, _ = make_box_scene(bodies=800, depth=8)
with rg.Scene(data) as sc:
    sc.set_accel(rg.ACCEL_GRID)
    img = sc.render_image(256, 144)
    st = sc.last_stats
open(sys.argv[2], "wb").write(img.tobytes())
print(json.dumps({"exact_tests": st.exact_tests, "accel": st.accel_used}))
"""


def test_host_built_grid_equals_device_built_grid(tmp_path):
    data, _ = make_box_scene(bodies=800, depth=8)
    img, st = _render(data, 256, 144, rg.PIPELINE_AUTO, rg.ACCEL_GRID)
    out = tmp_path / "host.rgba"
    env = dict(os.environ, RG_GRID_BUILD="host")
    r = subprocess.run([sys.executable, "-c", _HOST_BUILD, ROOT, str(out)], env=env, capture_output=True, text=True,
                       check=True)
    got = json.loads(r.stdout.strip().splitlines()[-1])
    assert got["accel"] == rg.ACCEL_GRID and st.accel_used == rg.ACCEL_GRID
    assert got["exact_tests"] == st.exact_tests
    assert out.read_bytes() == img.tobytes()


def test_device_lanes_equal_the_single_device_frame():
    data, _ = make_box_scene(bodies=800, depth=6)
    ref, st = _render(data, 256, 147, rg.PIPELINE_AUTO, rg.ACCEL_AUTO)
    assert st.accel_used == rg.ACCEL_GRID
    with rg.Scene(data, devices=[0, 0, 0]) as sc:
        for schedule in (1, 2):
            sc.set_option(rg._native.OPT_SCHEDULE, schedule)
            img = sc.render_image(256, 147)
            assert np.array_equal(img, ref), schedule
            assert sc.last_stats.rays == st.rays
    with rg.Scene(data, device=rg.DEVICE_ALL) as sc:
        assert np.array_equal(sc.render_image(256, 147), ref)
