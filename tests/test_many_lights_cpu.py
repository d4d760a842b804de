"""Scenes with any number of lights (the reference's Scene::lights is a Vec of any length, rendering.rs:132-172).
CPU-only: the C ABI accepts them and stops at the device check, and the YAML loaders and the oracle take them."""
import ctypes

import numpy as np
import pytest

from raingun_b200 import _native, host
from raingun_b200 import scene as pyscene
from raingun_b200.examples import bundled_texture_loader
from raingun_b200.synth import make_light_scene, make_light_scene_doc, to_yaml

FIELDS = ("body_kind", "body_geom", "coloration_kind", "color", "texture_id", "texture_offset", "albedo",
          "surface_kind", "surface_param", "light_kind", "light_vec", "light_color", "light_intensity")


@pytest.mark.parametrize("lights", [33, 100, 10000])
def test_scene_create_accepts_any_light_count(lights):
    """Validation no longer refuses more than RG_MAX_LIGHTS lights.  Without a device the call gets as far as the
    device check (validation runs first: test_validation_without_device) and fails there with RG_E_CUDA."""
    lib = _native.lib()
    data, _ = make_light_scene(lights, spheres=20)
    assert data.n_lights == lights
    desc, keep = data.to_desc()
    out = ctypes.c_void_p()
    rc = lib.rg_scene_create(ctypes.byref(desc), 0, ctypes.byref(out))
    assert rc != _native.E_LIGHTS
    if lib.rg_device_count() > 0:
        assert rc == 0
        lib.rg_scene_destroy(out)
    else:
        assert rc == _native.E_CUDA
        assert b"no CPU path" in lib.rg_last_error()


def test_every_light_is_still_validated():
    """The per-light checks stay: a bad kind past the 32nd light is refused before the device is looked at."""
    lib = _native.lib()
    data, _ = make_light_scene(100, spheres=20)
    data.light_kind = data.light_kind.copy()
    data.light_kind[77] = 9
    desc, keep = data.to_desc()
    out = ctypes.c_void_p()
    assert lib.rg_scene_create(ctypes.byref(desc), 0, ctypes.byref(out)) == _native.E_INVALID
    assert b"lights[77]" in lib.rg_last_error()


def test_light_scene_generator_is_seeded_and_has_the_special_lights():
    a, b = make_light_scene_doc(40, spheres=30), make_light_scene_doc(40, spheres=30)
    assert a == b
    lights = a["lights"]
    assert len(lights) == 40
    assert all(("Directional" if i % 2 == 0 else "Spherical") in l for i, l in enumerate(lights))
    first_sphere = next(x["Sphere"] for x in a["bodies"] if "Sphere" in x)
    assert lights[1]["Spherical"]["position"] == first_sphere["center"]      # inside a body
    assert lights[3]["Spherical"]["position"][2] > 0.0                       # behind the camera (it looks along -z)
    assert lights[2]["Directional"]["intensity"] == 0.0
    assert len({l[next(iter(l))]["color"] for l in lights}) == 40            # distinct colours
    # the bodies do not depend on the light count
    assert make_light_scene_doc(3, spheres=30)["bodies"] == a["bodies"]


def test_hundred_light_yaml_loads_identically_and_the_oracle_renders_it():
    from oracle import oracle

    text = to_yaml(make_light_scene_doc(100, spheres=40, depth=4))
    native = host.parse_scene(text, bundled_texture_loader)
    py = pyscene.parse_scene(text, bundled_texture_loader)
    assert native.n_lights == py.n_lights == 100
    assert native.fov == py.fov and native.max_recursion_depth == py.max_recursion_depth
    for f in FIELDS:
        x, y = getattr(native, f), getattr(py, f)
        assert x.dtype == y.dtype and x.shape == y.shape, f
        assert x.tobytes() == y.tobytes(), f
    img, st, _ = oracle().render(py, 64, 36)
    assert img.shape == (36, 64, 4)
    lit = st.rays_shadow // 100
    assert st.rays_shadow == lit * 100 and lit > 0   # one shadow ray per (lit hit, light)
    assert len(np.unique(img.reshape(-1, 4), axis=0)) > 16
