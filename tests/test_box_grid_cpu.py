"""Boxes and disks in the grid, the CPU side: the reference behaviour the grid has to preserve (the box test's
hit outside the box when 1.0 / d_k is infinite and the origin lies on a face plane) and the B4 scene."""
import numpy as np

from raingun_b200 import host
from raingun_b200 import scene as pyscene
from raingun_b200.examples import bundled_texture_loader
from raingun_b200.synth import B4, make_box_scene, make_box_scene_doc, to_yaml

SKY = np.array([0x66, 0x7F, 0xFF, 0xFF], np.uint8)


def assert_same_scene(a, b):
    assert (a.fov, a.max_recursion_depth, a.n_bodies) == (b.fov, b.max_recursion_depth, b.n_bodies)
    for f in ("body_kind", "body_geom", "coloration_kind", "color", "texture_id", "texture_offset", "albedo",
              "surface_kind", "surface_param", "light_kind", "light_vec", "light_color", "light_intensity"):
        x, y = getattr(a, f), getattr(b, f)
        assert x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes(), f


def test_box_test_hits_outside_the_box_for_an_origin_on_a_face(oracle):
    """d.x = +0 (1.0 / d.x = inf) and o.x on the box's lo_x face: (lo_x - o.x) * inf = NaN drops an overlap check,
    and the reference reports a hit whose point lies far outside the unit box."""
    g = np.array([0, 0, 0, 1, 1, 1, 0, 0], float)
    o = np.array([1.0, -1.6852268020417216, -0.25255756791192274])
    d = np.array([0.0, -0.617810741873622, 0.7863268323194655])
    t = oracle.intersect(3, g, o, d)
    assert t is not None
    p = o + t * d
    assert p[1] < -1.8, p                     # y = -1.88: nearly two units below the box
    # the same ray moved off the face plane misses
    assert oracle.intersect(3, g, o + np.array([1e-9, 0, 0]), d) is None


def _face_doc(box):
    mat = {"coloration": {"Color": "#ffffff"}, "albedo": 0.5, "surface": "Diffuse"}
    bodies = [{"Plane": {"origin": [0.0, -2.0, -5.0], "normal": [0.0, -1.0, 0.0], "material": mat}}]
    if box:
        bodies.append({"AABB": {"bounds": [[0.0, 3.0, -40.0], [1.0, 4.0, -39.0]], "material": mat}})
    return {"fov": 90.0, "defaultColor": "#667fff", "maxRecursionDepth": 3,
            "lights": [{"Directional": {"direction": {"x": 0.0, "y": -1.0, "z": 0.0}, "color": "#ffffff",
                                        "intensity": 5.0}}],
            "bodies": bodies}


def test_box_on_the_face_plane_darkens_one_ground_column(oracle):
    """225 x 126 (odd width: the centre column's primary rays have d.x = +0 and hit the ground at x = 0), a sun
    straight overhead (shadow rays with d.x = -0) and a box whose lo_x face is the plane x = 0, 30 units away:
    the reference blacks out 60 ground pixels of column 112 through the NaN case of its box test.  No other
    ground pixel changes; the rest of the difference is the box itself, seen against the sky."""
    a, _, _ = oracle.render(pyscene.scene_from_dict(_face_doc(False)), 225, 126)
    b, _, _ = oracle.render(pyscene.scene_from_dict(_face_doc(True)), 225, 126)
    diff = (a != b).any(axis=2)
    sky = (a == SKY).all(axis=2)
    ys, xs = np.nonzero(diff & ~sky)
    assert len(ys) == 60 and set(xs.tolist()) == {112}
    assert (b[ys, xs, :3] == 0).all()
    ys, xs = np.nonzero(diff & sky)
    assert 0 < len(ys) < 12 and set(xs.tolist()) <= {112, 113} and ys.max() < 63


def test_b4_generator_is_deterministic_and_matches_its_definition():
    d1, spec = make_box_scene(bodies=400)
    d2, _ = make_box_scene(bodies=400)
    assert_same_scene(d1, d2)
    assert spec is B4 and (spec.width, spec.height, spec.seed, spec.depth) == (3840, 2160, 1004, 8)
    kinds = np.bincount(d1.body_kind, minlength=4)
    assert kinds[0] == 0 and kinds[1] == 1 and kinds[2] + kinds[3] == 400
    assert 0.6 < kinds[3] / 400 < 0.8                           # selector < 0.7: AABB
    boxes = d1.body_geom[d1.body_kind == 3]
    half = (boxes[:, 3:6] - boxes[:, 0:3]) / 2
    assert (half > 0.06 - 1e-6).all() and (half < 0.3 + 1e-6).all()
    centre = (boxes[:, 3:6] + boxes[:, 0:3]) / 2
    assert (np.abs(centre[:, 0]) <= 24.0 + 1e-6).all() and (centre[:, 2] < -4.0 + 1e-6).all()
    disks = d1.body_geom[d1.body_kind == 2]
    assert (disks[:, 6] >= 0.08).all() and (disks[:, 6] <= 0.35).all()
    # a shorter scene is a prefix of the same stream
    d3, _ = make_box_scene(bodies=100)
    assert np.array_equal(d3.body_geom, d1.body_geom[:101])
    assert len(make_box_scene_doc()["bodies"]) == 10001


def test_native_loader_equals_python_loader_on_b4_yaml():
    data, _ = make_box_scene(bodies=500, texture_loader=bundled_texture_loader)
    text = to_yaml(make_box_scene_doc(500))
    native = host.parse_scene(text, bundled_texture_loader)
    assert_same_scene(native, data)
    assert native.n_bodies == 501
