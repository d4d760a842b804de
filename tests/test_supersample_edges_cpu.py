"""RG_OPT_SUPERSAMPLE_EDGES without a device: the key in every mirror, the mask the GPU tests expect, and the oracle's
per-pixel ray counts they build counters from."""
import importlib.util
import os
import re

import numpy as np
import pytest

from raingun_b200 import _native
from raingun_b200.examples import example_scene
from raingun_b200.synth import make_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_spec = importlib.util.spec_from_file_location("edge_oracle", os.path.join(ROOT, "tests", "edge_oracle.py"))
eo = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(eo)


def test_key_is_16_everywhere():
    with open(os.path.join(ROOT, "include", "raingun_b200.h"), encoding="utf-8") as f:
        assert re.search(r"\bRG_OPT_SUPERSAMPLE_EDGES\s*=\s*16\b", f.read())
    with open(os.path.join(ROOT, "integration", "raingun-b200-sys", "src", "lib.rs"), encoding="utf-8") as f:
        assert "pub const RG_OPT_SUPERSAMPLE_EDGES: i32 = 16;" in f.read()
    assert _native.OPT_SUPERSAMPLE_EDGES == 16


def _frame(h, w, fill=100):
    img = np.full((h, w, 4), fill, np.uint8)
    img[..., 3] = 255
    return img


def test_flat_frame_refines_nothing():
    assert not eo.mask(_frame(5, 7), 0).any()


@pytest.mark.parametrize("y,x", [(0, 0), (0, 6), (4, 0), (4, 6), (2, 3), (0, 3), (2, 0)])
def test_one_pixel_refines_its_in_image_neighbourhood(y, x):
    img = _frame(5, 7)
    img[y, x, 1] = 130
    m = eo.mask(img, 10)
    want = np.zeros((5, 7), bool)
    want[max(0, y - 1):y + 2, max(0, x - 1):x + 2] = True
    assert np.array_equal(m, want)


def test_diagonal_neighbours_count():
    img = _frame(3, 3)
    img[0, 0, 0] = 200
    m = eo.mask(img, 50)
    assert m[1, 1] and m[0, 0] and m[0, 1] and m[1, 0]
    assert not m[2, 2] and not m[0, 2] and not m[2, 0]


def test_threshold_is_strict():
    img = _frame(3, 4)
    img[1, 1, 2] = 100 + 16
    assert not eo.mask(img, 16).any()     # a difference of exactly T does not refine
    assert eo.mask(img, 15)[1, 1]
    img[1, 1, 2] = 100 - 17               # nor does the sign matter
    assert eo.mask(img, 16)[1, 1]


def test_alpha_is_ignored_and_255_refines_nothing():
    img = _frame(4, 4)
    img[2, 2, 3] = 0
    assert not eo.mask(img, 0).any()
    rng = np.random.default_rng(7)
    noise = rng.integers(0, 256, (6, 9, 4), dtype=np.uint8)
    assert not eo.mask(noise, 255).any()
    assert eo.mask(noise, 0).mean() > 0.9


def test_oracle_counts_sum_to_frame_totals(oracle):
    for scene, w, h in ((example_scene("test2"), 64, 48), (make_scene("C4", spheres=60, depth=5)[0], 48, 27)):
        img, st, f32 = oracle.render(scene, w, h, want_f32=True)
        rgba, got32, counts = eo.render_counts(scene, w, h)
        assert np.array_equal(rgba, img)
        assert np.array_equal(got32.view(np.uint32), f32.view(np.uint32))
        assert tuple(int(v) for v in counts.sum(axis=(0, 1))) == eo.counters(st)
        assert (counts[..., 0] == 1).all()
        # a band: the same pixels and counts as the full frame's rows
        band, _, bc = eo.render_counts(scene, w, h, 5, 11)
        assert np.array_equal(band, img[5:11]) and np.array_equal(bc, counts[5:11])
