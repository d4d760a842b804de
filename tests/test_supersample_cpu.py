"""RG_OPT_SUPERSAMPLE without a device: the key is the same in the C header, the Python binding and the Rust
bindings, and the test reduction of tests/test_gpu_supersample.py sums in the header's order."""
import importlib.util
import os
import re

import numpy as np

import raingun_b200 as rg
from raingun_b200 import _native

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def test_option_key_agrees_everywhere():
    header = open(os.path.join(ROOT, "include", "raingun_b200.h")).read()
    rust = open(os.path.join(ROOT, "integration", "raingun-b200-sys", "src", "lib.rs")).read()
    assert re.search(r"\bRG_OPT_SUPERSAMPLE\s*=\s*14\b", header)
    assert re.search(r"\bRG_OPT_SUPERSAMPLE:\s*i32\s*=\s*14;", rust)
    assert _native.OPT_SUPERSAMPLE == 14
    assert callable(rg.Scene.set_supersample)


def test_reduction_order():
    """Float addition is not associative: the reference sums sub-rows, then sub-columns, from 0, then divides."""
    spec = importlib.util.spec_from_file_location("supersample_gpu_tests", os.path.join(HERE, "test_gpu_supersample.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    reduce = mod.reduce
    rng = np.random.default_rng(7)
    for n in (1, 2, 3):
        samples = rng.random((2 * n, 3 * n, 3), dtype=np.float32) * np.float32(1.7)
        got = reduce(samples, n)
        assert got.dtype == np.float32 and got.shape == (2, 3, 3)
        for y in range(2):
            for x in range(3):
                for c in range(3):
                    s = np.float32(0.0)
                    for j in range(n):
                        for i in range(n):
                            s = np.float32(s + samples[n * y + j, n * x + i, c])
                    assert got[y, x, c].view(np.uint32) == np.float32(s / np.float32(n * n)).view(np.uint32)
        if n == 1:
            assert np.array_equal(got.view(np.uint32), samples.view(np.uint32))
