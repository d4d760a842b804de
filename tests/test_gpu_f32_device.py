"""Unquantised f32 frames delivered to device memory and to row-list destinations: rg_render_rows_f32_device,
rg_render_rowlist_f32_device, rg_render_rowlist_f32_scatter and rg_render_rowlist_f32_host.  Each is the f32 twin of
an RGBA8 entry point: it must accept and refuse what its twin does, report its twin's counters, and deliver the bits
rg_render_rows_f32 (and the oracle) delivers for the same pixels.  f32 results are compared as uint32 views, so NaN
and -0 are compared by their bits; every frame a row list writes into is pre-filled with 0xFF bytes, and every word
outside the listed rows must still be 0xFFFFFFFF afterwards (no stray stores)."""
import ctypes

import numpy as np
import pytest

import raingun_b200 as rg
from raingun_b200 import _native
from raingun_b200.dist import rows_of_tiles
from raingun_b200.examples import example_scene
from raingun_b200.synth import make_scene

pytestmark = pytest.mark.gpu

# test1 at its own size (RG_PIPELINE_AUTO takes the megakernel for it), and a 400-sphere C4 scene on the wavefront
CASES = {"test1-auto": ("test1", 800, 600, rg.PIPELINE_AUTO, rg.ACCEL_AUTO),
         "c4-grid": ("C4", 256, 144, rg.PIPELINE_WAVEFRONT, rg.ACCEL_GRID),
         "c4-brute": ("C4", 256, 144, rg.PIPELINE_WAVEFRONT, rg.ACCEL_BRUTE)}
SENTINEL = 0xFFFFFFFF

_data, _refs = {}, {}


def scene_data(name):
    if name not in _data:
        _data[name] = example_scene("test1") if name == "test1" else make_scene("C4", spheres=400, depth=8)[0]
    return _data[name]


def reference(oracle, name, w, h):
    """(RGBA8, oracle stats, f32) of the whole frame."""
    if (name, w, h) not in _refs:
        _refs[(name, w, h)] = oracle.render(scene_data(name), w, h, want_f32=True)
    return _refs[(name, w, h)]


def open_scene(case, n=None):
    name, _, _, pipeline, accel = CASES[case]
    sc = rg.Scene(scene_data(name))
    sc.set_pipeline(pipeline)
    sc.set_accel(accel)
    if n is not None:
        sc.set_supersample(n)
    return sc


def list_rows(h):
    return np.array([h - 1, 0, 5, 6, 7, 40, 99], np.uint32)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def counters(st):
    return (st.rays_primary, st.rays_shadow, st.rays_reflection, st.rays_transmission,
            st.err_nan_distance, st.err_transmission_none, st.err_aabb_normal)


def side_stream():
    import torch

    return torch.cuda.Stream()


def device_frame(h, w):
    """A full (h, w, 3) float32 frame on cuda:0, every word 0xFFFFFFFF (compared only with words outside the listed
    rows)."""
    import torch

    t = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
    t.view(torch.int32).fill_(-1)
    torch.cuda.synchronize()
    return t


def host_frame(h, w):
    a = np.empty((h, w, 3), np.float32)
    a.view(np.uint32)[:] = SENTINEL
    return a


def check_scattered(got, rows, ref32, label):
    got = bits(got)
    assert np.array_equal(got[rows], bits(ref32)[rows]), label
    rest = np.setdiff1d(np.arange(got.shape[0]), rows)
    assert (got[rest] == SENTINEL).all(), f"{label}: stores outside the listed rows"


@pytest.mark.parametrize("case", list(CASES))
def test_rows_f32_device_is_the_oracle(oracle, case):
    import torch

    name, w, h = CASES[case][:3]
    _, ost, ref32 = reference(oracle, name, w, h)
    s = side_stream()
    with open_scene(case) as sc:
        for y0, y1 in ((0, h), (h // 3, 2 * h // 3)):
            out = torch.empty((y1 - y0, w, 3), dtype=torch.float32, device="cuda")
            torch.cuda.synchronize()
            sc.render_rows_f32_device(w, h, y0, y1, out.data_ptr(), s.cuda_stream)
            assert np.array_equal(bits(out.cpu().numpy()), bits(ref32[y0:y1])), (case, y0, y1)
            if (y0, y1) == (0, h):
                assert counters(sc.last_stats) == counters(ost), case


@pytest.mark.parametrize("case", list(CASES))
def test_rowlist_f32_device_is_compacted_in_list_order(oracle, case):
    import torch

    name, w, h = CASES[case][:3]
    _, _, ref32 = reference(oracle, name, w, h)
    rows = list_rows(h)
    s = side_stream()
    out = torch.empty((rows.size, w, 3), dtype=torch.float32, device="cuda")
    torch.cuda.synchronize()
    with open_scene(case) as sc:
        sc.render_rowlist_f32_device(w, h, rows, out.data_ptr(), s.cuda_stream)
    assert np.array_equal(bits(out.cpu().numpy()), bits(ref32[rows]))


@pytest.mark.parametrize("case,w", [("test1-auto", 800), ("c4-grid", 256), ("c4-grid", 250), ("c4-brute", 256),
                                    ("c4-brute", 250)])
def test_rowlist_f32_scatter_stores_the_listed_rows_only(oracle, case, w):
    """W = 256: every group of 4 pixels is 16-byte aligned (three 128-bit stores); W = 250: every other row starts
    8 bytes off alignment (scalar stores) and a group of 4 crosses each row's end."""
    name, _, h = CASES[case][:3]
    _, _, ref32 = reference(oracle, name, w, h)
    rows = list_rows(h)
    frame = device_frame(h, w)
    s = side_stream()
    with open_scene(case) as sc:
        sc.render_rowlist_f32_scatter(w, h, rows, frame.data_ptr(), s.cuda_stream)
    check_scattered(frame.cpu().numpy(), rows, ref32, f"{case} W={w}")


@pytest.mark.parametrize("case", list(CASES))
def test_rowlist_f32_host_copies_the_listed_rows_only(oracle, case):
    """A contiguous run (one copy) and an interleaved share, every third 8-row tile (one strided copy), into a
    pinned host frame."""
    name, w, h = CASES[case][:3]
    _, _, ref32 = reference(oracle, name, w, h)
    for label, rows in (("run", np.arange(10, 42, dtype=np.uint32)),
                        ("every third tile", rows_of_tiles(list(range(0, (h + 7) // 8, 3)), 8, h))):
        frame = host_frame(h, w)
        rg.host_register(frame.ctypes.data, frame.nbytes)
        try:
            with open_scene(case) as sc:
                sc.render_rowlist_f32_host(w, h, rows, frame.ctypes.data)
        finally:
            rg.host_unregister(frame.ctypes.data)
        check_scattered(frame, rows, ref32, f"{case} {label}")


@pytest.mark.parametrize("n", [2, 3])
@pytest.mark.parametrize("case", ["c4-grid", "c4-brute", "mega"])
def test_supersampled_f32_entries_equal_render_rows_f32(case, n):
    """RG_OPT_SUPERSAMPLE = n: every f32 entry delivers render_rows_f32's n x n averages, bit for bit, and counts the
    same rays.  The scatter entry (wavefront only) runs k_resolve_ss<F32Scatter>."""
    import torch

    mega = case == "mega"
    w, h = 256, 144
    rows = list_rows(h)
    s = side_stream()
    with open_scene("c4-brute" if mega else case, n) as sc:
        if mega:
            sc.set_pipeline(rg.PIPELINE_MEGAKERNEL)
        ref32 = sc.render_rows_f32(w, h)
        ref_counts = counters(sc.last_stats)
        out = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
        torch.cuda.synchronize()
        sc.render_rows_f32_device(w, h, 0, h, out.data_ptr(), s.cuda_stream)
        assert np.array_equal(bits(out.cpu().numpy()), bits(ref32)), "rows_f32_device"
        assert counters(sc.last_stats) == ref_counts
        sc.render_rowlist_f32_device(w, h, rows, out.data_ptr(), s.cuda_stream)
        assert np.array_equal(bits(out[:rows.size].cpu().numpy()), bits(ref32[rows])), "rowlist_f32_device"
        frame = host_frame(h, w)
        rg.host_register(frame.ctypes.data, frame.nbytes)
        try:
            sc.render_rowlist_f32_host(w, h, rows, frame.ctypes.data)
        finally:
            rg.host_unregister(frame.ctypes.data)
        check_scattered(frame, rows, ref32, "rowlist_f32_host")
        if not mega:
            dframe = device_frame(h, w)
            sc.render_rowlist_f32_scatter(w, h, rows, dframe.data_ptr(), s.cuda_stream)
            check_scattered(dframe.cpu().numpy(), rows, ref32, "rowlist_f32_scatter")


@pytest.mark.parametrize("case", list(CASES))
def test_f32_entries_report_their_twins_counters(oracle, case):
    """The ray and error counters of each f32 entry equal its RGBA8 twin's for the same rows, and over the whole
    frame (a row list holding every row, in reverse) the oracle's."""
    import torch

    name, w, h = CASES[case][:3]
    _, ost, _ = reference(oracle, name, w, h)
    s = side_stream().cuda_stream
    dev = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
    host = host_frame(h, w)
    torch.cuda.synchronize()
    with open_scene(case) as sc:
        for rows in (list_rows(h), np.arange(h, dtype=np.uint32)[::-1].copy()):
            pairs = {"device": (lambda: sc.render_rowlist_device(w, h, rows, dev.data_ptr(), s),
                                lambda: sc.render_rowlist_f32_device(w, h, rows, dev.data_ptr(), s)),
                     "scatter": (lambda: sc.render_rowlist_scatter(w, h, rows, dev.data_ptr(), s),
                                 lambda: sc.render_rowlist_f32_scatter(w, h, rows, dev.data_ptr(), s)),
                     "host": (lambda: sc.render_rowlist_host(w, h, rows, host.ctypes.data),
                              lambda: sc.render_rowlist_f32_host(w, h, rows, host.ctypes.data))}
            for label, (twin, f32) in pairs.items():
                a, b = counters(twin()), counters(f32())
                assert a == b, (case, label, rows.size)
                if rows.size == h:
                    assert b == counters(ost), (case, label)
        a = counters(sc.render_rows_device(w, h, 0, h, dev.data_ptr(), s))
        b = counters(sc.render_rows_f32_device(w, h, 0, h, dev.data_ptr(), s))
        assert a == b == counters(ost), case


def test_scatter_kinds_on_one_buffer_replay_their_own_graphs(oracle):
    """RGBA8 and f32 scatter batches with the same rows into the same device buffer must never share a CUDA graph:
    each stays right for three interleaved rounds, and by the third each is a replay of its own graph."""
    import torch

    name, w, h = CASES["c4-grid"][:3]
    ref, _, ref32 = reference(oracle, name, w, h)
    rows = list_rows(h)
    buf = torch.empty(h * w * 12, dtype=torch.uint8, device="cuda")
    s = side_stream().cuda_stream
    with open_scene("c4-grid") as sc:
        for it in range(3):
            buf.fill_(0xFF)
            torch.cuda.synchronize()
            sc.render_rowlist_scatter(w, h, rows, buf.data_ptr(), s)
            rgba_replays = sc.last_stats.graph_replays
            assert np.array_equal(buf[:h * w * 4].cpu().numpy().reshape(h, w, 4)[rows], ref[rows]), it
            buf.fill_(0xFF)
            torch.cuda.synchronize()
            sc.render_rowlist_f32_scatter(w, h, rows, buf.data_ptr(), s)
            f32_replays = sc.last_stats.graph_replays
            check_scattered(buf.view(torch.float32).view(h, w, 3).cpu().numpy(), rows, ref32, f"round {it}")
            if it == 2:
                assert (rgba_replays, f32_replays) == (1, 1)


def _codes(call_pairs):
    """[(code of the RGBA8 twin, code of the f32 entry)] for (twin, f32) pairs of zero-argument calls."""
    out = []
    for twin, f32 in call_pairs:
        got = []
        for fn in (twin, f32):
            try:
                fn()
                got.append(_native.RG_OK)
            except rg.RaingunError as e:
                got.append(e.code)
        out.append(tuple(got))
    return out


def test_f32_entries_refuse_what_their_twins_refuse():
    import torch

    data = scene_data("C4")
    w, h = 256, 144
    dev = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
    host = host_frame(h, w)
    torch.cuda.synchronize()
    p, hp = dev.data_ptr(), host.ctypes.data
    rows = list_rows(h)

    def pairs(sc, w, h, rows, y1):
        return [(lambda: sc.render_rows_device(w, h, 0, y1, p), lambda: sc.render_rows_f32_device(w, h, 0, y1, p)),
                (lambda: sc.render_rowlist_device(w, h, rows, p), lambda: sc.render_rowlist_f32_device(w, h, rows, p)),
                (lambda: sc.render_rowlist_scatter(w, h, rows, p), lambda: sc.render_rowlist_f32_scatter(w, h, rows, p)),
                (lambda: sc.render_rowlist_host(w, h, rows, hp), lambda: sc.render_rowlist_f32_host(w, h, rows, hp))]

    E_INVALID, E_PORTRAIT = _native.E_INVALID, _native.E_PORTRAIT
    with rg.Scene(data, devices=[0, 0]) as sc:   # a multi-device handle
        assert _codes(pairs(sc, w, h, rows, h)) == [(E_INVALID, E_INVALID)] * 4
    with rg.Scene(data) as sc:
        sc.set_pipeline(rg.PIPELINE_WAVEFRONT)
        bad = np.array([0, h], np.uint32)   # a row >= height
        assert _codes(pairs(sc, w, h, bad, h + 1)) == [(E_INVALID, E_INVALID)] * 4
        assert _codes(pairs(sc, h - 1, h, rows[rows < h - 1], h)) == [(E_PORTRAIT, E_PORTRAIT)] * 4
        # NULL rows with n_rows > 0
        L, st = _native.lib(), rg.Stats()
        for twin, f32 in (("rg_render_rowlist_device", "rg_render_rowlist_f32_device"),
                          ("rg_render_rowlist_scatter", "rg_render_rowlist_f32_scatter")):
            codes = [getattr(L, e)(sc._h, w, h, None, 3, ctypes.c_void_p(p), None, ctypes.byref(st)) for e in (twin, f32)]
            assert codes == [E_INVALID, E_INVALID], twin
        codes = [getattr(L, e)(sc._h, w, h, None, 3, ctypes.c_void_p(hp), ctypes.byref(st))
                 for e in ("rg_render_rowlist_host", "rg_render_rowlist_f32_host")]
        assert codes == [E_INVALID, E_INVALID]
        sc.set_pipeline(rg.PIPELINE_MEGAKERNEL)
        assert _codes(pairs(sc, w, h, rows, h)[2:3]) == [(E_INVALID, E_INVALID)]


def test_f32_scatter_gathers_across_two_devices(oracle):
    """GPU 1 stores an interleaved half of the rows straight into a frame on GPU 0 (peer access), GPU 0 renders the
    other half; the assembled f32 frame is the oracle's, bit for bit.  Needs two GPUs."""
    import torch

    if rg.device_count() < 2:
        pytest.skip("needs two GPUs")
    if not torch.cuda.can_device_access_peer(1, 0):
        pytest.skip("no peer access between GPU 1 and GPU 0")
    name, w, h = CASES["c4-grid"][:3]
    _, _, ref32 = reference(oracle, name, w, h)
    frame = device_frame(h, w)
    _native.check(_native.lib().rg_device_enable_peer(1, 0))
    tiles = [np.arange(y, min(h, y + 8), dtype=np.uint32) for y in range(0, h, 8)]
    rows0, rows1 = np.concatenate(tiles[0::2]), np.concatenate(tiles[1::2])
    data = scene_data(name)
    with rg.Scene(data, device=0) as s0, rg.Scene(data, device=1) as s1:
        for s_ in (s0, s1):
            s_.set_pipeline(rg.PIPELINE_WAVEFRONT)
        with torch.cuda.device(1):
            s1.render_rowlist_f32_scatter(w, h, rows1, frame.data_ptr(), torch.cuda.current_stream(1).cuda_stream)
        with torch.cuda.device(0):
            s0.render_rowlist_f32_scatter(w, h, rows0, frame.data_ptr(), torch.cuda.current_stream(0).cuda_stream)
    torch.cuda.synchronize(1)
    torch.cuda.synchronize(0)
    assert np.array_equal(bits(frame.cpu().numpy()), bits(ref32))
