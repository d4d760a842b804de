"""raingun_b200 — B200-native render hot path of the raingun ray tracer.

Python host-side mirror of raingun-lib's public surface for this path
(raingun-lib/src/scene.rs:11-51, rendering.rs:18-22):

    scene = Scene.from_yaml_file("examples/test1.yml")     # serde_yaml::from_reader, main.rs:117-118
    image = scene.render_image(800, 600)                   # Scene::render_image, scene.rs:41-43
    scene.streaming_render(800, 600, on_rows)              # Scene::streaming_render, scene.rs:45-51

Everything that computes pixels happens in libraingun_b200.so (hand-written sm_100a CUDA)
behind the C ABI of include/raingun_b200.h; this module only flattens scenes and moves
buffers.  There is no CPU path.
"""
from __future__ import annotations

import ctypes
from typing import Callable, Optional

import numpy as np

from . import _native
from ._native import (ACCEL_AUTO, ACCEL_BRUTE, ACCEL_GRID, DEVICE_ALL, PIPELINE_AUTO, PIPELINE_MEGAKERNEL, PIPELINE_WAVEFRONT,
                      RaingunError)
from .scene import SceneData, SceneError, Stats, load_scene, parse_scene, scene_from_dict

__all__ = ["Scene", "SharedFrame", "host_register", "host_unregister", "trim", "SceneData", "SceneError", "RaingunError", "Stats", "load_scene", "parse_scene",
           "scene_from_dict", "device_count", "measure_peaks", "ACCEL_AUTO", "ACCEL_BRUTE", "ACCEL_GRID",
           "PIPELINE_WAVEFRONT", "PIPELINE_MEGAKERNEL", "PIPELINE_AUTO", "DEVICE_ALL"]


def device_count() -> int:
    return int(_native.lib().rg_device_count())


def measure_peaks(device: int = 0):
    """(fp32 TFLOP/s, fp64 TFLOP/s, SM MHz) of a register-resident FMA loop — roofline denominators."""
    a, b, c = ctypes.c_double(), ctypes.c_double(), ctypes.c_double()
    _native.check(_native.lib().rg_measure_peaks(device, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)))
    return a.value, b.value, c.value


def trim() -> int:
    """Frees the device-side contexts destroyed scenes have parked for reuse (rg_trim); returns how many."""
    return int(_native.lib().rg_trim())


def host_register(ptr: int, nbytes: int) -> None:
    """Pins host memory for full-speed device-to-host copies (rg_host_register)."""
    _native.check(_native.lib().rg_host_register(ctypes.c_void_p(ptr), nbytes))


def host_unregister(ptr: int) -> None:
    _native.check(_native.lib().rg_host_unregister(ctypes.c_void_p(ptr)))


class SharedFrame:
    """A device frame on ``device`` that the other ranks of a box map through CUDA IPC and write
    over NVLink (rg_shared_frame_*).  ``SharedFrame.create`` on the owner, ``handle`` (64 bytes) to
    the peers by any channel, ``SharedFrame.open`` there."""

    def __init__(self, device: int, ptr: int, nbytes: int, owner: bool, handle: bytes = b"") -> None:
        self.device, self.ptr, self.nbytes, self.owner, self.handle = device, ptr, nbytes, owner, handle

    @classmethod
    def create(cls, device: int, nbytes: int) -> "SharedFrame":
        p = ctypes.c_void_p()
        h = ctypes.create_string_buffer(_native.IPC_HANDLE_BYTES)
        _native.check(_native.lib().rg_shared_frame_create(device, nbytes, ctypes.byref(p), h))
        return cls(device, p.value, nbytes, True, h.raw)

    @classmethod
    def open(cls, device: int, handle: bytes, nbytes: int) -> "SharedFrame":
        p = ctypes.c_void_p()
        _native.check(_native.lib().rg_shared_frame_open(device, handle, ctypes.byref(p)))
        return cls(device, p.value, nbytes, False, handle)

    @property
    def __cuda_array_interface__(self):   # zero-copy view for torch.as_tensor(frame, device=...)
        return {"shape": (self.nbytes,), "typestr": "|u1", "data": (self.ptr, False), "version": 2}

    def close(self) -> None:
        if self.ptr:
            _native.check(_native.lib().rg_shared_frame_close(self.device, ctypes.c_void_p(self.ptr), 1 if self.owner else 0))
            self.ptr = 0


class Scene:
    """A scene resident on one GPU — or on several (``device=DEVICE_ALL`` / ``devices=[...]``): renders into
    host memory are then split into row tiles across the GPUs inside the library (rayon's ``par_iter``,
    rendering.rs:27-35).  The uploaded counterpart of raingun-lib's ``Scene``."""

    def __init__(self, data: SceneData, device: int = 0, devices=None) -> None:
        self.data = data
        self.device = device
        self._h = ctypes.c_void_p()
        self.last_stats = Stats()
        desc, keep = data.to_desc()
        if devices is not None:
            arr = (ctypes.c_int32 * len(devices))(*devices)
            _native.check(_native.lib().rg_scene_create_multi(ctypes.byref(desc), arr, len(devices), ctypes.byref(self._h)))
        else:
            _native.check(_native.lib().rg_scene_create(ctypes.byref(desc), device, ctypes.byref(self._h)))
        del keep

    @property
    def device_count(self) -> int:
        return int(_native.lib().rg_scene_device_count(self._h))

    # -- construction, as src/main.rs:117-125 does it
    @classmethod
    def from_yaml(cls, text: str, device: int = 0, texture_loader=None, max_depth: Optional[int] = None,
                  texture_root: Optional[str] = None) -> "Scene":
        """The scene is parsed by the native host library (C++ YAML reader + texture decoders,
        include/raingun_host.h); ``scene.parse_scene`` is the independent Python implementation the
        tests compare it with."""
        from . import host

        return cls(host.parse_scene(text, texture_loader, texture_root, max_depth), device)

    @classmethod
    def from_yaml_file(cls, path: str, device: int = 0, texture_root: Optional[str] = None,
                       max_depth: Optional[int] = None) -> "Scene":
        with open(path, "r", encoding="utf-8") as f:
            return cls.from_yaml(f.read(), device, None, max_depth, texture_root)

    def close(self) -> None:
        if getattr(self, "_h", None) is not None and self._h.value:
            _native.lib().rg_scene_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self) -> None:  # pragma: no cover - best effort
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self) -> "Scene":
        return self

    def __exit__(self, *exc) -> None:
        self.close()

    def set_option(self, key: int, value: int) -> None:
        _native.check(_native.lib().rg_scene_set_option(self._h, key, int(value)))

    def set_pipeline(self, pipeline: int) -> None:
        self.set_option(_native.OPT_PIPELINE, pipeline)

    def set_accel(self, accel: int) -> None:
        self.set_option(_native.OPT_ACCEL, accel)

    def set_max_depth_limit(self, limit: int) -> None:
        self.set_option(_native.OPT_MAX_DEPTH, limit)

    def set_supersample(self, n: int) -> None:
        """Anti-aliasing (RG_OPT_SUPERSAMPLE, 1 <= n <= 8): every render then delivers the reference's frame at
        n x width by n x height, averaged n x n per pixel in f32 on the GPU, in arrays of unchanged shape.  1 (the
        default) is the reference's own frame."""
        self.set_option(_native.OPT_SUPERSAMPLE, n)

    def set_supersample_edges(self, t: Optional[int]) -> None:
        """Edge-adaptive anti-aliasing (RG_OPT_SUPERSAMPLE_EDGES): with ``set_supersample(n)``, n > 1, only pixels on an
        edge of the reference's own frame get their n x n samples: a pixel whose r, g or b byte differs by more than
        ``t`` (0 <= t <= 255) from one of its 8 neighbours in that frame.  Every other pixel is the reference's pixel.
        ``None`` (the default) supersamples every pixel."""
        self.set_option(_native.OPT_SUPERSAMPLE_EDGES, -1 if t is None else t)

    # -- Scene::render_image (scene.rs:41-43)
    def render_image(self, width: int, height: int, out: Optional[np.ndarray] = None) -> np.ndarray:
        return self.render_rows(width, height, 0, height, out)

    def render_rows(self, width: int, height: int, y0: int, y1: int, out: Optional[np.ndarray] = None) -> np.ndarray:
        rows = max(0, y1 - y0)
        if out is None:
            out = np.empty((rows, width, 4), np.uint8)
        if out.dtype != np.uint8 or not out.flags.c_contiguous or out.size != rows * width * 4:
            raise ValueError("out must be a C-contiguous uint8 array of rows*width*4 bytes")
        st = Stats()
        _native.check(_native.lib().rg_render_rows(self._h, width, height, y0, y1, out.ctypes.data, ctypes.byref(st)))
        self.last_stats = st
        return out

    def render_rows_into(self, width: int, height: int, y0: int, y1: int, host_ptr: int) -> Stats:
        """Same, into a raw HOST pointer (e.g. a pinned torch tensor's data_ptr())."""
        st = Stats()
        _native.check(_native.lib().rg_render_rows(self._h, width, height, y0, y1, ctypes.c_void_p(host_ptr),
                                                   ctypes.byref(st)))
        self.last_stats = st
        return st

    def render_rows_device(self, width: int, height: int, y0: int, y1: int, device_ptr: int,
                           cuda_stream: int = 0) -> Stats:
        """Result stays in HBM at ``device_ptr`` (e.g. a torch CUDA tensor's data_ptr())."""
        st = Stats()
        _native.check(_native.lib().rg_render_rows_device(self._h, width, height, y0, y1, ctypes.c_void_p(device_ptr),
                                                          ctypes.c_void_p(cuda_stream), ctypes.byref(st)))
        self.last_stats = st
        return st

    def _render_rowlist(self, entry, width: int, height: int, rows, ptr: int, *stream) -> Stats:
        rows = np.ascontiguousarray(rows, np.uint32)
        st = Stats()
        _native.check(entry(self._h, width, height, ctypes.c_void_p(rows.ctypes.data), int(rows.size), ctypes.c_void_p(ptr),
                            *stream, ctypes.byref(st)))
        self.last_stats = st
        return st

    def render_rows_f32_device(self, width: int, height: int, y0: int, y1: int, device_ptr: int,
                               cuda_stream: int = 0) -> Stats:
        """``render_rows_device`` with the unquantised f32 colours: (y1-y0)*width*3 floats in HBM at ``device_ptr``."""
        st = Stats()
        _native.check(_native.lib().rg_render_rows_f32_device(self._h, width, height, y0, y1, ctypes.c_void_p(device_ptr),
                                                              ctypes.c_void_p(cuda_stream), ctypes.byref(st)))
        self.last_stats = st
        return st

    def render_rowlist_device(self, width: int, height: int, rows, device_ptr: int, cuda_stream: int = 0) -> Stats:
        """Row-tile sharding unit: renders the listed image rows, compacted in list order, into
        HBM at ``device_ptr`` (len(rows)*width*4 bytes)."""
        return self._render_rowlist(_native.lib().rg_render_rowlist_device, width, height, rows, device_ptr,
                                    ctypes.c_void_p(cuda_stream))

    def render_rowlist_scatter(self, width: int, height: int, rows, frame_ptr: int, cuda_stream: int = 0) -> Stats:
        """As render_rowlist_device, but row ``rows[k]`` lands at its own place in the FULL frame at
        ``frame_ptr`` — which may be another GPU's memory (``SharedFrame``): the gather of a sharded
        frame fused into the last kernel."""
        return self._render_rowlist(_native.lib().rg_render_rowlist_scatter, width, height, rows, frame_ptr,
                                    ctypes.c_void_p(cuda_stream))

    def render_rowlist_f32_device(self, width: int, height: int, rows, device_ptr: int, cuda_stream: int = 0) -> Stats:
        """``render_rowlist_device`` with f32 colours: len(rows)*width*3 floats, compacted in list order."""
        return self._render_rowlist(_native.lib().rg_render_rowlist_f32_device, width, height, rows, device_ptr,
                                    ctypes.c_void_p(cuda_stream))

    def render_rowlist_f32_scatter(self, width: int, height: int, rows, frame_ptr: int, cuda_stream: int = 0) -> Stats:
        """``render_rowlist_scatter`` with f32 colours: row ``rows[k]`` lands at ``frame_ptr + rows[k]*width*12`` bytes
        of a full width*height*3 float frame (device memory, possibly another GPU's, or pinned host memory)."""
        return self._render_rowlist(_native.lib().rg_render_rowlist_f32_scatter, width, height, rows, frame_ptr,
                                    ctypes.c_void_p(cuda_stream))

    def render_rowlist_f32_host(self, width: int, height: int, rows, frame_ptr: int) -> Stats:
        """``render_rowlist_host`` with f32 colours: row ``rows[k]`` is copied to ``frame_ptr + rows[k]*width*12`` bytes
        of a full width*height*3 float frame in HOST memory."""
        return self._render_rowlist(_native.lib().rg_render_rowlist_f32_host, width, height, rows, frame_ptr)

    def render_rows_f32(self, width: int, height: int, y0: int = 0, y1: Optional[int] = None) -> np.ndarray:
        """The unquantised f32 colours (``RenderedPixel.color``, rendering.rs:18-22): (rows, width, 3) float32."""
        y1 = height if y1 is None else y1
        out = np.empty((max(0, y1 - y0), width, 3), np.float32)
        st = Stats()
        _native.check(_native.lib().rg_render_rows_f32(self._h, width, height, y0, y1, out.ctypes.data, ctypes.byref(st)))
        self.last_stats = st
        return out

    def streaming_render_f32(self, width: int, height: int, on_rows: Callable[[int, np.ndarray], bool], band_rows: int = 0) -> bool:
        """``streaming_render`` with the colours as the reference's channel carries them: unquantised f32 RGB."""
        return self._stream(_native.lib().rg_render_stream_f32, _native.ROWS_F32_CB, 3, width, height, on_rows, band_rows)

    def render_rowlist_host(self, width: int, height: int, rows, frame_ptr: int) -> Stats:
        """Renders the listed image rows and copies row ``rows[k]`` to ``frame_ptr + rows[k]*width*4`` in HOST
        memory (a full frame, ideally pinned / ``host_register``-ed; may be shared by one process per GPU)."""
        return self._render_rowlist(_native.lib().rg_render_rowlist_host, width, height, rows, frame_ptr)

    # -- Scene::streaming_render (scene.rs:45-51): finished row bands instead of single pixels
    def streaming_render(self, width: int, height: int, on_rows: Callable[[int, np.ndarray], bool],
                         band_rows: int = 0) -> bool:
        """Calls ``on_rows(y0, rgba_rows)`` per finished band; return False from it to cancel
        (the closed channel of rendering.rs:53-54,67).  Returns False if cancelled."""
        return self._stream(_native.lib().rg_render_stream, _native.ROWS_CB, 4, width, height, on_rows, band_rows)

    def _stream(self, entry, cb_type, channels: int, width: int, height: int, on_rows, band_rows: int) -> bool:
        failure = []

        def trampoline(y0, rows, w, ptr, _user):
            try:
                arr = np.ctypeslib.as_array(ptr, shape=(rows, w, channels))
                keep_going = on_rows(int(y0), arr)
                return 0 if (keep_going is None or keep_going) else 1
            except BaseException as e:  # never unwind through C
                failure.append(e)
                return 1

        cb = cb_type(trampoline)
        st = Stats()
        rc = entry(self._h, width, height, band_rows, cb, None, ctypes.byref(st))
        self.last_stats = st
        if failure:
            raise failure[0]
        if rc == _native.E_CANCELLED:
            return False
        _native.check(rc)
        return True
