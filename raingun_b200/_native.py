"""ctypes binding of libraingun_b200.so — the C ABI of include/raingun_b200.h.

There is no fallback: if the CUDA library is missing this module raises at import time
of the symbols, and every render call fails loudly when no sm_100 device is present.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

from .scene import SceneDesc, Stats

_HERE = os.path.dirname(os.path.abspath(__file__))
# RAINGUN_B200_LIB selects another build of the same library (tuning experiments: tools/build_variants.sh)
LIB_PATH = os.environ.get("RAINGUN_B200_LIB") or os.path.join(_HERE, "libraingun_b200.so")

RG_OK = 0
ERRORS = {0: "RG_OK", -1: "RG_E_INVALID", -2: "RG_E_PORTRAIT", -3: "RG_E_TOO_LARGE", -4: "RG_E_DEPTH",
          -5: "RG_E_CUDA", -6: "RG_E_NOMEM", -7: "RG_E_CANCELLED", -8: "RG_E_LIGHTS", -9: "RG_E_BUSY"}
# E_LIGHTS is obsolete: scenes may have any number of lights, and the library no longer returns it
E_INVALID, E_PORTRAIT, E_TOO_LARGE, E_DEPTH, E_CUDA, E_NOMEM, E_CANCELLED, E_LIGHTS, E_BUSY = -1, -2, -3, -4, -5, -6, -7, -8, -9
DEVICE_ALL = -1

PIPELINE_WAVEFRONT, PIPELINE_MEGAKERNEL, PIPELINE_AUTO = 0, 1, 2
ACCEL_AUTO, ACCEL_BRUTE, ACCEL_GRID = 0, 1, 2
OPT_PIPELINE, OPT_ACCEL, OPT_MAX_DEPTH, OPT_BATCH_PIXELS, OPT_VERIFY_CULL, OPT_OVERLAP = 1, 2, 3, 4, 5, 6
OPT_HOST_FREE, OPT_GRAPH, OPT_TRACE_STATS, OPT_SCHEDULE, OPT_TILE_ROWS, OPT_ORIGIN_HINTS = 7, 8, 9, 11, 12, 13
OPT_SUPERSAMPLE, OPT_LIGHT_GRIDS, OPT_SUPERSAMPLE_EDGES = 14, 15, 16

ROWS_CB = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32,
                           ctypes.POINTER(ctypes.c_uint8), ctypes.c_void_p)

ROWS_F32_CB = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32,
                               ctypes.POINTER(ctypes.c_float), ctypes.c_void_p)

# every symbol include/raingun_b200.h declares
EXPORTS = ("rg_scene_create", "rg_scene_create_multi", "rg_scene_device_count", "rg_scene_destroy", "rg_scene_set_option", "rg_render", "rg_render_rows",
           "rg_render_rows_device", "rg_render_rowlist_device", "rg_render_rowlist_scatter", "rg_render_rowlist_host", "rg_host_register", "rg_host_unregister", "rg_device_enable_peer", "rg_shm_barrier_open", "rg_shm_barrier_wait", "rg_shm_barrier_close", "rg_shared_frame_create",
           "rg_shared_frame_open", "rg_shared_frame_close", "rg_render_stream", "rg_render_rows_f32", "rg_render_stream_f32",
           "rg_render_rows_f32_device", "rg_render_rowlist_f32_device", "rg_render_rowlist_f32_scatter", "rg_render_rowlist_f32_host", "rg_trim", "rg_last_error", "rg_measure_peaks",
           "rg_device_count")
IPC_HANDLE_BYTES = 64


class RaingunError(RuntimeError):
    def __init__(self, code: int, message: str) -> None:
        super().__init__(f"{ERRORS.get(code, code)}: {message}")
        self.code = code


_lib: Optional[ctypes.CDLL] = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
                          "g.build()'` (or make -C raingun_b200/csrc). There is no CPU fallback.")
    L = ctypes.CDLL(LIB_PATH)
    vp, u32, i32 = ctypes.c_void_p, ctypes.c_uint32, ctypes.c_int32
    L.rg_scene_create.restype = ctypes.c_int
    L.rg_scene_create.argtypes = [ctypes.POINTER(SceneDesc), i32, ctypes.POINTER(vp)]
    L.rg_scene_create_multi.restype = ctypes.c_int
    L.rg_scene_create_multi.argtypes = [ctypes.POINTER(SceneDesc), ctypes.POINTER(i32), u32, ctypes.POINTER(vp)]
    L.rg_scene_device_count.restype = ctypes.c_int
    L.rg_scene_device_count.argtypes = [vp]
    L.rg_scene_destroy.restype = None
    L.rg_scene_destroy.argtypes = [vp]
    L.rg_scene_set_option.restype = ctypes.c_int
    L.rg_scene_set_option.argtypes = [vp, i32, ctypes.c_int64]
    L.rg_render.restype = ctypes.c_int
    L.rg_render.argtypes = [vp, u32, u32, vp, ctypes.POINTER(Stats)]
    L.rg_render_rows.restype = ctypes.c_int
    L.rg_render_rows.argtypes = [vp, u32, u32, u32, u32, vp, ctypes.POINTER(Stats)]
    L.rg_render_rows_device.restype = ctypes.c_int
    L.rg_render_rows_device.argtypes = [vp, u32, u32, u32, u32, vp, vp, ctypes.POINTER(Stats)]
    L.rg_render_rowlist_device.restype = ctypes.c_int
    L.rg_render_rowlist_device.argtypes = [vp, u32, u32, vp, u32, vp, vp, ctypes.POINTER(Stats)]
    L.rg_render_rowlist_scatter.restype = ctypes.c_int
    L.rg_render_rowlist_scatter.argtypes = [vp, u32, u32, vp, u32, vp, vp, ctypes.POINTER(Stats)]
    L.rg_render_rowlist_host.restype = ctypes.c_int
    L.rg_render_rowlist_host.argtypes = [vp, u32, u32, vp, u32, vp, ctypes.POINTER(Stats)]
    L.rg_host_register.restype = ctypes.c_int
    L.rg_host_register.argtypes = [vp, ctypes.c_size_t]
    L.rg_host_unregister.restype = ctypes.c_int
    L.rg_host_unregister.argtypes = [vp]
    L.rg_shm_barrier_open.restype = ctypes.c_int
    L.rg_shm_barrier_open.argtypes = [ctypes.c_char_p, u32, i32, ctypes.POINTER(vp)]
    L.rg_shm_barrier_wait.restype = ctypes.c_int
    L.rg_shm_barrier_wait.argtypes = [vp]
    L.rg_shm_barrier_close.restype = ctypes.c_int
    L.rg_shm_barrier_close.argtypes = [vp]
    L.rg_device_enable_peer.restype = ctypes.c_int
    L.rg_device_enable_peer.argtypes = [i32, i32]
    L.rg_shared_frame_create.restype = ctypes.c_int
    L.rg_shared_frame_create.argtypes = [i32, ctypes.c_size_t, ctypes.POINTER(vp), ctypes.c_char_p]
    L.rg_shared_frame_open.restype = ctypes.c_int
    L.rg_shared_frame_open.argtypes = [i32, ctypes.c_char_p, ctypes.POINTER(vp)]
    L.rg_shared_frame_close.restype = ctypes.c_int
    L.rg_shared_frame_close.argtypes = [i32, vp, i32]
    L.rg_render_stream.restype = ctypes.c_int
    L.rg_render_stream.argtypes = [vp, u32, u32, u32, ROWS_CB, vp, ctypes.POINTER(Stats)]
    L.rg_render_rows_f32.restype = ctypes.c_int
    L.rg_render_rows_f32.argtypes = [vp, u32, u32, u32, u32, vp, ctypes.POINTER(Stats)]
    L.rg_render_stream_f32.restype = ctypes.c_int
    L.rg_render_stream_f32.argtypes = [vp, u32, u32, u32, ROWS_F32_CB, vp, ctypes.POINTER(Stats)]
    L.rg_render_rows_f32_device.restype = ctypes.c_int
    L.rg_render_rows_f32_device.argtypes = [vp, u32, u32, u32, u32, vp, vp, ctypes.POINTER(Stats)]
    L.rg_render_rowlist_f32_device.restype = ctypes.c_int
    L.rg_render_rowlist_f32_device.argtypes = [vp, u32, u32, vp, u32, vp, vp, ctypes.POINTER(Stats)]
    L.rg_render_rowlist_f32_scatter.restype = ctypes.c_int
    L.rg_render_rowlist_f32_scatter.argtypes = [vp, u32, u32, vp, u32, vp, vp, ctypes.POINTER(Stats)]
    L.rg_render_rowlist_f32_host.restype = ctypes.c_int
    L.rg_render_rowlist_f32_host.argtypes = [vp, u32, u32, vp, u32, vp, ctypes.POINTER(Stats)]
    L.rg_trim.restype = ctypes.c_int
    L.rg_trim.argtypes = []
    L.rg_last_error.restype = ctypes.c_char_p
    L.rg_last_error.argtypes = []
    L.rg_measure_peaks.restype = ctypes.c_int
    L.rg_measure_peaks.argtypes = [i32, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double),
                                   ctypes.POINTER(ctypes.c_double)]
    L.rg_device_count.restype = ctypes.c_int
    L.rg_device_count.argtypes = []
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != RG_OK:
        msg = lib().rg_last_error()
        raise RaingunError(rc, msg.decode("utf-8", "replace") if msg else "")
