"""Sharded f32 frames on CPU: world_size 2, gloo backend, the CPU oracle's unquantised colours standing in for the
per-rank renderer (``Scene.render_rowlist_f32_device`` / ``render_rowlist_f32_host`` on a GPU).  Under test is
raingun_b200/dist.py with ``pixel_format="f32"``: rows of 12-byte pixels through the p2p and host gathers, the
(H, W, 3) float32 frame on rank 0, and the refusal of the MAX-reduce gather.  Frames are compared as uint32 views,
so NaN and -0 are compared by their bits."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from raingun_b200.dist import render_frame_sharded

W, H, TILE = 96, 54, 4


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _f32_rows(O, data, rows):
    return np.concatenate([O.render_rows(data, W, H, int(y), int(y) + 1, threads=1, want_f32=True)[2] for y in rows], axis=0)


def _worker(rank, world, port, schedule, out_dir, gather_mode):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from oracle import oracle
    from raingun_b200.synth import make_scene

    data, _ = make_scene("C4", spheres=40, depth=4)
    O = oracle()

    def render_rowlist(rows, out):   # out: len(rows) * W * 12 bytes, compacted in list order
        out.copy_(torch.from_numpy(_f32_rows(O, data, rows).view(np.uint8).reshape(-1)))
        return len(rows)

    host_frames = host_barrier = None
    if gather_mode == "host":
        from raingun_b200.dist import HostBarrier, SharedHostFrame
        host_frames = SharedHostFrame(W, H, rank, world, pin=False, pixel_format="f32")
        host_barrier = HostBarrier(rank, world)

        def render_rowlist(rows, frame_ptr):   # noqa: F811 - row y goes to frame_ptr + y * W * 12
            frame = np.ctypeslib.as_array(ctypes.cast(frame_ptr, ctypes.POINTER(ctypes.c_float)), shape=(H, W, 3))
            frame[rows.astype(np.int64)] = _f32_rows(O, data, rows)
            return len(rows)

    if gather_mode == "reduce":
        with pytest.raises(ValueError):
            render_frame_sharded(render_rowlist, W, H, rank, world, 1, torch.device("cpu"), tile_rows=TILE,
                                 schedule=schedule, gather_mode="reduce", pixel_format="f32")
        np.save(os.path.join(out_dir, f"refused{rank}.npy"), np.array([1]))
    else:
        for it, frame_id in enumerate((1, 2)):
            res = render_frame_sharded(render_rowlist, W, H, rank, world, frame_id, torch.device("cpu"), tile_rows=TILE,
                                       schedule=schedule, gather_mode=gather_mode, peer_frames=host_frames,
                                       host_barrier=host_barrier, pixel_format="f32")
            if rank == 0:
                assert res.frame.dtype == torch.float32 and tuple(res.frame.shape) == (H, W, 3)
                np.save(os.path.join(out_dir, f"frame{it}.npy"), np.array(res.frame.numpy()))
            if host_frames is not None:
                dist.barrier()   # rank 0 has copied the frame out before anyone overwrites it
                host_frames.array(frame_id)[:] = 0
                dist.barrier()
    if host_frames is not None:
        host_frames.close()
        host_barrier.close()
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("gather_mode", ["p2p", "host"])
@pytest.mark.parametrize("schedule", ["static", "steal"])
def test_two_ranks_gather_the_f32_frame(tmp_path, oracle, schedule, gather_mode):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), schedule, str(tmp_path), gather_mode), nprocs=world, join=True)
    from raingun_b200.synth import make_scene

    data, _ = make_scene("C4", spheres=40, depth=4)
    _, _, ref32 = oracle.render(data, W, H, want_f32=True)
    for it in range(2):
        got = np.load(tmp_path / f"frame{it}.npy")
        assert got.dtype == np.float32 and got.shape == (H, W, 3)
        assert np.array_equal(got.view(np.uint32), ref32.view(np.uint32)), f"frame {it}"


def test_reduce_refuses_f32_on_every_rank(tmp_path):
    world = 2
    mp.spawn(_worker, args=(world, _free_port(), "steal", str(tmp_path), "reduce"), nprocs=world, join=True)
    assert all((tmp_path / f"refused{r}.npy").exists() for r in range(world))


def test_f32_entry_points_refuse_a_null_scene():
    """The four f32 entry points check their handle before anything touches a device."""
    from raingun_b200 import _native
    from raingun_b200.scene import Stats

    L = _native.lib()
    rows = (ctypes.c_uint32 * 1)(0)
    st = Stats()
    assert L.rg_render_rows_f32_device(None, 8, 4, 0, 4, None, None, ctypes.byref(st)) == _native.E_INVALID
    for entry in (L.rg_render_rowlist_f32_device, L.rg_render_rowlist_f32_scatter):
        assert entry(None, 8, 4, rows, 1, None, None, ctypes.byref(st)) == _native.E_INVALID
    assert L.rg_render_rowlist_f32_host(None, 8, 4, rows, 1, None, ctypes.byref(st)) == _native.E_INVALID
