"""Row-tile sharding of one frame across the GPUs of a box — the multi-GPU form of
render_image's ``par_iter`` over pixels (raingun-lib/src/rendering.rs:27-35).

Pixels are independent, so the path shards with NO data-path collective: the scene is
replicated, the image is cut into tiles of ``tile_rows`` rows, and every rank renders the
tiles it claims.  Cost per row is very uneven (sky vs sphere field), so tiles are handed out
by a work-stealing counter — an atomic fetch-add on the c10d store all ranks already share —
in guided chunks (large first, small last).  The only exchange is the final gather of the
finished tiles into rank 0's frame: point-to-point sends over NVLink (NCCL send/recv), i.e.
rayon's ``collect`` (rendering.rs:34-35).

A batch of few rows cannot fill a B200 (its 8 bounce levels are ~40 short, latency-bound launches
with a host read-back each), so a rank may keep SEVERAL batches in flight: ``render_rowlist`` can
be a list of renderers (one scene handle + CUDA stream each), driven by one host thread each.  The
static share is split between them and the stealable tail is claimed by whichever thread runs dry,
so the fixed cost of a small batch hides under the other thread's kernels.

Gather.  ``peer`` (GPUs): rank 0 owns the frame (two, alternating per frame), every other rank
maps it through CUDA IPC and its last kernel stores each finished row at its place in rank 0's
memory over NVLink (``rg_render_rowlist_scatter``) — compute and "collective" are one kernel, and a
barrier is all that is left.  ``reduce`` / ``p2p``: NCCL (or gloo) collectives on packed rows.

Pixel formats.  ``pixel_format="rgba8"`` (the default) gathers the reference's RGBA8 bytes, 4 per pixel;
``"f32"`` the unquantised f32 colours (``RenderedPixel.color``), 3 floats per pixel.  Rows travel as bytes
either way: ``row_bytes = width * bytes_per_pixel`` is the only place the format enters, and only the
finished frame is viewed as (H, W, 4) uint8 or (H, W, 3) float32.

One process per GPU (torchrun); works unchanged on the gloo backend with CPU tensors, which
is how the host logic is tested without GPUs (tests/test_dist_gloo.py).
"""
from __future__ import annotations

import pickle
import threading
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass, field
from typing import Callable, List, Optional, Sequence, Union

import numpy as np
import torch
import torch.distributed as dist

DEFAULT_TILE_ROWS = 8
# "auto" schedule: with at least this many interleaved tiles per rank the static shares are
# balanced by the law of large numbers (measured on C4 at 4K, 8-row tiles: 2 % spread over 4 ranks),
# while every stolen tail batch costs ~1 ms of latency-bound launches (measured: +0.5..0.9 ms per
# 4K frame at 4-8 GPUs); below it, cost per tile is too uneven to trust static ownership.
AUTO_STATIC_MIN_TILES_PER_RANK = 16

# pixel_format -> (bytes per pixel, channels, numpy dtype, torch dtype) of a finished frame
PIXEL_FORMATS = {"rgba8": (4, 4, np.uint8, torch.uint8), "f32": (12, 3, np.float32, torch.float32)}


def _format(pixel_format: str):
    if pixel_format not in PIXEL_FORMATS:
        raise ValueError(f"pixel_format must be one of {sorted(PIXEL_FORMATS)}, not {pixel_format!r}")
    return PIXEL_FORMATS[pixel_format]


def bytes_per_pixel(pixel_format: str) -> int:
    return _format(pixel_format)[0]


def frame_view(buf: torch.Tensor, height: int, width: int, pixel_format: str) -> torch.Tensor:
    """The finished frame over the bytes of a contiguous uint8 buffer: (H, W, 4) uint8 or (H, W, 3) float32."""
    _, channels, _, dtype = _format(pixel_format)
    return buf.view(dtype).view(height, width, channels)


def n_tiles(height: int, tile_rows: int) -> int:
    return (height + tile_rows - 1) // tile_rows


def tile_rows_range(tile: int, tile_rows: int, height: int) -> range:
    return range(tile * tile_rows, min(height, (tile + 1) * tile_rows))


_ROWS_CACHE: dict = {}


def rows_of_tiles(tiles: Sequence[int], tile_rows: int, height: int) -> np.ndarray:
    """Image rows of the listed tiles, in list order (read-only array: static shares repeat every
    frame, so the result is memoised)."""
    if len(tiles) == 0:
        return np.zeros(0, np.uint32)
    key = (tuple(tiles), tile_rows, height)
    rows = _ROWS_CACHE.get(key)
    if rows is None:
        if len(_ROWS_CACHE) > 256:
            _ROWS_CACHE.clear()
        rows = np.concatenate([np.arange(r.start, r.stop, dtype=np.uint32)
                               for r in (tile_rows_range(t, tile_rows, height) for t in tiles)])
        rows.setflags(write=False)
        _ROWS_CACHE[key] = rows
    return rows


def resolve_schedule(schedule: str, num_tiles: int, world: int) -> str:
    if schedule != "auto":
        return schedule
    return "static" if num_tiles >= AUTO_STATIC_MIN_TILES_PER_RANK * max(world, 1) else "steal"


def guided_chunks(num_tiles: int, world: int, min_chunk: int = 1) -> List[List[int]]:
    """Deterministic guided self-scheduling: each chunk takes ``max(min_chunk, remaining //
    (2 * world))`` consecutive tiles.  Every rank computes the same list, so a claim is just
    an index into it."""
    chunks, start = [], 0
    while start < num_tiles:
        size = min(num_tiles - start, max(min_chunk, (num_tiles - start) // (2 * max(world, 1))))
        chunks.append(list(range(start, start + size)))
        start += size
    return chunks


def static_chunk(num_tiles: int, world: int, rank: int) -> List[int]:
    """Interleaved static ownership: tile t belongs to rank t % world."""
    return list(range(rank, num_tiles, world))


_POOLS = {}


def _pool(workers: int) -> ThreadPoolExecutor:
    if workers not in _POOLS:
        _POOLS[workers] = ThreadPoolExecutor(max_workers=workers, thread_name_prefix="raingun-batch")
    return _POOLS[workers]


def split_share(tiles: Sequence[int], workers: int, lead: float = 0.0) -> List[List[int]]:
    """A rank's static share dealt to its in-flight batches, each staying interleaved over the
    image.  ``lead`` (0 = equal shares) is the fraction the first batch gets: the other batches then
    run dry first and claim the stealable tail WHILE the lead batch still fills the GPU, which is
    what hides the fixed cost of the small tail batches."""
    if workers <= 1:
        return [list(tiles)]
    if not (0.0 < lead < 1.0):
        return [list(tiles[k::workers]) for k in range(workers)]
    out: List[List[int]] = [[] for _ in range(workers)]
    rest = 0
    for i, t in enumerate(tiles):
        if int((i + 1) * lead) > int(i * lead):
            out[0].append(t)
        else:
            out[1 + rest % (workers - 1)].append(t)
            rest += 1
    return out


def hybrid_plan(num_tiles: int, world: int, tail_every: int = 16, min_chunk: int = 2):
    """Work stealing without paying for it when the load is balanced: 1 - 1/tail_every of the
    tiles are owned statically (interleaved over the image and over the ranks: one large batch per
    rank, no counter traffic); every ``tail_every``-th tile forms the tail that is handed out by
    the work-stealing counter in guided chunks, which absorbs whatever imbalance remains.
    Returns ``(static_tiles_per_rank, tail_chunks)``."""
    if world <= 1 or num_tiles < 4 * world:
        return [list(range(num_tiles))] + [[] for _ in range(max(world, 1) - 1)], []
    static = [t for t in range(num_tiles) if t % tail_every != tail_every - 1]
    tail = [t for t in range(num_tiles) if t % tail_every == tail_every - 1]
    per_rank = [static[r::world] for r in range(world)]
    # one tail chunk per rank on average: a claim is a whole wavefront batch (~1 ms of fixed cost)
    per = max(min_chunk, (len(tail) + world - 1) // world)
    chunks = [tail[i:i + per] for i in range(0, len(tail), per)]
    return per_rank, chunks


class TileCounter:
    """Work-stealing counter over a c10d store: ``store.add`` is an atomic fetch-add."""

    def __init__(self, store, key: str, chunks: Sequence[Sequence[int]]) -> None:
        self.store, self.key, self.chunks = store, key, [list(c) for c in chunks]

    def claim(self) -> Optional[List[int]]:
        idx = int(self.store.add(self.key, 1)) - 1
        return self.chunks[idx] if idx < len(self.chunks) else None


# Counter keys must never be reused: a key left over from an earlier frame is already past its last chunk, every
# claim on it returns None and the stealable tiles would silently stay unrendered.  So a key is made of a
# session nonce (rank 0 draws it once per store, the others read it) and a call sequence number that every rank
# advances in step (render_frame_sharded is collective); `frame_id` is only a label.  Keys two calls old are
# deleted by rank 0, and in the stealing schedule the rows all ranks rendered are added up and checked.
_SESSIONS: dict = {}
_CALL_SEQ = [0]


def _session_nonce(store, rank: int) -> str:
    sid = id(store)
    if sid not in _SESSIONS:
        if rank == 0:
            import secrets
            nonce = secrets.token_hex(8)
            store.set("raingun/session", nonce)
        else:
            nonce = bytes(store.get("raingun/session")).decode()
        _SESSIONS[sid] = nonce
    return _SESSIONS[sid]


class HostBarrier:
    """End-of-frame barrier of the ranks of one box in shared memory (rg_shm_barrier_*): a few microseconds where a
    collective on the GPUs takes 60-100.  Valid only after every rank's own device work is complete, which the
    blocking render calls guarantee.  Rank 0 creates it and publishes the name through the store."""

    def __init__(self, rank: int, world: int, store=None, tag: str = "0") -> None:
        import ctypes
        import os

        from . import _native
        self._native, self.world = _native, world
        self._h = ctypes.c_void_p()
        key = f"raingun/host_barrier/{tag}"
        store = store or (default_store() if world > 1 else None)
        if rank == 0:
            name = f"/raingun_bar_{os.getpid()}_{tag}"
            _native.check(_native.lib().rg_shm_barrier_open(name.encode(), world, 1, ctypes.byref(self._h)))
            if world > 1:
                store.set(key, name)
        else:
            name = bytes(store.get(key)).decode()
            _native.check(_native.lib().rg_shm_barrier_open(name.encode(), world, 0, ctypes.byref(self._h)))

    def wait(self) -> None:
        self._native.check(self._native.lib().rg_shm_barrier_wait(self._h))

    def close(self) -> None:
        if self._h:
            if self.world > 1:
                dist.barrier()   # nobody is still waiting on the page
            self._native.lib().rg_shm_barrier_close(self._h)
            self._h = None


class SharedHostFrame:
    """One frame in HOST memory that every rank of the box writes its rows into: a shared-memory file mapped
    and pinned (``rg_host_register``) in each process, so every GPU delivers its rows over its own PCIe link
    (``Scene.render_rowlist_host``) and nothing is gathered on one GPU first.  Two frames alternate like
    ``PeerFrames``.  Rank 0 reads the finished frame after the end-of-frame barrier."""

    def __init__(self, width: int, height: int, rank: int, world: int, store=None, tag: str = "0", pin: bool = True,
                 pixel_format: str = "rgba8") -> None:
        import os

        self.width, self.height, self.rank, self.world = width, height, rank, world
        bpp, channels, np_dtype, _ = _format(pixel_format)
        self.pixel_format = pixel_format
        self.nbytes = width * height * bpp
        self.maps, self.paths, self.pinned = [], [], []
        for k in range(2):
            key = f"raingun/host_frame/{tag}/{k}"
            if rank == 0:
                path = f"/dev/shm/raingun_{os.getpid()}_{tag}_{k}"
                with open(path, "wb") as f:
                    f.truncate(self.nbytes)
                if world > 1:
                    (store or default_store()).set(key, path)
            else:
                path = bytes((store or default_store()).get(key)).decode()
            mm = np.memmap(path, dtype=np_dtype, mode="r+", shape=(height, width, channels))
            self.maps.append(mm)
            self.paths.append(path)
            if pin:
                from . import host_register
                host_register(mm.ctypes.data, self.nbytes)
                self.pinned.append(mm.ctypes.data)

    def ptr(self, frame_id: int) -> int:
        return self.maps[frame_id & 1].ctypes.data

    def array(self, frame_id: int) -> np.ndarray:
        return self.maps[frame_id & 1]

    def close(self) -> None:
        import os

        from . import host_unregister
        if self.world > 1:
            dist.barrier()
        for p in self.pinned:
            host_unregister(p)
        self.pinned, self.maps = [], []
        if self.world > 1:
            dist.barrier()
        if self.rank == 0:
            for path in self.paths:
                try:
                    os.unlink(path)
                except OSError:
                    pass


class PeerFrames:
    """Rank 0's frame buffers as every rank of the box sees them (CUDA IPC, written over NVLink).
    Two frames alternate (``frame_id & 1``): a rank that is already storing rows of frame k+1 cannot
    disturb rank 0 still reading frame k, and the end-of-frame barrier keeps everyone within one
    frame of each other."""

    def __init__(self, width: int, height: int, rank: int, world: int, device_index: int, store=None,
                 tag: str = "0", pixel_format: str = "rgba8") -> None:
        from . import SharedFrame

        self.width, self.height, self.rank, self.world, self.device_index = width, height, rank, world, device_index
        self.pixel_format = pixel_format
        nbytes = width * height * bytes_per_pixel(pixel_format)
        self.frames = []
        for k in range(2):
            key = f"raingun/peer_frame/{tag}/{k}"
            if rank == 0:
                try:
                    f = SharedFrame.create(device_index, nbytes)
                except Exception:
                    if world > 1:   # never leave the peers blocked on the key
                        (store or default_store()).set(key, b"!")
                    raise
                if world > 1:
                    (store or default_store()).set(key, f.handle)
            else:
                handle = bytes((store or default_store()).get(key))
                if len(handle) != 64:
                    raise RuntimeError("rank 0 could not create the shared frame")
                f = SharedFrame.open(device_index, handle, nbytes)
            self.frames.append(f)

    def ptr(self, frame_id: int) -> int:
        return self.frames[frame_id & 1].ptr

    def tensor(self, frame_id: int) -> torch.Tensor:
        """Zero-copy (H, W, 4) uint8 or (H, W, 3) float32 view of the frame (meaningful on rank 0, which owns the
        memory)."""
        t = torch.as_tensor(self.frames[frame_id & 1], device=torch.device("cuda", self.device_index))
        return frame_view(t, self.height, self.width, self.pixel_format)

    def close(self, sync: bool = True) -> None:
        """``sync=False`` only when no peer can be using the frames (e.g. set-up failed on some rank)."""
        sync = sync and self.world > 1
        if sync:
            dist.barrier()   # nobody unmaps or frees while a peer may still be storing
        for f in self.frames:
            if not f.owner:
                f.close()
        if sync:
            dist.barrier()
        for f in self.frames:
            if f.owner:
                f.close()
        self.frames = []


@dataclass
class ShardResult:
    frame: Optional[torch.Tensor]          # (H, W, 4) uint8 or (H, W, 3) float32 on rank 0, None elsewhere
    my_tiles: List[int] = field(default_factory=list)
    claims: int = 0
    schedule: str = ""                     # the schedule actually used ("auto" resolved)
    stats: list = field(default_factory=list)   # whatever render_rowlist returned, per call
    rows_seen: int = 0                     # steal schedule: rows all ranks had reported when this rank finished
    rows_total_key: str = ""


def default_store():
    return dist.distributed_c10d._get_default_store()


def render_frame_sharded(render_rowlist: Union[Callable[[np.ndarray, torch.Tensor], object], Sequence[Callable]],
                         width: int, height: int,
                         rank: int, world: int, frame_id: int, device: torch.device, store=None,
                         tile_rows: int = DEFAULT_TILE_ROWS, schedule: str = "auto",
                         gather: bool = True, staging: Optional[torch.Tensor] = None,
                         gather_mode: str = "reduce", frame_buf: Optional[torch.Tensor] = None,
                         lead: float = 0.6, peer_frames: Optional[PeerFrames] = None,
                         host_barrier: Optional["HostBarrier"] = None, pixel_format: str = "rgba8") -> ShardResult:
    """Renders one frame across ``world`` ranks.

    ``render_rowlist(rows, out)`` must fill ``out`` (a uint8 tensor of ``len(rows)*row_bytes``
    bytes on ``device``, ``row_bytes = width * bytes_per_pixel(pixel_format)``) with the listed image rows,
    compacted in list order, and return once they are there — on a GPU that is ``Scene.render_rowlist_device``
    (``"rgba8"``) or ``Scene.render_rowlist_f32_device`` (``"f32"``).  A LIST of such callables keeps
    that many batches in flight on this rank (one host thread each; see the module docstring).
    ``schedule`` is ``"steal"`` (static interleaved share first, then the
    work-stealing counter for the tail — see ``hybrid_plan``), ``"static"`` (interleaved
    ownership only, one batch per rank) or ``"auto"`` (static when every rank owns at least
    ``AUTO_STATIC_MIN_TILES_PER_RANK`` tiles, else steal).

    ``gather_mode``: ``"peer"`` — needs ``peer_frames``; the renderers are then called as
    ``render_rowlist(rows, frame_ptr)`` and must store row ``rows[k]`` at ``frame_ptr + rows[k]*row_bytes``
    (``Scene.render_rowlist_scatter`` / ``render_rowlist_f32_scatter``); the frame is complete on rank 0 after one
    barrier.
    ``"host"`` — as ``"peer"`` with ``peer_frames`` a ``SharedHostFrame``: the renderers
    (``Scene.render_rowlist_host`` / ``render_rowlist_f32_host``) copy every row to its place in ONE pinned host frame all ranks map, each GPU
    over its own PCIe link; the frame is complete in rank 0's host memory after one barrier.
    ``"reduce"`` — every rank scatters its rows into a zeroed full frame and ONE
    NCCL reduce (MAX over disjoint rows, i.e. a gather that needs no ownership exchange) lands the
    frame on rank 0 over NVLink; ``"p2p"`` — the row lists travel through the store and rank 0
    receives each rank's packed rows point to point.  ``"peer"``, ``"host"`` and ``"p2p"`` move bytes and serve
    either ``pixel_format``; ``"reduce"`` is RGBA8 only (a MAX over zero-filled rows does not carry the f32 NaN
    bits the reference's colours can hold) and raises ``ValueError`` for ``"f32"`` before any collective.
    """
    row_bytes = width * bytes_per_pixel(pixel_format)
    if gather and gather_mode == "reduce" and pixel_format != "rgba8":
        raise ValueError(f"gather_mode='reduce' cannot gather pixel_format={pixel_format!r}: a MAX reduction does not "
                         "carry NaN bits; use 'p2p', 'peer' or 'host'")
    nt = n_tiles(height, tile_rows)
    schedule = resolve_schedule(schedule, nt, world)
    res = ShardResult(frame=None, schedule=schedule)
    renderers = list(render_rowlist) if isinstance(render_rowlist, (list, tuple)) else [render_rowlist]
    workers = len(renderers)
    host = gather_mode == "host"     # like "peer", but the shared frame lives in pinned host memory (SharedHostFrame)
    peer = gather_mode == "peer" or host
    if peer and peer_frames is None:
        raise ValueError(f"gather_mode={gather_mode!r} needs peer_frames")
    if staging is None and not peer:
        staging = torch.empty((height * row_bytes,), dtype=torch.uint8, device=device)
    # first[k]: the batch worker k starts with (no counter traffic); claim(): the stealable rest
    if world == 1:
        first = split_share(list(range(nt)), workers)
        claim = lambda: None
    elif schedule == "steal":
        if store is None:
            store = default_store()
        per_rank, tail_chunks = hybrid_plan(nt, world, min_chunk=2 if workers == 1 else 1)
        _CALL_SEQ[0] += 1
        seq = _CALL_SEQ[0]
        prefix = f"raingun/{_session_nonce(store, rank)}"
        steal_key = f"{prefix}/tiles/{seq}"
        counter = TileCounter(store, steal_key, tail_chunks)
        first = split_share(per_rank[rank], workers, lead)
        claim = counter.claim
    elif schedule == "static":
        first = split_share(static_chunk(nt, world, rank), workers)
        claim = lambda: None
    else:
        raise ValueError(f"unknown schedule {schedule!r}")

    lock, claim_lock = threading.Lock(), threading.Lock()
    state = {"filled": 0}
    my_rows: List[np.ndarray] = []

    def run_worker(k: int) -> None:
        tiles = first[k]
        while tiles is not None:
            if tiles:
                rows = rows_of_tiles(tiles, tile_rows, height)
                with lock:   # reserve the output rows of this batch
                    at = state["filled"]
                    state["filled"] = at + int(rows.size)
                if peer:
                    stat = renderers[k](rows, peer_frames.ptr(frame_id))
                else:
                    out = staging[at * row_bytes:(at + int(rows.size)) * row_bytes]
                    stat = renderers[k](rows, out)
                with lock:
                    res.claims += 1
                    res.stats.append(stat)
                    res.my_tiles.extend(tiles)
                    my_rows.append((at, rows))
            with claim_lock:   # one store round trip at a time per rank
                tiles = claim()

    if workers == 1:
        run_worker(0)
    else:
        for f in [_pool(workers).submit(run_worker, k) for k in range(workers)]:
            f.result()
    filled_rows = state["filled"]
    my_rows = [r for _, r in sorted(my_rows, key=lambda ar: ar[0])]   # staging order
    rows_all = np.concatenate(my_rows) if my_rows else np.zeros(0, np.uint32)
    if world > 1 and schedule == "steal":
        # every row must have been rendered by exactly one rank: add up what the ranks did (the barrier of the
        # gather below — or the caller's — orders the read after every rank's add), drop counters two calls old
        total = int(store.add(f"{prefix}/rows/{seq}", int(rows_all.size)))
        res.rows_total_key = f"{prefix}/rows/{seq}"
        if rank == 0 and seq > 2:
            for old_key in (f"{prefix}/tiles/{seq - 2}", f"{prefix}/rows/{seq - 2}"):
                try:
                    store.delete_key(old_key)
                except Exception:   # not every store can delete
                    pass
        res.rows_seen = total   # a lower bound until every rank has added; checked after the barrier
    if not gather:
        return res
    def check_all_rows_rendered():
        if world > 1 and schedule == "steal":
            total = int(store.add(res.rows_total_key, 0))
            if total != height:
                raise RuntimeError(f"sharded frame {frame_id}: the ranks rendered {total} rows of {height} "
                                   "(work-stealing counter out of step)")

    if peer:   # the rows are already in rank 0's frame (GPU memory, or pinned host memory); make that known
        if world > 1:
            if host_barrier is not None:   # every rank's render call has synchronised its own stream: a CPU barrier is enough
                host_barrier.wait()
            else:
                dist.barrier()
        check_all_rows_rendered()
        if host:
            res.frame = torch.from_numpy(peer_frames.array(frame_id)) if rank == 0 else None
        else:
            res.frame = peer_frames.tensor(frame_id) if rank == 0 else None
        return res

    # ---- gather: ownership is dynamic, so the row lists travel first (tiny), then the pixels
    packed = staging[: filled_rows * row_bytes]
    if world == 1:
        frame = packed if np.array_equal(rows_all, np.arange(height)) else \
            _scatter_rows(torch.empty((height, row_bytes), dtype=torch.uint8, device=device), rows_all, packed, width)
        res.frame = frame_view(frame, height, width, pixel_format)
        return res
    if gather_mode == "reduce":
        frame = frame_buf if frame_buf is not None else torch.empty((height, width, 4), dtype=torch.uint8, device=device)
        frame.zero_()
        _scatter_rows(frame, rows_all, packed, width)
        dist.reduce(frame, dst=0, op=dist.ReduceOp.MAX)
        res.frame = frame if rank == 0 else None
        if rank == 0:
            check_all_rows_rendered()
        return res
    if store is None:
        store = default_store()
    store.set(f"raingun/rows/{frame_id}/{rank}", pickle.dumps(rows_all))
    if rank == 0:
        frame = torch.empty((height, row_bytes), dtype=torch.uint8, device=device)
        _scatter_rows(frame, rows_all, packed, width)
        lists = {r: pickle.loads(store.get(f"raingun/rows/{frame_id}/{r}")) for r in range(1, world)}
        recv_bufs, ops = {}, []
        for r, rl in lists.items():
            if rl.size:
                recv_bufs[r] = torch.empty((int(rl.size) * row_bytes,), dtype=torch.uint8, device=device)
                ops.append(dist.P2POp(dist.irecv, recv_bufs[r], r))
        if ops:
            for req in dist.batch_isend_irecv(ops):
                req.wait()
        for r, buf in recv_bufs.items():
            _scatter_rows(frame, lists[r], buf, width)
        res.frame = frame_view(frame, height, width, pixel_format)
        check_all_rows_rendered()
    elif filled_rows:
        for req in dist.batch_isend_irecv([dist.P2POp(dist.isend, packed, 0)]):
            req.wait()
    return res


_IDX_CACHE: dict = {}


def _scatter_rows(frame: torch.Tensor, rows: np.ndarray, packed: torch.Tensor, width: int) -> torch.Tensor:
    """Copies packed row ``k`` to row ``rows[k]`` of ``frame`` (contiguous, one image row per index of dim 0; rows
    are moved as bytes, whatever the pixel format)."""
    if rows.size:
        key = (str(frame.device), rows.tobytes())   # static ownership repeats every frame: keep the index on the device
        idx = _IDX_CACHE.get(key)
        if idx is None:
            if len(_IDX_CACHE) > 64:
                _IDX_CACHE.clear()
            idx = _IDX_CACHE[key] = torch.from_numpy(rows.astype(np.int64)).to(frame.device)
        frame.view(frame.shape[0], -1).index_copy_(0, idx, packed.view(int(rows.size), -1))
    return frame
