"""What the f32 output kinds cost: C4 (raingun_b200.synth.make_scene("C4"), 10,000 mixed spheres) at 3840x2160,
device-resident, delivered as RGBA8 (4 bytes per pixel) and as unquantised f32 RGB (12 bytes per pixel).

    python tools/gpu_f32_device.py [--res 3840x2160] [--frames 5] [--warmup 2] [--out r.json]

Kinds, one handle each (wavefront pipeline, grid tracer, as the scene's AUTO choice):
  rows_device           rg_render_rows_device, the whole frame into HBM (RGBA8)
  rows_f32_device       rg_render_rows_f32_device, the same in f32
  rowlist_scatter       rg_render_rowlist_scatter, an interleaved 1/8 share (every 8th 8-row tile: one GPU of eight)
                        stored at its place in a full RGBA8 frame
  rowlist_f32_scatter   rg_render_rowlist_f32_scatter, the same share into a full f32 frame
  rowlist_f32_host      rg_render_rowlist_f32_host, the whole frame into a pinned host frame (one copy per run of rows)
For each: the median over --frames frames after --warmup frames of the call's wall time (the call returns when the
work is done) and of rg_stats.ms_device, the bytes of the destination frame, and a CRC of it.  Then the last kernel of
a batch (k_quantise, k_export_f32, k_quantise_scatter, k_export_f32_scatter) alone: every frame of a second pass runs
with CUDA graphs off under torch.profiler, which records each launch's device duration; the median per launch is
printed.  The card's name, power limit and maximum SM clock are read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LAST_KERNEL = {"rows_device": "k_quantise(", "rows_f32_device": "k_export_f32(", "rowlist_scatter": "k_quantise_scatter(",
               "rowlist_f32_scatter": "k_export_f32_scatter("}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--res", default="3840x2160")
    ap.add_argument("--frames", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--kernel-frames", type=int, default=20)
    ap.add_argument("--out", default="")
    a = ap.parse_args()

    import torch

    import raingun_b200 as rg
    from raingun_b200.dist import rows_of_tiles
    from raingun_b200.examples import bundled_texture_loader
    from raingun_b200.synth import make_scene

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    print("card:", q, flush=True)
    w, h = map(int, a.res.split("x"))
    data = make_scene("C4", texture_loader=bundled_texture_loader)[0]
    share = rows_of_tiles(list(range(0, (h + 7) // 8, 8)), 8, h)   # tile t of 8 rows belongs to GPU t mod 8
    stream = torch.cuda.current_stream().cuda_stream
    rgba = torch.zeros(h * w * 4, dtype=torch.uint8, device="cuda")
    f32 = torch.zeros(h * w * 12, dtype=torch.uint8, device="cuda")
    host = np.zeros(h * w * 12, np.uint8)
    rg.host_register(host.ctypes.data, host.nbytes)
    calls = {
        "rows_device": (rgba, lambda sc: sc.render_rows_device(w, h, 0, h, rgba.data_ptr(), stream)),
        "rows_f32_device": (f32, lambda sc: sc.render_rows_f32_device(w, h, 0, h, f32.data_ptr(), stream)),
        "rowlist_scatter": (rgba, lambda sc: sc.render_rowlist_scatter(w, h, share, rgba.data_ptr(), stream)),
        "rowlist_f32_scatter": (f32, lambda sc: sc.render_rowlist_f32_scatter(w, h, share, f32.data_ptr(), stream)),
        "rowlist_f32_host": (host, lambda sc: sc.render_rowlist_f32_host(w, h, np.arange(h, dtype=np.uint32), host.ctypes.data)),
    }
    res = {"card": q, "width": w, "height": h, "share_rows": int(share.size), "runs": []}
    f32_frame = None
    try:
        for kind, (buf, call) in calls.items():
            if isinstance(buf, torch.Tensor):
                buf.zero_()
            else:
                buf[:] = 0
            torch.cuda.synchronize()
            with rg.Scene(data) as sc:
                for _ in range(a.warmup):
                    call(sc)
                wall, dev = [], []
                for _ in range(a.frames):
                    t0 = time.perf_counter()
                    st = call(sc)
                    wall.append((time.perf_counter() - t0) * 1e3)
                    dev.append(st.ms_device)
            torch.cuda.synchronize()
            frame = buf.cpu().numpy() if isinstance(buf, torch.Tensor) else buf
            if kind == "rows_f32_device":
                f32_frame = frame.copy()
            same = None
            if kind in ("rowlist_f32_scatter", "rowlist_f32_host") and f32_frame is not None:
                rows = share if kind == "rowlist_f32_scatter" else np.arange(h)
                same = bool(np.array_equal(frame.reshape(h, -1)[rows], f32_frame.reshape(h, -1)[rows]))
            r = {"kind": kind, "wall_ms": wall, "ms_device": dev, "median_ms": statistics.median(wall),
                 "median_ms_device": statistics.median(dev), "frame_bytes": int(frame.nbytes),
                 "rows": int(share.size) if "scatter" in kind else h, "rays": st.rays, "launches": st.gpu_launches,
                 "batches": st.batches, "graph_replays": st.graph_replays, "pipeline": st.pipeline_used,
                 "crc32": "%08x" % zlib.crc32(frame.tobytes()), "f32_bits_equal_rows_f32_device": same}
            res["runs"].append(r)
            print(json.dumps(r), flush=True)

        # the last kernel alone: eager launches (graphs off) under the profiler, every launch's device time
        from torch.profiler import ProfilerActivity, profile
        kernel_us = {}
        for kind, name in LAST_KERNEL.items():
            with rg.Scene(data) as sc:
                sc.set_option(rg._native.OPT_GRAPH, 1)
                calls[kind][1](sc)
                torch.cuda.synchronize()
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(a.kernel_frames):
                        calls[kind][1](sc)
                    torch.cuda.synchronize()
            durs = [e.duration_ns() / 1e3 for e in prof.profiler.kineto_results.events()
                    if name in e.name() and e.device_type() == torch.autograd.DeviceType.CUDA]
            kernel_us[kind] = {"kernel": name.rstrip("("), "launches": len(durs),
                               "median_us": statistics.median(durs) if durs else None}
            print(json.dumps({"last_kernel": kind, **kernel_us[kind]}), flush=True)
        res["last_kernel"] = kernel_us
    finally:
        rg.host_unregister(host.ctypes.data)

    print("%-20s %10s %10s %12s %6s %9s %12s" % ("kind", "ms/frame", "ms_device", "frame MB", "rows", "crc32",
                                                 "last kernel us"))
    for r in res["runs"]:
        k = res["last_kernel"].get(r["kind"], {}).get("median_us")
        print("%-20s %10.3f %10.3f %12.1f %6d %9s %12s" % (r["kind"], r["median_ms"], r["median_ms_device"],
                                                           r["frame_bytes"] / 1e6, r["rows"], r["crc32"],
                                                           "-" if k is None else "%.1f" % k), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
