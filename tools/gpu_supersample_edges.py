"""The cost of edge-adaptive anti-aliasing (RG_OPT_SUPERSAMPLE_EDGES = T with RG_OPT_SUPERSAMPLE = n) against the full
n x n frame and the n = 1 frame.

    python tools/gpu_supersample_edges.py [--cases C4:3840x2160,C3:3840x2160,test1:800x600,test1:3840x2160]
                                          [--factors 2,4] [--thresholds 0,4,16,64] [--out r.json]

Per scene and setting: ms per frame device-resident (rg_render_rows_device, host clock around the call and a device
synchronise; median of --frames after --warmup, graphs on), the refined share ((rays_primary - w h) / (n n w h)),
rays, Grays/s, launches, batches, graph replays, CRC of the frame.  Then, in a separate run under torch.profiler, the
device time per frame of the mask kernels (k_edge_emit, k_edge_scan, k_edge_compact).  The card's name, power limit
and max SM clock are printed first."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

MASK_KERNELS = ("k_edge_emit", "k_edge_scan", "k_edge_compact")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="C4:3840x2160,C3:3840x2160,test1:800x600,test1:3840x2160")
    ap.add_argument("--factors", default="2,4")
    ap.add_argument("--thresholds", default="0,4,16,64")
    ap.add_argument("--frames", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--prof-frames", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    import raingun_b200 as rg
    from raingun_b200.examples import bundled_texture_loader, example_scene
    from raingun_b200.synth import make_scene

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    print("card (name, power limit, max SM clock):", q, flush=True)
    factors = [int(x) for x in a.factors.split(",") if x]
    thresholds = [int(x) for x in a.thresholds.split(",") if x]
    stream = torch.cuda.current_stream().cuda_stream
    res = {"card": q, "runs": []}
    for case in a.cases.split(","):
        name, size = case.split(":")
        w, h = map(int, size.split("x"))
        data = (example_scene(name) if name.startswith("test")
                else make_scene(name, texture_loader=bundled_texture_loader)[0])
        out = torch.empty(w * h * 4, dtype=torch.uint8, device="cuda")
        settings = [(1, None)] + [(n, t) for n in factors for t in [None] + thresholds]
        with rg.Scene(data) as sc:
            for n, t in settings:
                sc.set_supersample(n)
                sc.set_supersample_edges(t)
                for _ in range(a.warmup):
                    sc.render_rows_device(w, h, 0, h, out.data_ptr(), stream)
                ms = []
                for _ in range(a.frames):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    st = sc.render_rows_device(w, h, 0, h, out.data_ptr(), stream)
                    torch.cuda.synchronize()
                    ms.append((time.perf_counter() - t0) * 1e3)
                med = statistics.median(ms)
                r = {"scene": name, "width": w, "height": h, "n": n, "T": t, "ms": ms, "median_ms": med,
                     "refined_share": (st.rays_primary - w * h) / (n * n * w * h) if t is not None else (1.0 if n > 1 else 0.0),
                     "rays": st.rays, "rays_primary": st.rays_primary, "grays_per_s": st.rays / (med * 1e-3) / 1e9,
                     "launches": st.gpu_launches, "batches": st.batches, "graph_replays": st.graph_replays,
                     "pipeline": st.pipeline_used, "accel": st.accel_used,
                     "crc32": "%08x" % zlib.crc32(out.cpu().numpy().tobytes())}
                if t is not None:   # the mask kernels alone, in a run of their own under the profiler
                    torch.cuda.synchronize()
                    with profile(activities=[ProfilerActivity.CUDA]) as prof:
                        for _ in range(a.prof_frames):
                            sc.render_rows_device(w, h, 0, h, out.data_ptr(), stream)
                        torch.cuda.synchronize()
                    us = sum(e.duration_ns() / 1e3 for e in prof.profiler.kineto_results.events()
                             if e.device_type() == torch.autograd.DeviceType.CUDA and any(k in e.name() for k in MASK_KERNELS))
                    r["mask_ms_per_frame"] = us / 1e3 / a.prof_frames
                res["runs"].append(r)
                print(json.dumps(r), flush=True)
    print("%-6s %10s %2s %4s %9s %7s %13s %8s %8s %7s %7s %8s" % ("scene", "size", "n", "T", "ms/frame", "share", "rays",
                                                                 "Grays/s", "launches", "batches", "replays", "mask ms"))
    for r in res["runs"]:
        print("%-6s %10s %2d %4s %9.2f %7.3f %13d %8.2f %8d %7d %7d %8s" % (
            r["scene"], "%dx%d" % (r["width"], r["height"]), r["n"], "-" if r["T"] is None else r["T"], r["median_ms"],
            r["refined_share"], r["rays"], r["grays_per_s"], r["launches"], r["batches"], r["graph_replays"],
            "%.3f" % r["mask_ms_per_frame"] if "mask_ms_per_frame" in r else "-"), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
