"""The cost of anti-aliasing: C4 (raingun_b200.synth.make_scene("C4"), 10,000 mixed spheres) at 3840x2160 with
RG_OPT_SUPERSAMPLE = n for each n in --factors (n x n primary rays per pixel, averaged on the GPU).

    python tools/gpu_supersample.py [--factors 1,2,3,4] [--res 3840x2160] [--out r.json]

Frames are rendered into device memory (rg_render_rows_device); times are rg_stats.ms_device, the median of --frames
frames after --warmup frames, on one handle per n.  The card's name and power limit are printed with the numbers."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--factors", default="1,2,3,4")
    ap.add_argument("--res", default="3840x2160")
    ap.add_argument("--frames", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="")
    a = ap.parse_args()

    import torch

    import raingun_b200 as rg
    from raingun_b200.examples import bundled_texture_loader
    from raingun_b200.synth import make_scene

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    print("card:", q, flush=True)
    w, h = map(int, a.res.split("x"))
    data = make_scene("C4", texture_loader=bundled_texture_loader)[0]
    out = torch.empty(w * h * 4, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    res = {"card": q, "width": w, "height": h, "runs": []}
    for n in [int(x) for x in a.factors.split(",") if x]:
        with rg.Scene(data) as sc:
            sc.set_supersample(n)
            for _ in range(a.warmup):
                sc.render_rows_device(w, h, 0, h, out.data_ptr(), stream)
            ms = []
            for _ in range(a.frames):
                st = sc.render_rows_device(w, h, 0, h, out.data_ptr(), stream)
                ms.append(st.ms_device)
            torch.cuda.synchronize()
            crc = zlib.crc32(out.cpu().numpy().tobytes())
        med = statistics.median(ms)
        r = {"n": n, "ms": ms, "median_ms": med, "rays": st.rays, "rays_primary": st.rays_primary,
             "grays_per_s": st.rays / (med * 1e-3) / 1e9, "launches": st.gpu_launches, "batches": st.batches,
             "graph_replays": st.graph_replays, "pipeline": st.pipeline_used, "crc32": "%08x" % crc}
        res["runs"].append(r)
        print(json.dumps(r), flush=True)
    print("%3s %10s %14s %12s %9s %8s %8s %9s" % ("n", "ms/frame", "rays", "Grays/s", "launches", "batches", "replays",
                                                 "crc32"))
    for r in res["runs"]:
        print("%3d %10.2f %14d %12.3f %9d %8d %8d %9s" % (r["n"], r["median_ms"], r["rays"], r["grays_per_s"], r["launches"],
                                                          r["batches"], r["graph_replays"], r["crc32"]), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
