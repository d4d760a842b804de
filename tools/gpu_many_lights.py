"""The cost of many lights: the many-light scene (raingun_b200.synth.make_light_scene: C4's 10,000 mixed spheres, L
lights) at 3840x2160 for L in --lights, and optionally C4 and the shipped examples at 800x600 with this build and
another build of the library, alternating.

    python tools/gpu_many_lights.py [--lights 3,8,32,33,64,128] [--baseline-lib path/to/libraingun_b200.so] [--out r.json]

Frames are rendered into device memory (rg_render_rows_device); times are rg_stats.ms_device, the median of --frames
frames after --warmup frames.  Each (build, scene) measurement runs in a fresh process because a process loads one
library (RAINGUN_B200_LIB selects it).  The card's name and power limit are printed with the numbers."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def worker(scene, width, height, frames, warmup):
    sys.path.insert(0, ROOT)
    import torch

    import raingun_b200 as rg
    from raingun_b200.examples import bundled_texture_loader, example_scene
    from raingun_b200.synth import make_light_scene, make_scene

    if scene.startswith("L"):
        data = make_light_scene(int(scene[1:]), texture_loader=bundled_texture_loader)[0]
    elif scene.startswith("C"):
        data = make_scene(scene, texture_loader=bundled_texture_loader)[0]
    else:
        data = example_scene(scene)
    out = torch.empty(width * height * 4, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream
    with rg.Scene(data) as sc:
        for _ in range(warmup):
            sc.render_rows_device(width, height, 0, height, out.data_ptr(), stream)
        ms = []
        for _ in range(frames):
            st = sc.render_rows_device(width, height, 0, height, out.data_ptr(), stream)
            ms.append(st.ms_device)
        torch.cuda.synchronize()
        crc = zlib.crc32(out.cpu().numpy().tobytes())
    print(json.dumps({"ms": ms, "rays": st.rays, "rays_shadow": st.rays_shadow, "launches": st.gpu_launches,
                      "batches": st.batches, "graph_replays": st.graph_replays, "pipeline": st.pipeline_used,
                      "crc32": "%08x" % crc}))


def run(lib, scene, width, height, frames, warmup):
    env = dict(os.environ)
    if lib:
        env["RAINGUN_B200_LIB"] = os.path.abspath(lib)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", scene, str(width), str(height), str(frames),
                        str(warmup)], env=env, capture_output=True, text=True)
    if r.returncode:
        sys.stderr.write(r.stderr)
        r.check_returncode()
    res = json.loads(r.stdout.strip().splitlines()[-1])
    res.update(scene=scene, width=width, height=height, lib=lib or "this build", median_ms=statistics.median(res["ms"]),
               spread_ms=max(res["ms"]) - min(res["ms"]))
    res["shadow_rays_per_s"] = res["rays_shadow"] / (res["median_ms"] * 1e-3)
    print(json.dumps({k: v for k, v in res.items() if k != "ms"}), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worker", nargs=5)
    ap.add_argument("--lights", default="3,8,32,33,64,128")
    ap.add_argument("--res", default="3840x2160")
    ap.add_argument("--frames", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--baseline-lib", default="")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if a.worker:
        s, w, h, f, wu = a.worker
        return worker(s, int(w), int(h), int(f), int(wu))

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    print("card:", q, flush=True)
    out = {"card": q, "runs": []}
    w, h = map(int, a.res.split("x"))
    for n in [int(x) for x in a.lights.split(",") if x]:
        out["runs"].append(run("", "L%d" % n, w, h, a.frames, a.warmup))
    print("%6s %10s %12s %12s %14s %9s %8s %8s %9s" % ("lights", "ms/frame", "rays", "shadow", "shadow/s", "launches",
                                                      "batches", "replays", "crc32"))
    for r in out["runs"]:
        print("%6s %10.2f %12d %12d %14.4g %9d %8d %8d %9s" % (r["scene"][1:], r["median_ms"], r["rays"], r["rays_shadow"],
                                                              r["shadow_rays_per_s"], r["launches"], r["batches"],
                                                              r["graph_replays"], r["crc32"]), flush=True)
    if a.baseline_lib:
        scenes = ("C4", "test1", "test2", "test3")
        for _ in range(a.rounds):
            for lib in (a.baseline_lib, ""):
                for scene in scenes:
                    out["runs"].append(run(lib, scene, 800, 600, 10, 3))
        for scene in scenes:
            for lib in (a.baseline_lib, ""):
                rs = [r for r in out["runs"] if r["scene"] == scene and r["lib"] == (lib or "this build")]
                meds = [r["median_ms"] for r in rs]
                print("%s 800x600 %s: median of rounds %.3f ms, range %.3f-%.3f, crc32 %s" % (
                    scene, lib or "this build", statistics.median(meds), min(meds), max(meds),
                    ",".join(sorted({r["crc32"] for r in rs}))), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
