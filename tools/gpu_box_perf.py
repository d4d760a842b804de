"""B4 (10,000 boxes and disks, raingun_b200.synth.make_box_scene) on the grid and by brute force, and C4 / C3
timed with this build and with another build of the library, alternating, in one run.

    python tools/gpu_box_perf.py [--baseline-lib path/to/libraingun_b200.so] [--out result.json]

Every number is device time per frame (rg_stats.ms_device) of a warm scene, the median of --frames frames.
Each (build, scene) measurement runs in a fresh process because a process loads one library
(RAINGUN_B200_LIB selects it).  The card's name and power limit are recorded with the numbers."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def worker(scene, width, height, accel, frames, warmup):
    sys.path.insert(0, ROOT)
    import raingun_b200 as rg
    from raingun_b200.examples import bundled_texture_loader
    from raingun_b200.synth import make_box_scene, make_scene

    data = (make_box_scene(scene) if scene == "B4" else make_scene(scene, texture_loader=bundled_texture_loader))[0]
    with rg.Scene(data) as sc:
        sc.set_accel({"grid": rg.ACCEL_GRID, "brute": rg.ACCEL_BRUTE}[accel])
        for _ in range(warmup):
            sc.render_image(width, height)
        ms = []
        for _ in range(frames):
            sc.render_image(width, height)
            ms.append(sc.last_stats.ms_device)
        st = sc.last_stats
    print(json.dumps({"ms": ms, "rays": st.rays, "exact_tests": st.exact_tests, "accel_used": st.accel_used}))


def run(lib, scene, width, height, accel, frames, warmup):
    env = dict(os.environ)
    if lib:
        env["RAINGUN_B200_LIB"] = os.path.abspath(lib)
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", scene, str(width), str(height), accel,
                        str(frames), str(warmup)], env=env, capture_output=True, text=True, check=True)
    res = json.loads(r.stdout.strip().splitlines()[-1])
    res.update(scene=scene, width=width, height=height, accel=accel, lib=lib or "this build",
               median_ms=statistics.median(res["ms"]))
    print(json.dumps({k: v for k, v in res.items() if k != "ms"}), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worker", nargs=6)
    ap.add_argument("--baseline-lib", default="")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--frames", type=int, default=5)
    ap.add_argument("--brute-res", default="640x360")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if a.worker:
        s, w, h, acc, f, wu = a.worker
        return worker(s, int(w), int(h), acc, int(f), int(wu))

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    print("card:", q, flush=True)
    out = {"card": q, "runs": []}
    bw, bh = map(int, a.brute_res.split("x"))
    out["runs"].append(run("", "B4", 3840, 2160, "grid", a.frames, 2))
    out["runs"].append(run("", "B4", bw, bh, "grid", a.frames, 2))
    out["runs"].append(run("", "B4", bw, bh, "brute", 2, 1))
    g, b = out["runs"][1], out["runs"][2]
    out["b4_speedup_rays_per_s"] = (g["rays"] / g["median_ms"]) / (b["rays"] / b["median_ms"])
    print("B4 %dx%d: grid %.3f ms, brute %.1f ms: %.0fx (rays/s)" % (bw, bh, g["median_ms"], b["median_ms"],
                                                                     out["b4_speedup_rays_per_s"]), flush=True)
    if a.baseline_lib:
        for _ in range(a.rounds):
            for lib in (a.baseline_lib, ""):
                for scene in ("C4", "C3"):
                    out["runs"].append(run(lib, scene, 3840, 2160, "grid", a.frames, 2))
        for scene in ("C4", "C3"):
            for lib in (a.baseline_lib, ""):
                meds = [r["median_ms"] for r in out["runs"] if r["scene"] == scene and r["lib"] == (lib or "this build")]
                print("%s %s: median of rounds %.3f ms, range %.3f-%.3f" % (scene, lib or "this build", statistics.median(meds),
                                                                           min(meds), max(meds)), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
