"""Shadow rays through per-light light grids: what the any-hit trace costs with and without them.

For each workload (default C4): per-ray walk counters of the any-hit and the nearest-hit launches separately
(RG_OPT_TRACE_STATS = 2 / 3), exact tests per frame, the per-launch kernel times of one frame (torch.profiler), the
scene-upload time, and a short timed loop, each with RG_OPT_LIGHT_GRIDS on and off.  Prints the card's name, power
limit and clocks first.  Usage: python tools/gpu_light_grids.py [C4 C5 ...]"""
import collections
import subprocess
import sys
import time

sys.path.insert(0, ".")
import torch

import raingun_b200 as rg
from raingun_b200 import _native as N
from raingun_b200.examples import bundled_texture_loader
from raingun_b200.synth import make_scene

OPT_LIGHT_GRIDS = getattr(N, "OPT_LIGHT_GRIDS", None)
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,clocks.mem", "--format=csv"],
                     capture_output=True, text=True).stdout.strip())


def scene(sd, light_grids):
    sc = rg.Scene(sd)
    sc.set_option(N.OPT_GRAPH, 1)
    if OPT_LIGHT_GRIDS is not None:
        sc.set_option(OPT_LIGHT_GRIDS, light_grids)
    return sc


def walk_counters(sd, w, h, out, light_grids):
    res = {}
    for mode, kind in ((2, "any-hit"), (3, "nearest-hit")):
        with scene(sd, light_grids) as sc:
            sc.set_option(N.OPT_TRACE_STATS, mode)
            st = sc.render_rows_device(w, h, 0, h, out.data_ptr(), 0)
        r = st.rays_shadow if mode == 2 else st.rays - st.rays_shadow
        res[kind] = (r, st.grid_cells / r, st.grid_fetches / r, st.grid_culls / r)
    return res, st.exact_tests


def launch_times(sd, w, h, out, light_grids):
    from torch.profiler import ProfilerActivity, profile

    with scene(sd, light_grids) as sc:
        for _ in range(2):
            sc.render_rows_device(w, h, 0, h, out.data_ptr(), 0)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            sc.render_rows_device(w, h, 0, h, out.data_ptr(), 0)
            torch.cuda.synchronize()
    per = collections.defaultdict(list)
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and "k_" in e.name:
            name = e.name
            if "k_trace_grid" in name:
                name = "k_trace_grid<any-hit>" if "k_trace_grid<true" in name else "k_trace_grid<nearest>"
            else:
                name = name.split("(")[0].split("<")[0].replace("void ", "").replace("rg::", "")
            per[name].append(e.device_time_total / 1000.0)
    return per


def timed(sd, w, h, out, light_grids, steps=20):
    with scene(sd, light_grids) as sc:
        for _ in range(3):
            sc.render_rows_device(w, h, 0, h, out.data_ptr(), 0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            sc.render_rows_device(w, h, 0, h, out.data_ptr(), 0)
        torch.cuda.synchronize()
        ms = (time.perf_counter() - t0) * 1e3 / steps
        frame = out.clone()
    return ms, frame


def upload_ms(sd, light_grids, reps=5):
    best = 1e30
    for _ in range(reps):
        t0 = time.perf_counter()
        with scene(sd, light_grids):
            best = min(best, (time.perf_counter() - t0) * 1e3)
    return best


for name in (sys.argv[1:] or ["C4"]):
    sd, spec = make_scene(name, texture_loader=bundled_texture_loader)
    w, h = spec.width, spec.height
    out = torch.empty(h * w * 4, dtype=torch.uint8, device="cuda")
    settings = (1, 0) if OPT_LIGHT_GRIDS is not None else (0,)
    frames = {}
    for lg in settings:
        tag = f"{name} light grids {'on' if lg else 'off'}" if OPT_LIGHT_GRIDS is not None else f"{name}"
        ctr, exact = walk_counters(sd, w, h, out, lg)
        for kind, (r, cells, fetches, culls) in ctr.items():
            print(f"{tag}: {kind:11s} rays {r:11d}  cells/ray {cells:6.2f}  records/ray {fetches:6.2f}  culls/ray {culls:6.2f}")
        print(f"{tag}: exact tests per frame {exact}")
        per = launch_times(sd, w, h, out, lg)
        for k in sorted(per, key=lambda k: -sum(per[k])):
            v = per[k]
            print(f"{tag}: {k:24s} launches {len(v):3d}  sum {sum(v):8.3f} ms  each " + " ".join(f"{x:.3f}" for x in v[:16]))
        print(f"{tag}: scene upload (best of 5) {upload_ms(sd, lg):.2f} ms")
        ms, frames[lg] = timed(sd, w, h, out, lg)
        print(f"{tag}: frame {ms:.3f} ms (mean of 20, graph off)")
    if len(frames) == 2:
        print(f"{name}: frames identical: {bool(torch.equal(frames[0], frames[1]))}")
