#!/usr/bin/env python
"""bench.py — the hot path's headline benchmark (BASELINE.json: Mrays/s over all bounces and
ms/frame at 4K, 1/2/4/8 B200, beside the reference's CPU path).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU algorithm
                                                              # (the oracle port; no Rust here)
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...     # N > 1
    python bench.py ... --dump-outputs DIR                    # + the last timed frame as DIR/*.npy

A step = one full frame of the workload (default C4 = BASELINE.json configs[3]: 3840x2160,
10,000 mixed reflective/refractive spheres + ground plane, 3 lights, depth 8; synthetic,
raingun_b200/synth.py).  A ray = one Scene::trace call (rendering.rs:73,126,150).
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "Mrays/sec (all bounces) at 4K; ms/frame in ms_per_step"
UNIT = "Mrays/s"
# pixels of the frame --dump-outputs writes: 32 MiB of float32 RGBA + 16 MiB of float64 indices (a quarter of a 4K frame)
DUMP_PIXELS = 1 << 21


def dump_outputs(out_dir, frame, stats) -> None:
    """--dump-outputs: what the device-resident arm's last timed step delivered, comparable between two builds.
    frame_sample.npy is float32 RGBA (0..255) of a fixed, seeded sample of the frame's pixels, frame_sample_index.npy
    their flat indices y * width + x; ray_counts.npy (one GPU) the frame's primary, shadow, reflection and
    transmission rays."""
    os.makedirs(out_dir, exist_ok=True)
    h, w, _ = frame.shape
    idx = np.sort(np.random.default_rng(0).choice(h * w, size=min(DUMP_PIXELS, h * w), replace=False))
    np.save(os.path.join(out_dir, "frame_sample.npy"), frame.reshape(h * w, 4)[idx].astype(np.float32))
    np.save(os.path.join(out_dir, "frame_sample_index.npy"), idx.astype(np.float64))
    if stats is not None:
        np.save(os.path.join(out_dir, "ray_counts.npy"), np.array(
            [stats.rays_primary, stats.rays_shadow, stats.rays_reflection, stats.rays_transmission], np.float64))


def flops_per_ray(data) -> float:
    """SURVEY.md 8(d): F_ray = 17 N_sphere + 16 N_plane + 32 N_disk + 22 N_aabb + 6, every ray
    charged the full body list (brute-force semantics)."""
    kinds = np.bincount(np.asarray(data.body_kind, np.int64), minlength=4)
    return float(17 * kinds[0] + 16 * kinds[1] + 32 * kinds[2] + 22 * kinds[3] + 6)


def workload_config(name, spec, data, extra):
    cfg = {"workload": f"{name}: synthetic {spec.width}x{spec.height}, {spec.spheres} "
                       f"{'mixed reflecting/refractive/diffuse' if spec.mixed else 'diffuse'} spheres + ground plane, "
                       f"{spec.lights} lights with shadow rays, depth {spec.depth} (BASELINE.json configs, SURVEY 8d, seed {spec.seed})",
           "width": spec.width, "height": spec.height, "bodies": int(data.n_bodies), "lights": int(data.n_lights),
           "max_depth": int(data.max_recursion_depth)}
    cfg.update(extra)
    return cfg


def profiled_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel's first launch (level-0
    nearest-hit k_trace_brute: 8.29 M rays) from the committed `ncu --set full` capture, per launch;
    None when no summary is present.  Not measured in this run: ncu cannot run inside the bench."""
    import glob
    import re
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_summary.md")), reverse=True):
        text = open(path).read()
        m = re.search(r"capture `prof_brute_r\w+\.ncu-rep`.*?k_trace_brute(?:_resident)?<0.*?DRAM read: ([\d.]+) (M|G)byte.*?DRAM written: ([\d.]+) (M|G)byte",
                      text, re.S)
        if m:
            unit = {"M": 1e6, "G": 1e9}
            return int(float(m.group(1)) * unit[m.group(2)] + float(m.group(3)) * unit[m.group(4)]), os.path.basename(path)
    return None, None


def profiled_grid_kernel():
    """Key ncu metrics of the kernel that dominates the `value` arm (k_trace_grid, nearest + any-hit
    variants) from the newest committed `--set full` capture; {} when no summary is present."""
    import glob
    import re
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_summary.md")), reverse=True):
        text = open(path).read()
        out = {}
        for variant, label in (("0", "nearest"), ("1", "any_hit")):
            ms = list(re.finditer(r"### `void k_trace_grid<%s(?:, 0)?>.*?\n\n(.*?)\n\n" % variant, text, re.S))
            if not ms:
                continue
            m = ms[-1]   # the last captured launch of the variant: a deep level (level 0 is the coherent exception)
            vals = {}
            for key, pat in (("ipc", r"IPC \(per SM, active\): ([\d.]+)"), ("issue_slots_busy_pct", r"issue slots busy %: ([\d.]+)"),
                             ("active_threads_per_warp", r"avg active threads / warp instr: ([\d.]+)"),
                             ("achieved_occupancy_pct", r"achieved occupancy %: ([\d.]+)"),
                             ("l1_hit_pct", r"L1/TEX hit rate %: ([\d.]+)"), ("dram_pct_of_peak", r"DRAM throughput % of peak: ([\d.]+)")):
                mm = re.search(pat, m.group(1))
                if mm:
                    vals[key] = round(float(mm.group(1)), 2)
            sm = re.search(r"top stall reasons.*?: (.*)", m.group(1))
            if sm:
                vals["top_stalls"] = sm.group(1).strip()
            out[label] = vals
        if out:
            out["source"] = f"profiles/{os.path.basename(path)}"
            return out
    return {}


class ClockSampler:
    """nvidia-smi sampling DURING the timed region (B200_PROFILING.md clocks line)."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int) -> None:
        self.proc, self.gpu = None, gpu_index

    def start(self) -> None:
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "nvidia-smi unavailable"}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.splitlines():
            p = [x.strip() for x in line.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2])); power.append(float(p[3]))
            except ValueError:
                continue
            for name, v in zip(names, p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "note": "no samples"}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "power_w_max": max(power), "samples": len(sm)}


def host_description() -> dict:
    """CPU model, logical cores and the oracle's compiler flags (BASELINE.md section 3 asks for them)."""
    model = None
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.lower().startswith("model name"):
                    model = line.split(":", 1)[1].strip()
                    break
    except OSError:
        pass
    flags = None
    try:
        with open(os.path.join(ROOT, "oracle", "Makefile")) as f:
            for line in f:
                if line.startswith("CXXFLAGS"):
                    flags = line.split("=", 1)[1].strip()
                    break
    except OSError:
        pass
    return {"cpu_model": model, "logical_cores": os.cpu_count(), "oracle_cxxflags": flags}


# ------------------------------------------------------------------------------------------ CPU arm
def oracle_sample(data, spec, target_seconds: float, threads=None):
    """Times the CPU oracle (the restated reference algorithm, all host threads, work-stealing
    over rows like rayon's par_iter) on a centred row band sized for ~target_seconds."""
    from oracle import oracle
    O = oracle()
    threads = threads or O.hardware_threads()
    w, h = spec.width, spec.height
    mid = h // 2
    probe_rows = max(1, min(h, threads // 4))
    t0 = time.perf_counter()
    _, st, _ = O.render_rows(data, w, h, mid, min(h, mid + probe_rows), threads=threads)
    dt = max(time.perf_counter() - t0, 1e-6)
    rows = int(max(probe_rows, min(h, target_seconds / dt * probe_rows)))
    y0 = max(0, mid - rows // 2)
    y1 = min(h, y0 + rows)
    return O, threads, y0, y1


def run_reference(args, rank):
    if rank != 0:
        return 0
    from raingun_b200.examples import bundled_texture_loader
    from raingun_b200.synth import make_scene
    data, spec = make_scene(args.workload, texture_loader=bundled_texture_loader)
    total = max(1, args.steps + args.warmup)
    per_step = max(1.0, min(15.0, args.reference_budget / total))
    O, threads, y0, y1 = oracle_sample(data, spec, per_step)
    w, h = spec.width, spec.height
    for _ in range(args.warmup):
        O.render_rows(data, w, h, y0, y1, threads=threads)
    rays = 0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        _, st, _ = O.render_rows(data, w, h, y0, y1, threads=threads)
        rays += st.rays
    dt = time.perf_counter() - t0
    value = rays / dt / 1e6
    sample = f"rows [{y0},{y1}) of {h} ({y1 - y0} rows x {w} px) per step, all bounces"
    rays_per_row = rays / max(1, args.steps) / max(1, y1 - y0)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / max(1, args.steps) * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.workload, spec, data, {"sample": sample, "parallelism": f"cpu{threads}"}),
        "cpu_baseline": dict({"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
                             **host_description()),
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "ms_per_frame_extrapolated": (rays_per_row * h) / (value * 1e6) * 1e3 if value > 0 else None,
        "note": "reference = CPU restatement of raingun's algorithm (oracle/); cargo/rustc are not in this image",
    }
    print(json.dumps(line), flush=True)
    return 0


def profiled_thread_instructions():
    """Thread instructions k_trace_grid executes per ray, from the newest committed ncu capture
    (profiles/r*_grid_counters.json: smsp__thread_inst_executed.sum and the rays of the captured launches);
    None when absent.  ncu cannot run inside the bench, so this one factor of the issue roofline is a
    profile constant of the same code on the same workload; everything else is measured in this run."""
    import glob
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_grid_counters.json")), reverse=True):
        try:
            with open(path) as f:
                d = json.load(f)
            return float(d["thread_inst_per_ray"]), os.path.basename(path), d
        except (OSError, ValueError, KeyError):
            continue
    return None, None, None


def grid_issue_roofline(rg, _native, data, w, h, staging, sptr, local_rank, value_mrays, clocks):
    """k_trace_grid does no dense arithmetic and moves ~0.2 TB/s: neither the FP32 pipe nor HBM bounds it.  What
    bounds a divergent traversal is the chip's LANE-ISSUE rate: 148 SMs x 4 schedulers x 32 lanes x clock
    thread-instructions per second.  achieved = thread instructions per ray (ncu, committed profile) x rays/s
    (this run); frac = IPC/4 x active lanes/32.  The per-ray walk counters come from one instrumented frame."""
    sc = rg.Scene(data, device=local_rank)
    sc.set_option(_native.OPT_TRACE_STATS, 1)
    st = sc.render_rows_device(w, h, 0, h, staging.data_ptr(), sptr)
    sc.close()
    # the kernel's own launch durations, measured live: one stream, eager launches, CUDA events around every trace launch
    sc = rg.Scene(data, device=local_rank)
    sc.set_option(_native.OPT_OVERLAP, 1)
    sc.set_option(_native.OPT_GRAPH, 1)
    kt = None
    for _ in range(3):
        kt = sc.render_rows_device(w, h, 0, h, staging.data_ptr(), sptr)
    sc.close()
    r = max(1, st.rays)
    tipr, src, prof = profiled_thread_instructions()
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    peak = 148 * 4 * 32 * sm_mhz * 1e6
    out = {"bound": "lane-issue slots (148 SM x 4 schedulers x 32 lanes x SM clock)", "peak": peak / 1e12, "unit": "T thread-instr/s",
           "sm_mhz_used": sm_mhz,
           "per_ray": {"cells_visited": st.grid_cells / r, "records_fetched_nonempty": st.grid_fetches / r, "cull_tests": st.grid_culls / r,
                       "exact_fp64_tests": st.exact_tests / r, "rays_per_refill": r / max(1, st.grid_refills),
                       "scan_lane_use": st.grid_lane_steps / max(1, st.grid_lane_slots),
                       "l2_bytes_algorithmic": 48.0 * st.grid_cells / r + 48.0 + 12.0},
           "per_ray_note": "l2_bytes_algorithmic = 48 B per cell visited (chained records of crowded cells add a few per cent) "
                           "+ 48 B ray + 12 B hit"}
    if tipr and kt and kt.ms_trace > 0:
        launches = 2 * (kt.max_level + 1)
        achieved = tipr * kt.rays / (kt.ms_trace * 1e-3)        # thread instructions / second while the kernel runs
        out.update({"achieved": achieved / 1e12, "frac": achieved / peak,
                    "kernel_ms_per_frame": kt.ms_trace, "launches_per_frame": launches, "avg_launch_ms": kt.ms_trace / max(1, launches),
                    "thread_instr_per_ray": tipr, "thread_instr_source": f"profiles/{src}",
                    "frac_under_ncu": (prof or {}).get("ipc_lanes_product"), "avg_active_lanes_under_ncu": (prof or {}).get("avg_active_lanes"),
                    # the same numerator against the WHOLE step (k_shade etc. included, streams overlapped): what the frame leaves unused
                    "frac_of_step": tipr * value_mrays * 1e6 / peak,
                    "how": "achieved = thread instructions per ray (ncu, committed capture) x rays of the frame / sum of the trace launches' "
                           "durations (CUDA events, one stream, this run)"})
    return out


def run_configs(rg, _native, torch, device, local_rank, world, sha):
    """BASELINE.json configs beside the headline one: the three shipped scenes at their native 800x600 (configs[0..1];
    test1 also on the CPU oracle, full frame), C3 at 4K on one GPU (configs[2]) and C5 at 8K (configs[4]) — on one GPU
    and, at N > 1, row-tile sharded over all N GPUs inside the library.  Device-resident ms/frame (CUDA events),
    best of a few frames after a warm-up."""
    from oracle import oracle
    from raingun_b200.examples import bundled_texture_loader, example_scene
    from raingun_b200.synth import make_scene
    out = {}
    buf = torch.empty(7680 * 4320 * 4, dtype=torch.uint8, device=device)
    stream = torch.cuda.current_stream(device).cuda_stream

    def timed(sc, w_, h_, reps):
        best, st_ = 1e30, None
        for _ in range(reps):
            st_ = sc.render_rows_device(w_, h_, 0, h_, buf.data_ptr(), stream)
            best = min(best, st_.ms_device)
        return best, st_

    for name in ("test1", "test2", "test3"):
        sd = example_scene(name)
        with rg.Scene(sd, device=local_rank) as sc:
            ms, st_ = timed(sc, 800, 600, 6)
        entry = {"width": 800, "height": 600, "ms_per_frame": ms, "mrays_per_s": st_.rays / ms / 1e3, "rays": int(st_.rays),
                 "pipeline": {0: "wavefront", 1: "megakernel"}.get(st_.pipeline_used, "?"), "launches": int(st_.gpu_launches)}
        if name == "test1":   # BASELINE.json configs[0]: the reference CLI's own CPU case, here the oracle on all host threads
            O = oracle()
            t0 = time.perf_counter()
            ref, ost, _ = O.render(sd, 800, 600)
            dt = time.perf_counter() - t0
            img = buf[: 800 * 600 * 4].view(600, 800, 4).cpu().numpy()
            entry["cpu_oracle"] = {"ms_per_frame": dt * 1e3, "mrays_per_s": ost.rays / dt / 1e6, "threads": O.hardware_threads(),
                                   "identical_to_gpu_frame": bool(np.array_equal(ref, img))}
        out[f"{name}@800x600"] = entry
    for wl in ("C3", "C5"):
        sd, spec_ = make_scene(wl, texture_loader=bundled_texture_loader)
        with rg.Scene(sd, device=local_rank) as sc:
            ms, st_ = timed(sc, spec_.width, spec_.height, 4 if wl == "C3" else 2)
        single_sha = sha(buf[: spec_.width * spec_.height * 4].cpu().numpy())
        entry = {"width": spec_.width, "height": spec_.height, "bodies": int(sd.n_bodies), "ms_per_frame": ms,
                 "mrays_per_s": st_.rays / ms / 1e3, "rays": int(st_.rays), "batches": int(st_.batches), "n_gpus": 1}
        if wl == "C5" and world > 1 and rg.device_count() >= world:
            host = torch.empty((spec_.height, spec_.width, 4), dtype=torch.uint8).pin_memory()
            with rg.Scene(sd, devices=list(range(world))) as msc:
                best = 1e30
                for _ in range(3):
                    t0 = time.perf_counter()
                    mst = msc.render_rows_into(spec_.width, spec_.height, 0, spec_.height, host.data_ptr())
                    best = min(best, (time.perf_counter() - t0) * 1e3)
            entry["sharded"] = {"n_gpus": world, "ms_per_frame_wall_incl_d2h": best, "mrays_per_s": mst.rays / best / 1e3,
                                "identical_to_one_gpu_frame": sha(host.numpy()) == single_sha,
                                "how": "row tiles across the GPUs inside the library (rg_scene_create_multi), frame delivered to pinned host memory"}
            del host
        out[f"{wl}@{spec_.width}x{spec_.height}"] = entry
    del buf
    return out


# ------------------------------------------------------------------------------------------ GPU arm
def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C4", choices=["C3", "C4", "C5"])
    ap.add_argument("--accel", default="auto", choices=["auto", "grid", "brute"])
    ap.add_argument("--schedule", default="auto", choices=["auto", "steal", "static"])
    ap.add_argument("--tile-rows", type=int, default=8)
    ap.add_argument("--gather", default="peer", choices=["peer", "reduce", "p2p"],
                    help="N>1: peer = rows stored straight into rank 0's frame over NVLink by the last kernel (CUDA IPC)")
    ap.add_argument("--e2e-gather", default="host", choices=["host", "device"],
                    help="N>1 end-to-end arm: host = every rank copies its rows over its own PCIe link into ONE pinned "
                         "shared-memory frame; device = gather on rank 0's GPU (--gather) and one D2H from there")
    ap.add_argument("--frames-inflight", type=int, default=1,
                    help="device-resident arm: frames in flight per GPU (each on its own scene handle(s), host thread, frame "
                         "buffers and end-of-frame barrier); 1 (default) = one frame after the other, ms_per_step is then the "
                         "latency of a frame.  Measured on 8 B200: 2.817 / 2.788 / 2.785 ms per frame with 1 / 2 / 3 in flight - "
                         "the device-resident arm is bound on the GPUs, not by the host between frames")
    ap.add_argument("--e2e-inflight", type=int, default=3,
                    help="end-to-end arm: steps in flight per GPU (each a complete upload -> render -> frame-to-host step "
                         "on its own scene handle and host thread; 1 = strictly one after the other)")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config table (test1/2/3, C3, C5)")
    ap.add_argument("--no-in-library", action="store_true", help="skip the in-library multi-GPU arm (N>1)")
    ap.add_argument("--lead", type=float, default=0.6, help="share of a rank's static tiles given to its first in-flight batch")
    ap.add_argument("--inflight", type=int, default=1,
                    help="N>1: wavefront batches each rank keeps in flight (scene handle + stream + host thread each)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU-baseline sample budget (N=1)")
    ap.add_argument("--reference-budget", type=float, default=150.0, help="--impl reference: total seconds")
    ap.add_argument("--no-roofline", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed frame (a fixed, seeded sample of its pixels, float32) and its ray counts "
                         "to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference(args, rank)

    import torch
    import torch.distributed as dist

    import raingun_b200 as rg
    from raingun_b200 import _native
    from raingun_b200.dist import render_frame_sharded
    from raingun_b200.examples import bundled_texture_loader
    from raingun_b200.synth import make_scene

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: this benchmark has no CPU fallback"}), flush=True)
        return 2
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    n_gpus = world

    data, spec = make_scene(args.workload, texture_loader=bundled_texture_loader)
    w, h = spec.width, spec.height
    accel = {"auto": rg.ACCEL_AUTO, "grid": rg.ACCEL_GRID, "brute": rg.ACCEL_BRUTE}[args.accel]
    stream = torch.cuda.current_stream(device)
    sptr = stream.cuda_stream

    def barrier():
        torch.cuda.synchronize(device)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(device)

    section = [0]

    def rank0_only(work):
        """Runs `work()` on rank 0 while the other ranks wait ON THE CPU (a key in the c10d store): an NCCL barrier
        would park a spinning kernel on every idle GPU, and the rank-0 sections below use those GPUs themselves."""
        barrier()
        section[0] += 1
        result = None
        if world == 1:
            return work()
        store = dist.distributed_c10d._get_default_store()
        key = f"raingun/bench/section{section[0]}"
        if rank == 0:
            try:
                result = work()
            finally:
                store.set(key, b"done")
        else:
            store.wait([key])
        barrier()
        return result

    def reduce_max(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def reduce_sum(xs):
        if world == 1:
            return [int(x) for x in xs]
        t = torch.tensor(xs, dtype=torch.int64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [int(x) for x in t.tolist()]

    scene = rg.Scene(data, device=local_rank)
    scene.set_accel(accel)
    inflight = max(1, args.inflight) if world > 1 else 1
    side_streams = [torch.cuda.Stream(device) for _ in range(inflight - 1)]

    def make_lanes(first_scene):
        """The rank's in-flight batch lanes: (scene handle, CUDA stream) each; lane 0 is the given scene."""
        lanes = [(first_scene, sptr)]
        for s_ in side_streams:
            extra = rg.Scene(data, device=local_rank)
            extra.set_accel(accel)
            lanes.append((extra, s_.cuda_stream))
        return lanes

    peer_frames = None
    gather_note = None
    if world > 1 and args.gather == "peer":
        from raingun_b200.dist import PeerFrames
        try:
            peer_frames = PeerFrames(w, h, rank, world, local_rank)
        except Exception as e:   # CUDA IPC unavailable (e.g. restricted container): every rank falls back together
            gather_note = f"peer gather unavailable on rank {rank}: {e}"
        ok = torch.tensor([0 if peer_frames is None else 1], dtype=torch.int32, device=device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            if peer_frames is not None and rank != 0:   # importers unmap first ...
                peer_frames.close(sync=False)
                peer_frames = None
            dist.barrier()
            if peer_frames is not None:                 # ... then the owner frees
                peer_frames.close(sync=False)
                peer_frames = None
            args.gather = "reduce"
            gather_note = gather_note or "peer gather unavailable on another rank"
            print(f"[bench] {gather_note}; using the NCCL reduce gather", file=sys.stderr, flush=True)

    host_barrier = None
    if world > 1:   # end-of-frame barrier of the ranks in shared memory (microseconds) instead of a GPU collective
        from raingun_b200.dist import HostBarrier
        try:
            host_barrier = HostBarrier(rank, world, tag="bench")
        except Exception as e:
            print(f"[bench] shared-memory barrier unavailable on rank {rank}: {e}", file=sys.stderr, flush=True)
        ok = torch.tensor([0 if host_barrier is None else 1], dtype=torch.int32, device=device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0 and host_barrier is not None:
            host_barrier.close()
            host_barrier = None

    def run_threads(jobs):
        """Runs the callables on one thread each; an exception in any of them is re-raised here (not lost with its thread)."""
        import threading
        errors = []

        def guarded(job):
            try:
                job()
            except BaseException as e:   # noqa: BLE001 - reported below
                errors.append(e)
        th = [threading.Thread(target=guarded, args=(j,)) for j in jobs]
        for x in th:
            x.start()
        for x in th:
            x.join()
        if errors:
            raise errors[0]

    def lane_renderers(lanes, peer):
        if peer is not None:
            return [(lambda rows, fptr, sc_=sc_, st_=st_: sc_.render_rowlist_scatter(w, h, rows, fptr, st_))
                    for sc_, st_ in lanes]
        return [(lambda rows, out, sc_=sc_, st_=st_: sc_.render_rowlist_device(w, h, rows, out.data_ptr(), st_))
                for sc_, st_ in lanes]

    lanes = make_lanes(scene)
    staging = torch.empty((h * w * 4,), dtype=torch.uint8, device=device)
    frame_buf = torch.empty((h, w, 4), dtype=torch.uint8, device=device) if world > 1 else None
    host_frame = torch.empty((h, w, 4), dtype=torch.uint8).pin_memory()

    gathered = {}

    # Frames in flight.  A frame is one blocking call of the public API per rank plus the end-of-frame barrier; a host
    # that renders a SEQUENCE of frames hides the host-side part of a frame (launch, the final synchronisation, the
    # barrier and the skew between the ranks) behind the next frame by driving it from a second thread on its own scene
    # handle, frame buffers and barrier.  Every frame is still rendered completely; ms_per_step is wall time / frames and
    # the latency of a frame is reported beside it (frame_latency_ms).  With a collective gather (NCCL) frames go one by one.
    F = max(1, args.frames_inflight)
    if world > 1 and (peer_frames is None or host_barrier is None):
        F = 1
    ctxs = [{"lanes": lanes, "peer": peer_frames, "bar": host_barrier, "staging": staging, "frame_no": 0, "id": 0}]
    for f in range(1, F):
        sc_f = rg.Scene(data, device=local_rank)
        sc_f.set_accel(accel)
        peer_f = bar_f = None
        if world > 1:
            from raingun_b200.dist import HostBarrier, PeerFrames
            peer_f = PeerFrames(w, h, rank, world, local_rank, tag=f"v{f}")
            bar_f = HostBarrier(rank, world, tag=f"v{f}")
        ctxs.append({"lanes": make_lanes(sc_f), "peer": peer_f, "bar": bar_f, "frame_no": 0, "id": f,
                     "staging": torch.empty((h * w * 4,), dtype=torch.uint8, device=device)})

    def step_resident(ctx):
        """One frame, inputs (scene) and output resident in HBM.  Returns (rays, launches, stats)."""
        if world == 1:
            st = ctx["lanes"][0][0].render_rows_device(w, h, 0, h, ctx["staging"].data_ptr(), sptr)
            return st.rays, st.gpu_launches, st
        ctx["frame_no"] += 1
        res = render_frame_sharded(
            lane_renderers(ctx["lanes"], ctx["peer"]), w, h, rank, world,
            ctx["frame_no"], device, tile_rows=args.tile_rows, schedule=args.schedule if F == 1 else "static", staging=ctx["staging"],
            gather_mode=args.gather, frame_buf=frame_buf, lead=args.lead, peer_frames=ctx["peer"], host_barrier=ctx["bar"])
        if ctx["id"] == 0:
            gathered["frame"] = res.frame   # rank 0: the gathered (H, W, 4) frame in HBM
            gathered["schedule"] = res.schedule
        return (sum(s.rays for s in res.stats), sum(s.gpu_launches for s in res.stats),
                res.stats[-1] if res.stats else None)

    def run_frames(n_total, acc):
        """n_total frames dealt to the F in-flight streams (the same split on every rank); acc collects per stream
        (rays, launches, last stats, per-frame wall seconds)."""
        per = [n_total // F + (1 if f < n_total % F else 0) for f in range(F)]

        def body(f):
            rays_ = launches_ = 0
            last_ = None
            lat = []
            for _ in range(per[f]):
                t_ = time.perf_counter()
                r_, l_, last_ = step_resident(ctxs[f])
                lat.append(time.perf_counter() - t_)
                rays_ += r_
                launches_ += l_
            acc[f] = (rays_, launches_, last_, lat)
        if F == 1:
            body(0)
        else:
            run_threads([lambda f=f: body(f) for f in range(F)])

    # ---- device-resident arm: `value`
    run_frames(args.warmup * F, [None] * F)
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    acc = [None] * F
    run_frames(args.steps, acc)
    e1.record(stream)
    barrier()
    ms_total = reduce_max(e0.elapsed_time(e1))
    rays = sum(a_[0] for a_ in acc if a_)
    launches = sum(a_[1] for a_ in acc if a_)
    last_stats = acc[0][2]
    step_ms = [x * 1e3 / F for a_ in acc if a_ for x in a_[3]]   # this rank's view of each frame's share of the wall clock
    frame_latency_ms = float(np.median([x * 1e3 for a_ in acc if a_ for x in a_[3]]))
    clocks = sampler.stop() if rank == 0 else None
    rays, launches = reduce_sum([rays, launches])
    ms_per_step = ms_total / max(1, args.steps)
    value = rays / (ms_total * 1e-3) / 1e6 if ms_total > 0 else 0.0
    accel_used = {1: "brute", 2: "grid"}.get(last_stats.accel_used if last_stats else 0, "?")

    # ---- end-to-end arm: every step re-uploads the scene from host arrays through the C ABI
    # (rg_scene_create = H2D), renders, and reads the RGBA8 frame back into pinned host memory.
    desc_bytes = int(sum(np.asarray(a).nbytes for a in (
        data.body_kind, data.body_geom, data.coloration_kind, data.color, data.texture_id, data.texture_offset,
        data.albedo, data.surface_kind, data.surface_param, data.light_kind, data.light_vec, data.light_color,
        data.light_intensity)) + sum(t.nbytes for t in data.textures))
    for ctx in ctxs:
        for sc_, _ in ctx["lanes"]:
            sc_.close()
    for ctx in ctxs[1:]:   # the extra in-flight streams' frames and barriers (collective closes: same order on every rank)
        if ctx["peer"] is not None:
            ctx["peer"].close()
        if ctx["bar"] is not None:
            ctx["bar"].close()
        ctx["staging"] = None

    import hashlib

    def sha(arr) -> str:
        return hashlib.sha256(np.ascontiguousarray(arr).tobytes()).hexdigest()

    # the frame of the device-resident arm, for the equality check of all arms below
    value_frame_sha = None
    if rank == 0:
        value_frame = (gathered["frame"] if world > 1 else staging.view(h, w, 4)).cpu().numpy()
        value_frame_sha = sha(value_frame)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, value_frame, last_stats if world == 1 else None)
        del value_frame

    # Steps in flight.  A step is upload -> render -> frame in host memory -> destroy, each a blocking call of the public
    # API; a host that renders a sequence of frames keeps the GPU busy during the host-side parts of a step (scene
    # flattening, the final copy, the synchronisations) by running the next step on a second scene handle from a second
    # thread.  Every step still does all of its own copies inside the timed region; `ms_per_step` is wall time / steps.
    e2e_T = max(1, args.e2e_inflight)
    upload_s = [0.0] * e2e_T
    host_frames = None          # world > 1: one SharedHostFrame (+ end-of-frame barrier) per in-flight stream of steps
    e2e_barriers = None
    host_frame_t = [host_frame] + [torch.empty((h, w, 4), dtype=torch.uint8).pin_memory() for _ in range(e2e_T - 1)]
    e2e_gather = args.e2e_gather if world > 1 else "single"
    if world > 1 and args.e2e_gather == "host":
        from raingun_b200.dist import HostBarrier, SharedHostFrame
        try:
            host_frames = [SharedHostFrame(w, h, rank, world, tag=f"e2e{t}") for t in range(e2e_T)]
            e2e_barriers = [HostBarrier(rank, world, tag=f"e2e{t}") for t in range(e2e_T)]
        except Exception as e:   # /dev/shm or pinning unavailable: every rank falls back together
            print(f"[bench] shared host frame unavailable on rank {rank}: {e}", file=sys.stderr, flush=True)
            host_frames = None
        ok = torch.tensor([0 if host_frames is None else 1], dtype=torch.int32, device=device)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 0:
            host_frames = None
            e2e_gather = "device"
    if world > 1 and host_frames is None:
        e2e_T = 1   # the device gather is an NCCL collective: one stream of steps

    e2e_frame_no = [0] * e2e_T

    def step_e2e(t=0):
        t_up = time.perf_counter()
        sc = rg.Scene(data, device=local_rank)
        sc.set_accel(accel)
        upload_s[t] += time.perf_counter() - t_up   # reported separately as well (SURVEY 8d)
        if world == 1:
            r = sc.render_rows_into(w, h, 0, h, host_frame_t[t].data_ptr()).rays
            sc.close()
        elif host_frames is not None:
            # every rank delivers its own rows over its own PCIe link into the one pinned host frame (of stream t)
            e2e_frame_no[t] += 1
            res = render_frame_sharded(
                [lambda rows, fptr, sc_=sc: sc_.render_rowlist_host(w, h, rows, fptr)], w, h, rank, world, e2e_frame_no[t], device,
                tile_rows=args.tile_rows, schedule="static" if e2e_T > 1 else args.schedule, gather_mode="host",
                peer_frames=host_frames[t], host_barrier=e2e_barriers[t])
            if t == 0:
                gathered["host_frame"] = res.frame
            r = sum(s_.rays for s_ in res.stats)
            sc.close()
        else:
            ls = make_lanes(sc)            # every lane re-uploads the scene (counted in h2d_bytes_per_step)
            ctxs[0]["lanes"] = ls
            r, _, _ = step_resident(ctxs[0])    # row tiles gathered on rank 0's GPU
            if rank == 0:
                host_frame.copy_(gathered["frame"])
            for sc_, _ in ls:
                sc_.close()
        return r

    def e2e_stream(t, nsteps, out):
        out[t] = sum(step_e2e(t) for _ in range(nsteps))

    def run_e2e(nsteps_total):
        """nsteps_total steps, dealt round-robin to the in-flight streams (the same split on every rank)."""
        per = [nsteps_total // e2e_T + (1 if t < nsteps_total % e2e_T else 0) for t in range(e2e_T)]
        out = [0] * e2e_T
        if e2e_T == 1:
            e2e_stream(0, per[0], out)
        else:
            run_threads([lambda t=t: e2e_stream(t, per[t], out) for t in range(e2e_T) if per[t]])
        return sum(out)

    run_e2e(max(min(args.warmup, 2), 1) * e2e_T)
    for t in range(e2e_T):
        upload_s[t] = 0.0
    barrier()
    t0 = time.perf_counter()
    e2e_rays = run_e2e(args.steps)
    barrier()
    e2e_s = reduce_max(time.perf_counter() - t0)
    # ... and, for the record, the same steps strictly one after the other (the latency of one step)
    e2e_serial_ms = None
    if e2e_T > 1:
        n_serial = max(2, min(args.steps, 6))
        barrier()
        t0 = time.perf_counter()
        out_ = [0] * e2e_T
        e2e_stream(0, n_serial, out_)
        barrier()
        e2e_serial_ms = reduce_max(time.perf_counter() - t0) / n_serial * 1e3
    (e2e_rays,) = reduce_sum([e2e_rays])
    e2e_value = e2e_rays / e2e_s / 1e6 if e2e_s > 0 else 0.0
    e2e_frame_sha = None
    if rank == 0:
        e2e_frame_sha = sha(gathered["host_frame"].numpy() if host_frames is not None else host_frame.numpy())
        for t in range(1, e2e_T):   # every in-flight stream delivered the same frame
            other = host_frames[t].array(e2e_frame_no[t]) if host_frames is not None else host_frame_t[t].numpy()
            if e2e_frame_no[t] or host_frames is None:
                if sha(other) != e2e_frame_sha:
                    e2e_frame_sha = "streams differ"
        if e2e_frame_sha != value_frame_sha:
            print(json.dumps({"error": "the end-to-end frame differs from the device-resident frame",
                              "value_frame_sha256": value_frame_sha, "e2e_frame_sha256": e2e_frame_sha}), flush=True)
            return 3
    if host_frames is not None:
        for b_ in e2e_barriers:
            b_.close()
        for f_ in host_frames:
            f_.close()

    # ---- the same frame rendered on all N GPUs INSIDE the library (rank 0 only; the other ranks idle at the
    # barrier): rg_scene_create_multi + rg_render — what a host without torchrun gets (rendering.rs:27-35)
    in_library = None

    def in_library_arm():
        if rg.device_count() < world:
            return None
        if True:
            in_library = {}
            for label, schedule in (("static", 1), ("steal", 2)):
                with rg.Scene(data, devices=list(range(world))) as msc:
                    msc.set_accel(accel)
                    msc.set_option(_native.OPT_SCHEDULE, schedule)
                    for _ in range(max(2, min(args.warmup, 3))):
                        msc.render_rows_into(w, h, 0, h, host_frame.data_ptr())
                    t0 = time.perf_counter()
                    mrays = 0
                    for _ in range(args.steps):
                        mrays += msc.render_rows_into(w, h, 0, h, host_frame.data_ptr()).rays
                    dt = time.perf_counter() - t0
                    st_ = msc.last_stats
                    in_library[label] = {"ms_per_frame": dt / max(1, args.steps) * 1e3, "value": mrays / dt / 1e6, "unit": UNIT,
                                         "devices_used": int(st_.devices_used), "batches_last_frame": int(st_.batches),
                                         "frame_sha256_equal": sha(host_frame.numpy()) == value_frame_sha}
            in_library["what"] = ("one process, one library thread per GPU, row tiles owned statically (static) or a 1/16 tail claimed "
                                  "from a std::atomic counter (steal); scene already uploaded; timed: rg_render into pinned host memory, "
                                  "every GPU copying its rows over its own PCIe link (wall clock)")
        return in_library

    if world > 1 and not args.no_in_library:
        in_library = rank0_only(in_library_arm)

    # ---- roofline arm (rank 0): the reference algorithm itself — brute force, every ray x every
    # body — whose dominant kernel k_trace_brute is FP32-pipe bound (SURVEY 8d).
    roofline = None
    brute = None
    if not args.no_roofline:
        barrier()
        if rank == 0:
            fp32_peak, fp64_peak, _ = rg.measure_peaks(local_rank)
            sc = rg.Scene(data, device=local_rank)
            sc.set_accel(rg.ACCEL_BRUTE)
            sc.set_option(_native.OPT_GRAPH, 1)   # eager launches: the trace kernels are timed one by one with CUDA events
            bsteps = max(1, min(3, args.steps))
            sc.render_rows_device(w, h, 0, h, staging.data_ptr(), sptr)
            torch.cuda.synchronize(device)
            tr_ms = dev_ms = 0.0
            brays = blaunch = bexact = btests = 0
            for _ in range(bsteps):
                st = sc.render_rows_device(w, h, 0, h, staging.data_ptr(), sptr)
                tr_ms += st.ms_trace
                dev_ms += st.ms_device
                brays += st.rays
                bexact += st.exact_tests
                btests += st.body_tests
                blaunch += 2 * (st.max_level + 1)
            sc.close()
            fl = flops_per_ray(data)
            traffic, traffic_src = profiled_traffic()
            achieved = brays * fl / (tr_ms * 1e-3) / 1e12
            roofline = {"bound": "fp32", "kernel": "k_trace_brute_resident / k_trace_brute (nearest + shadow variants), accel=brute",
                        "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s", "frac": achieved / fp32_peak,
                        "traffic": traffic, "traffic_source": traffic_src and
                        f"profiles/{traffic_src}: DRAM read + written by the level-0 nearest-hit launch (8.29 M rays; algorithmic 60 B/ray "
                        "= 48 B ray + 12 B hit = 498 MB) - the kernel re-reads nothing from HBM",
                        "algorithmic_flops_per_ray": fl,
                        "pair_tests_per_s": brays * float(data.n_bodies) / (tr_ms * 1e-3),
                        "peak_source": "rg_measure_peaks: register-resident FFMA loop on this GPU, this run (MEASURED_PEAKS.json "
                                       "has no FP32 figure; nominal 74.4 TFLOP/s at 1965 MHz)",
                        "fp64_peak_tflops": fp64_peak,
                        "fp64_fallthrough_frac": bexact / btests if btests else None,   # pairs the FP32 cull could not reject
                        # the 17 algorithmic flop of a pair are executed as 7 FFMA (14 flop) + compare: the FMA pipe's own utilisation
                        "executed_ffma_frac": (brays * float(data.n_bodies) * 14.0 / (tr_ms * 1e-3) / 1e12) / fp32_peak,
                        "share_of_step": tr_ms / dev_ms if dev_ms > 0 else None}
            brute = {"value": brays / (dev_ms * 1e-3) / 1e6, "unit": UNIT, "ms_per_step": dev_ms / bsteps,
                     "ms_trace_kernels": tr_ms / bsteps, "steps": bsteps}
        barrier()

    # ---- every BASELINE.json config in the one run (rank 0; the other ranks idle at the barrier) ----------
    configs = None
    if not args.no_configs:
        configs = rank0_only(lambda: run_configs(rg, _native, torch, device, local_rank, world, sha))

    # ---- the kernel behind `value` (k_trace_grid) against ITS ceiling: lane-issue slots -------------------
    grid_roofline = None
    if rank == 0 and accel_used == "grid":
        grid_roofline = grid_issue_roofline(rg, _native, data, w, h, staging, sptr, local_rank, value, clocks)

    # ---- CPU baseline beside it (rank 0, N = 1): the oracle on all host threads, bounded sample
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        O, threads, y0, y1 = oracle_sample(data, spec, args.cpu_seconds)
        t0 = time.perf_counter()
        _, ost, _ = O.render_rows(data, w, h, y0, y1, threads=threads)
        dt = time.perf_counter() - t0
        cpu_baseline = dict({"value": ost.rays / dt / 1e6, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": f"rows [{y0},{y1}) of {h} ({(y1 - y0) * w} px, {ost.rays} rays) in {dt:.1f} s",
                             "ms_per_frame_extrapolated": dt * 1e3 * h / max(1, y1 - y0)}, **host_description())

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "ms_per_step_median": statistics.median(step_ms) if step_ms else None,
            "frames_in_flight": F, "frame_latency_ms": frame_latency_ms,
            "higher_is_better": True, "scaling": "strong",   # one fixed frame split N ways
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args.workload, spec, data, {
                "accel": accel_used, "pipeline": "wavefront",
                "parallelism": f"row-tiles x{world} ({args.schedule}->{gathered.get('schedule', '?')}, {args.tile_rows}-row tiles, {inflight} batches in flight per GPU, gather={args.gather}, end-of-frame barrier={'shared memory' if host_barrier is not None else 'nccl'})" if world > 1 else "1 GPU",
                "l2": "per-frame working set (ray queues + nodes, several GB) exceeds the 126 MB L2; no explicit flush",
                "frames_in_flight": f"{F} per GPU (own scene handle, host thread, frame buffers and end-of-frame barrier each): ms_per_step = wall time / frames; frame_latency_ms = one frame, start to end"}),
            "rays_per_frame": rays // max(1, args.steps),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": desc_bytes * world * inflight,
                    "d2h_bytes_per_step": h * w * 4, "ms_per_step": e2e_s / max(1, args.steps) * 1e3,
                    "scene_upload_ms_per_step": sum(upload_s) / max(1, args.steps) * 1e3,
                    "scene_upload_note": "wall time of rg_scene_create per step; with steps in flight it includes waiting for the GPU, which is rendering the other step",
                    "gather": e2e_gather, "steps_in_flight": e2e_T, "ms_per_step_one_in_flight": e2e_serial_ms,
                    "what": "rg_scene_create (scene H2D) + render + RGBA8 frame D2H into pinned host memory + rg_scene_destroy, per step"
                            + (f"; {e2e_T} steps in flight per GPU (each on its own scene handle and host thread), ms_per_step = wall time / steps" if e2e_T > 1 else "")
                            + ("; N>1: every rank copies its rows into ONE pinned shared-memory frame over its own PCIe link" if e2e_gather == "host" else "")},
            "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "brute_force": brute,
            # the kernel that dominates the `value` arm is latency / issue bound, not FP32- or HBM-bound: its
            # figure of merit is rays/s; the ncu numbers that say so come from the committed capture
            "value_arm_kernel": {"kernel": "k_trace_grid (exact grid traversal, nearest + any-hit)", "bound": "latency/issue",
                                 "trace_ms_per_step_sum_of_spans": (last_stats.ms_trace if last_stats else None),
                                 "device_ms_last_step": (last_stats.ms_device if last_stats else None),
                                 "rays_per_s": value * 1e6, "roofline": grid_roofline, "ncu": profiled_grid_kernel()},
            "cpu_baseline": cpu_baseline, "frame_sha256": value_frame_sha,
            "frame_sha256_equal_across_arms": True,   # device-resident, end-to-end (and gathered, N > 1) frames: checked above
            "in_library_multi_gpu": in_library, "configs": configs,
        }
        print(json.dumps(line), flush=True)
    if peer_frames is not None:
        peer_frames.close()
    if host_barrier is not None:
        host_barrier.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
