"""Host-free level loop, eager vs CUDA-graph replay: device ms of the C4 frame, of 1/N of it
(one interleaved row-list batch, the multi-GPU unit) and of the shipped examples at 800x600."""
import sys, time
sys.path.insert(0, ".")
import numpy as np, torch
import raingun_b200 as rg
from raingun_b200 import _native as N
from raingun_b200.synth import make_scene
from raingun_b200.examples import example_scene
from raingun_b200.dist import rows_of_tiles, n_tiles

MODES = (("host-free eager", 1), ("host-free graph", 2))


def timed(fn, reps=6):
    best_dev = best_wall = 1e9
    st = None
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        st = fn()
        torch.cuda.synchronize()
        best_wall = min(best_wall, (time.perf_counter() - t0) * 1e3)
        best_dev = min(best_dev, st.ms_device)
    return best_dev, best_wall, st


sd, spec = make_scene("C4")
w, h = spec.width, spec.height
out = torch.empty(h * w * 4, dtype=torch.uint8, device="cuda")
nt = n_tiles(h, 8)
stream = torch.cuda.current_stream().cuda_stream
for label, graph in MODES:
    sc = rg.Scene(sd)
    sc.set_option(N.OPT_GRAPH, graph)
    for frac in (1, 2, 4, 8, 16, 32):
        rows = rows_of_tiles(list(range(0, nt, frac)), 8, h)
        dev, wall, st = timed(lambda: sc.render_rowlist_device(w, h, rows, out.data_ptr(), stream))
        print(f"C4 {label:16s} 1/{frac:<2d}: device {dev:7.3f} ms  wall {wall:7.3f} ms  launches {st.gpu_launches} replays {st.graph_replays} "
              f"host_free {st.host_free}  Mrays/s {st.rays / dev / 1e3:.0f}", flush=True)
    sc.close()

for name in ("test1", "test2", "test3"):
    data = example_scene(name)
    for label, graph in MODES:
        sc = rg.Scene(data)
        sc.set_option(N.OPT_GRAPH, graph)
        for (ww, hh) in ((800, 600), (3840, 2160)):
            dev, wall, st = timed(lambda: sc.render_rows_device(ww, hh, 0, hh, out.data_ptr(), stream), reps=8)
            print(f"{name} {ww}x{hh} {label:16s}: device {dev:.3f} ms wall {wall:.3f} ms rays {st.rays} launches {st.gpu_launches} "
                  f"levels {st.max_level + 1} -> {st.rays / dev / 1e3:.0f} Mrays/s", flush=True)
        sc.close()
    sc = rg.Scene(data)
    sc.set_pipeline(rg.PIPELINE_MEGAKERNEL)
    dev, wall, st = timed(lambda: sc.render_rows_device(800, 600, 0, 600, out.data_ptr(), stream), reps=4)
    print(f"{name} 800x600 megakernel: device {dev:.3f} ms wall {wall:.3f} ms", flush=True)
    sc.close()

# instrumented grid tracer: where do the rays spend their steps?
for wl in ("C3", "C4"):
    sd, spec = make_scene(wl)
    sc = rg.Scene(sd)
    sc.set_option(N.OPT_TRACE_STATS, 1)
    st = sc.render_rows_device(spec.width, spec.height, 0, spec.height, out.data_ptr(), stream)
    r = st.rays
    print(f"{wl} trace stats: rays {r}  cells/ray {st.grid_cells / r:.2f}  fetches(occupied)/ray {st.grid_fetches / r:.2f}  culls/ray {st.grid_culls / r:.2f} "
          f" exact/ray {st.exact_tests / r:.2f}  rays/refill {r / max(1, st.grid_refills):.2f}  scan-lane use {st.grid_lane_steps / max(1, st.grid_lane_slots):.3f} "
          f" device {st.ms_device:.2f} ms", flush=True)
    sc.close()
