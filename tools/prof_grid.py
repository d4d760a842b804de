import sys
sys.path.insert(0, ".")
import raingun_b200 as rg
from raingun_b200 import _native as N
from raingun_b200.synth import make_scene
sd, spec = make_scene(sys.argv[1] if len(sys.argv) > 1 else "C4")
sc = rg.Scene(sd); sc.set_accel(2)
sc.set_option(N.OPT_GRAPH, 1)      # ncu sees kernels inside graphs too, but keep the launch order plain
for it in range(2):
    sc.render_rows(spec.width, spec.height, 0, spec.height)
print("trace ms", sc.last_stats.ms_trace, "device ms", sc.last_stats.ms_device)
