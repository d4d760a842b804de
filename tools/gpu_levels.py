"""Per-launch times of one C4 frame (events around every trace launch are not exported, so this
uses the launch list under ncu instead) -- here: just total ms and trace-span sum for a few orderings."""
import sys
sys.path.insert(0, ".")
import torch
import raingun_b200 as rg
from raingun_b200 import _native as N
from raingun_b200.synth import make_scene
sd, spec = make_scene(sys.argv[1] if len(sys.argv) > 1 else "C4")
w, h = spec.width, spec.height
out = torch.empty(h * w * 4, dtype=torch.uint8, device="cuda")
sc = rg.Scene(sd)
sc.set_option(N.OPT_GRAPH, 1)
for it in range(3):
    st = sc.render_rows_device(w, h, 0, h, out.data_ptr(), 0)
print(f"device {st.ms_device:.3f} ms, trace spans {st.ms_trace:.3f} ms, rays {st.rays}")
