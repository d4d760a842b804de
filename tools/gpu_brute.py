import sys, zlib
sys.path.insert(0, ".")
import numpy as np
import raingun_b200 as rg
from raingun_b200.synth import make_scene
# gpu_brute.py [config [spheres [width height]]]: a config shrunk to `spheres` (same generator stream) and/or `width x height`
name = sys.argv[1] if len(sys.argv) > 1 else "C4"
spheres = int(sys.argv[2]) if len(sys.argv) > 2 else None
from raingun_b200.examples import bundled_texture_loader
sd, spec = make_scene(name, spheres=spheres, texture_loader=bundled_texture_loader)
w, h = (int(sys.argv[3]), int(sys.argv[4])) if len(sys.argv) > 4 else (spec.width, spec.height)
with rg.Scene(sd) as sc:
    sc.set_accel(rg.ACCEL_BRUTE)
    for it in range(3):
        img = sc.render_image(w, h)
        st = sc.last_stats
print(name, "brute dev %.2f ms trace %.2f ms rays %d exact %d crc %08x" % (st.ms_device, st.ms_trace, st.rays, st.exact_tests, zlib.crc32(img.tobytes())), flush=True)
