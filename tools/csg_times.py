"""Kernel time of the CSG scenes beyond the whole-tree evaluator's limits (evaluated by csg_sweep) at 1920x1080
(device-resident frames; best of the renders after the first).
    python tools/csg_times.py"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ray_tracer_challenge_b200 as rt  # noqa: E402
from ray_tracer_challenge_b200 import scenes  # noqa: E402

SCENES = [
    ("csg_die (opaque, point light)", scenes.csg_die, dict()),
    ("csg_die (glass, point light)", scenes.csg_die, dict(glassy=True)),
    ("csg_die (opaque, 3x3 area light)", scenes.csg_die, dict(area_light=True)),
    ("csg_die (glass, 20 marbles: tree scene)", scenes.csg_die, dict(glassy=True, surrounded=True)),
    ("csg_carved_mesh (576 triangles - cylinder)", scenes.csg_carved_mesh, dict()),
    ("csg_chain (40 glass spheres)", scenes.csg_chain, dict()),
]
api = rt.new_session()
api.set_render_options(device_ids=[0])
for name, build, kw in SCENES:
    cam, world = build(api, width=1920, height=1080, **kw)
    p = cam.prepare(world)
    ms = []
    for _ in range(6):
        p.render(5, want_rgb=False, want_u8=False)
        ms.append(p.last_stats.kernel_ms)
    st = p.last_stats
    assert st.capacity_overflows == 0
    print(f"{name:45s} 1920x1080  {min(ms[1:]):8.3f} ms  {st.rays:>10d} rays  {st.rays / min(ms[1:]) / 1e3:9.1f} Mrays/s", flush=True)
    p.release()
