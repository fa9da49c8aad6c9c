"""Kernel time with RTC_OPT_EXACT_GROUPS off, on with every chain walked (RTC_EXACT_GROUPS_CERT=0: no node marked for
the one-box certificate) and on with the certificate, alternating in one process: three runs of each, every run the
best of five device-resident renders after a warm-up (L2 flushed before each).  Prints the card's name and power limit.
    python tools/exact_groups_times.py [scene ...]"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ray_tracer_challenge_b200 as rt  # noqa: E402
from bench import build_scene  # noqa: E402
from ray_tracer_challenge_b200 import scenes  # noqa: E402

SCENES = {
    "c1": lambda api: build_scene(api, "c1")[:2],
    "c3": lambda api: build_scene(api, "c3")[:2],
    "c4": lambda api: build_scene(api, "c4")[:2],
    "c5": lambda api: build_scene(api, "c5")[:2],
    "here_be_dragons": lambda api: scenes.here_be_dragons(api, width=1920, height=1080, n_u=320, n_v=160),
    "field_20k": lambda api: scenes.stress(api, width=640, height=360, n_spheres=20_000, n_each=16, n_csg=8),
}

print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip(), flush=True)


def best_ms(p):
    ms = []
    for _ in range(5):
        p.flush_l2()
        p.render(5, want_rgb=False, want_u8=False)
        ms.append(p.last_stats.kernel_ms)
    return min(ms)


MODES = {"off": (False, "1"), "walk": (True, "0"), "cert": (True, "1")}
for name in sys.argv[1:] or list(SCENES):
    prepared = {}
    for mode, (exact, cert) in MODES.items():
        os.environ["RTC_EXACT_GROUPS_CERT"] = cert  # read at commit
        api = rt.new_session()
        api.set_render_options(device_ids=[0])
        api.set_exact_groups(exact)
        cam, world = SCENES[name](api)
        p = cam.prepare(world)
        p.render(5, want_rgb=False, want_u8=False)  # warm-up: module load, learnt tile order
        prepared[mode] = (api, cam, world, p)
    runs = {mode: [] for mode in MODES}
    for _ in range(3):
        for mode in MODES:
            runs[mode].append(best_ms(prepared[mode][3]))
    rays = {mode: prepared[mode][3].last_stats.rays for mode in MODES}
    assert len(set(rays.values())) == 1, rays
    off = min(runs["off"])
    cols = "   ".join(f"{mode} {' '.join(f'{x:8.3f}' for x in runs[mode])} ms ({100 * (min(runs[mode]) / off - 1):+.1f} %)"
                      for mode in MODES)
    print(f"{name:16s} {cols}   rays {rays['off']}", flush=True)
    for _, _, _, p in prepared.values():
        p.release()
