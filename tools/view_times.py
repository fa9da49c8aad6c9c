"""A 36-view turntable of the bench workloads three ways, alternating in one process: (a) today's way, rtc_set_camera +
rtc_scene_commit + rtc_render per view; (b) rtc_render_views with one view per call; (c) one rtc_render_views call for all 36
views.  Each both device-resident (NULL, NULL) and into a pinned 8-bit canvas; host wall time of the whole turntable, best
of three alternating runs, reported per view.  The turntable: the workload camera's eye turned about the vertical axis
through its look-at point (scenes.orbit_cameras).  Prints the card's name and power limit.
    python tools/view_times.py [workload ...]   (c1 c3 c4 c5)"""
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ray_tracer_challenge_b200 as rt  # noqa: E402
from bench import build_scene  # noqa: E402
from ray_tracer_challenge_b200 import scenes  # noqa: E402

N_VIEWS = 36
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip(), flush=True)

lib = rt.device_library()
lib.rtc_last_error.restype = C.c_char_p
lib.rtc_host_alloc.restype = C.c_void_p
lib.rtc_host_free.argtypes = [C.c_void_p]
lib.rtc_set_camera.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_float)]
lib.rtc_scene_commit.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_int32)]
lib.rtc_render.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(rt.RtcStats)]
lib.rtc_render_views.argtypes = [C.c_void_p, C.c_int32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.POINTER(rt.RtcStats)]
lib.rtc_scene_destroy.argtypes = [C.c_void_p]


def check(rc):
    if rc < 0:
        raise RuntimeError(lib.rtc_last_error().decode())


def run(name):
    api = rt.new_session()
    api.set_render_options(device_ids=[0])
    cam, world = build_scene(api, name)[:2]
    w, h = cam.width_pixels, cam.height_pixels
    cams = scenes.orbit_cameras(api, cam, N_VIEWS)
    views = (rt.RtcView * N_VIEWS)(*[api.camera_view(c) for c in cams])
    far = cams[api.farthest_camera(cams)]
    # (a) one raw scene, re-committed for every view (the host SAH tree, as a prepared scene builds it)
    raw = api.export_scene(far, world)
    dev0 = (C.c_int32 * 1)(0)
    check(lib.rtc_scene_commit(raw, 1, dev0))
    # (b), (c) a scene committed once with the farthest camera
    once = api.export_scene(far, world)
    check(lib.rtc_scene_commit(once, 1, dev0))
    pinned = lib.rtc_host_alloc(C.c_size_t(N_VIEWS * w * h * 3))
    st = rt.RtcStats()

    def a(u8):
        for i in range(N_VIEWS):
            v = views[i]
            check(lib.rtc_set_camera(raw, w, h, v.half_width, v.half_height, v.pixel_size, v.transform_inverse))
            check(lib.rtc_scene_commit(raw, 1, dev0))
            check(lib.rtc_render(raw, 5, None, (u8 + i * w * h * 3) if u8 else None, C.byref(st)))

    def b(u8):
        for i in range(N_VIEWS):
            check(lib.rtc_render_views(once, 5, 1, C.addressof(views) + i * C.sizeof(rt.RtcView), None,
                                       (u8 + i * w * h * 3) if u8 else None, C.byref(st)))

    def c(u8):
        check(lib.rtc_render_views(once, 5, N_VIEWS, C.addressof(views), None, u8 if u8 else None, C.byref(st)))

    modes = {"a": a, "b": b, "c": c}
    for f in modes.values():  # warm-up: module load, first-touch of every buffer
        f(None), f(pinned)
    best = {(m, d): float("inf") for m in modes for d in ("device", "pinned_u8")}
    for _ in range(3):
        for m, f in modes.items():
            for d, dst in (("device", None), ("pinned_u8", pinned)):
                t0 = time.perf_counter()
                f(dst)
                best[(m, d)] = min(best[(m, d)], (time.perf_counter() - t0) * 1e3 / N_VIEWS)
    # the three ways render the same 36 frames
    frames = {}
    for m, f in modes.items():
        f(pinned)
        frames[m] = np.ctypeslib.as_array((C.c_uint8 * (N_VIEWS * w * h * 3)).from_address(pinned)).copy()
    same = frames["a"].tobytes() == frames["b"].tobytes() == frames["c"].tobytes()
    c(None)
    launches = st.launches
    cols = "  ".join(f"{m}: {best[(m, 'device')]:8.3f} / {best[(m, 'pinned_u8')]:8.3f}" for m in modes)
    print(f"{name:4s} {w}x{h}  ms per view (device / pinned u8)  {cols}   (c) launches {launches}  frames equal {same}", flush=True)
    lib.rtc_host_free(C.c_void_p(pinned))
    lib.rtc_scene_destroy(raw)
    lib.rtc_scene_destroy(once)


for workload in sys.argv[1:] or ["c1", "c3", "c4", "c5"]:
    run(workload)
