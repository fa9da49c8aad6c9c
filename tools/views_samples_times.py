"""Anti-aliased turntables: a 36-view turntable (scenes.orbit_cameras, as tools/view_times.py builds it) of the bench workloads
at n samples per axis, three ways alternating in one process: (a) rtc_set_camera + rtc_scene_commit + rtc_render_samples per
view; (b) rtc_render_views_samples with one view per call; (c) one rtc_render_views_samples call for all 36 views.  Each both
device-resident (NULL, NULL) and into a pinned 8-bit canvas; host wall time of the whole turntable, best of three alternating
runs, reported per view.  Then the texts: rtc_render_views_samples_ppm of the 36 views into pageable memory, against (c)
into the pinned canvas followed by the host writer (ppm_from_u8) of every view.  Prints the card's name, power limit and
clock in the same run.
    python tools/views_samples_times.py [--samples 1 2 4] [workload ...]   (default: c1 c3 c4)"""
import argparse
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

lib = rt.device_library()
lib.rtc_last_error.restype = C.c_char_p
lib.rtc_host_alloc.restype = C.c_void_p
lib.rtc_host_free.argtypes = [C.c_void_p]
lib.rtc_set_camera.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_float)]
lib.rtc_scene_commit.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_int32)]
lib.rtc_render_samples.argtypes = [C.c_void_p, C.c_int32, C.c_uint32, C.c_void_p, C.c_void_p, C.POINTER(rt.RtcStats)]
lib.rtc_render_views_samples.argtypes = [C.c_void_p, C.c_int32, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p,
                                         C.POINTER(rt.RtcStats)]
lib.rtc_render_views_samples_ppm.argtypes = [C.c_void_p, C.c_int32, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t,
                                             C.c_void_p, C.POINTER(rt.RtcStats)]
lib.rtc_ppm_bound.restype = C.c_size_t
lib.rtc_ppm_bound.argtypes = [C.c_uint32, C.c_uint32]
lib.rtc_scene_destroy.argtypes = [C.c_void_p]


def check(rc):
    if rc < 0:
        raise RuntimeError(lib.rtc_last_error().decode())


def run(name, samples):
    api = rt.new_session()
    api.set_render_options(device_ids=[0])
    cam, world = build_scene(api, name)[:2]
    w, h = cam.width_pixels, cam.height_pixels
    cams = scenes.orbit_cameras(api, cam, N_VIEWS)
    views = (rt.RtcView * N_VIEWS)(*[api.camera_view(c) for c in cams])
    far = cams[api.farthest_camera(cams)]
    dev0 = (C.c_int32 * 1)(0)
    raw = api.export_scene(far, world)  # (a): re-committed for every view
    check(lib.rtc_scene_commit(raw, 1, dev0))
    once = api.export_scene(far, world)  # (b), (c), text: committed once with the farthest camera
    check(lib.rtc_scene_commit(once, 1, dev0))
    frame = w * h * 3
    pinned = lib.rtc_host_alloc(C.c_size_t(N_VIEWS * frame))
    bound = lib.rtc_ppm_bound(w, h)
    text = np.empty(N_VIEWS * bound, np.uint8)
    offsets = (C.c_size_t * (N_VIEWS + 1))()
    st = rt.RtcStats()
    for n in samples:
        def a(u8):
            for i in range(N_VIEWS):
                v = views[i]
                check(lib.rtc_set_camera(raw, w, h, v.half_width, v.half_height, v.pixel_size, v.transform_inverse))
                check(lib.rtc_scene_commit(raw, 1, dev0))
                check(lib.rtc_render_samples(raw, 5, n, None, (u8 + i * frame) if u8 else None, C.byref(st)))

        def b(u8):
            for i in range(N_VIEWS):
                check(lib.rtc_render_views_samples(once, 5, 1, C.addressof(views) + i * C.sizeof(rt.RtcView), n, None,
                                                   (u8 + i * frame) if u8 else None, C.byref(st)))

        def c(u8):
            check(lib.rtc_render_views_samples(once, 5, N_VIEWS, C.addressof(views), n, None, u8 if u8 else None, C.byref(st)))

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
        frames = {}
        for m, f in modes.items():  # the three ways render the same 36 frames
            f(pinned)
            frames[m] = np.ctypeslib.as_array((C.c_uint8 * (N_VIEWS * frame)).from_address(pinned)).copy()
        same = frames["a"].tobytes() == frames["b"].tobytes() == frames["c"].tobytes()
        c(None)
        launches = st.launches
        cols = "  ".join(f"{m}: {best[(m, 'device')]:8.3f} / {best[(m, 'pinned_u8')]:8.3f}" for m in modes)
        print(f"{name:4s} {w}x{h} n={n}  ms per view (device / pinned u8)  {cols}   (c) launches {launches}  frames equal {same}",
              flush=True)

        # the texts: on the device, against (c) into the pinned canvas then the host writer of every view
        def device_text():
            check(lib.rtc_render_views_samples_ppm(once, 5, N_VIEWS, C.addressof(views), n, text.ctypes.data, text.nbytes, offsets,
                                                   C.byref(st)))

        def host_text():
            c(pinned)
            u8 = np.ctypeslib.as_array((C.c_uint8 * (N_VIEWS * frame)).from_address(pinned)).reshape(N_VIEWS, h, w, 3)
            return [rt.CanvasU8(w, h, u8[i], api).to_ppm() for i in range(N_VIEWS)]

        device_text()
        t_dev = float("inf")
        for _ in range(3):
            t0 = time.perf_counter()
            device_text()
            t_dev = min(t_dev, (time.perf_counter() - t0) * 1e3 / N_VIEWS)
        t0 = time.perf_counter()
        want = host_text()
        t_host = (time.perf_counter() - t0) * 1e3 / N_VIEWS
        got = [text[offsets[i]:offsets[i + 1]].tobytes().decode("ascii") for i in range(N_VIEWS)]
        print(f"{name:4s} {w}x{h} n={n}  text ms per view: rtc_render_views_samples_ppm {t_dev:8.3f}   (c) + host writer {t_host:8.3f}"
              f"   texts equal {got == want}", flush=True)
    lib.rtc_host_free(C.c_void_p(pinned))
    lib.rtc_scene_destroy(raw)
    lib.rtc_scene_destroy(once)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("workloads", nargs="*", default=["c1", "c3", "c4"])
    ap.add_argument("--samples", type=int, nargs="+", default=[1, 2, 4])
    args = ap.parse_args()
    print(subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip(), flush=True)
    for workload in args.workloads:
        run(workload, args.samples)


if __name__ == "__main__":
    main()
