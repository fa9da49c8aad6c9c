"""A 36-view turntable of c1, c3 and c4 written as PPM text (`Canvas::to_ppm` of every view) three ways, alternating in one
process:

    (a) per view    rtc_set_camera + rtc_scene_commit + rtc_render_ppm
    (b) planes      one rtc_render_views into a pinned 8-bit plane, then the host writer (sg_ppm_from_u8) per view
    (c) views_ppm   one rtc_render_views_ppm

Each flow writes its 36 texts one after the other into pinned memory and into a (reused) pageable array.  Host wall time of
the whole turntable, best of three alternating runs, reported per view.  The three flows must produce the same 36 texts.
Then, in a separate profiled pass (torch.profiler with CUDA activities), the text kernels of one (c) call into pinned
memory.  The turntable: the workload camera's eye turned about the vertical axis through its look-at point
(scenes.orbit_cameras), committed once with the farthest camera for (b) and (c).  The card's name, power limit and max SM
clock are read in the same call.

    python tools/views_ppm_times.py [workload ...]   (c1 c3 c4)   [--out results.json]
"""
import argparse
import ctypes as C
import hashlib
import json
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
REPS = 3

lib = rt.device_library()
lib.rtc_last_error.restype = C.c_char_p
lib.rtc_host_alloc.restype = C.c_void_p
lib.rtc_host_alloc.argtypes = [C.c_size_t]
lib.rtc_host_free.argtypes = [C.c_void_p]
lib.rtc_ppm_bound.restype = C.c_size_t
lib.rtc_ppm_bound.argtypes = [C.c_uint32, C.c_uint32]
lib.rtc_set_camera.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_float)]
lib.rtc_scene_commit.argtypes = [C.c_void_p, C.c_int32, C.POINTER(C.c_int32)]
lib.rtc_render_ppm.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(rt.RtcStats)]
lib.rtc_render_views.argtypes = [C.c_void_p, C.c_int32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.POINTER(rt.RtcStats)]
lib.rtc_render_views_ppm.argtypes = [C.c_void_p, C.c_int32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_size_t,
                                     C.POINTER(C.c_size_t), C.POINTER(rt.RtcStats)]
lib.rtc_scene_destroy.argtypes = [C.c_void_p]


def check(rc):
    if rc < 0:
        raise RuntimeError(lib.rtc_last_error().decode())
    return rc


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def text_kernels_ms(fn):
    """ppm_row_bytes and ppm_write device time of one call (torch.profiler, CUDA activities), summed per kernel name."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {"ppm_row_bytes": 0.0, "ppm_write": 0.0}
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        for k in out:
            if k in e.name:
                out[k] += e.device_time_total / 1000.0  # us -> ms
    return out


def run(api, name):
    cam, world = build_scene(api, name)[:2]
    w, h = cam.width_pixels, cam.height_pixels
    cams = scenes.orbit_cameras(api, cam, N_VIEWS)
    views = (rt.RtcView * N_VIEWS)(*[api.camera_view(c) for c in cams])
    far = cams[api.farthest_camera(cams)]
    dev0 = (C.c_int32 * 1)(0)
    raw = api.export_scene(far, world)  # (a): re-committed for every view
    check(lib.rtc_scene_commit(raw, 1, dev0))
    once = api.export_scene(far, world)  # (b), (c): committed once with the farthest camera
    check(lib.rtc_scene_commit(once, 1, dev0))
    bound = lib.rtc_ppm_bound(w, h)
    cap = N_VIEWS * bound
    plane = lib.rtc_host_alloc(N_VIEWS * w * h * 3)
    pinned_ptr = lib.rtc_host_alloc(cap)
    assert plane and pinned_ptr, "rtc_host_alloc failed"
    pageable = np.empty(cap, np.uint8)
    pageable[:] = 0  # first touch outside the timed runs
    dests = {"pinned": pinned_ptr, "pageable": pageable.ctypes.data}
    st = rt.RtcStats()
    offsets = (C.c_size_t * (N_VIEWS + 1))()

    def a(dst):
        at = 0
        n = C.c_size_t()
        for i in range(N_VIEWS):
            v = views[i]
            check(lib.rtc_set_camera(raw, w, h, v.half_width, v.half_height, v.pixel_size, v.transform_inverse))
            check(lib.rtc_scene_commit(raw, 1, dev0))
            check(lib.rtc_render_ppm(raw, 5, dst + at, cap - at, C.byref(n), C.byref(st)))
            offsets[i] = at
            at += n.value
        offsets[N_VIEWS] = at

    def b(dst):
        check(lib.rtc_render_views(once, 5, N_VIEWS, C.addressof(views), None, plane, C.byref(st)))
        at = 0
        for i in range(N_VIEWS):
            n = check(api.lib.sg_ppm_from_u8(api.ctx, w, h, C.cast(plane + i * w * h * 3, rt._api.U8P),
                                             C.cast(dst + at, C.c_char_p), cap - at))
            offsets[i] = at
            at += n
        offsets[N_VIEWS] = at

    def c(dst):
        check(lib.rtc_render_views_ppm(once, 5, N_VIEWS, C.addressof(views), dst, cap, offsets, C.byref(st)))

    def texts(dst):  # each view's text as its digest (c3's 36 texts are 2.8 GB)
        return [hashlib.sha256((C.c_char * (offsets[i + 1] - offsets[i])).from_address(dst + offsets[i]).raw).hexdigest()
                for i in range(N_VIEWS)]

    flows = {"a": a, "b": b, "c": c}
    out = {}
    for m, f in flows.items():  # warm-up (module load, first touch of every buffer), and the texts of each flow
        for d, dst in dests.items():
            f(dst)
            out[(m, d)] = texts(dst)
    same = all(t == out[("a", "pinned")] for t in out.values())
    launches = None
    best = {(m, d): float("inf") for m in flows for d in dests}
    for _ in range(REPS):
        for m, f in flows.items():
            for d, dst in dests.items():
                t0 = time.perf_counter()
                f(dst)
                best[(m, d)] = min(best[(m, d)], (time.perf_counter() - t0) * 1e3 / N_VIEWS)
                if m == "c":
                    launches = st.launches
    c(pinned_ptr)
    row = {"size": f"{w}x{h}", "text_MB_per_view": round(offsets[N_VIEWS] / N_VIEWS / 1e6, 3),
           "ms_per_view": {f"{m}_{d}": round(v, 3) for (m, d), v in best.items()},
           "c_render_launches": launches, "c_kernel_ms_per_view": round(st.kernel_ms / N_VIEWS, 4), "texts_equal": same}
    try:
        k = text_kernels_ms(lambda: c(pinned_ptr))
        row["c_text_kernels_ms_per_view"] = {n: round(v / N_VIEWS, 4) for n, v in k.items()}
    except Exception as e:  # a separate pass: report what failed, keep the wall times
        row["c_text_kernels_ms_per_view"] = f"not captured: {type(e).__name__}: {e}"
    lib.rtc_host_free(C.c_void_p(plane))
    lib.rtc_host_free(C.c_void_p(pinned_ptr))
    lib.rtc_scene_destroy(raw)
    lib.rtc_scene_destroy(once)
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("workloads", nargs="*", default=["c1", "c3", "c4"])
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    args = ap.parse_args()
    result = {"card": card(), "n_views": N_VIEWS, "workloads": {}}
    print("card:", result["card"], flush=True)
    api = rt.new_session()
    api.set_render_options(device_ids=[0])
    for name in args.workloads:
        row = run(api, name)
        result["workloads"][name] = row
        print(name, json.dumps(row), flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
