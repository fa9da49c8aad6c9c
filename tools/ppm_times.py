"""Times the demos' last step, `camera.render(world, 5).to_ppm()`, two ways, on c3, c3_counter (generated jitter), c1 and c4:

    (a) u8   one-shot Camera.render_b200_u8 (the 8-bit plane leaves the device), then CanvasU8.to_ppm on the host
    (b) ppm  one-shot Camera.render_b200_ppm (rtc_render_ppm: the text is written on the device and copied out)

For each flow the host wall time of the whole Python call (flatten, commit, render, text as a str) into pinned and into
pageable memory, best of --reps runs with the flows alternating; for (a) also the host writer alone.  Then, in a separate
profiled pass (torch.profiler with CUDA activities), the kernels and device-to-host copies of one call of each flow: the
encode kernels' time and the text copy.  The card's name and power limit are read in the same call.

    python tools/ppm_times.py [--reps 5] [--out results.json]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import ray_tracer_challenge_b200 as rt  # noqa: E402
from ray_tracer_challenge_b200 import scenes  # noqa: E402

WORKLOADS = {  # bench.py's definitions
    "c3": ("soft_shadows", dict(width=3840, height=2160, u_steps=4, v_steps=4)),
    "c3_counter": ("soft_shadows", dict(width=3840, height=2160, u_steps=4, v_steps=4, jitter=None, seed=7)),
    "c1": ("soft_shadows", dict(width=1000, height=400, u_steps=10, v_steps=10)),
    "c4": ("dragon_element", dict(width=1920, height=1080, n_u=320, n_v=160)),
}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def pinned(nbytes):
    lib = rt.device_library()
    lib.rtc_host_alloc.restype = C.c_void_p
    lib.rtc_host_alloc.argtypes = [C.c_size_t]
    ptr = lib.rtc_host_alloc(nbytes)
    if not ptr:
        raise RuntimeError("rtc_host_alloc failed")
    return np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(ptr))


def flows(gpu, name):
    build, kw = WORKLOADS[name]
    cam, world = getattr(scenes, build)(gpu, **kw)
    w, h = cam.width_pixels, cam.height_pixels
    u8_pinned = pinned(w * h * 3).reshape(h, w, 3)
    text_pinned = pinned(gpu.lib.rtc_ppm_bound(w, h))
    return cam, world, {
        "u8_pageable": lambda: cam.render_b200_u8(world, 5).to_ppm(),
        "u8_pinned": lambda: cam.render_b200_u8(world, 5, out_u8=u8_pinned).to_ppm(),
        "ppm_pageable": lambda: cam.render_b200_ppm(world, 5),
        "ppm_pinned": lambda: cam.render_b200_ppm(world, 5, out=text_pinned),
    }


def profile(fn):
    """Kernel and copy times of one call (torch.profiler, CUDA activities): per kernel name, and device-to-host copies."""
    import torch
    from torch.profiler import ProfilerActivity, profile as tprofile

    torch.cuda.init()
    with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        name = e.name if not e.name.lower().startswith("memcpy") else e.name.split()[0] + " " + ("DtoH" if "DtoH" in e.name else e.name)
        key = "ppm_write" if "ppm_write" in name else "ppm_row_bytes" if "ppm_row_bytes" in name else \
            ("memcpy DtoH" if "DtoH" in name or "Device -> Pageable" in name or "Device -> Pinned" in name else
             "render kernels" if "render" in name else name[:40])
        out[key] = out.get(key, 0.0) + e.device_time_total / 1000.0  # us -> ms
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    ap.add_argument("--workloads", default="c3,c3_counter,c1,c4")
    args = ap.parse_args()
    gpu = rt.new_session()
    gpu.set_render_options(n_devices=1)
    result = {"card": card(), "workloads": {}}
    print("card:", result["card"], flush=True)
    for name in args.workloads.split(","):
        cam, world, fs = flows(gpu, name)
        texts = {k: f() for k, f in fs.items()}  # warm-up, and every flow writes the same text
        assert len(set(texts.values())) == 1, name
        text_mb = len(texts["ppm_pinned"]) / 1e6
        best = {k: float("inf") for k in fs}
        lib_ms = {k: float("inf") for k in fs}
        canvas = cam.render_b200_u8(world, 5)
        writer = float("inf")
        for _ in range(args.reps):
            for k, f in fs.items():
                t0 = time.perf_counter()
                f()
                best[k] = min(best[k], (time.perf_counter() - t0) * 1e3)
                if k.startswith("ppm"):
                    lib_ms[k] = min(lib_ms[k], cam.last_rtc_stats.total_ms)
            t0 = time.perf_counter()
            canvas.to_ppm()
            writer = min(writer, (time.perf_counter() - t0) * 1e3)
        row = {"text_MB": round(text_mb, 2), "wall_ms_best": {k: round(v, 3) for k, v in best.items()},
               "host_writer_ms_best": round(writer, 3),
               "rtc_render_ppm_total_ms_best": {k: round(v, 3) for k, v in lib_ms.items() if v != float("inf")}}
        try:
            row["profile_ms"] = {k: {n: round(v, 4) for n, v in profile(f).items()} for k, f in fs.items() if k.startswith("ppm")}
        except Exception as e:  # the profile is a separate pass: report what failed, keep the wall times
            row["profile_ms"] = f"not captured: {type(e).__name__}: {e}"
        result["workloads"][name] = row
        print(name, json.dumps(row), flush=True)
    if args.out:
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
