"""One frame's `Canvas::to_ppm` text written by N processes, one shard each, timed per rank:

    torchrun --nproc_per_node N tools/shard_ppm_times.py [workload ...]   (c1 c3 c4)   [--out results.json]

Rank r commits the workload on device r % device_count and runs multi.render_ppm_shared: rtc_render_shard_ppm_rows into the
row lengths of a multi.SharedText, a barrier, rtc_write_shard_ppm into its text, a barrier.  Timed per rank: phase 1, the wait
at the first barrier, phase 2, the wait at the second, and the whole frame; median of REPS frames, then the max over ranks.
Into the shared text registered with rtc_host_register (pinned) and unregistered (pageable).  For comparison, in the same
run: the single-process rtc_render_ppm (rank 0 alone, into pinned and pageable memory) and the N-rank rtc_render_shard of the
8-bit plane into a registered multi.SharedCanvas.  Rank 0 checks the shared text against rtc_render_ppm's.  The card's name
and power limit are read in the same run.  Ranks beyond the device count share devices: their times are not those of one
GPU per rank.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ctypes as C  # noqa: E402

import torch.distributed as dist  # noqa: E402

import ray_tracer_challenge_b200 as rt  # noqa: E402
from bench import build_scene  # noqa: E402
from ray_tracer_challenge_b200 import multi  # noqa: E402

REPS = 15
WARMUP = 3

lib = rt.device_library()
lib.rtc_host_register.argtypes = [C.c_void_p, C.c_size_t]
lib.rtc_host_unregister.argtypes = [C.c_void_p]
lib.rtc_host_alloc.restype = C.c_void_p
lib.rtc_host_alloc.argtypes = [C.c_size_t]
lib.rtc_host_free.argtypes = [C.c_void_p]
lib.rtc_ppm_bound.restype = C.c_size_t
lib.rtc_ppm_bound.argtypes = [C.c_uint32, C.c_uint32]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip()


def gather(value):
    out = [None] * dist.get_world_size()
    dist.all_gather_object(out, value)
    return out


def ms(t0, t1):
    return (t1 - t0) * 1e3


def shared_frames(prepared, text, rank, n):
    """REPS frames of render_ppm_shared's two phases and two barriers, each part timed on this rank (medians, ms)."""
    parts = {"phase1": [], "wait1": [], "phase2": [], "wait2": [], "frame": []}
    for k in range(WARMUP + REPS):
        dist.barrier()
        t0 = time.perf_counter()
        prepared.render_shard_ppm_rows(rank, n, text.row_bytes, 5)
        t1 = time.perf_counter()
        dist.barrier()
        t2 = time.perf_counter()
        length = prepared.write_shard_ppm(rank, n, text.row_bytes, text.buf)
        t3 = time.perf_counter()
        dist.barrier()
        t4 = time.perf_counter()
        if k >= WARMUP:
            for key, v in (("phase1", ms(t0, t1)), ("wait1", ms(t1, t2)), ("phase2", ms(t2, t3)), ("wait2", ms(t3, t4)),
                           ("frame", ms(t0, t4))):
                parts[key].append(v)
    return {k: float(np.median(v)) for k, v in parts.items()}, length


def run(api, name, rank, n):
    cam, world = build_scene(api, name)[:2]
    w, h = cam.width_pixels, cam.height_pixels
    prepared = cam.prepare(world)
    port = os.environ.get("MASTER_PORT", "0")
    text = multi.open_shared_text(dist, rank, f"rtc_shard_ppm_times_{port}_{name}", w, h)
    row = {"size": f"{w}x{h}", "ranks": n}
    for mode in ("unregistered", "registered"):
        if mode == "registered":
            assert lib.rtc_host_register(text.address, text.nbytes) == 0
        parts, length = shared_frames(prepared, text, rank, n)
        per_rank = gather(parts)
        if rank == 0:
            row[mode] = {"max_over_ranks": {k: round(max(p[k] for p in per_rank), 3) for k in parts},
                         "per_rank": [{k: round(v, 3) for k, v in p.items()} for p in per_rank]}
            row["text_MB"] = round(length / 1e6, 3)
            row.setdefault("text_equals_render_ppm", True)
            row["text_equals_render_ppm"] &= text.text(length) == prepared.render_ppm(5)
        dist.barrier()
        if mode == "registered":
            lib.rtc_host_unregister(text.address)
    # the single-process rtc_render_ppm, rank 0 alone
    if rank == 0:
        bound = lib.rtc_ppm_bound(w, h)
        ptr = lib.rtc_host_alloc(bound)
        pinned = np.ctypeslib.as_array((C.c_uint8 * bound).from_address(ptr))
        pageable = np.zeros(bound, np.uint8)
        st = rt.SgStats()
        for dest, buf in (("pinned", pinned), ("pageable", pageable)):
            times = []
            for k in range(WARMUP + REPS):  # the library call alone (PreparedScene.render_ppm also decodes the text to a str)
                t0 = time.perf_counter()
                api.check(api.lib.sg_render_prepared_ppm(api.ctx, prepared.handle, 5, 0, buf.ctypes.data, buf.nbytes, C.byref(st)))
                if k >= WARMUP:
                    times.append(ms(t0, time.perf_counter()))
            row[f"render_ppm_one_process_{dest}"] = round(float(np.median(times)), 3)
        lib.rtc_host_free(C.c_void_p(ptr))
    dist.barrier()
    # the N-rank rtc_render_shard of the 8-bit plane into a registered shared canvas
    canvas = multi.open_shared_canvas(dist, rank, f"rtc_shard_ppm_times_canvas_{port}_{name}", w, h)
    assert lib.rtc_host_register(canvas.address, canvas.nbytes) == 0
    times = []
    for k in range(WARMUP + REPS):
        dist.barrier()
        t0 = time.perf_counter()
        prepared.render(5, out_u8=canvas.u8, want_rgb=False, shard=rank, n_shards=n)
        dist.barrier()
        if k >= WARMUP:
            times.append(ms(t0, time.perf_counter()))
    frame = gather(float(np.median(times)))
    if rank == 0:
        row["render_shard_u8_frame_max_over_ranks"] = round(max(frame), 3)
    lib.rtc_host_unregister(canvas.address)
    dist.barrier()
    canvas.close()
    text.close()
    prepared.release()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("workloads", nargs="*", default=["c1", "c3", "c4"])
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file (rank 0)")
    args = ap.parse_args()
    dist.init_process_group("gloo")
    rank, n = dist.get_rank(), dist.get_world_size()
    devices = lib.rtc_device_count()
    api = rt.new_session()
    api.set_render_options(device_ids=[rank % devices])
    result = {"card": card() if rank == 0 else None, "ranks": n, "devices": devices, "workloads": {}}
    if rank == 0:
        print("card:", result["card"], "| ranks:", n, "| devices:", devices, flush=True)
    for name in args.workloads:
        row = run(api, name, rank, n)
        if rank == 0:
            result["workloads"][name] = row
            print(name, json.dumps(row), flush=True)
    if rank == 0 and args.out:
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
