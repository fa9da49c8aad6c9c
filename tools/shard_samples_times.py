"""Anti-aliased frames rendered by N processes, one shard each, timed per rank:

    torchrun --nproc-per-node N tools/shard_samples_times.py [workload ...]   (c1 c3 c4)   [--samples 2 4] [--out results.json]

Rank r commits the workload on device r % device_count.  For each workload and n samples per axis:
  - kernel: RtcStats.kernel_ms of rtc_render_shard_samples (shard r of N, the frame left on the device), FRAMES frames after a
    barrier each; per rank the median and range, then the max over ranks;
  - frame: host wall time of one frame's 8-bit plane into a registered multi.SharedCanvas (every rank's render, then a
    barrier), median of FRAMES frames, max over ranks;
  - text: host wall time of multi.render_ppm_shared(samples=n) into a registered multi.SharedText (both phases and both
    barriers), median, max over ranks;
  - baseline, in the same run: rank 0 alone, the single-process rtc_render_samples on one GPU — its kernel_ms, its 8-bit plane
    into the same registered canvas, and its text (rtc_render_views_samples_ppm of the committed camera, the path of
    render_samples_ppm) into the registered shared text — while the other ranks wait.
Speed-up = baseline / N-rank figure.  Rank 0 checks the shared frame and text against the single-process ones.  The card's
name, power limit and max SM clock are read in the same run.  Ranks beyond the device count share devices: their times are
not those of one GPU per rank.
"""
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
import torch.distributed as dist  # noqa: E402

import ray_tracer_challenge_b200 as rt  # noqa: E402
from bench import WORKLOADS  # noqa: E402
from ray_tracer_challenge_b200 import multi, scenes  # noqa: E402

FRAMES = 25
WARMUP = 3

lib = rt.device_library()
lib.rtc_host_register.argtypes = [C.c_void_p, C.c_size_t]
lib.rtc_host_unregister.argtypes = [C.c_void_p]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return q.stdout.strip()


def gather(value):
    out = [None] * dist.get_world_size()
    dist.all_gather_object(out, value)
    return out


def spread(v):
    return {"median_ms": round(float(np.median(v)), 4), "min_ms": round(float(np.min(v)), 4), "max_ms": round(float(np.max(v)), 4)}


def timed(fn, barrier=True):
    """FRAMES host wall times (ms) of fn() after WARMUP calls; each call starts behind a barrier"""
    out = []
    for k in range(WARMUP + FRAMES):
        if barrier:
            dist.barrier()
        t0 = time.perf_counter()
        fn()
        if k >= WARMUP:
            out.append((time.perf_counter() - t0) * 1e3)
    return out


def kernel_times(p, fn, barrier=True):
    out = []
    for k in range(WARMUP + FRAMES):
        if barrier:
            dist.barrier()
        fn()
        if k >= WARMUP:
            out.append(p.last_stats.kernel_ms)
    return out


def run(api, name, samples, rank, n_ranks):
    builder, kw, depth, _ = WORKLOADS[name]
    cam, world = getattr(scenes, builder)(api, **kw)
    w, h = cam.width_pixels, cam.height_pixels
    p = cam.prepare(world)
    port = os.environ.get("MASTER_PORT", "0")
    canvas = multi.open_shared_canvas(dist, rank, f"rtc_shard_samples_times_canvas_{port}_{name}", w, h)
    text = multi.open_shared_text(dist, rank, f"rtc_shard_samples_times_text_{port}_{name}", w, h)
    assert lib.rtc_host_register(canvas.address, canvas.nbytes) == 0
    assert lib.rtc_host_register(text.address, text.nbytes) == 0
    rows = []
    for n in samples:
        row = {"workload": name, "size": f"{w}x{h}", "n": n, "ranks": n_ranks}
        kern = kernel_times(p, lambda: p.render_samples(n, depth, want_rgb=False, want_u8=False, shard=rank, n_shards=n_ranks))

        def frame():
            p.render_samples(n, depth, want_rgb=False, out_u8=canvas.u8, shard=rank, n_shards=n_ranks)
            dist.barrier()

        wall = timed(frame)
        length = 0

        def shared_text():
            nonlocal length
            length = multi.render_ppm_shared(dist, rank, n_ranks, p, text, depth, samples=n)

        txt = timed(shared_text)
        per_rank = gather({"kernel": spread(kern), "frame": spread(wall), "text": spread(txt)})
        if rank == 0:
            for key in ("kernel", "frame", "text"):
                row[key] = {"max_over_ranks_median_ms": max(r[key]["median_ms"] for r in per_rank),
                            "per_rank": [r[key] for r in per_rank]}
            whole = p.render_samples(n, depth)
            row["frame_equals_render_samples"] = bool(np.array_equal(canvas.u8, whole.to_u8()))
            row["text_equals_render_samples_ppm"] = text.text(length) == p.render_samples_ppm(n, depth)
            # the single-process baseline on one GPU, rank 0 alone
            base_kern = kernel_times(p, lambda: p.render_samples(n, depth, want_rgb=False, want_u8=False), barrier=False)
            base_wall = timed(lambda: p.render_samples(n, depth, want_rgb=False, out_u8=canvas.u8), barrier=False)
            # the library call alone (PreparedScene.render_samples_ppm also decodes the text to a str)
            offsets, st = (C.c_size_t * 2)(), rt.SgStats()
            one = (C.c_int * 1)(cam.handle)
            base_txt = timed(lambda: api.check(api.lib.sg_render_prepared_views_samples_ppm(
                api.ctx, p.handle, depth, 1, one, n, 0, text.buf.ctypes.data, text.buf.nbytes, offsets, C.byref(st))), barrier=False)
            row["baseline_one_process"] = {"kernel": spread(base_kern), "frame": spread(base_wall), "text": spread(base_txt)}
            row["speedup"] = {k: round(row["baseline_one_process"][k]["median_ms"] / row[k]["max_over_ranks_median_ms"], 3)
                              for k in ("kernel", "frame", "text")}
            print(json.dumps(row), flush=True)
        dist.barrier()
        rows.append(row)
    lib.rtc_host_unregister(canvas.address)
    lib.rtc_host_unregister(text.address)
    dist.barrier()
    canvas.close()
    text.close()
    p.release()
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("workloads", nargs="*", default=["c1", "c3", "c4"])
    ap.add_argument("--samples", type=int, nargs="+", default=[2, 4])
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file (rank 0)")
    args = ap.parse_args()
    dist.init_process_group("gloo")
    rank, n_ranks = dist.get_rank(), dist.get_world_size()
    devices = lib.rtc_device_count()
    api = rt.new_session()
    api.set_render_options(device_ids=[rank % devices])
    result = {"card": card() if rank == 0 else None, "ranks": n_ranks, "devices": devices, "rows": []}
    if rank == 0:
        print("card:", result["card"], "| ranks:", n_ranks, "| devices:", devices, flush=True)
    for name in args.workloads:
        result["rows"] += run(api, name, args.samples, rank, n_ranks)
    if rank == 0 and args.out:
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
