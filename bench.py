#!/usr/bin/env python
"""bench.py — the reference's headline metric on B200: Mrays/s and frame ms of `Camera::render`
(lib/src/camera.rs:76-91), beside the CPU render of the same frame.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c3] [--impl ours|reference] [--dump-outputs DIR]

A *step* is one frame of the workload (default c3 = BASELINE.json configs[2]: the soft-shadow scene at
3840x2160 with a 4x4 = 16-cell jittered area light, reflections, depth 5 — the frame the north-star target is
quoted on).  A *ray* is one World::intersect query: primary + reflect/refract + shadow (SURVEY.md §8d).

    value        Mrays/s with the scene resident in HBM and the frame left on the device; per-step time = the
                 CUDA-event duration of the render kernel, max over ranks
    e2e          the same frame through Camera::render_b200 (flatten + commit + render + D2H of the f32 and 8-bit
                 canvases into pinned host memory), host wall clock
    roofline     algorithmic FP32 flops of the frame (detailed pass, SURVEY.md Appendix E) / kernel time, against
                 the FP32 peak measured live by the K5 FMA micro-benchmark
    cpu_baseline the CPU oracle (a C++ port of the reference; Rust is not installed) on a bounded row sample

Multi-GPU: one process per GPU (torchrun), the frame's 8-row bands interleaved over the ranks (strong scaling of
one frame, no collective on the data path; every rank writes its bands into one shared host canvas).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (scene builder name, kwargs, depth, description)
    "c1": ("soft_shadows", dict(width=1000, height=400, u_steps=10, v_steps=10), 5,
           "soft_shadows demo as shipped: 1000x400, 10x10-cell area light, depth 5"),
    "c2": ("reflect_refract", dict(width=1920, height=1080), 5,
           "chapter-11 reflect/refract scene at 1920x1080, point light, depth 5"),
    "c3": ("soft_shadows", dict(width=3840, height=2160, u_steps=4, v_steps=4), 5,
           "soft-shadow + reflection scene at 3840x2160, 4x4 = 16 jittered light cells, depth 5"),
    "c3_counter": ("soft_shadows", dict(width=3840, height=2160, u_steps=4, v_steps=4, jitter=None, seed=7), 5,
                   "the c3 frame with the light as the demo ships it: jitter_fn = None (rectangle_light.rs:46), i.e. 32 generated "
                   "jitter values per shade instead of a fixed table"),
    "c4": ("dragon_element", dict(width=1920, height=1080, n_u=320, n_v=160), 5,
           "synthetic 102k-triangle OBJ mesh in divided groups (here_be_dragons element) at 1920x1080"),
    "c5": ("stress", dict(width=3840, height=2160, n_spheres=100_000), 5,
           "100k-sphere field + cylinders/cones/cubes + CSG + checker plane at 3840x2160"),
}


def sample_clocks(stop: threading.Event, out: list, gpu_index: int) -> None:
    """One streaming nvidia-smi (-lms 50) for the whole timed region; every line is one sample."""
    q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    try:
        proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(gpu_index),
                                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except Exception:
        return

    def reader():
        for line in proc.stdout:
            parts = [p.strip() for p in line.strip().split(",")]
            if len(parts) >= 6:
                out.append(parts)

    t = threading.Thread(target=reader, daemon=True)
    t.start()
    stop.wait()
    proc.terminate()
    t.join(timeout=2)


def clocks_summary(samples: list) -> dict:
    if not samples:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
    sm = sorted(int(s[0]) for s in samples if s[0].isdigit())
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in samples)]
    return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": int(samples[0][1]) if samples[0][1].isdigit() else None,
            "reasons": reasons, "samples": len(samples)}


def config_of(workload: str, w: int, h: int, depth: int, n_gpus: int, fma: bool = False) -> dict:
    """The `config` object of the JSON line — the SAME dict for this arm and for `--impl reference`, so the two lines
    name one workload (the keys describing the GPU run say so)."""
    return {"workload": f"{workload}: {WORKLOADS[workload][3]}", "resolution": [w, h], "depth": depth,
            "kernel_build": "fma-contracted" if fma else "ieee (no contraction, bit-exact vs the oracle)",
            "l2": "GPU arm: flushed between timed iterations (256 MiB memset); CPU arm: n/a",
            "sharding": f"{n_gpus} rank(s), interleaved 8-row bands (GPU arm)"}


def build_scene(api, workload: str):
    from ray_tracer_challenge_b200 import scenes

    name, kw, depth, desc = WORKLOADS[workload]
    cam, world = getattr(scenes, name)(api, **kw)
    return cam, world, depth, desc


def cpu_baseline(workload: str, threads: int, target_seconds: float = 12.0) -> dict:
    """The oracle (C++ port of the reference) on a bounded sample: every `ystep`-th row of the same frame."""
    from tests.oracle_binding import load_oracle

    oracle = load_oracle()
    cam, world, depth, _ = build_scene(oracle, workload)
    h = cam.height_pixels
    oracle.probe.set_threads(threads)
    # calibrate on a very sparse sample, then choose the row stride for ~target_seconds of work
    probe_step = max(1, h // 16)
    t0 = time.perf_counter()
    _, _, st = oracle.probe.render_rows(cam, world, depth, probe_step // 2, h, probe_step)
    dt = max(time.perf_counter() - t0, 1e-4)
    rows_probe = max(1, len(range(probe_step // 2, h - 1, probe_step)))
    per_row = dt / rows_probe
    rows_target = int(max(8, min(h - 1, target_seconds / per_row)))
    ystep = max(1, (h - 1) // rows_target)
    t0 = time.perf_counter()
    _, _, st = oracle.probe.render_rows(cam, world, depth, ystep // 2, h, ystep)
    dt = time.perf_counter() - t0
    rows = len(range(ystep // 2, h - 1, ystep))
    mrays = st.rays / dt / 1e6
    return {"value": round(mrays, 4), "unit": "Mrays/s", "cores": threads, "kind": "port",
            "sample": f"rows {ystep // 2}::{ystep} of the {cam.width_pixels}x{h} frame ({rows} rows, {st.rays} rays, {dt:.2f} s)",
            "est_frame_ms": round(dt * (h - 1) / rows * 1e3, 1),
            # the reference algorithm's own work for the frame (every ray against every object, Appendix E units)
            "reference_flops_per_frame": float(st.flops) * (h - 1) / rows}


def run_reference(args) -> None:
    """--impl reference: the reference's CPU algorithm (oracle port; Rust is not installed) with every host thread."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from tests.oracle_binding import load_oracle

    oracle = load_oracle()
    threads = oracle.probe.max_threads()
    oracle.probe.set_threads(threads)
    cam, world, depth, desc = build_scene(oracle, args.workload)
    h = cam.height_pixels
    # one step = every `ystep`-th row; size the stride so warmup+steps finish within a few minutes
    t0 = time.perf_counter()
    probe_step = max(1, h // 16)
    oracle.probe.render_rows(cam, world, depth, 0, h, probe_step)
    per_row = (time.perf_counter() - t0) / max(1, len(range(0, h - 1, probe_step)))
    budget = 150.0 / max(1, args.steps + args.warmup)
    ystep = max(1, int(np.ceil((h - 1) * per_row / budget)))
    rays = 0
    for _ in range(args.warmup):
        oracle.probe.render_rows(cam, world, depth, 0, h, ystep)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        _, _, st = oracle.probe.render_rows(cam, world, depth, 0, h, ystep)
        rays += st.rays
    dt = time.perf_counter() - t0
    value = rays / dt / 1e6
    rows = len(range(0, h - 1, ystep))
    line = {
        "impl": "reference", "metric": "Mrays/s (Camera::render: primary + reflect/refract + shadow rays per second)",
        "value": round(value, 4), "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(dt / args.steps * 1e3, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": config_of(args.workload, cam.width_pixels, h, depth, args.gpus),
        "cpu_baseline": {"value": round(value, 4), "unit": "Mrays/s", "cores": threads, "kind": "port",
                         "sample": f"each step renders rows 0::{ystep} ({rows} of {h - 1} rows) of the frame"},
        "e2e": {"value": round(value, 4), "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


class Ctx:
    """Per-process plumbing shared by every measurement of a run."""

    def __init__(self, args):
        import torch

        self.torch = torch
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world_size = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.dist = None
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the renderer has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        if self.world_size > 1:
            import torch.distributed as dist

            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
            self.dist = dist
        import ray_tracer_challenge_b200 as rt
        from ray_tracer_challenge_b200 import multi

        self.rt, self.multi = rt, multi
        self.api = rt.new_session()
        self.api.set_render_options(device_ids=[self.local_rank], fma=args.fma)
        self.lib = rt.device_library()
        import ctypes as C

        self.lib.rtc_host_alloc.restype = C.c_void_p
        self.lib.rtc_host_alloc.argtypes = [C.c_size_t]
        self.lib.rtc_host_free.argtypes = [C.c_void_p]
        self.lib.rtc_host_register.argtypes = [C.c_void_p, C.c_size_t]
        self.lib.rtc_host_unregister.argtypes = [C.c_void_p]
        self.lib.rtc_measure_fp32_peak.argtypes = [C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
        self.n_shards = self.world_size if self.world_size > 1 else 0
        self._peak = None

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()

    def reduce(self, value, op):
        return self.multi.reduce_scalar(self.dist, value, op, "cuda")

    def fp32_peak(self):
        """(measured TFLOP/s of the K5 FMA micro-benchmark, nominal TFLOP/s at the device's clock)"""
        if self._peak is None:
            import ctypes as C

            tflops, mhz = C.c_double(), C.c_double()
            self.lib.rtc_measure_fp32_peak(self.local_rank, C.byref(tflops), C.byref(mhz))
            props = self.torch.cuda.get_device_properties(self.local_rank)
            self._peak = (tflops.value, props.multi_processor_count * 128 * 2 * mhz.value * 1e6 / 1e12)
        return self._peak


DUMP_PIXELS = 1 << 20  # sampled pixels of a larger frame: 32 bytes each over the three arrays, 32 MiB in all


def dump_frame(ctx: Ctx, prepared, depth: int, out_dir: str) -> None:
    """Writes the frame of the last timed step as a caller of PreparedScene.render receives it: the f32 canvas and its
    8-bit plane at every pixel, or at a fixed seeded sample of DUMP_PIXELS pixels of a larger frame, plus the ray counts.
    The timed steps leave the frame on the device, so it is rendered once more with a copy to the host.  A host canvas
    would otherwise cut the frame into sliced launches in natural tile order.  With RTC_OPT_RENDER_SLICES = 1 the render
    is the timed steps' single launch, in the tile order they learnt.  Equal ray and launch counts are a sanity check,
    not a proof."""
    timed = prepared.last_stats
    prepared.set_option(4, 1)  # RTC_OPT_RENDER_SLICES
    frame = prepared.render(depth, shard=ctx.rank, n_shards=ctx.n_shards, fma=ctx.args.fma)
    st = prepared.last_stats
    counts = [st.primary_rays, st.secondary_rays, st.shadow_rays]
    if counts != [timed.primary_rays, timed.secondary_rays, timed.shadow_rays] or st.launches != timed.launches:
        raise RuntimeError("the frame rendered for --dump-outputs is not the timed one")
    n = frame.width * frame.height
    pixel = np.arange(n) if n <= DUMP_PIXELS else np.sort(np.random.default_rng(0).choice(n, DUMP_PIXELS, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "rgb.npy"), frame.data.reshape(n, 3)[pixel])
    np.save(os.path.join(out_dir, "u8.npy"), frame.to_u8().reshape(n, 3)[pixel].astype(np.float32))
    np.save(os.path.join(out_dir, "pixel.npy"), pixel.astype(np.float64))
    np.save(os.path.join(out_dir, "ray_counts.npy"), np.array(counts, np.float64))


def measure_device(ctx: Ctx, prepared, depth: int, steps: int, warmup: int, spin_s: float = 0.0) -> dict:
    """Device-resident throughput of one workload: `steps` frames, L2 flushed before each, CUDA-event time of the render
    kernel per frame, max over ranks; rays summed over ranks."""
    a = ctx.args
    for _ in range(warmup):
        prepared.render(depth, want_rgb=False, want_u8=False, shard=ctx.rank, n_shards=ctx.n_shards, fma=a.fma)
    t_spin = time.perf_counter()
    while time.perf_counter() - t_spin < spin_s:  # same load while the clock sampler spins up
        prepared.render(depth, want_rgb=False, want_u8=False, shard=ctx.rank, n_shards=ctx.n_shards, fma=a.fma)
    ctx.barrier()
    kernel_ms, rays, launches = 0.0, 0, 0
    wall0 = time.perf_counter()
    for _ in range(steps):
        prepared.flush_l2()  # evict the scene and the previous frame between timed iterations
        prepared.render(depth, want_rgb=False, want_u8=False, shard=ctx.rank, n_shards=ctx.n_shards, fma=a.fma)
        kernel_ms += prepared.last_stats.kernel_ms
        rays += prepared.last_stats.rays
        launches += prepared.last_stats.launches
    ctx.barrier()
    wall_ms = (time.perf_counter() - wall0) * 1e3
    kernel_ms_max = ctx.reduce(kernel_ms, "max")
    rays_total = ctx.reduce(rays, "sum")
    return {"kernel_ms_per_step": kernel_ms_max / steps, "rays_per_frame": rays_total / steps,
            "mrays": rays_total / (kernel_ms_max * 1e-3) / 1e6, "launches": int(ctx.reduce(launches, "sum")),
            "wall_ms_per_step": wall_ms / steps}


def scene_bytes(ctx: Ctx, world) -> int:
    """Host-to-device bytes of one commit: the flattened arrays the C ABI receives (prims, nodes, refs, materials)."""
    import ctypes as C

    _, _, _, _, counts = ctx.api.flatten(world)
    return int(counts[0] * C.sizeof(ctx.rt.RtcPrim) + counts[1] * C.sizeof(ctx.rt.RtcNode) + counts[2] * 4 + counts[3] * 44)


def measure_e2e(ctx: Ctx, workload: str, cam, world, depth: int, rays_per_frame: float, e_steps: int, variants: bool) -> dict:
    """The one-shot call a user makes — Camera::render_b200 (flatten + commit + render + device-to-host copy into pinned host
    canvases) — on every rank for its bands of ONE shared frame; wall clock, max over ranks.  `value` is the render -> to_ppm
    flow of the reference's demos (the 8-bit plane comes back; the f32 plane stays on the device until pixel_at asks for it);
    `f32_canvas` is the same with the f32 plane copied as well."""
    import ctypes as C

    from ray_tracer_challenge_b200.api import U8P, fptr

    api, lib, rank, a = ctx.api, ctx.lib, ctx.rank, ctx.args
    w, h = cam.width_pixels, cam.height_pixels
    n_sh = max(ctx.world_size, 1)
    canvas = None
    if ctx.world_size == 1:
        p_rgb, p_u8 = lib.rtc_host_alloc(w * h * 12), lib.rtc_host_alloc(w * h * 3)
        rgb = np.ctypeslib.as_array(C.cast(p_rgb, C.POINTER(C.c_float)), shape=(h, w, 3))
        u8 = np.ctypeslib.as_array(C.cast(p_u8, C.POINTER(C.c_uint8)), shape=(h, w, 3))
        registered = True
    else:
        # every rank copies its bands straight into one shared host canvas (POSIX shared memory, page-locked by each
        # rank): the "simple host gather" of SURVEY.md §8e with no extra copy
        canvas = ctx.multi.open_shared_canvas(ctx.dist, rank, f"rtc_bench_{os.environ.get('MASTER_PORT', '0')}_{workload}", w, h)
        rgb, u8 = canvas.rgb, canvas.u8
        registered = lib.rtc_host_register(canvas.address, canvas.nbytes) == 0
    stats = ctx.rt.SgStats()

    def one_shot(with_f32: bool, into=None):
        api.check(api.lib.sg_camera_render_shard(api.ctx, cam.handle, world.handle, depth, rank, n_sh, fptr(rgb) if with_f32 else None,
                                                 (u8 if into is None else into).ctypes.data_as(U8P), C.byref(stats)))

    def timed(with_f32: bool, into=None) -> float:
        one_shot(with_f32, into)
        t_w = time.perf_counter()
        one_shot(with_f32, into)
        # the closing barrier (an NCCL all-reduce and a synchronize: ~0.1 ms) is inside the timed region, so a 0.3 ms frame is
        # timed over enough calls for it not to matter: at least e_steps, up to 200, about 30 ms of work (every rank agrees
        # on the count: the slowest rank's estimate decides)
        est = ctx.reduce(time.perf_counter() - t_w, "max")
        n = int(max(e_steps, min(200, 0.03 / max(est, 1e-6))))
        ctx.barrier()
        t0 = time.perf_counter()
        for _ in range(n):
            one_shot(with_f32, into)
        ctx.barrier()
        return ctx.reduce(time.perf_counter() - t0, "max") / n

    dt_u8 = timed(False)
    h2d = scene_bytes(ctx, world) * n_sh
    out = {"value": round(rays_per_frame / dt_u8 / 1e6, 3), "unit": "Mrays/s", "ms_per_frame": round(dt_u8 * 1e3, 3),
           "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(w * h * 3),
           "path": "Camera::render_b200 on every rank (flatten + commit + render of its bands + D2H of the 8-bit canvas into one "
                   "pinned host canvas): the reference demos' render -> to_ppm flow; the f32 plane stays on the device"
                   + ("" if registered else " (cudaHostRegister failed: pageable copy)")}
    if variants:
        dt_f32 = timed(True)
        out["f32_canvas"] = {"value": round(rays_per_frame / dt_f32 / 1e6, 3), "ms_per_frame": round(dt_f32 * 1e3, 3),
                             "d2h_bytes_per_step": int(w * h * 15),
                             "path": "the same with the f32 Canvas (canvas.rs:6-10) copied to the host as well"}
        if ctx.world_size == 1:
            heap = np.zeros((h, w, 3), np.uint8)  # what the glue's CanvasU8 owns, like the reference's Vec: pageable memory
            dt_heap = timed(False, heap)
            out["heap_canvas"] = {"value": round(rays_per_frame / dt_heap / 1e6, 3), "ms_per_frame": round(dt_heap * 1e3, 3),
                                  "d2h_bytes_per_step": int(w * h * 3),
                                  "path": "the 8-bit canvas into a plain heap array instead of pinned memory (staged through a "
                                          "pinned frame by the host's threads)"}
    if ctx.world_size == 1:
        lib.rtc_host_free(p_rgb)
        lib.rtc_host_free(p_u8)
    else:
        if registered:
            lib.rtc_host_unregister(canvas.address)
        del rgb, u8
        ctx.dist.barrier()
        canvas.close()
    return out


def roofline_of(ctx: Ctx, workload: str, detail: dict, ms_frame: float) -> dict:
    peak, nominal = ctx.fp32_peak()
    achieved = detail["flops"] / (ms_frame * 1e-3) / 1e12
    prof = {}
    for rnd in ("r02", "r01"):  # the committed ncu capture of this workload's kernel (tools/ncu_profile_json.py)
        try:
            with open(os.path.join(ROOT, "profiles", f"{rnd}_{workload}_profile.json")) as fh:
                prof = json.load(fh)
            break
        except Exception:
            pass
    return {"bound": "fp32", "achieved": round(achieved, 3), "peak": round(peak, 2), "unit": "TFLOP/s",
            "frac": round(achieved / peak, 4), "traffic": prof.get("dram_bytes"),
            "traffic_source": prof.get("source"),
            "issue_slot_utilisation_pct": prof.get("issue_active_pct"),
            "fma_pipe_utilisation_pct": prof.get("pipe_fma_pct"),
            # what the hardware executed (ncu SASS counts of the committed capture: FADD + FMUL + 2 FFMA + FMNMX +
            # MUFU, predicated-on threads, packed forms counted per lane) over this run's kernel time
            "executed_fp32_tflops": round(prof["executed_fp32_flops"] / (ms_frame * 1e-3) / 1e12, 3) if prof.get("executed_fp32_flops") else None,
            "what": "achieved = algorithmic FP32 flops of the units the kernel EXECUTED (SURVEY.md Appendix E table x the "
                    "detailed pass's counters: tests skipped by the shadow filter's bundle reject are not counted) / kernel time",
            "peak_kind": "measured live: K5 FMA micro-benchmark (MEASURED_PEAKS.json has no FP32 figure)",
            "nominal_peak": round(nominal, 2), "frac_of_nominal": round(achieved / nominal, 4),
            "flops_per_frame": detail["flops"], "rays_per_frame": detail["rays"],
            "flops_per_ray": round(detail["flops"] / max(detail["rays"], 1), 1),
            "node_visits_per_ray": round(detail["node_visits"] / max(detail["rays"], 1), 2),
            "prim_tests_per_ray": round(sum(detail["prim_tests"]) / max(detail["rays"], 1), 2)}


def run_workload(ctx: Ctx, workload: str, steps: int, warmup: int, headline: bool, dump_dir: str | None = None) -> dict:
    """Everything measured for one workload.  headline: the long form (clock sampling, e2e variants)."""
    a = ctx.args
    cam, world, depth, desc = build_scene(ctx.api, workload)
    w, h = cam.width_pixels, cam.height_pixels
    prepared = cam.prepare(world)
    detail = None
    if ctx.world_size == 1:  # rays / flops of the frame (deterministic): one detailed pass, untimed
        prepared.render(depth, want_rgb=False, want_u8=False, detailed=True, fma=a.fma)
        detail = prepared.last_stats.as_dict()
    clock_samples: list = []
    stop = threading.Event()
    sampler = None
    if headline:
        sampler = threading.Thread(target=sample_clocks, args=(stop, clock_samples, ctx.local_rank), daemon=True)
        sampler.start()
    dev = measure_device(ctx, prepared, depth, steps, warmup, spin_s=0.4 if headline else 0.0)
    stop.set()
    if sampler:
        sampler.join(timeout=2)
    if dump_dir is not None:
        dump_frame(ctx, prepared, depth, dump_dir)
    # the first frame of a shard, before anything about the frame has been learnt (the reference API is one-shot):
    # a fresh commit, one untimed-by-us render whose own CUDA-event time is read
    first = cam.prepare(world)
    first.flush_l2()
    first.render(depth, want_rgb=False, want_u8=False, shard=ctx.rank, n_shards=ctx.n_shards, fma=a.fma)
    first_ms = ctx.reduce(first.last_stats.kernel_ms, "max")
    first.release()
    prepared.release()
    e2e = measure_e2e(ctx, workload, cam, world, depth, dev["rays_per_frame"], max(3, min(steps, 10)), variants=headline)
    out = {"workload": workload, "desc": desc, "resolution": [w, h], "depth": depth, "dev": dev, "e2e": e2e, "detail": detail,
           "first_frame_kernel_ms": round(first_ms, 4), "clocks": clocks_summary(clock_samples) if headline else None}
    if detail is not None and ctx.rank == 0:
        out["roofline"] = roofline_of(ctx, workload, detail, dev["kernel_ms_per_step"])
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed frames of the headline workload")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="c3", choices=sorted(WORKLOADS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--fma", action="store_true", help="time the FMA-contracted kernel build instead of the IEEE one")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-per-workload", action="store_true", help="skip the short runs of the other BASELINE configs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed frame of the headline workload to DIR as .npy "
                                                          "(one process only), to compare two builds output for output")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.dump_outputs and (args.impl != "ours" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs needs --impl ours and one process (a rank renders only its own bands)")

    if args.impl == "reference":
        run_reference(args)
        return

    ctx = Ctx(args)
    rank, world_size = ctx.rank, ctx.world_size
    main_run = run_workload(ctx, args.workload, args.steps, args.warmup, headline=True, dump_dir=args.dump_outputs)
    dev, detail = main_run["dev"], main_run["detail"]
    w, h = main_run["resolution"]

    # ---- the other BASELINE configs and the as-shipped jitter mode, a few frames each (same process, same clocks)
    per_workload = {}
    if not args.no_per_workload:
        for name in ("c1", "c2", "c3", "c3_counter", "c4", "c5"):
            if name == args.workload:
                continue
            # 8 warm-up frames: the launch-order trial of a shard (one cold frame, one that records the tile costs, three
            # timed) is over before the timed ones
            r = run_workload(ctx, name, 5, 8, headline=False)
            if rank == 0:
                per_workload[name] = {
                    "desc": r["desc"], "ms_per_step": round(r["dev"]["kernel_ms_per_step"], 4), "mrays": round(r["dev"]["mrays"], 1),
                    "rays_per_frame": r["dev"]["rays_per_frame"], "first_frame_kernel_ms": r["first_frame_kernel_ms"],
                    "e2e_ms": r["e2e"]["ms_per_frame"], "e2e_mrays": r["e2e"]["value"],
                    "h2d_bytes_per_step": r["e2e"]["h2d_bytes_per_step"], "d2h_bytes_per_step": r["e2e"]["d2h_bytes_per_step"],
                    "roofline_frac": r["roofline"]["frac"] if r.get("roofline") else None,
                    "achieved_tflops": r["roofline"]["achieved"] if r.get("roofline") else None, "steps": 5, "warmup": 8}

    # ---- CPU baseline (rank 0, N = 1 only)
    roofline, cpu = main_run.get("roofline"), None
    if rank == 0 and world_size == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(args.workload, 1)
        if roofline and cpu.get("reference_flops_per_frame"):
            ref_flops = cpu["reference_flops_per_frame"]
            ref_tf = ref_flops / (dev["kernel_ms_per_step"] * 1e-3) / 1e12
            roofline["reference_algorithm"] = {
                "flops_per_frame": ref_flops, "achieved": round(ref_tf, 3), "frac": round(ref_tf / roofline["peak"], 4),
                "what": "the same frame's flops as the REFERENCE algorithm spends them (the oracle's counters: every ray "
                        "against every object) / our kernel time: work-equivalent throughput, not hardware utilisation"}
        try:
            from tests.oracle_binding import load_oracle

            n_threads = load_oracle().probe.max_threads()
            cpu["all_cores"] = cpu_baseline(args.workload, n_threads, 6.0)
        except Exception as e:  # pragma: no cover
            cpu["all_cores"] = {"error": str(e)}

    if rank == 0:
        line = {
            "metric": "Mrays/s (Camera::render: primary + reflect/refract + shadow rays per second)",
            "value": round(dev["mrays"], 2), "unit": "Mrays/s", "n_gpus": world_size, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(dev["kernel_ms_per_step"], 4), "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_of(args.workload, w, h, main_run["depth"], world_size, args.fma),
            "rays_per_frame": dev["rays_per_frame"], "wall_ms_per_step_incl_flush": round(dev["wall_ms_per_step"], 3),
            "first_frame_kernel_ms": main_run["first_frame_kernel_ms"],
            "e2e": main_run["e2e"], "gpu_launches": dev["launches"], "clocks": main_run["clocks"],
        }
        if roofline:
            line["roofline"] = roofline
        if cpu:
            line["cpu_baseline"] = cpu
        if per_workload:
            line["per_workload"] = per_workload
        print(json.dumps(line), flush=True)
    if ctx.dist is not None:
        ctx.dist.destroy_process_group()


if __name__ == "__main__":
    main()
