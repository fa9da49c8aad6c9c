"""Kernel time of anti-aliased frames (rtc_render_samples) on one device, frames left on the device, in alternating runs:
(a) rtc_render_samples with n samples per axis; (b) rtc_render of the committed camera; (c) rtc_render of the scene
committed with the sample camera C_n (n times the canvas size): the same rays as (a), with the big frame written to HBM.
Each figure is RtcStats.kernel_ms: median and range over the rounds.  Prints the card's name and power limit, and with
--json PATH also writes the table there as JSON.
    python tools/sample_times.py [--rounds R] [--samples 1 2 4] [--json PATH] [workload ...]   (default: c1 c3 c4)"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ray_tracer_challenge_b200 as rt  # noqa: E402
from bench import WORKLOADS  # noqa: E402
from ray_tracer_challenge_b200 import scenes  # noqa: E402


def kernel_ms(p, fn, rounds):
    fn()  # warm-up
    out = []
    for _ in range(rounds):
        fn()
        out.append(p.last_stats.kernel_ms)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("workloads", nargs="*", default=["c1", "c3", "c4"])
    ap.add_argument("--samples", type=int, nargs="+", default=[1, 2, 4])
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=5, help="kernel times per figure per round")
    ap.add_argument("--json", help="also write the table to this file")
    args = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    print(card, flush=True)
    api = rt.new_session()
    api.set_render_options(device_ids=[0])
    rows = []
    for name in args.workloads:
        builder, kw, depth, _ = WORKLOADS[name]
        build = getattr(scenes, builder)
        cam, world = build(api, **kw)
        p = cam.prepare(world)
        for n in args.samples:
            big = None
            if n > 1:
                bcam, bworld = build(api, **dict(kw, width=n * kw["width"], height=n * kw["height"]))
                big = bcam.prepare(bworld)
            t = {"a": [], "b": [], "c": []}
            for _ in range(args.rounds):  # alternate the three within every round
                t["a"] += kernel_ms(p, lambda: p.render_samples(n, depth, want_rgb=False, want_u8=False), args.reps)
                t["b"] += kernel_ms(p, lambda: p.render(depth, want_rgb=False, want_u8=False), args.reps)
                if big is not None:
                    t["c"] += kernel_ms(big, lambda: big.render(depth, want_rgb=False, want_u8=False), args.reps)
            if big is not None:
                big.release()
            row = {"workload": name, "n": n}
            for k, v in t.items():
                if v:
                    row[k] = {"median_ms": float(np.median(v)), "min_ms": float(np.min(v)), "max_ms": float(np.max(v))}
            rows.append(row)
            line = f"{name} n={n}: " + "  ".join(
                f"({k}) {row[k]['median_ms']:.3f} ms [{row[k]['min_ms']:.3f}, {row[k]['max_ms']:.3f}]" for k in "abc" if k in row)
            print(line, flush=True)
        p.release()
    if args.json:
        with open(args.json, "w") as f:
            json.dump({"card": card, "rows": rows}, f, indent=1)


if __name__ == "__main__":
    main()
