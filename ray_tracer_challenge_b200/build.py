"""In-tree build of the native libraries (sm_100a only; nvcc cross-compiles without a GPU).

    librtc_b200.so  the C ABI of include/rtc_b200.h: csrc/rtc_api.cu + csrc/rtc_commit.cu (host half of a commit) + csrc/rtc_lbvh.cu (device tree builder) +
                    csrc/rtc_ppm.cu (PPM text kernels) +
                    csrc/rtc_kernels.cu compiled four times
                    (FMA-contracting `fast` build and -fmad=false `strict` build, each again with csg_sweep's call sites
                    for scenes holding a CSG beyond csg_eval's limits)
    librtc_host.so  the C++ host mirror of the reference API + flattener (csrc/host/), linked against
                    librtc_b200.so

Run as `python -m ray_tracer_challenge_b200.build [--force]`.
"""
from __future__ import annotations

import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
BUILD = os.path.join(PKG, "build")
LIB_DEVICE = os.path.join(PKG, "librtc_b200.so")
LIB_HOST = os.path.join(PKG, "librtc_host.so")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
# tuning aid: RTC_NVCC_DEFINES="-DRTC_SMALL_MINBLOCKS=8 ..." is appended to every nvcc compile line
EXTRA_DEFINES = os.environ.get("RTC_NVCC_DEFINES", "").split()
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-ffp-contract=off", "--expt-relaxed-constexpr", *EXTRA_DEFINES,
]


def _newer(target: str, sources: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _run(cmd: list[str]) -> None:
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("build failed: " + " ".join(cmd) + "\n" + proc.stdout + proc.stderr)


def build(force: bool = False, verbose: bool = False) -> None:
    os.makedirs(BUILD, exist_ok=True)
    headers = [os.path.join(CSRC, h) for h in sorted(os.listdir(CSRC)) if h.endswith((".h", ".cuh"))]
    headers.append(os.path.join(ROOT, "include", "rtc_b200.h"))
    kernels = os.path.join(CSRC, "rtc_kernels.cu")
    api = os.path.join(CSRC, "rtc_api.cu")
    commit = os.path.join(CSRC, "rtc_commit.cu")
    lbvh = os.path.join(CSRC, "rtc_lbvh.cu")
    ppm = os.path.join(CSRC, "rtc_ppm.cu")
    objs = {
        os.path.join(BUILD, "kernels_fast.o"): [NVCC, *NVCC_FLAGS, "-c", kernels],
        os.path.join(BUILD, "kernels_strict.o"): [NVCC, *NVCC_FLAGS, "-DRTC_STRICT", "-fmad=false", "-c", kernels],
        os.path.join(BUILD, "kernels_fast_sweep.o"): [NVCC, *NVCC_FLAGS, "-DRTC_CSG_SWEEP_BUILD", "-c", kernels],
        os.path.join(BUILD, "kernels_strict_sweep.o"): [NVCC, *NVCC_FLAGS, "-DRTC_STRICT", "-fmad=false", "-DRTC_CSG_SWEEP_BUILD", "-c",
                                                        kernels],
        os.path.join(BUILD, "api.o"): [NVCC, *NVCC_FLAGS, "-c", api],
        os.path.join(BUILD, "commit.o"): [NVCC, *NVCC_FLAGS, "-c", commit],
        os.path.join(BUILD, "lbvh.o"): [NVCC, *NVCC_FLAGS, "-c", lbvh],
        os.path.join(BUILD, "ppm.o"): [NVCC, *NVCC_FLAGS, "-c", ppm],
    }
    jobs = []
    for obj, cmd in objs.items():
        src = cmd[-1]
        if force or _newer(obj, [src, *headers]):
            jobs.append(cmd + ["-o", obj])
    if jobs:
        if verbose:
            print(f"compiling {len(jobs)} CUDA translation unit(s) for sm_100a ...", flush=True)
        with ThreadPoolExecutor(max_workers=7) as pool:
            list(pool.map(_run, jobs))
    if force or jobs or _newer(LIB_DEVICE, list(objs)):
        _run([NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB_DEVICE, *objs, "-cudart", "shared"])
    host_src = os.path.join(CSRC, "host", "rtc_host.cpp")
    host_deps = [host_src, os.path.join(CSRC, "host", "rtc_host.hpp"), os.path.join(CSRC, "rtc_parallel.h"),
                 os.path.join(ROOT, "include", "rtc_b200.h"), os.path.join(ROOT, "include", "rtc_scene.h"), LIB_DEVICE]
    if force or _newer(LIB_HOST, host_deps):
        _run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-Wall",
              "-pthread",
              "-o", LIB_HOST, host_src, "-L" + PKG, "-lrtc_b200", "-Wl,-rpath,$ORIGIN"])


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
    print("built", LIB_DEVICE, "and", LIB_HOST)
