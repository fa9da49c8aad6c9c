"""rtc_render_samples' kernels (dev_kernels.cuh: render_tiles_samples, render_stream_samples) on the HOST in 128-thread
blocks of 32-lane warps (tests/emu/emu_samples.cpp): with n samples per axis every pixel is, bit for bit in f32 and in 8
bits, the box filter — summed in f32 from sample (0, 0), j outer and i inner, then divided by n * n — of the oracle's
Camera::render at n times the canvas size, and n = 1 is render_tiles' frame.  Also: the sample camera's derived fields
against the oracle's Camera::new, and every argument check of rtc_render_samples without a device.  The module runs again
under AddressSanitizer + UBSan.  Test infrastructure only."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from ray_tracer_challenge_b200 import scenes
from tests.test_device_code_on_host import _build
from tests.test_kernels_on_host import (FRAME_CASES, U8_UNWRITTEN, UNWRITTEN, DevCounters, _bind, _check_frame,
                                        _code, _dragon, _Lean, _ptr, _render, _same, _scene, _soft_lean, _soft_table,
                                        _stress)

SAMPLES, STREAM_SAMPLES = 6, 7   # emu_samples.cpp: kSamples, kStreamSamples
RTC_ERR_INVALID, RTC_ERR_STATE = -1, -4
SANITIZED = bool(os.environ.get("RTC_EMU_SANITIZE"))


def _bind_samples(lib):
    P = C.c_void_p
    lib.emu_render_samples.argtypes = [P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, P, P,
                                       C.POINTER(DevCounters), C.POINTER(C.c_int)]
    lib.emu_sample_camera.argtypes = [P, C.c_uint, C.POINTER(C.c_float)]
    return _bind(lib)


@pytest.fixture(scope="module")
def kern(tmp_path_factory):
    device, lib = _build(tmp_path_factory, "emu_samples.cpp")
    return device, _bind_samples(lib)


@pytest.fixture(scope="module")
def kern_sweep(tmp_path_factory):
    device, lib = _build(tmp_path_factory, "emu_samples.cpp", ["-DRTC_CSG_SWEEP_BUILD"])
    return device, _bind_samples(lib)


@pytest.fixture(scope="module")
def host():
    import ray_tracer_challenge_b200 as rt

    return rt.new_session()


RAN = set()  # (kind, variant code) of every samples launch of this module


def _render_samples(kern, scene, w, h, n, converge=-1, stream=-1, lean=1):
    device, lib = kern
    rgb = np.full((h, w, 3), UNWRITTEN, np.uint32).view(np.float32)
    u8 = np.full((h, w, 3), U8_UNWRITTEN, np.uint8)
    ctr, var = DevCounters(), C.c_int(-1)
    with _Lean(lean):
        rc = lib.emu_render_samples(scene, 5, 0, 1, 0, (h + 7) // 8, n, converge, stream, _ptr(rgb), _ptr(u8), C.byref(ctr),
                                    C.byref(var))
    assert rc == 0, device.rtc_last_error()
    RAN.add((var.value >> 5, var.value & 31))
    return rgb, u8, ctr, var.value


def box_filter(big, w, h, n):
    """rtc_render_samples' mean of the n W x n H frame `big`, summed sequentially in f32; last row and column zero"""
    b = np.asarray(big, np.float32)[:n * h, :n * w].reshape(h, n, w, n, 3)
    s = b[:, 0, :, 0].copy()
    for j in range(n):
        for i in range(n):
            if i or j:
                s = (s + b[:, j, :, i]).astype(np.float32)
    s = (s / np.float32(n * n)).astype(np.float32)
    s[h - 1, :], s[:, w - 1] = 0.0, 0.0
    return s


def _csg_die(rt, width, height):
    return scenes.csg_die(rt, width=width, height=height)


# name -> (scene, options (converge, stream, RTC_LEAN), the variant (kind, stats, small, converge, drawn, lean))
CASES = {
    "lean_drawn": (_soft_lean, (-1, -1, 1), (SAMPLES, 0, 1, 0, 1, 1)),
    "lean_table": (_soft_table, (-1, -1, 1), (SAMPLES, 0, 1, 0, 0, 1)),
    "drawn_small": (_soft_lean, (-1, -1, 0), (SAMPLES, 0, 1, 0, 1, 0)),
    "drawn_converging": (_soft_lean, (1, -1, 1), (SAMPLES, 0, 1, 1, 1, 0)),
    "small": (FRAME_CASES["reflect_refract"][0], (0, -1, 1), (SAMPLES, 0, 1, 0, 0, 0)),
    "small_converging": (FRAME_CASES["reflect_refract"][0], (1, -1, 1), (SAMPLES, 0, 1, 1, 0, 0)),
    "tree_tiles": (_dragon, (0, 0, 1), (SAMPLES, 0, 0, 0, 0, 0)),
    "tree_converging": (_dragon, (1, 0, 1), (SAMPLES, 0, 0, 1, 0, 0)),
    "tree_stream": (_stress, (-1, -1, 1), (STREAM_SAMPLES, 0, 0, 1, 0, 0)),
}
SIZES = [(24, 13), (21, 10)]  # a width divisible by 8 (the staged epilogue) and an odd one (per-pixel stores)


def _want(oracle, make, w, h, n):
    ocam, oworld = make(oracle, n * w, n * h)
    return box_filter(ocam.render(oworld, 5).data, w, h, n)


@pytest.mark.parametrize("n", [1, 2, 3])
@pytest.mark.parametrize("size", SIZES, ids=["24x13", "21x10"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_samples_match_oracle_box_filter(name, size, n, kern, host, oracle):
    """Every variant launch_samples picks — lean, drawn, table, general small, converging, tree tiles, tree stream — at n =
    1, 2 and 3 (a mean that is not a power of two): the box filter of the oracle's render at n W x n H, which also pins
    the jitter key of every sample in the generated-jitter scenes."""
    device, _ = kern
    make, (converge, stream, lean), (kind, *flags) = CASES[name]
    w, h = size
    want = _want(oracle, make, w, h, n)
    scene = _scene(host, make, w, h)
    try:
        rgb, u8, _, var = _render_samples(kern, scene, w, h, n, converge, stream, lean)
    finally:
        device.rtc_scene_destroy(scene)
    assert (var >> 5, var & 31) == (kind, _code(*flags)), (name, var)
    _check_frame(oracle, rgb, u8, want, (name, size, n))


@pytest.mark.parametrize("n", [1, 2, 3])
def test_sweep_build_samples_csg_die(n, kern_sweep, oracle, host):
    """The strict_sweep build (csg_sweep's call sites) on a CSG beyond csg_eval's limits, both converge modes."""
    device, _ = kern_sweep
    w, h = 24, 13
    want = _want(oracle, _csg_die, w, h, n)
    scene = _scene(host, _csg_die, w, h)
    try:
        for converge in (0, 1):
            rgb, u8, _, var = _render_samples(kern_sweep, scene, w, h, n, converge, 0)
            assert var >> 5 == SAMPLES
            _check_frame(oracle, rgb, u8, want, ("csg_die", n, converge))
    finally:
        device.rtc_scene_destroy(scene)


@pytest.mark.parametrize("name", sorted(CASES))
def test_one_sample_is_the_render_kernel_frame(name, kern, host):
    """n = 1 gives render_tiles' / render_stream's frame bit for bit in both planes, and the same secondary rays and shades."""
    device, _ = kern
    make, (converge, stream, lean), _ = CASES[name]
    w, h = 24, 13
    scene = _scene(host, make, w, h)
    try:
        rgb, u8, ctr, _ = _render_samples(kern, scene, w, h, 1, converge, stream, lean)
        want, want_u8, want_ctr, _ = _render(kern, scene, w, h, converge=converge, stream=stream, lean=lean)
    finally:
        device.rtc_scene_destroy(scene)
    assert _same(rgb, want).all() and (u8 == want_u8).all(), name
    assert (ctr.secondary, ctr.shades) == (want_ctr.secondary, want_ctr.shades)


@pytest.mark.parametrize("size", [(40, 21), (21, 40), (32, 32)], ids=["landscape", "portrait", "square"])
def test_sample_camera_is_the_oracle_camera_at_n_times_the_size(size, kern, host, oracle):
    """C_n's pixel_size, half_width and half_height are those of the oracle's Camera::new(n W, n H, fov, transform)."""
    device, lib = kern
    w, h = size
    fov = 1.0471975
    eye, at = (0.3, 1.5, -5.0), (0.0, 1.0, 0.0)
    cam = host.Camera(w, h, fov, host.view_transform(eye, at, (0, 1, 0)))
    world = scenes.soft_shadows(host, width=w, height=h, u_steps=2, v_steps=2)[1]
    scene = host.export_scene(cam, world)
    try:
        for n in (1, 2, 3, 4, 7, 16):
            got = (C.c_float * 3)()
            lib.emu_sample_camera(scene, n, got)
            want = oracle.probe.camera_info(oracle.Camera(n * w, n * h, fov, oracle.view_transform(eye, at, (0, 1, 0))))
            assert (np.float32(got[0]), np.float32(got[1]), np.float32(got[2])) == \
                (np.float32(want["pixel_size"]), np.float32(want["half_width"]), np.float32(want["half_height"])), (size, n)
    finally:
        device.rtc_scene_destroy(scene)


def test_render_samples_checks_its_arguments_before_the_scene_state():
    import ray_tracer_challenge_b200 as rt

    lib = rt.device_library()
    lib.rtc_last_error.restype = C.c_char_p
    lib.rtc_render_samples.argtypes = [C.c_void_p, C.c_int32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.rtc_set_camera.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_float)]
    lib.rtc_scene_destroy.argtypes = [C.c_void_p]
    scene = C.c_void_p()
    assert lib.rtc_scene_create(C.byref(scene)) == 0
    ident = (C.c_float * 16)(*[1.0 if i % 5 == 0 else 0.0 for i in range(16)])
    rgb = np.full((32, 64, 3), 7.0, np.float32)
    try:
        assert lib.rtc_set_camera(scene, 64, 32, 1.0, 0.5, 2.0 / 64, ident) == 0
        assert lib.rtc_render_samples(None, 5, 2, _ptr(rgb), None, None) == RTC_ERR_INVALID
        for n in (0, 17, 1 << 31):
            assert lib.rtc_render_samples(scene, 5, n, _ptr(rgb), None, None) == RTC_ERR_INVALID, n
            assert b"samples_per_axis" in lib.rtc_last_error()
        for depth in (-1, 24):
            assert lib.rtc_render_samples(scene, depth, 2, _ptr(rgb), None, None) == RTC_ERR_INVALID, depth
            assert b"reflection_recursion_depth" in lib.rtc_last_error()
        # valid arguments: the scene is not committed
        for n in (1, 16):
            for depth in (0, 23):
                assert lib.rtc_render_samples(scene, depth, n, _ptr(rgb), None, None) == RTC_ERR_STATE, (n, depth)
        assert b"before rtc_scene_commit" in lib.rtc_last_error()
        # a sample canvas rtc_set_camera would refuse: 16384 x 8192 is allowed, 4 x 4 samples of it are not
        assert lib.rtc_set_camera(scene, 16384, 8192, 1.0, 0.5, 2.0 / 16384, ident) == 0
        assert lib.rtc_render_samples(scene, 5, 1, None, None, None) == RTC_ERR_STATE
        assert lib.rtc_render_samples(scene, 5, 2, None, None, None) == RTC_ERR_STATE  # 2^29 <= 2^31 / 3
        assert lib.rtc_render_samples(scene, 5, 3, None, None, None) == RTC_ERR_INVALID
        assert b"sample canvas" in lib.rtc_last_error()
        assert lib.rtc_render_samples(scene, 99, 3, None, None, None) == RTC_ERR_INVALID  # the canvas before the depth
        assert b"sample canvas" in lib.rtc_last_error()
        assert (rgb == 7.0).all()  # nothing written on a refused call
    finally:
        lib.rtc_scene_destroy(scene)


def test_every_samples_variant_ran(kern):
    """The samples kernels this module ran are all launch_samples can select in the strict build."""
    if not RAN or os.environ.get("PYTEST_XDIST_WORKER"):
        pytest.skip("needs the whole module in one process")
    out = (C.c_int * 64)()
    n = kern[1].emu_sample_variants(out)
    want = {(v >> 5, v & 31) for v in out[:n]}
    assert n == 8 + 1 and len(want) == n
    assert RAN == want, (sorted(want - RAN), sorted(RAN - want))


def test_samples_under_address_sanitizer():
    """This module again with the harnesses built with -fsanitize=address,undefined."""
    import subprocess

    if SANITIZED or os.environ.get("RTC_EMU_TSAN"):
        pytest.skip("already inside a sanitized run")
    libasan = subprocess.run(["g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not libasan or not os.path.exists(libasan):
        pytest.skip("no libasan")
    env = dict(os.environ, LD_PRELOAD=libasan, RTC_EMU_SANITIZE="1", ASAN_OPTIONS="detect_leaks=0:abort_on_error=1",
               UBSAN_OPTIONS="print_stacktrace=1:halt_on_error=1")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    proc = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-s", "-p", "no:cacheprovider"],
                          cwd=root, env=env, capture_output=True, text=True, timeout=1800)
    tail = (proc.stdout + proc.stderr)[-4000:]
    assert proc.returncode == 0, tail
    assert "passed" in proc.stdout and "AddressSanitizer" not in tail and "runtime error" not in tail, tail
