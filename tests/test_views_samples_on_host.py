"""rtc_render_views_samples' kernels (dev_kernels.cuh: render_tiles_views_samples, render_stream_views_samples) on the HOST
in 128-thread blocks of 32-lane warps (tests/emu/emu_views_samples.cpp): view v of a batch with n samples per axis is, bit
for bit in f32 and in 8 bits, the box filter of the oracle's Camera::render with view v's camera at n times the canvas size,
and n = 1 is render_tiles_views' batch.  Also: launches of a sub-range of views and of bands as the host's plan cuts them,
the per-view sample camera against the oracle's Camera::new, and every argument check of rtc_render_views_samples(_ppm)
without a device.  The module runs again under AddressSanitizer + UBSan.  Test infrastructure only."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from ray_tracer_challenge_b200 import scenes
from tests.test_device_code_on_host import _build
from tests.test_kernels_on_host import (STREAM_VIEWS, U8_UNWRITTEN, UNWRITTEN, VIEWS, DevCounters, _check_frame, _code, _Lean,
                                        _orbit, _ptr, _same)
from tests.test_samples_on_host import CASES, SAMPLES, SIZES, STREAM_SAMPLES, _bind_samples, _csg_die, box_filter

VIEWS_SAMPLES, STREAM_VIEWS_SAMPLES = 8, 9   # emu_views_samples.cpp: kViewsSamples, kStreamViewsSamples
BAND_ROWS = 8
RTC_ERR_INVALID, RTC_ERR_STATE = -1, -4
SANITIZED = bool(os.environ.get("RTC_EMU_SANITIZE"))


def _bind_views_samples(lib):
    P = C.c_void_p
    lib.emu_render_views_samples.argtypes = [P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, P, C.c_int, C.c_int, C.c_int, C.c_int,
                                             P, P, C.POINTER(DevCounters), C.POINTER(C.c_int)]
    lib.emu_view_sample_camera.argtypes = [P, C.c_uint, C.c_uint, C.POINTER(C.c_float)]
    return _bind_samples(lib)


@pytest.fixture(scope="module")
def kern(tmp_path_factory):
    device, lib = _build(tmp_path_factory, "emu_views_samples.cpp")
    return device, _bind_views_samples(lib)


@pytest.fixture(scope="module")
def kern_sweep(tmp_path_factory):
    device, lib = _build(tmp_path_factory, "emu_views_samples.cpp", ["-DRTC_CSG_SWEEP_BUILD"])
    return device, _bind_views_samples(lib)


@pytest.fixture(scope="module")
def host():
    import ray_tracer_challenge_b200 as rt

    return rt.new_session()


RAN = set()  # (kind, variant code) of every batch samples launch of this module


def _batch(kern, scene, cams, w, h, n, converge=-1, stream=-1, lean=1, band_begin=0, n_bands=None, out=None):
    """One launch of views cams (exported scenes) over bands [band_begin, band_begin + n_bands), into out (rgb, u8) or new
    planes"""
    device, lib = kern
    n_views = len(cams)
    if n_bands is None:
        n_bands = (h + BAND_ROWS - 1) // BAND_ROWS - band_begin
    if out is None:
        out = (np.full((n_views, h, w, 3), UNWRITTEN, np.uint32).view(np.float32), np.full((n_views, h, w, 3), U8_UNWRITTEN, np.uint8))
    rgb, u8 = out
    ctr, var = DevCounters(), C.c_int(-1)
    table = (C.c_void_p * n_views)(*[c.value for c in cams])
    with _Lean(lean):
        rc = lib.emu_render_views_samples(scene, 5, 0, 1, band_begin, n_bands, table, n_views, n, converge, stream, _ptr(rgb), _ptr(u8),
                                          C.byref(ctr), C.byref(var))
    assert rc == 0, device.rtc_last_error()
    RAN.add((var.value >> 5, var.value & 31))
    return rgb, u8, ctr, var.value


def _poses(host, cam):
    """The batch's three cameras as (eye, look-at, fov), None for the committed camera itself: it, an orbit position, and the
    committed eye with another field of view"""
    orbit = _orbit(host, cam, 3, 60.0)
    e0, p0, fov = orbit[0]
    return [None, orbit[1], (e0, p0, fov * 0.75)]


def _cameras(rt, make, w, h, n, poses):
    """(committed camera, world, the batch's cameras at n W x n H) in either API"""
    cam, world = make(rt, n * w, n * h)
    return cam, world, [cam if p is None else rt.Camera(n * w, n * h, p[2], rt.view_transform(p[0], p[1], (0, 1, 0))) for p in poses]


def _export_batch(host, make, w, h, poses):
    cam, world, cams = _cameras(host, make, w, h, 1, poses)
    return host.export_scene(cam, world), [host.export_scene(c, world) for c in cams]


def _destroy(device, scene, views):
    for v in views:
        device.rtc_scene_destroy(v)
    device.rtc_scene_destroy(scene)


@pytest.mark.parametrize("n", [1, 2, 3])
@pytest.mark.parametrize("size", SIZES, ids=["24x13", "21x10"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_views_samples_match_oracle_box_filter(name, size, n, kern, host, oracle):
    """Every variant launch_views_samples picks, for a batch of the committed camera, an orbit position and another field of
    view: view v is the box filter of the oracle's render with view v's camera at n W x n H, which also pins each sample's
    jitter key to its index in its own view's sample frame."""
    device, _ = kern
    make, (converge, stream, lean), (kind, *flags) = CASES[name]
    w, h = size
    hcam, _ = make(host, w, h)
    poses = _poses(host, hcam)
    _, oworld, ocams = _cameras(oracle, make, w, h, n, poses)
    wants = [box_filter(c.render(oworld, 5).data, w, h, n) for c in ocams]
    scene, views = _export_batch(host, make, w, h, poses)
    try:
        rgb, u8, _, var = _batch(kern, scene, views, w, h, n, converge, stream, lean)
    finally:
        _destroy(device, scene, views)
    want_kind = STREAM_VIEWS_SAMPLES if kind == STREAM_SAMPLES else VIEWS_SAMPLES
    assert (var >> 5, var & 31) == (want_kind, _code(*flags)), (name, var)
    for v in range(len(views)):
        _check_frame(oracle, rgb[v], u8[v], wants[v], (name, size, n, v))


@pytest.mark.parametrize("n", [1, 2, 3])
def test_sweep_build_views_samples_csg_die(n, kern_sweep, oracle, host):
    """The strict_sweep build (csg_sweep's call sites) on a CSG beyond csg_eval's limits, both converge modes."""
    device, _ = kern_sweep
    w, h = 24, 13
    hcam, _ = _csg_die(host, w, h)
    poses = _poses(host, hcam)
    _, oworld, ocams = _cameras(oracle, _csg_die, w, h, n, poses)
    wants = [box_filter(c.render(oworld, 5).data, w, h, n) for c in ocams]
    scene, views = _export_batch(host, _csg_die, w, h, poses)
    try:
        for converge in (0, 1):
            rgb, u8, _, var = _batch(kern_sweep, scene, views, w, h, n, converge, 0)
            assert var >> 5 == VIEWS_SAMPLES
            for v in range(len(views)):
                _check_frame(oracle, rgb[v], u8[v], wants[v], ("csg_die", n, converge, v))
    finally:
        _destroy(device, scene, views)


@pytest.mark.parametrize("name", sorted(CASES))
def test_one_sample_is_the_views_kernel_batch(name, kern, host):
    """n = 1 gives render_tiles_views' / render_stream_views' batch bit for bit in both planes, with the same secondary
    rays and shades."""
    device, lib = kern
    make, (converge, stream, lean), _ = CASES[name]
    w, h = 24, 13
    hcam, _ = make(host, w, h)
    scene, views = _export_batch(host, make, w, h, _poses(host, hcam))
    n_views = len(views)
    try:
        rgb, u8, ctr, _ = _batch(kern, scene, views, w, h, 1, converge, stream, lean)
        want = np.full((n_views, h, w, 3), UNWRITTEN, np.uint32).view(np.float32)
        want_u8 = np.full((n_views, h, w, 3), U8_UNWRITTEN, np.uint8)
        want_ctr, var = DevCounters(), C.c_int(-1)
        table = (C.c_void_p * n_views)(*[v.value for v in views])
        with _Lean(lean):
            assert lib.emu_render_views(scene, 5, 0, 1, 0, (h + 7) // 8, table, n_views, converge, stream, _ptr(want), _ptr(want_u8),
                                        C.byref(want_ctr), C.byref(var)) == 0
        assert var.value >> 5 in (VIEWS, STREAM_VIEWS)
    finally:
        _destroy(device, scene, views)
    assert _same(rgb, want).all() and (u8 == want_u8).all(), name
    assert (ctr.secondary, ctr.shades) == (want_ctr.secondary, want_ctr.shades)


@pytest.mark.parametrize("name", ["lean_drawn", "small_converging", "tree_tiles", "tree_stream"])
def test_sub_range_launches_make_the_whole_batch(name, kern, host):
    """The launches the host's plan makes: runs of whole views (the view table and the planes from view v0 on) and a view
    cut by bands.  Pieced together they are the one-launch batch bit for bit.  In the stream scene a 7-view batch of a
    21x10 canvas has 12 8x4 blocks per view, so refills of the persistent grid's warps cross view boundaries."""
    device, _ = kern
    make, (converge, stream, lean), _ = CASES[name]
    w, h, n = 21, 10, 2
    hcam, _ = make(host, w, h)
    orbit = _orbit(host, hcam, 7, 90.0)
    poses = [None] + orbit[1:]
    scene, views = _export_batch(host, make, w, h, poses)
    n_views, nb = len(views), (h + BAND_ROWS - 1) // BAND_ROWS
    try:
        want, want_u8, _, _ = _batch(kern, scene, views, w, h, n, converge, stream, lean)
        rgb = np.full((n_views, h, w, 3), UNWRITTEN, np.uint32).view(np.float32)
        u8 = np.full((n_views, h, w, 3), U8_UNWRITTEN, np.uint8)
        for v0, v1 in [(0, 3), (3, 6)]:  # runs of whole views
            _batch(kern, scene, views[v0:v1], w, h, n, converge, stream, lean, out=(rgb[v0:v1], u8[v0:v1]))
        for b0 in range(nb):  # the last view, band by band
            _batch(kern, scene, views[6:], w, h, n, converge, stream, lean, band_begin=b0, n_bands=1, out=(rgb[6:], u8[6:]))
    finally:
        _destroy(device, scene, views)
    assert nb == 2 and _same(rgb, want).all() and (u8 == want_u8).all(), name


@pytest.mark.parametrize("size", [(40, 21), (21, 40), (32, 32)], ids=["landscape", "portrait", "square"])
def test_view_sample_camera_is_the_oracle_camera_at_n_times_the_size(size, kern, host, oracle):
    """A view's sample camera (sample_camera's RtcView overload): pixel_size, half_width and half_height of the oracle's
    Camera::new(n W, n H, fov, transform), for views of other fields of view than the committed one."""
    device, lib = kern
    w, h = size
    eye, at = (0.3, 1.5, -5.0), (0.0, 1.0, 0.0)
    world = scenes.soft_shadows(host, width=w, height=h, u_steps=2, v_steps=2)[1]
    for fov in (0.5, 1.0471975, 2.0):
        cam = host.Camera(w, h, fov, host.view_transform(eye, at, (0, 1, 0)))
        scene = host.export_scene(cam, world)
        try:
            for n in (1, 2, 3, 4, 7, 16):
                got = (C.c_float * 3)()
                lib.emu_view_sample_camera(scene, w, n, got)
                want = oracle.probe.camera_info(oracle.Camera(n * w, n * h, fov, oracle.view_transform(eye, at, (0, 1, 0))))
                assert (np.float32(got[0]), np.float32(got[1]), np.float32(got[2])) == \
                    (np.float32(want["pixel_size"]), np.float32(want["half_width"]), np.float32(want["half_height"])), (size, fov, n)
        finally:
            device.rtc_scene_destroy(scene)


class _View(C.Structure):
    _fields_ = [("half_width", C.c_float), ("half_height", C.c_float), ("pixel_size", C.c_float), ("transform_inverse", C.c_float * 16)]


def test_views_samples_check_their_arguments_in_order_before_the_scene_state():
    """NULL scene; rtc_render_views' checks of n_views and views; samples_per_axis; the sample canvas; the depth; then, for the
    text call, ppm / view_offsets and the capacity — each RTC_ERR_INVALID, before the uncommitted scene's RTC_ERR_STATE."""
    import ray_tracer_challenge_b200 as rt

    lib = rt.device_library()
    lib.rtc_last_error.restype = C.c_char_p
    P = C.c_void_p
    lib.rtc_render_views_samples.argtypes = [P, C.c_int32, C.c_uint32, P, C.c_uint32, P, P, P]
    lib.rtc_render_views_samples_ppm.argtypes = [P, C.c_int32, C.c_uint32, P, C.c_uint32, P, C.c_size_t, P, P]
    lib.rtc_set_camera.argtypes = [P, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_float)]
    lib.rtc_ppm_bound.restype = C.c_size_t
    lib.rtc_ppm_bound.argtypes = [C.c_uint32, C.c_uint32]
    lib.rtc_scene_destroy.argtypes = [P]
    scene = C.c_void_p()
    assert lib.rtc_scene_create(C.byref(scene)) == 0
    ident = [1.0 if i % 5 == 0 else 0.0 for i in range(16)]
    good = (_View * 2)(*[_View(1.0, 0.5, 2.0 / 64, (C.c_float * 16)(*ident)) for _ in range(2)])
    bad = (_View * 2)(good[0], _View(1.0, 0.5, 0.0, (C.c_float * 16)(*ident)))
    nan = (_View * 1)(_View(float("nan"), 0.5, 2.0 / 64, (C.c_float * 16)(*ident)))
    rgb = np.full((2, 32, 64, 3), 7.0, np.float32)
    bound = lib.rtc_ppm_bound(64, 32)
    text = np.full(2 * bound, 9, np.uint8)
    offsets = (C.c_size_t * 3)(5, 5, 5)
    cap = text.nbytes

    def frames(*args):
        return lib.rtc_render_views_samples(*args[:5], _ptr(rgb), None, None)

    def ppm(*args, buf=_ptr(text), offs=offsets, capacity=cap):
        return lib.rtc_render_views_samples_ppm(*args[:5], buf, capacity, offs, None)

    def refused(call, args, msg, **kw):
        assert call(*args, **kw) == RTC_ERR_INVALID, (args, kw)
        assert msg in lib.rtc_last_error(), (lib.rtc_last_error(), msg)

    try:
        assert lib.rtc_set_camera(scene, 64, 32, 1.0, 0.5, 2.0 / 64, (C.c_float * 16)(*ident)) == 0
        for call in (frames, ppm):
            refused(call, (None, 5, 2, good, 2), b"null scene")
            refused(call, (scene, 5, 0, good, 2), b"n_views")
            refused(call, (scene, 5, 2, None, 2), b"n_views")
            refused(call, (scene, 5, 2, bad, 2), b"pixel_size <= 0")
            refused(call, (scene, 5, 1, nan, 2), b"non-finite")
            refused(call, (scene, 99, 2, bad, 0), b"pixel_size <= 0")  # the views before samples_per_axis and depth
            for n in (0, 17, 1 << 31):
                refused(call, (scene, 99, 2, good, n), b"samples_per_axis")  # samples before the depth
            for depth in (-1, 24):
                refused(call, (scene, depth, 2, good, 2), b"reflection_recursion_depth")
        # the text call's own checks come last
        refused(ppm, (scene, 5, 2, good, 2), b"ppm and view_offsets", buf=None)
        refused(ppm, (scene, 5, 2, good, 2), b"ppm and view_offsets", offs=None)
        refused(ppm, (scene, 99, 2, good, 2), b"reflection_recursion_depth", buf=None)  # the depth before them
        refused(ppm, (scene, 5, 2, good, 2), b"below n_views * rtc_ppm_bound", capacity=2 * bound - 1)
        # valid arguments: the scene is not committed
        for n in (1, 16):
            for depth in (0, 23):
                assert frames(scene, depth, 2, good, n) == RTC_ERR_STATE, (n, depth)
                assert ppm(scene, depth, 2, good, n) == RTC_ERR_STATE, (n, depth)
        assert ppm(scene, 5, 2, good, 2, capacity=2 * bound) == RTC_ERR_STATE
        assert b"before rtc_scene_commit" in lib.rtc_last_error()
        # a sample canvas rtc_set_camera would refuse, before the depth and the text's checks
        assert lib.rtc_set_camera(scene, 16384, 8192, 1.0, 0.5, 2.0 / 16384, (C.c_float * 16)(*ident)) == 0
        assert frames(scene, 5, 2, good, 2) == RTC_ERR_STATE  # 2^29 <= 2^31 / 3
        refused(frames, (scene, 99, 2, good, 3), b"sample canvas")
        refused(ppm, (scene, 99, 2, good, 3), b"sample canvas", buf=None)
        refused(ppm, (scene, 5, 1, good, 1), b"below n_views * rtc_ppm_bound", capacity=1000)
        assert (rgb == 7.0).all() and (text == 9).all() and list(offsets) == [5, 5, 5]  # nothing written on a refused call
    finally:
        lib.rtc_scene_destroy(scene)


def test_every_views_samples_variant_ran(kern):
    """The batch samples kernels this module ran are all launch_views_samples can select in the strict build."""
    if not RAN or os.environ.get("PYTEST_XDIST_WORKER"):
        pytest.skip("needs the whole module in one process")
    out = (C.c_int * 64)()
    n = kern[1].emu_views_sample_variants(out)
    want = {(v >> 5, v & 31) for v in out[:n]}
    assert n == 8 + 1 and len(want) == n
    ran = {r for r in RAN if r[0] in (VIEWS_SAMPLES, STREAM_VIEWS_SAMPLES)}
    assert ran == want, (sorted(want - ran), sorted(ran - want))


def test_views_samples_under_address_sanitizer():
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
