"""rtc_render_views_ppm's text kernels and host scan on the HOST (tests/emu/emu_ppm_views.cpp: emu_ppm_views, dev_ppm.cuh in
128-thread blocks of 32-lane warps, rtc_internal.h: ppm_layout): a batch of n_views 8-bit planes, split over 1, 2 or 3
devices, is encoded in one launch of each kernel per device, and each view's text must be byte for byte the host writer's
(CanvasU8.to_ppm) and the oracle's Canvas::to_ppm (canvas.rs:58-96).  The module runs again under AddressSanitizer + UBSan.
Also: every argument check of rtc_render_views_ppm comes before the scene's state, and the Python wrappers reject a bad
`out`, without a device."""
import ctypes as C
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.test_device_code_on_host import _build

SANITIZED = bool(os.environ.get("RTC_EMU_SANITIZE"))
RTC_ERR_INVALID, RTC_ERR_STATE = -1, -4
SENTINEL = 0x7F


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    device, lib = _build(tmp_path_factory, "emu_ppm_views.cpp")
    lib.emu_ppm_views.restype = C.c_longlong
    lib.emu_ppm_views.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_longlong, C.c_void_p]
    device.rtc_ppm_bound.restype = C.c_size_t
    device.rtc_ppm_bound.argtypes = [C.c_uint32, C.c_uint32]
    return device, lib


@pytest.fixture(scope="module")
def host():
    import ray_tracer_challenge_b200 as rt

    return rt.new_session()


def _emu_views(emu, planes, n_dev):
    """The texts of a batch (planes: n, h, w, 3) as emu_ppm_views writes them; checks the offsets and the bytes past the text."""
    device, lib = emu
    n, h, w, _ = planes.shape
    planes = np.ascontiguousarray(planes)
    cap = n * device.rtc_ppm_bound(w, h)
    out = np.full(cap + 16, SENTINEL, np.uint8)
    at = np.full(n + 1, 2**63, np.uint64)
    total = lib.emu_ppm_views(planes.ctypes.data, w, h, n, n_dev, out.ctypes.data, cap, at.ctypes.data)
    assert total >= 0, "the text outgrew n_views * rtc_ppm_bound" if total == -1 else "ppm_write wrote past its device's text"
    assert at[n] == 2**63, "view_at written past its n entries"
    assert np.all(out[total:] == SENTINEL), "bytes written past the batch's text"
    offsets = [int(x) for x in at[:n]] + [total]
    assert offsets[0] == 0 and all(a < b for a, b in zip(offsets, offsets[1:])), offsets
    return [out[offsets[v]:offsets[v + 1]].tobytes().decode("ascii") for v in range(n)]


def _host_ppm(host, u8):
    import ray_tracer_challenge_b200 as rt

    h, w, _ = u8.shape
    return rt.CanvasU8(w, h, np.ascontiguousarray(u8), host).to_ppm()


def _oracle_ppm(oracle, u8):
    """Canvas::to_ppm of an f32 canvas whose scale_color values are u8: (v + 0.5) / 255 truncates back to v."""
    h, w, _ = u8.shape
    c = oracle.new_canvas(w, h)
    c.data[:] = ((u8.astype(np.float32) + np.float32(0.5)) / np.float32(255.0)).astype(np.float32)
    return c.to_ppm()


def _batch(rng, n, h, w):
    """n planes that differ from view to view and from row to row: each view has its own random values and its own share of
    one-digit runs, so a view or a row taken from the wrong place changes the text."""
    planes = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    for v in range(n):
        planes[v][rng.random((h, w)) < 0.15 * (v % 4)] = v % 10
        planes[v, :, 0, 0] = (np.arange(h) * 7 + v * 31) % 256  # every row's first value: its own
    return planes


# ragged heights, heights below one band of 8, and heights where a device owns no band (h <= 8: devices 1 and 2; h <= 16:
# device 2)
HEIGHTS = (1, 3, 5, 7, 8, 9, 12, 16, 17, 23, 26)


def test_batches_equal_the_host_writer_and_the_oracle(emu, host, oracle):
    rng = np.random.default_rng(17)
    checked_oracle = 0
    for w in range(1, 41):
        for k, n in enumerate((1, 2, 3, 7)):
            h = HEIGHTS[(w + 3 * k) % len(HEIGHTS)]
            planes = _batch(rng, n, h, w)
            want = [_host_ppm(host, planes[v]) for v in range(n)]
            if (w + k) % 3 == 0 or SANITIZED:  # the oracle agrees with the host writer (a third of the batches: it is slow)
                for v in range(n):
                    assert _oracle_ppm(oracle, planes[v]) == want[v], (w, h, n, v)
                checked_oracle += 1
            for n_dev in (1, 2, 3):
                got = _emu_views(emu, planes, n_dev)
                for v in range(n):
                    assert got[v] == want[v], (w, h, n, n_dev, v)
    assert checked_oracle >= 50


def test_every_device_count_meets_every_view_count_on_one_plane_size(emu, host):
    """All of n_views 1, 2, 3, 7 x devices 1, 2, 3 at a size whose bands split unevenly (37 rows: 5 bands), wider than one
    warp step (100 px = 300 values)."""
    rng = np.random.default_rng(19)
    for n in (1, 2, 3, 7):
        planes = _batch(rng, n, 37, 100)
        want = [_host_ppm(host, planes[v]) for v in range(n)]
        for n_dev in (1, 2, 3):
            assert _emu_views(emu, planes, n_dev) == want, (n, n_dev)


def test_a_batch_is_its_views_encoded_one_by_one(emu):
    """The text of view v of a batch does not depend on the other views: it equals the one-view batch of that plane."""
    rng = np.random.default_rng(23)
    planes = _batch(rng, 7, 19, 33)
    for n_dev in (1, 2, 3):
        batch = _emu_views(emu, planes, n_dev)
        assert batch == [_emu_views(emu, planes[v:v + 1], n_dev)[0] for v in range(7)], n_dev


def _lib():
    import ray_tracer_challenge_b200 as rt

    lib = rt.device_library()
    lib.rtc_last_error.restype = C.c_char_p
    lib.rtc_ppm_bound.restype = C.c_size_t
    lib.rtc_ppm_bound.argtypes = [C.c_uint32, C.c_uint32]
    lib.rtc_render_views_ppm.argtypes = [C.c_void_p, C.c_int32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_size_t,
                                         C.POINTER(C.c_size_t), C.c_void_p]
    lib.rtc_set_camera.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_float)]
    lib.rtc_scene_destroy.argtypes = [C.c_void_p]
    return rt, lib


def test_render_views_ppm_checks_its_arguments_before_the_scene_state():
    rt, lib = _lib()
    scene = C.c_void_p()
    assert lib.rtc_scene_create(C.byref(scene)) == 0
    ident = [1.0 if i % 5 == 0 else 0.0 for i in range(16)]
    assert lib.rtc_set_camera(scene, 64, 32, 1.0, 0.5, 2.0 / 64, (C.c_float * 16)(*ident)) == 0
    n = 3
    views = (rt.RtcView * n)(*[rt.RtcView(1.0, 0.5, 2.0 / 64, (C.c_float * 16)(*ident)) for _ in range(n)])
    bound = lib.rtc_ppm_bound(64, 32)
    buf = C.create_string_buffer(n * bound)
    offsets = (C.c_size_t * (n + 1))(*[777] * (n + 1))

    def call(scene=scene, depth=5, n_views=n, views=views, ppm=buf, capacity=n * bound, offsets=offsets):
        return lib.rtc_render_views_ppm(scene, depth, n_views, views, ppm, capacity, offsets, None)

    def refused(code, text, **kw):
        assert call(**kw) == code, kw
        assert text.encode() in lib.rtc_last_error(), (kw, lib.rtc_last_error())

    try:
        assert call(scene=None) == RTC_ERR_INVALID
        refused(RTC_ERR_INVALID, "non-null", ppm=None)
        refused(RTC_ERR_INVALID, "non-null", offsets=None)
        refused(RTC_ERR_INVALID, "n_views must be >= 1", n_views=0)
        refused(RTC_ERR_INVALID, "n_views must be >= 1", views=None)
        for field, value, text in (("half_width", math.inf, "non-finite"), ("pixel_size", math.nan, "non-finite"),
                                   ("pixel_size", 0.0, "pixel_size <= 0"), ("pixel_size", -1.0, "pixel_size <= 0")):
            bad = (rt.RtcView * n)(*views)
            setattr(bad[2], field, value)
            refused(RTC_ERR_INVALID, f"view 2 has a {text}" if text == "non-finite" else text, views=bad)
        bad = (rt.RtcView * n)(*views)
        bad[1].transform_inverse[7] = math.inf
        refused(RTC_ERR_INVALID, "view 1 has a non-finite field", views=bad)
        refused(RTC_ERR_INVALID, "rtc_ppm_bound", capacity=n * bound - 1)
        refused(RTC_ERR_INVALID, "rtc_ppm_bound", capacity=0)
        more = (rt.RtcView * (n + 1))(*views, views[0])
        refused(RTC_ERR_INVALID, "rtc_ppm_bound", n_views=n + 1, views=more)  # the same capacity is one view short
        for depth in (-1, 24):
            refused(RTC_ERR_INVALID, "reflection_recursion_depth", depth=depth)
        # valid arguments: the scene is not committed (a capacity of exactly n_views * bound is enough)
        for depth in (0, 23):
            refused(RTC_ERR_STATE, "before rtc_scene_commit", depth=depth)
        refused(RTC_ERR_STATE, "before rtc_scene_commit", capacity=n * bound + 1)
        assert list(offsets) == [777] * (n + 1) and buf.raw == b"\0" * (n * bound)  # nothing written on a refused call
    finally:
        lib.rtc_scene_destroy(scene)


def test_an_overflowing_capacity_product_is_refused():
    """n_views * rtc_ppm_bound beyond size_t: the largest canvas rtc_set_camera takes (w * h <= 2^31 / 3, a bound of 8.6 GB)
    and 2^32 - 1 views.  Refused before any view is read (the views array holds one)."""
    rt, lib = _lib()
    scene = C.c_void_p()
    assert lib.rtc_scene_create(C.byref(scene)) == 0
    ident = [1.0 if i % 5 == 0 else 0.0 for i in range(16)]
    w, h = 65535, 10922
    assert w * h <= 2**31 // 3
    assert lib.rtc_set_camera(scene, w, h, 1.0, 0.5, 2.0 / w, (C.c_float * 16)(*ident)) == 0
    bound = lib.rtc_ppm_bound(w, h)
    n_views = 2**32 - 1
    assert n_views * bound >= 2**64
    views = (rt.RtcView * 1)(rt.RtcView(1.0, 0.5, 2.0 / w, (C.c_float * 16)(*ident)))
    buf = C.create_string_buffer(16)
    offsets = (C.c_size_t * 2)()
    wrapped = (n_views * bound) % 2**64  # the capacity a wrapped product would ask for
    try:
        for capacity in (wrapped, 2**64 - 1):
            assert lib.rtc_render_views_ppm(scene, 5, n_views, views, buf, capacity, offsets, None) == RTC_ERR_INVALID, capacity
            assert b"overflows" in lib.rtc_last_error()
    finally:
        lib.rtc_scene_destroy(scene)


def test_python_wrappers_reject_a_bad_out(host):
    import ray_tracer_challenge_b200 as rt
    from ray_tracer_challenge_b200 import scenes

    cam, world = scenes.soft_shadows(host, width=40, height=20, u_steps=2, v_steps=2)
    views = scenes.orbit_cameras(host, cam, 3)
    need = 3 * host.lib.rtc_ppm_bound(40, 20)
    read_only = np.zeros(need, np.uint8)
    read_only.flags.writeable = False
    bad = (np.zeros(need - 1, np.uint8), np.zeros(need, np.int8), np.zeros(need // 2 + 1, np.uint16),
           np.zeros(2 * need, np.uint8)[::2], read_only, bytearray(need))
    prepared = object.__new__(rt.PreparedScene)  # the check comes before the library is reached: no commit needed
    prepared.api, prepared.camera, prepared.world, prepared.handle = host, cam, world, -1
    for out in bad:
        with pytest.raises(ValueError, match="rtc_ppm_bound"):
            host.render_views_ppm(world, views, 5, out=out)
        with pytest.raises(ValueError, match="rtc_ppm_bound"):
            prepared.render_views_ppm(views, 5, out=out)
    with pytest.raises(ValueError, match="at least one camera"):
        host.render_views_ppm(world, [], 5)


def test_views_ppm_on_host_under_address_sanitizer():
    """This module again in a child process whose harness is built with -fsanitize=address,undefined."""
    if SANITIZED or os.environ.get("RTC_EMU_TSAN"):
        pytest.skip("already inside a sanitized run")
    libasan = subprocess.run(["g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not libasan or not os.path.exists(libasan):
        pytest.skip("no libasan")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RTC_EMU_SANITIZE="1", LD_PRELOAD=libasan, ASAN_OPTIONS="detect_leaks=0:abort_on_error=1",
               UBSAN_OPTIONS="print_stacktrace=1:halt_on_error=1")
    proc = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-p", "no:cacheprovider"],
                          cwd=root, env=env, capture_output=True, text=True)
    tail = (proc.stdout + proc.stderr)[-3000:]
    assert proc.returncode == 0, tail
    assert "passed" in proc.stdout and "AddressSanitizer" not in tail and "runtime error" not in tail, tail
