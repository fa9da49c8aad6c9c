"""rtc_render_ppm's text kernels (dev_ppm.cuh: ppm_row_bytes, ppm_write) on the HOST in 128-thread blocks of 32-lane warps
(tests/emu/emu_ppm.cpp, tests/emu/simt.h), with the host scan rtc_render_ppm runs between them (rtc_internal.h:
ppm_layout).  The text must be byte for byte the host writer's (ppm_from_u8, CanvasU8.to_ppm) and the oracle's
Canvas::to_ppm (canvas.rs:58-96), also for a frame split over 2 and 3 devices.  The module runs again under
AddressSanitizer + UBSan.  Also: rtc_ppm_bound and every argument check of rtc_render_ppm, without a device."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.test_device_code_on_host import _build

SANITIZED = bool(os.environ.get("RTC_EMU_SANITIZE"))
BAND_ROWS = 8  # rtc_types.h: kBandRows
RTC_ERR_INVALID, RTC_ERR_STATE = -1, -4


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    device, lib = _build(tmp_path_factory, "emu_ppm.cpp")
    lib.emu_ppm.restype = C.c_longlong
    lib.emu_ppm.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_longlong]
    lib.emu_ppm_row_bytes.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    device.rtc_ppm_bound.restype = C.c_size_t
    device.rtc_ppm_bound.argtypes = [C.c_uint32, C.c_uint32]
    return device, lib


@pytest.fixture(scope="module")
def host():
    import ray_tracer_challenge_b200 as rt

    return rt.new_session()


def _emu_ppm(emu, u8, n_dev=1):
    device, lib = emu
    h, w, _ = u8.shape
    u8 = np.ascontiguousarray(u8)
    cap = device.rtc_ppm_bound(w, h)
    out = np.zeros(cap, np.uint8)
    n = lib.emu_ppm(u8.ctypes.data, w, h, n_dev, out.ctypes.data, cap)
    assert n >= 0, "the text outgrew rtc_ppm_bound" if n == -1 else "ppm_write wrote past its device's text"
    return out[:n].tobytes().decode("ascii")


def _host_ppm(host, u8):
    import ray_tracer_challenge_b200 as rt

    h, w, _ = u8.shape
    return rt.CanvasU8(w, h, np.ascontiguousarray(u8), host).to_ppm()


def _oracle_ppm(oracle, u8):
    """Canvas::to_ppm of an f32 canvas whose scale_color values are u8: (v + 0.5) / 255 truncates back to v."""
    h, w, _ = u8.shape
    c = oracle.new_canvas(w, h)
    data = ((u8.astype(np.float32) + np.float32(0.5)) / np.float32(255.0)).astype(np.float32)
    assert np.array_equal(np.clip(np.minimum(data * np.float32(255.0), np.float32(255.0)), 0.0, None).astype(np.uint8), u8)
    c.data[:] = data
    return c.to_ppm()


def _planes(rng, w, h):
    return {"zeros": np.zeros((h, w, 3), np.uint8), "255": np.full((h, w, 3), 255, np.uint8),
            "100": np.full((h, w, 3), 100, np.uint8), "random": rng.integers(0, 256, (h, w, 3), dtype=np.uint8)}


def test_small_planes_equal_the_host_writer_and_the_oracle(emu, host, oracle):
    rng = np.random.default_rng(5)
    for w in range(1, 41):
        for h in range(1, 6):
            for name, u8 in _planes(rng, w, h).items():
                want = _host_ppm(host, u8)
                assert _emu_ppm(emu, u8) == want, (w, h, name)
                assert _oracle_ppm(oracle, u8) == want, (w, h, name)


def _first_line_ends(digits):
    """The columns at which the values of the first line end, by the rule of canvas.rs:47-55, for these digit counts."""
    line, ends = 0, []
    for i, d in enumerate(digits):
        line += d
        ends.append(line)
        if i + 1 == len(digits) or line >= 67:
            return ends
        line += 1


def test_values_ending_at_columns_66_to_69(emu, host, oracle):
    """Rows whose first line has a value ending at exactly column 66, 67, 68 and 69: the space / newline choice at the rule's
    edge (a line of 66 columns goes on, one of 67 or more ends), then the rest of the row from the shifted line start."""
    rng = np.random.default_rng(7)
    value = {1: 7, 2: 42, 3: 200}
    for target in (66, 67, 68, 69):
        rows = []
        while len(rows) < 6:
            digits = list(rng.choice([1, 2, 3], size=3 * 31, p=[0.2, 0.3, 0.5]))
            if target in _first_line_ends(digits):
                rows.append([value[d] for d in digits])
        u8 = np.array(rows, np.uint8).reshape(6, 31, 3)
        want = _host_ppm(host, u8)
        assert _oracle_ppm(oracle, u8) == want
        lines = want.splitlines()[3:]
        assert lines[0][target - 1] != " " and (len(lines[0]) == target or lines[0][target] == " ")
        assert (len(lines[0]) == target) == (target >= 67) and max(len(line) for line in lines) <= 70
        assert _emu_ppm(emu, u8) == want, target
        assert _emu_ppm(emu, u8, 2) == want, target


def test_rows_of_a_4k_frame(emu, host):
    """A 3840 x 2160 random plane (41 KB of text per row, 90 warp steps); under the sanitizers its first 64 rows."""
    rng = np.random.default_rng(9)
    u8 = rng.integers(0, 256, (64 if SANITIZED else 2160, 3840, 3), dtype=np.uint8)
    assert _emu_ppm(emu, u8) == _host_ppm(host, u8)


def test_frames_split_over_devices_assemble_through_the_host_scan(emu, host):
    """Each device encodes only its bands (b % n_dev == device) into its own text; the host scan places every band."""
    rng = np.random.default_rng(11)
    for w, h in ((23, 37), (1, 9), (300, 64), (57, 100), (5, 17), (40, 8)):
        u8 = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        u8[rng.random((h, w)) < 0.3] = 3  # runs of one-digit values: lines of up to 34 values
        want = _host_ppm(host, u8)
        for n_dev in (1, 2, 3):
            assert _emu_ppm(emu, u8, n_dev) == want, (w, h, n_dev)


def test_row_byte_lengths_in_band_order(emu):
    """ppm_row_bytes: device d's j-th row is frame row (d + j // 8 * n_dev) * 8 + j % 8, its length the digits of its values
    plus one separator each."""
    _, lib = emu
    rng = np.random.default_rng(13)
    h, w = 45, 29
    u8 = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    digits = 1 + (u8 >= 10) + (u8 >= 100)
    lengths = (digits + 1).reshape(h, -1).sum(axis=1)
    for n_dev in (1, 2, 3, 7):
        for d in range(n_dev):
            rows = [r for b in range(d, (h + BAND_ROWS - 1) // BAND_ROWS, n_dev) for r in range(b * BAND_ROWS, min(h, (b + 1) * BAND_ROWS))]
            out = np.full(h + 1, -1, np.int64)
            assert lib.emu_ppm_row_bytes(u8.ctypes.data, w, h, d, n_dev, out.ctypes.data) == len(rows)
            assert list(out[:len(rows)]) == list(lengths[rows]), (n_dev, d)
            assert out[len(rows)] == -1


def test_ppm_bound():
    import ray_tracer_challenge_b200 as rt

    lib = rt.device_library()
    lib.rtc_ppm_bound.restype = C.c_size_t
    lib.rtc_ppm_bound.argtypes = [C.c_uint32, C.c_uint32]
    for w, h in ((1, 1), (7, 3), (3840, 2160), (1920, 1080), (0, 0), (65535, 65535)):
        assert lib.rtc_ppm_bound(w, h) == len(f"P3\n{w} {h}\n255\n") + w * h * 12, (w, h)
    assert lib.rtc_ppm_bound(1, 1) == 11 + 12
    # the bound is reached: every value 3 digits and a separator
    host = rt.new_session()
    u8 = np.full((5, 9, 3), 200, np.uint8)
    assert len(_host_ppm(host, u8)) == lib.rtc_ppm_bound(9, 5)


def test_render_ppm_checks_its_arguments_before_the_scene_state():
    import ray_tracer_challenge_b200 as rt

    lib = rt.device_library()
    lib.rtc_last_error.restype = C.c_char_p
    lib.rtc_ppm_bound.restype = C.c_size_t
    lib.rtc_ppm_bound.argtypes = [C.c_uint32, C.c_uint32]
    lib.rtc_render_ppm.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t), C.c_void_p]
    lib.rtc_set_camera.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_float)]
    lib.rtc_scene_destroy.argtypes = [C.c_void_p]
    scene = C.c_void_p()
    assert lib.rtc_scene_create(C.byref(scene)) == 0
    ident = (C.c_float * 16)(*[1.0 if i % 5 == 0 else 0.0 for i in range(16)])
    assert lib.rtc_set_camera(scene, 64, 32, 1.0, 0.5, 2.0 / 64, ident) == 0
    bound = lib.rtc_ppm_bound(64, 32)
    buf = C.create_string_buffer(bound)
    n = C.c_size_t(12345)
    try:
        assert lib.rtc_render_ppm(None, 5, buf, bound, C.byref(n), None) == RTC_ERR_INVALID
        assert lib.rtc_render_ppm(scene, 5, None, bound, C.byref(n), None) == RTC_ERR_INVALID
        assert b"non-null" in lib.rtc_last_error()
        assert lib.rtc_render_ppm(scene, 5, buf, bound, None, None) == RTC_ERR_INVALID
        assert lib.rtc_render_ppm(scene, 5, buf, bound - 1, C.byref(n), None) == RTC_ERR_INVALID
        assert b"rtc_ppm_bound" in lib.rtc_last_error()
        assert lib.rtc_render_ppm(scene, 5, buf, 0, C.byref(n), None) == RTC_ERR_INVALID
        for depth in (-1, 24):
            assert lib.rtc_render_ppm(scene, depth, buf, bound, C.byref(n), None) == RTC_ERR_INVALID, depth
            assert b"reflection_recursion_depth" in lib.rtc_last_error()
        # valid arguments: the scene is not committed
        for depth in (0, 23):
            assert lib.rtc_render_ppm(scene, depth, buf, bound, C.byref(n), None) == RTC_ERR_STATE
        assert b"before rtc_scene_commit" in lib.rtc_last_error()
        assert n.value == 12345 and buf.raw == b"\0" * bound  # nothing written on a refused call
    finally:
        lib.rtc_scene_destroy(scene)


def test_ppm_on_host_under_address_sanitizer():
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
