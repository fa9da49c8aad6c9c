"""One frame's PPM text written by several processes, one shard each (rtc_render_shard_ppm_rows, rtc_write_shard_ppm), on the
HOST: tests/emu/emu_shard_ppm.cpp's emu_ppm_shards runs the text kernels (dev_ppm.cuh) in 128-thread blocks of 32-lane warps, puts
every shard's row lengths into one array in frame-row order, and has every shard lay out the whole text on its own from that
array (rtc_internal.h: ppm_layout_frame_rows) and copy only its bands.  The text must be the host writer's (CanvasU8.to_ppm),
every byte below its length written and none at or past it, and each shard must write only its bands (shard 0 also the
header).  The module runs again under AddressSanitizer + UBSan.  Also: every argument and state check of the two calls,
without a device."""
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
SENTINEL = 0x7F  # DEL: no byte of a PPM text


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    device, lib = _build(tmp_path_factory, "emu_shard_ppm.cpp")
    lib.emu_ppm_shards.restype = C.c_longlong
    lib.emu_ppm_shards.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_longlong]
    device.rtc_ppm_bound.restype = C.c_size_t
    device.rtc_ppm_bound.argtypes = [C.c_uint32, C.c_uint32]
    return device, lib


@pytest.fixture(scope="module")
def host():
    import ray_tracer_challenge_b200 as rt

    return rt.new_session()


def _shards(emu, u8, n_shards, only=-1):
    """The buffer (pre-filled with the sentinel, rtc_ppm_bound bytes) after the shards' writes, and the text's length."""
    device, lib = emu
    h, w, _ = u8.shape
    u8 = np.ascontiguousarray(u8)
    cap = device.rtc_ppm_bound(w, h)
    out = np.full(cap, SENTINEL, np.uint8)
    n = lib.emu_ppm_shards(u8.ctypes.data, w, h, n_shards, only, out.ctypes.data, cap)
    assert n >= 0, {-1: "the text outgrew rtc_ppm_bound", -2: "ppm_write wrote past a shard's text",
                    -3: "two shards laid out different lengths"}[n]
    return out, n


def _host_ppm(host, u8):
    import ray_tracer_challenge_b200 as rt

    h, w, _ = u8.shape
    return rt.CanvasU8(w, h, np.ascontiguousarray(u8), host).to_ppm()


def _row_spans(text, h):
    """The header's length and [start, end) of every frame row's text.  A row's values fill whole lines (its last value ends
    with a newline), so the rows are found by counting values: 3 * width per row."""
    lines = text.split("\n")
    w = int(lines[1].split(" ")[0])
    header = sum(len(line) + 1 for line in lines[:3])
    spans, at, line = [], header, 3
    for _ in range(h):
        start, values = at, 0
        while values < 3 * w:
            values += len(lines[line].split(" "))
            at += len(lines[line]) + 1
            line += 1
        spans.append((start, at))
    return header, spans


def _check_shards(emu, host, u8, n_shards):
    h = u8.shape[0]
    want = _host_ppm(host, u8)
    out, n = _shards(emu, u8, n_shards)
    assert n == len(want), (u8.shape, n_shards)
    assert not (out[:n] == SENTINEL).any(), "a byte of the text was not written"
    assert (out[n:] == SENTINEL).all(), "a byte at or past the text's length was written"
    assert out[:n].tobytes().decode("ascii") == want, (u8.shape, n_shards)
    if n_shards == 1:
        return
    # each shard alone: exactly its bands' bytes (and shard 0 the header), the rest untouched
    header, spans = _row_spans(want, h)
    for shard in range(n_shards):
        alone, m = _shards(emu, u8, n_shards, only=shard)
        assert m == n
        mine = np.zeros(len(alone), bool)
        if shard == 0:
            mine[:header] = True
        for y, (a, b) in enumerate(spans):
            if y // BAND_ROWS % n_shards == shard:
                mine[a:b] = True
        written = alone != SENTINEL
        assert np.array_equal(written, mine), (u8.shape, n_shards, shard)
        assert alone[mine].tobytes() == np.frombuffer(want.encode(), np.uint8)[mine[:n]].tobytes()


def test_shards_assemble_the_host_writers_text(emu, host):
    rng = np.random.default_rng(17)
    for w, h in ((23, 37), (1, 9), (300, 64), (57, 100), (5, 17), (40, 8)):
        u8 = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        u8[rng.random((h, w)) < 0.3] = 3  # runs of one-digit values: lines of up to 34 values
        for n_shards in range(1, 6):  # (40, 8) is one band: shards 1.. own none
            _check_shards(emu, host, u8, n_shards)


def test_a_4k_frame_in_eight_shards(emu, host):
    """A 3840 x 2160 random plane split 8 ways; under the sanitizers its first 64 rows."""
    rng = np.random.default_rng(19)
    u8 = rng.integers(0, 256, (64 if SANITIZED else 2160, 3840, 3), dtype=np.uint8)
    want = _host_ppm(host, u8)
    out, n = _shards(emu, u8, 8)
    assert n == len(want) and out[:n].tobytes().decode("ascii") == want
    assert (out[n:] == SENTINEL).all()


def test_row_spans_helper():
    """_row_spans finds each row's text (the per-shard checks above rest on it)."""
    text = "P3\n2 2\n255\n1 2 3 4 5 6\n7 8 9 10 11 12\n"
    header, spans = _row_spans(text, 2)
    assert header == len("P3\n2 2\n255\n")
    assert [text[a:b] for a, b in spans] == ["1 2 3 4 5 6\n", "7 8 9 10 11 12\n"]


def _lib():
    import ray_tracer_challenge_b200 as rt

    lib = rt.device_library()
    lib.rtc_last_error.restype = C.c_char_p
    lib.rtc_ppm_bound.restype = C.c_size_t
    lib.rtc_ppm_bound.argtypes = [C.c_uint32, C.c_uint32]
    lib.rtc_render_shard_ppm_rows.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    lib.rtc_write_shard_ppm.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t,
                                        C.POINTER(C.c_size_t)]
    lib.rtc_set_camera.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_float)]
    lib.rtc_scene_destroy.argtypes = [C.c_void_p]
    return lib


def test_shard_ppm_checks_its_arguments_before_the_scene_state():
    lib = _lib()
    scene = C.c_void_p()
    assert lib.rtc_scene_create(C.byref(scene)) == 0
    ident = (C.c_float * 16)(*[1.0 if i % 5 == 0 else 0.0 for i in range(16)])
    w, h = 64, 32
    assert lib.rtc_set_camera(scene, w, h, 1.0, 0.5, 2.0 / w, ident) == 0
    bound = lib.rtc_ppm_bound(w, h)
    buf = C.create_string_buffer(bound)
    n = C.c_size_t(12345)
    rows_in = np.full(h, 9 * w, np.uint64)  # lengths in range
    rows_out = np.full(h, 777, np.uint64)

    def phase1(scene=scene, depth=5, shard=0, n_shards=2, row_bytes=rows_out.ctypes.data):
        return lib.rtc_render_shard_ppm_rows(scene, depth, shard, n_shards, row_bytes, None)

    def phase2(scene=scene, shard=0, n_shards=2, row_bytes=rows_in.ctypes.data, ppm=buf, capacity=bound, ppm_bytes=C.byref(n)):
        return lib.rtc_write_shard_ppm(scene, shard, n_shards, row_bytes, ppm, capacity, ppm_bytes)

    def refused(call, code, text, **kw):
        assert call(**kw) == code, kw
        assert text.encode() in lib.rtc_last_error(), (kw, lib.rtc_last_error())

    try:
        assert phase1(scene=None) == RTC_ERR_INVALID
        refused(phase1, RTC_ERR_INVALID, "non-null", row_bytes=None)
        for shard, n_shards in ((0, 0), (0, -1), (-1, 2), (2, 2), (5, 3)):
            refused(phase1, RTC_ERR_INVALID, "n_shards must be >= 1", shard=shard, n_shards=n_shards)
        for depth in (-1, 24):
            refused(phase1, RTC_ERR_INVALID, "reflection_recursion_depth", depth=depth)

        assert phase2(scene=None) == RTC_ERR_INVALID
        for arg in ("row_bytes", "ppm", "ppm_bytes"):
            refused(phase2, RTC_ERR_INVALID, "non-null", **{arg: None})
        for shard, n_shards in ((0, 0), (-1, 2), (2, 2)):
            refused(phase2, RTC_ERR_INVALID, "n_shards must be >= 1", shard=shard, n_shards=n_shards)
        refused(phase2, RTC_ERR_INVALID, "rtc_ppm_bound", capacity=bound - 1)
        refused(phase2, RTC_ERR_INVALID, "rtc_ppm_bound", capacity=0)
        for row, value in ((0, 6 * w - 1), (h - 1, 12 * w + 1), (17, 0), (3, 2**64 - 1)):
            bad = rows_in.copy()
            bad[row] = value
            refused(phase2, RTC_ERR_INVALID, f"row_bytes[{row}] = {value} is outside", row_bytes=bad.ctypes.data)
        # the range's ends are valid
        edges = rows_in.copy()
        edges[0], edges[1] = 6 * w, 12 * w
        refused(phase2, RTC_ERR_STATE, "before rtc_scene_commit", row_bytes=edges.ctypes.data)

        # valid arguments: the scene is not committed
        for depth in (0, 23):
            refused(phase1, RTC_ERR_STATE, "before rtc_scene_commit", depth=depth)
        for shard, n_shards in ((0, 1), (1, 2), (7, 8)):
            refused(phase1, RTC_ERR_STATE, "before rtc_scene_commit", shard=shard, n_shards=n_shards)
            refused(phase2, RTC_ERR_STATE, "before rtc_scene_commit", shard=shard, n_shards=n_shards)
        refused(phase2, RTC_ERR_STATE, "before rtc_scene_commit", capacity=bound + 1)
        # nothing written on a refused call
        assert n.value == 12345 and buf.raw == b"\0" * bound and (rows_out == 777).all() and (rows_in == 9 * w).all()
    finally:
        lib.rtc_scene_destroy(scene)


def test_python_wrappers_check_their_arrays(host):
    import ray_tracer_challenge_b200 as rt
    from ray_tracer_challenge_b200 import scenes

    cam, world = scenes.soft_shadows(host, width=40, height=20, u_steps=2, v_steps=2)
    prepared = object.__new__(rt.PreparedScene)  # the checks come before the library is reached: no commit needed
    prepared.api, prepared.camera, prepared.world, prepared.handle = host, cam, world, -1
    read_only = np.zeros(20, np.uint64)
    read_only.flags.writeable = False
    for rows in (np.zeros(19, np.uint64), np.zeros(20, np.int64), np.zeros(40, np.uint64)[::2], read_only, [0] * 20):
        with pytest.raises(ValueError, match="row_bytes"):
            prepared.render_shard_ppm_rows(0, 2, rows)
        with pytest.raises(ValueError, match="row_bytes"):
            prepared.write_shard_ppm(0, 2, rows, np.zeros(host.lib.rtc_ppm_bound(40, 20), np.uint8))
    rows = np.zeros(20, np.uint64)
    with pytest.raises(ValueError, match="rtc_ppm_bound"):
        prepared.write_shard_ppm(0, 2, rows, np.zeros(host.lib.rtc_ppm_bound(40, 20) - 1, np.uint8))
    with pytest.raises(ValueError, match="needs out"):
        prepared.write_shard_ppm(0, 2, rows, None)


def test_shared_text_layout(tmp_path):
    """multi.SharedText: height uint64 row lengths, then rtc_ppm_bound bytes of text, in one segment both ranks see."""
    import ray_tracer_challenge_b200 as rt
    from ray_tracer_challenge_b200 import multi

    name = f"rtc_test_text_{os.getpid()}"
    owner = multi.SharedText(name, 40, 20, create=True)
    other = multi.SharedText(name, 40, 20, create=False)
    try:
        bound = rt.new_session().lib.rtc_ppm_bound(40, 20)
        assert owner.bound == bound and owner.nbytes == 20 * 8 + bound
        assert owner.row_bytes.dtype == np.uint64 and owner.row_bytes.shape == (20,) and owner.buf.nbytes == bound
        owner.row_bytes[3] = 12345
        other.buf[:5] = np.frombuffer(b"P3\n40", np.uint8)
        assert other.row_bytes[3] == 12345 and owner.text(5) == "P3\n40"
        assert owner.buf.ctypes.data == owner.address + 20 * 8
    finally:
        other.close()
        owner.close()


def test_shard_ppm_on_host_under_address_sanitizer():
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
