"""One anti-aliased frame shared by several processes, one shard each (rtc_render_shard_samples,
rtc_render_shard_samples_ppm_rows + rtc_write_shard_ppm), on the HOST: tests/emu/emu_shard_samples.cpp runs rtc_render_samples'
kernels in 128-thread blocks of 32-lane warps with DevFrame.shard / n_shards of shard s of N over the bands the host plans for
it, then the PPM text kernels over that shard's rows.  For every samples variant, N = 1, 2, 3, 5, 8 and n = 1, 2, 3:
  - the union of the shards is, bit for bit in f32 and 8 bits, the box filter of the oracle's render at n W x n H;
  - each shard writes only its bands (the sentinel elsewhere survives);
  - the shards' texts, laid out from the exchanged row lengths, are the oracle's Canvas::to_ppm of that box filter.
Also every argument check of the two new entry points, in order, without a device.  The module runs again under
AddressSanitizer + UBSan.  Test infrastructure only."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.test_device_code_on_host import _build
from tests.test_kernels_on_host import U8_UNWRITTEN, UNWRITTEN, DevCounters, _check_frame, _code, _Lean, _ptr, _scene
from tests.test_samples_on_host import CASES, SIZES, _bind_samples, _want

SANITIZED = bool(os.environ.get("RTC_EMU_SANITIZE"))
BAND_ROWS = 8  # rtc_types.h: kBandRows
RTC_ERR_INVALID, RTC_ERR_STATE = -1, -4
SENTINEL = 0x7F  # DEL: no byte of a PPM text
SHARDS = [1, 2, 3, 5, 8]


@pytest.fixture(scope="module")
def kern(tmp_path_factory):
    device, lib = _build(tmp_path_factory, "emu_shard_samples.cpp")
    P = C.c_void_p
    lib.emu_render_shard_samples.argtypes = [P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, P, P,
                                             C.POINTER(DevCounters), C.POINTER(C.c_int)]
    lib.emu_shard_ppm_rows.argtypes = [P, C.c_int, C.c_int, C.c_int, C.c_int, P]
    lib.emu_write_shard_ppm.restype = C.c_longlong
    lib.emu_write_shard_ppm.argtypes = [P, C.c_int, C.c_int, C.c_int, C.c_int, P, P, C.c_longlong]
    device.rtc_ppm_bound.restype = C.c_size_t
    device.rtc_ppm_bound.argtypes = [C.c_uint32, C.c_uint32]
    return device, _bind_samples(lib)


@pytest.fixture(scope="module")
def host():
    import ray_tracer_challenge_b200 as rt

    return rt.new_session()


def _owned_rows(h, shard, n_shards):
    return np.array([y // BAND_ROWS % n_shards == shard for y in range(h)])


def _render_shard(kern, scene, w, h, n, shard, n_shards, converge, stream, lean):
    """Shard `shard` of n_shards into fresh sentinel-filled planes, in two slices when it owns two bands or more."""
    device, lib = kern
    rgb = np.full((h, w, 3), UNWRITTEN, np.uint32).view(np.float32)
    u8 = np.full((h, w, 3), U8_UNWRITTEN, np.uint8)
    ctr, var = DevCounters(), C.c_int(-1)
    with _Lean(lean):
        rc = lib.emu_render_shard_samples(scene, 5, n, shard, n_shards, 2, converge, stream, _ptr(rgb), _ptr(u8), C.byref(ctr),
                                          C.byref(var))
    assert rc == 0, device.rtc_last_error()
    return rgb, u8, var.value


def _shard_text(kern, planes, w, h):
    """Every shard's phase 1 into one row-length array (the exchange), then every shard's phase 2 into one sentinel-filled
    buffer: the text."""
    device, lib = kern
    n_shards = len(planes)
    row_bytes = np.zeros(h, np.uint64)
    for s, u8 in enumerate(planes):
        lib.emu_shard_ppm_rows(_ptr(u8), w, h, s, n_shards, _ptr(row_bytes))
    cap = device.rtc_ppm_bound(w, h)
    out = np.full(cap, SENTINEL, np.uint8)
    total = None
    for s, u8 in enumerate(planes):
        n = lib.emu_write_shard_ppm(_ptr(u8), w, h, s, n_shards, _ptr(row_bytes), _ptr(out), cap)
        assert n >= 0, {-1: "the text outgrew rtc_ppm_bound", -2: "ppm_write wrote past a shard's text"}[n]
        assert total is None or n == total
        total = n
    assert (out[total:] == SENTINEL).all(), "a byte at or past the text's length was written"
    return out[:total].tobytes().decode("ascii")


def _oracle_ppm(oracle, want, w, h):
    c = oracle.new_canvas(w, h)
    c.data[:] = want
    return c.to_ppm()


@pytest.mark.parametrize("n", [1, 2, 3])
@pytest.mark.parametrize("size", SIZES, ids=["24x13", "21x10"])
@pytest.mark.parametrize("name", sorted(CASES))
def test_shards_make_up_the_oracle_box_filter(name, size, n, kern, host, oracle):
    """Every variant launch_samples picks, N = 1, 2, 3, 5, 8 shards: each shard's writes stay inside its bands, the union is
    the box filter of the oracle's render at n W x n H bit for bit, and the shards' texts are the oracle's to_ppm of it."""
    device, _ = kern
    make, (converge, stream, lean), (kind, *flags) = CASES[name]
    w, h = size
    want = _want(oracle, make, w, h, n)
    want_ppm = _oracle_ppm(oracle, want, w, h)
    scene = _scene(host, make, w, h)
    try:
        for n_shards in SHARDS:
            rgb = np.full((h, w, 3), UNWRITTEN, np.uint32).view(np.float32)
            u8 = np.full((h, w, 3), U8_UNWRITTEN, np.uint8)
            planes = []
            for s in range(n_shards):
                srgb, su8, var = _render_shard(kern, scene, w, h, n, s, n_shards, converge, stream, lean)
                mine = _owned_rows(h, s, n_shards)
                assert (srgb[~mine].view(np.uint32) == UNWRITTEN).all(), (name, n_shards, s, "f32 row outside the shard")
                assert (su8[~mine] == U8_UNWRITTEN).all(), (name, n_shards, s, "8-bit row outside the shard")
                if mine.any():
                    assert (var >> 5, var & 31) == (kind, _code(*flags)), (name, var)
                rgb[mine], u8[mine] = srgb[mine], su8[mine]
                planes.append(su8)
            _check_frame(oracle, rgb, u8, want, (name, size, n, n_shards))
            assert _shard_text(kern, planes, w, h) == want_ppm, (name, size, n, n_shards)
    finally:
        device.rtc_scene_destroy(scene)


def _lib():
    import ray_tracer_challenge_b200 as rt

    lib = rt.device_library()
    lib.rtc_last_error.restype = C.c_char_p
    lib.rtc_render_shard_samples.argtypes = [C.c_void_p, C.c_int32, C.c_uint32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                             C.c_void_p]
    lib.rtc_render_shard_samples_ppm_rows.argtypes = [C.c_void_p, C.c_int32, C.c_uint32, C.c_int32, C.c_int32, C.c_void_p,
                                                      C.c_void_p]
    lib.rtc_set_camera.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_float)]
    lib.rtc_scene_destroy.argtypes = [C.c_void_p]
    return lib


def test_shard_samples_check_their_arguments_in_order_before_the_scene_state():
    """NULL scene, (text) row_bytes, the shard, the samples and the sample canvas, the depth, then the uncommitted scene."""
    lib = _lib()
    scene = C.c_void_p()
    assert lib.rtc_scene_create(C.byref(scene)) == 0
    ident = (C.c_float * 16)(*[1.0 if i % 5 == 0 else 0.0 for i in range(16)])
    w, h = 64, 32
    rgb = np.full((h, w, 3), 7.0, np.float32)
    rows = np.full(h, 777, np.uint64)

    def frames(scene=scene, depth=5, n=2, shard=0, n_shards=2, rows=None):
        return lib.rtc_render_shard_samples(scene, depth, n, shard, n_shards, _ptr(rgb), None, None)

    def text(scene=scene, depth=5, n=2, shard=0, n_shards=2, rows=rows.ctypes.data):
        return lib.rtc_render_shard_samples_ppm_rows(scene, depth, n, shard, n_shards, rows, None)

    def refused(call, code, what, **kw):
        assert call(**kw) == code, (call.__name__, kw)
        assert what.encode() in lib.rtc_last_error(), (call.__name__, kw, lib.rtc_last_error())

    try:
        assert lib.rtc_set_camera(scene, w, h, 1.0, 0.5, 2.0 / w, ident) == 0
        for call in (frames, text):
            # every check fails at once: the first in the order decides
            assert call(scene=None, rows=None, shard=5, n=0, depth=-1) == RTC_ERR_INVALID
            assert b"null scene" in lib.rtc_last_error()
        refused(text, RTC_ERR_INVALID, "row_bytes must be non-null", rows=None, shard=5, n=0, depth=-1)
        for call in (frames, text):
            for shard, n_shards in ((0, 0), (0, -1), (-1, 2), (2, 2), (5, 3)):
                refused(call, RTC_ERR_INVALID, "n_shards must be >= 1", shard=shard, n_shards=n_shards, n=0, depth=-1)
            for n in (0, 17, 1 << 31):
                refused(call, RTC_ERR_INVALID, "samples_per_axis", n=n, depth=-1)
            for depth in (-1, 24):
                refused(call, RTC_ERR_INVALID, "reflection_recursion_depth", depth=depth)
            # valid arguments: the scene is not committed
            for n in (1, 16):
                for depth in (0, 23):
                    for shard, n_shards in ((0, 1), (1, 2), (7, 8)):
                        refused(call, RTC_ERR_STATE, "before rtc_scene_commit", n=n, depth=depth, shard=shard, n_shards=n_shards)
        assert b"rtc_render_shard_samples_ppm_rows" in lib.rtc_last_error()
        # a sample canvas rtc_set_camera would refuse, before the depth: 16384 x 8192 is allowed, 3 x 3 samples of it are not
        assert lib.rtc_set_camera(scene, 16384, 8192, 1.0, 0.5, 2.0 / 16384, ident) == 0
        for call in (frames, text):
            refused(call, RTC_ERR_STATE, "before rtc_scene_commit", n=2)
            refused(call, RTC_ERR_INVALID, "sample canvas", n=3, depth=99)
            refused(call, RTC_ERR_INVALID, "n_shards must be >= 1", n=3, n_shards=0)  # the shard before the canvas
        assert (rgb == 7.0).all() and (rows == 777).all()  # nothing written on a refused call
    finally:
        lib.rtc_scene_destroy(scene)


def test_python_wrappers_pass_shards_and_samples(host):
    """render_samples(shard=, n_shards=) and render_shard_ppm_rows(samples=) check their arrays and reach the host library
    with argument lists its ctypes signatures take (a mismatch raises TypeError); without a commit it refuses the handle."""
    import ray_tracer_challenge_b200 as rt
    from ray_tracer_challenge_b200 import scenes

    cam, world = scenes.soft_shadows(host, width=40, height=20, u_steps=2, v_steps=2)
    prepared = object.__new__(rt.PreparedScene)  # no commit: the calls stop at the host library's handle check
    prepared.api, prepared.camera, prepared.world, prepared.handle = host, cam, world, -1
    with pytest.raises(ValueError, match="row_bytes"):
        prepared.render_shard_ppm_rows(0, 2, np.zeros(19, np.uint64), samples=2)
    for call in (lambda: prepared.render_samples(2, shard=1, n_shards=2),
                 lambda: prepared.render_shard_ppm_rows(1, 2, np.zeros(20, np.uint64), samples=2)):
        with pytest.raises(rt.RtcError, match="bad prepared handle"):
            call()


def test_shard_samples_on_host_under_address_sanitizer():
    """This module again in a child process whose harness is built with -fsanitize=address,undefined."""
    if SANITIZED or os.environ.get("RTC_EMU_TSAN"):
        pytest.skip("already inside a sanitized run")
    libasan = subprocess.run(["g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not libasan or not os.path.exists(libasan):
        pytest.skip("no libasan")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RTC_EMU_SANITIZE="1", LD_PRELOAD=libasan, ASAN_OPTIONS="detect_leaks=0:abort_on_error=1",
               UBSAN_OPTIONS="print_stacktrace=1:halt_on_error=1")
    proc = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-s", "-p", "no:cacheprovider"],
                          cwd=root, env=env, capture_output=True, text=True, timeout=3600)
    tail = (proc.stdout + proc.stderr)[-4000:]
    assert proc.returncode == 0, tail
    assert "passed" in proc.stdout and "AddressSanitizer" not in tail and "runtime error" not in tail, tail
