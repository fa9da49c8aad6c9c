"""The kernels themselves (dev_kernels.cuh) on the HOST with real 128-thread blocks and 32-lane warps (tests/emu/simt.h,
tests/emu/emu_kernels.cpp): tile and band mapping, learnt tile order, the warp-transposed epilogue, the tile-cost probe,
the small-scene staging by three warps and the per-thread origin cache, the pixel streams' refill, warp-aggregated
counters, the detailed (counting) pass and the wavefront renderer's warp-aggregated appends and refills.  Every frame is
the oracle's Camera::render bit for bit, in f32 and in 8 bits, and the kernel that ran is the one the launch functions
pick for the same inputs.  Collectives are checked for convergence on every call (a lane at another collective or a
rendezvous that never completes aborts); the module runs again under AddressSanitizer + UBSan and under
ThreadSanitizer, the memcheck and racecheck passes the GPU pool cannot run.  Test infrastructure only."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from ray_tracer_challenge_b200 import scenes
from tests.test_device_code_on_host import COLOR_CASES, FP, ROOT, _build, _rays
from tests.wave_child import tight_glass_die

BAND_ROWS, TILE_W = 8, 16        # rtc_types.h: kBandRows, kTileW
WAVE_LEVELS = 25                 # rtc_types.h: kWaveLevels
UNWRITTEN = 0x7FBADBAD           # a NaN no render writes
U8_UNWRITTEN = 0xAB
TILES, VIEWS, TRACE, STREAM, STREAM_VIEWS = range(5)  # emu_kernels.cpp: Kind
RAY_COUNTS = 19                  # emu_color.cpp: kRayCounts
TSAN = bool(os.environ.get("RTC_EMU_TSAN"))


class DevCounters(C.Structure):  # rtc_types.h
    _fields_ = [(n, C.c_ulonglong) for n in ("primary", "secondary", "shadow", "shades", "node_visits")] + \
               [("prim_tests", C.c_ulonglong * 8)] + \
               [(n, C.c_ulonglong) for n in ("xforms", "patterns", "cells", "schlicks", "refr_dirs", "overflows")]


def _bind(lib):
    P = C.c_void_p
    lib.emu_render.argtypes = [P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, P, P, C.c_int, C.c_int, C.c_int, P, P,
                               C.POINTER(DevCounters), C.POINTER(C.c_int)]
    lib.emu_render_views.argtypes = [P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, P, C.c_int, C.c_int, C.c_int, P, P,
                                     C.POINTER(DevCounters), C.POINTER(C.c_int)]
    lib.emu_trace.argtypes = [P, C.c_int, P, P, C.c_int, P, P, P, C.POINTER(DevCounters), C.POINTER(C.c_int)]
    lib.emu_wave_chunk32.argtypes = [P, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, P, P, P]
    lib.emu_set_activemask.argtypes = [C.c_int, C.c_uint]
    lib.emu_set_approx.argtypes = [C.c_int, C.c_uint]
    return lib


@pytest.fixture(scope="module")
def kern(tmp_path_factory):
    device, lib = _build(tmp_path_factory, "emu_kernels.cpp")
    return device, _bind(lib)


@pytest.fixture(scope="module")
def kern_sweep(tmp_path_factory):
    device, lib = _build(tmp_path_factory, "emu_kernels.cpp", ["-DRTC_CSG_SWEEP_BUILD"])
    return device, _bind(lib)


@pytest.fixture(scope="module")
def emu_color(tmp_path_factory):
    device, lib = _build(tmp_path_factory, "emu_color.cpp")
    lib.emu_color_at.argtypes = [C.c_void_p, C.c_uint32, FP, FP, C.c_int, C.c_int, C.c_int, FP, FP, C.POINTER(C.c_int32)]
    lib.emu_color_at_counts.argtypes = [C.c_void_p, C.c_uint32, FP, FP, C.c_int, C.POINTER(C.c_uint)]
    lib.emu_set_approx.argtypes = [C.c_int, C.c_uint]
    return device, lib


@pytest.fixture(scope="module")
def host():
    import ray_tracer_challenge_b200 as rt

    return rt.new_session()


RAN = set()  # (kind, variant code) of every launch of this module


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _render(kern, scene, w, h, depth=5, shard=0, n_shards=1, band_begin=0, n_bands=None, order=None, cost=None, detailed=0,
            converge=-1, stream=-1, lean=1):
    device, lib = kern
    if n_bands is None:
        n_bands = len(range(shard, (h + BAND_ROWS - 1) // BAND_ROWS, n_shards)) - band_begin
    rgb = np.full((h, w, 3), UNWRITTEN, np.uint32).view(np.float32)
    u8 = np.full((h, w, 3), U8_UNWRITTEN, np.uint8)
    ctr, var = DevCounters(), C.c_int(-1)
    with _Lean(lean):
        rc = lib.emu_render(scene, depth, shard, n_shards, band_begin, n_bands, _ptr(order), _ptr(cost), detailed, converge,
                            stream, _ptr(rgb), _ptr(u8), C.byref(ctr), C.byref(var))
    assert rc == 0, device.rtc_last_error()
    RAN.add((var.value >> 5, var.value & 31))
    return rgb, u8, ctr, var.value


def _code(stats, small, converge, drawn, lean):
    return 16 * stats + 8 * small + 4 * converge + 2 * drawn + lean


def _scale(oracle, frame):
    return np.vectorize(lambda v: oracle.probe.scale_color(float(v)), otypes=[np.uint8])(frame)


def _same(a, b):
    return (np.ascontiguousarray(a).view(np.uint32) == np.ascontiguousarray(b).view(np.uint32)).all(axis=-1)


def _check_frame(oracle, rgb, u8, want, label):
    same = _same(rgb, want)
    assert same.all(), (label, int((~same).sum()), np.argwhere(~same)[:3], rgb[~same][:2], want[~same][:2])
    want_u8 = _scale(oracle, want)
    assert (u8 == want_u8).all(), (label, np.argwhere((u8 != want_u8).any(axis=2))[:3])


def _soft_lean(rt, width, height):
    return scenes.soft_shadows(rt, width=width, height=height, u_steps=4, v_steps=4, jitter=None, seed=3)


def _soft_table(rt, width, height):
    return scenes.soft_shadows(rt, width=width, height=height, u_steps=4, v_steps=4)


def _first_textures(rt, width, height):
    return scenes.first_textures(rt, width=width, height=height, u_steps=4, v_steps=4)


def _stress(rt, width, height):
    return scenes.stress(rt, width=width, height=height, n_spheres=1500, n_each=6, n_csg=6)


def _dragon(rt, width, height):
    return scenes.dragon_element(rt, width=width, height=height, n_u=24, n_v=12)


def _tight_die(rt, width, height):
    return tight_glass_die(rt, width, height)


def _filter_zoo_table(rt, width, height):
    return scenes.filter_zoo(rt, width=width, height=height, jitter="table")


# name -> (scene, {forced options: the variant each must select})
#   variant: (kind, stats, small, converge, drawn, lean); options: (converge, stream, RTC_LEAN)
FRAME_CASES = {
    "soft_lean_drawn": (_soft_lean, [((-1, -1, 1), (TILES, 0, 1, 0, 1, 1)), ((1, -1, 1), (TILES, 0, 1, 1, 1, 0)),
                                     ((-1, -1, 0), (TILES, 0, 1, 0, 1, 0))]),
    "soft_lean_table": (_soft_table, [((-1, -1, 1), (TILES, 0, 1, 0, 0, 1)), ((-1, -1, 0), (TILES, 0, 1, 0, 0, 0))]),
    "reflect_refract": (lambda rt, width, height: scenes.reflect_refract(rt, width=width, height=height),
                        [((0, -1, 1), (TILES, 0, 1, 0, 0, 0)), ((1, -1, 1), (TILES, 0, 1, 1, 0, 0))]),
    "first_textures": (_first_textures, [((-1, -1, 1), (TILES, 0, 1, 0, 0, 0)), ((1, -1, 1), (TILES, 0, 1, 1, 0, 0))]),
    "filter_zoo": (_filter_zoo_table, [((1, -1, 1), (TILES, 0, 1, 1, 0, 0))]),
    # an area light without the cell-mask loops: the per-cell shadow loop reads the per-thread origin cache
    "zoo_area_light": (lambda rt, width, height: scenes.shapes_zoo(rt, width=width, height=height, area_light=True),
                       [((-1, -1, 1), (TILES, 0, 1, 1, 0, 0)), ((0, -1, 1), (TILES, 0, 1, 0, 0, 0))]),
    "textured": (lambda rt, width, height: scenes.textured(rt, width=width, height=height), [((-1, -1, 1), (TILES, 0, 1, 0, 0, 0))]),
    "dragon_tree": (_dragon, [((0, 0, 1), (TILES, 0, 0, 0, 0, 0)), ((1, 0, 1), (TILES, 0, 0, 1, 0, 0)),
                              ((-1, 1, 1), (STREAM, 0, 0, 1, 0, 0))]),
    "stress_stream": (_stress, [((-1, -1, 1), (STREAM, 0, 0, 1, 0, 0)), ((1, 0, 1), (TILES, 0, 0, 1, 0, 0))]),
    "tight_die_stream": (_tight_die, [((-1, -1, 1), (STREAM, 0, 0, 1, 0, 0)), ((0, 0, 1), (TILES, 0, 0, 0, 0, 0))]),
}
SIZES = [(48, 24), (61, 37)]  # width divisible by 8 (the staged epilogue) and a ragged frame


def _scene(host, make, w, h):
    cam, world = make(host, width=w, height=h)
    return host.export_scene(cam, world)


class _Lean:
    """RTC_LEAN=0 keeps a lean-eligible scene on the general build; read whenever the harness flattens the scene"""

    def __init__(self, lean):
        self.lean = lean

    def __enter__(self):
        os.environ["RTC_LEAN"] = str(self.lean)

    def __exit__(self, *exc):
        del os.environ["RTC_LEAN"]


@pytest.mark.parametrize("size", SIZES, ids=["48x24", "61x37"])
@pytest.mark.parametrize("name", sorted(FRAME_CASES))
def test_kernel_frames_match_oracle_bit_for_bit(name, size, kern, host, oracle):
    """render_tiles and render_stream as launch_render picks them — lean, drawn, table, converging or not, small table or
    tree, pixel stream — over whole frames: the oracle's f32 and 8-bit canvases, and its secondary rays and shades."""
    if TSAN and size != SIZES[0]:
        pytest.skip("one size under ThreadSanitizer: the one with the staged epilogue")
    device, _ = kern
    make, options = FRAME_CASES[name]
    w, h = size
    ocam, oworld = make(oracle, w, h)
    want = np.asarray(ocam.render(oworld, 5).data, np.float32)
    st = ocam.last_stats
    for (converge, stream, lean), (kind, *flags) in options:
        scene = _scene(host, make, w, h)
        try:
            rgb, u8, ctr, var = _render(kern, scene, w, h, converge=converge, stream=stream, lean=lean)
        finally:
            device.rtc_scene_destroy(scene)
        assert (var >> 5, var & 31) == (kind, _code(*flags)), (name, converge, stream, lean, var)
        _check_frame(oracle, rgb, u8, want, (name, size, converge, stream, lean))
        assert (ctr.secondary, ctr.shades) == (st.secondary_rays, st.shades), (name, converge, stream, st.as_dict())


def test_shards_chunks_tile_order_and_probe(kern, host, oracle):
    """Three interleaved shards, one of them in two band_begin chunks, reassemble the frame exactly and write nothing
    outside their bands; a random learnt tile order renders the same frame; with the tile-cost probe on, every rendered
    tile's cost is non-zero and no other entry is written (lean and general builds)."""
    device, _ = kern
    w, h = 61, 37
    for make, lean in ((_soft_lean, 1), (_soft_lean, 0), (_dragon, 1)):
        ocam, oworld = make(oracle, w, h)
        want = np.asarray(ocam.render(oworld, 5).data, np.float32)
        scene = _scene(host, make, w, h)
        try:
            whole = np.full((h, w, 3), UNWRITTEN, np.uint32).view(np.float32)
            for shard, band_begin, n_bands in ((0, 0, 2), (1, 0, 1), (1, 1, 1), (2, 0, 1)):
                rgb, u8, _, _ = _render(kern, scene, w, h, shard=shard, n_shards=3, band_begin=band_begin, n_bands=n_bands, stream=0, lean=lean)
                rows = np.zeros(h, bool)
                for band in list(range(shard, (h + 7) // 8, 3))[band_begin:band_begin + n_bands]:
                    rows[band * BAND_ROWS:(band + 1) * BAND_ROWS] = True
                assert _same(rgb[rows], want[rows]).all() and (rgb[~rows].view(np.uint32) == UNWRITTEN).all(), shard
                assert (u8[~rows] == U8_UNWRITTEN).all()
                assert (whole[rows].view(np.uint32) == UNWRITTEN).all()
                whole[rows] = rgb[rows]
            assert _same(whole, want).all()
            tiles_x, bands = (w + TILE_W - 1) // TILE_W, (h + BAND_ROWS - 1) // BAND_ROWS
            order = np.random.default_rng(5).permutation(tiles_x * bands).astype(np.int32)
            cost = np.zeros(tiles_x * bands, np.uint32)
            rgb, u8, _, _ = _render(kern, scene, w, h, order=order, cost=cost, stream=0, lean=lean)
            _check_frame(oracle, rgb, u8, want, ("tile order", lean))
            assert (cost != 0).all(), cost
            cost[:] = 0
            rgb, _, _, _ = _render(kern, scene, w, h, n_bands=2, cost=cost, stream=0, lean=lean)
            assert (cost[:2 * tiles_x] != 0).all() and not cost[2 * tiles_x:].any(), cost
        finally:
            device.rtc_scene_destroy(scene)


COUNT_FIELDS = ["node_visits"] + [f"prim_tests[{i}]" for i in range(8)] + ["xforms", "patterns", "cells", "schlicks",
                                                                            "refr_dirs", "overflows"]


@pytest.mark.parametrize("name", ["soft_lean_drawn", "reflect_refract", "first_textures", "dragon_tree", "stress_stream"])
def test_detailed_pass_counts_every_ray_once(name, kern, emu_color, host, oracle):
    """The detailed (counting) pass renders the timed build's frame, counts the oracle's secondary rays and shades, and
    every work counter equals the sum over the frame's pixels of the one-lane color_at counts: per-lane work does not
    depend on convergence, so a difference is an aggregation or double-count bug."""
    device, lib = emu_color
    w, h = 40, 24
    make, _ = FRAME_CASES[name]
    ocam, oworld = make(oracle, w, h)
    want = np.asarray(ocam.render(oworld, 5).data, np.float32)
    st = ocam.last_stats
    scene = _scene(host, make, w, h)
    try:
        timed, _, _, _ = _render(kern, scene, w, h)
        rgb, u8, ctr, var = _render(kern, scene, w, h, detailed=1)
        assert var & 16, var
        assert _same(rgb, timed).all()
        _check_frame(oracle, rgb, u8, want, name)
        assert (ctr.secondary, ctr.shades) == (st.secondary_rays, st.shades)
        n = (w - 1) * (h - 1)
        o, d = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32)
        for i, (y, x) in enumerate(np.ndindex(h - 1, w - 1)):
            ro, rd = oracle.probe.camera_ray(ocam, x, y)
            o[i], d[i] = ro[:3], rd[:3]
        per = np.zeros((n, RAY_COUNTS), np.uint32)
        assert lib.emu_color_at_counts(scene, n, o.ctypes.data_as(FP), d.ctypes.data_as(FP), 5,
                                       per.ctypes.data_as(C.POINTER(C.c_uint))) == 0
        tot = per.astype(np.uint64).sum(axis=0)
        got = [ctr.node_visits] + list(ctr.prim_tests) + [ctr.xforms, ctr.patterns, ctr.cells, ctr.schlicks, ctr.refr_dirs,
                                                           ctr.overflows]
        ref = list(tot[0:8]) + [tot[8] + tot[15]] + list(tot[9:15])  # prim_tests[7] also counts the filter's re-tests
        assert [int(v) for v in got] == [int(v) for v in ref], dict(zip(COUNT_FIELDS, zip(got, ref)))
        assert (int(tot[16]), int(tot[17])) == (st.secondary_rays, st.shades)
        assert tot[0] > 0 or tot[1:9].sum() > 0
    finally:
        device.rtc_scene_destroy(scene)


def _orbit(host, cam, n, degrees):
    """scenes.orbit_cameras' turntable as (eye, look-at point, field of view) per view, for cameras of either API"""
    import math

    inv = np.asarray(host.camera_view(cam).transform_inverse, np.float64).reshape(4, 4)
    eye, fwd = inv[:3, 3], -inv[:3, 2]
    t = -(eye[0] * fwd[0] + eye[2] * fwd[2]) / (fwd[0] ** 2 + fwd[2] ** 2)
    pivot = tuple(float(c) for c in eye + t * fwd)
    out = []
    for i in range(n):
        a = math.radians(degrees * i / n)
        dx, dz = eye[0] - pivot[0], eye[2] - pivot[2]
        e = (pivot[0] + dx * math.cos(a) + dz * math.sin(a), eye[1], pivot[2] - dx * math.sin(a) + dz * math.cos(a))
        out.append((tuple(float(c) for c in e), pivot, cam.field_of_view))
    return out


@pytest.mark.parametrize("name", ["soft_lean_drawn", "soft_lean_table", "reflect_refract", "first_textures", "dragon_tree",
                                  "stress_stream"])
def test_views_match_oracle_per_camera(name, kern, host, oracle):
    """render_tiles_views / render_stream_views: view v of a batch is the oracle's render with camera v of an orbit."""
    device, lib = kern
    w, h, n_views = 40, 21, 3
    make, options = FRAME_CASES[name]
    cam, world = make(host, w, h)
    ocam, oworld = make(oracle, w, h)
    orbit = _orbit(host, cam, n_views, 60.0)
    cams = [host.Camera(w, h, fov, host.view_transform(e, p, (0, 1, 0))) for e, p, fov in orbit]
    ocams = [oracle.Camera(w, h, fov, oracle.view_transform(e, p, (0, 1, 0))) for e, p, fov in orbit]
    for (converge, stream, lean), (kind, *flags) in options:
        scene = host.export_scene(cam, world)
        views = [host.export_scene(c, world) for c in cams]
        try:
            rgb = np.full((n_views, h, w, 3), UNWRITTEN, np.uint32).view(np.float32)
            u8 = np.full((n_views, h, w, 3), U8_UNWRITTEN, np.uint8)
            ctr, var = DevCounters(), C.c_int(-1)
            table = (C.c_void_p * n_views)(*[v.value for v in views])
            with _Lean(lean):
                rc = lib.emu_render_views(scene, 5, 0, 1, 0, (h + 7) // 8, table, n_views, converge, stream, _ptr(rgb), _ptr(u8),
                                          C.byref(ctr), C.byref(var))
            assert rc == 0, device.rtc_last_error()
            RAN.add((var.value >> 5, var.value & 31))
            assert var.value >> 5 == (STREAM_VIEWS if kind == STREAM else VIEWS) and var.value & 31 == _code(*flags)
            secondary = shades = 0
            for v in range(n_views):
                want = np.asarray(ocams[v].render(oworld, 5).data, np.float32)
                secondary, shades = secondary + ocams[v].last_stats.secondary_rays, shades + ocams[v].last_stats.shades
                _check_frame(oracle, rgb[v], u8[v], want, (name, v, converge, stream, lean))
            assert (ctr.secondary, ctr.shades) == (secondary, shades)
        finally:
            for v in views:
                device.rtc_scene_destroy(v)
            device.rtc_scene_destroy(scene)


@pytest.mark.parametrize("name,make,kw,code", [
    ("drawn", scenes.soft_shadows, dict(width=40, height=17, u_steps=4, v_steps=4, jitter=None, seed=3), _code(0, 1, 1, 1, 0)),
    ("small", scenes.reflect_refract, dict(width=40, height=17), _code(0, 1, 1, 0, 0)),
    ("tree", scenes.stress, dict(width=40, height=17, n_spheres=1500, n_each=6, n_csg=6), _code(0, 0, 1, 0, 0)),
])
def test_trace_rays_match_oracle(name, make, kw, code, kern, host, oracle):
    """trace_rays for caller rays, n = 680 (not a multiple of the block): ray i is the primary ray of pixel i (the
    counter-mode jitter is keyed by it), so the colours are the oracle's frame; the never-rendered border's rays start
    far above the scene and point away."""
    device, lib = kern
    cam, world = make(host, **kw)
    ocam, oworld = make(oracle, **kw)
    want = np.asarray(ocam.render(oworld, 5).data, np.float32)
    h, w = want.shape[:2]
    n = w * h
    o, d = np.zeros((n, 3), np.float32), np.zeros((n, 3), np.float32)
    o[:, 1], d[:, 1] = 1.0e6, 1.0
    for y in range(h - 1):
        for x in range(w - 1):
            ro, rd = oracle.probe.camera_ray(ocam, x, y)
            o[y * w + x], d[y * w + x] = ro[:3], rd[:3]
    scene = host.export_scene(cam, world)
    try:
        rgb, t = np.zeros((n, 3), np.float32), np.zeros(n, np.float32)
        pos = np.zeros(n, np.int32)
        ctr, var = DevCounters(), C.c_int(-1)
        assert lib.emu_trace(scene, n, _ptr(o), _ptr(d), 5, _ptr(rgb), _ptr(t), _ptr(pos), C.byref(ctr), C.byref(var)) == 0
        RAN.add((var.value >> 5, var.value & 31))
        assert n % 128 and var.value == TRACE * 32 + code
        same = _same(rgb.reshape(h, w, 3), want)
        assert same.all(), (name, int((~same).sum()))
        assert ((t > 0) == (pos >= 0)).all() and (pos >= 0).sum() > n // 2
    finally:
        device.rtc_scene_destroy(scene)


def test_sweep_build_csg_die(kern_sweep, host, oracle):
    """The strict_sweep build (csg_sweep's call sites) on a CSG beyond csg_eval's limits."""
    device, _ = kern_sweep
    w, h = 40, 24
    cam, world = scenes.csg_die(host, width=w, height=h)
    ocam, oworld = scenes.csg_die(oracle, width=w, height=h)
    want = np.asarray(ocam.render(oworld, 5).data, np.float32)
    scene = host.export_scene(cam, world)
    try:
        for converge in (0, 1):
            rgb, u8, ctr, var = _render(kern_sweep, scene, w, h, converge=converge, stream=0)
            assert var >> 5 == TILES
            _check_frame(oracle, rgb, u8, want, ("csg_die", converge))
    finally:
        device.rtc_scene_destroy(scene)


WAVE_CASES = {
    "reflect_refract_csg": (scenes.reflect_refract, dict(width=40, height=24, with_csg=True)),
    "tight_glass_die": (tight_glass_die, dict(width=40, height=26)),
}


@pytest.mark.parametrize("mode", [0, 1, 2], ids=["all_live", "caller", "random"])
@pytest.mark.parametrize("name", sorted(WAVE_CASES))
def test_wavefront_with_warps_matches_oracle(name, mode, kern, host, oracle):
    """The wavefront renderer with 32-lane warps, the product's refill at 8 idle lanes, 2-3 blocks at once: at depths 0,
    1 and 5 the oracle's frame and ray counts, and through pools of exactly T and T - 1 rays (T: primary plus secondary)
    every level stays inside the pool and only the exact pool renders.  __activemask in each mode: frames must not depend
    on it."""
    if TSAN and mode != 2:
        pytest.skip("one mode under ThreadSanitizer")
    device, lib = kern
    make, kw = WAVE_CASES[name]
    cam, world = make(host, **kw)
    lib.emu_set_activemask(mode, 7)
    scene = host.export_scene(cam, world)
    try:
        for depth in ((5,) if TSAN else (0, 1, 5)):
            ocam, oworld = make(oracle, **kw)
            want = np.asarray(ocam.render(oworld, depth).data, np.float32)
            st = ocam.last_stats
            rays = st.primary_rays + st.secondary_rays
            h, w = want.shape[:2]
            for capacity in ((rays, rays - 1) if depth == 5 else (2 * rays,)):
                frame = np.full((h, w, 3), UNWRITTEN, np.uint32).view(np.float32)
                ints = np.zeros(4 * WAVE_LEVELS, np.int32)
                rec = (C.c_ulonglong * 3)()
                assert lib.emu_wave_chunk32(scene, depth, 0, 1, 0, (h + 7) // 8, capacity, 2, _ptr(frame), _ptr(ints), rec) == 0
                base, count = ints[:WAVE_LEVELS].astype(np.int64), ints[WAVE_LEVELS:2 * WAVE_LEVELS].astype(np.int64)
                assert (base + count <= capacity).all()
                assert (rec[0] == 0) == (capacity >= rays), (capacity, rays, rec[0])
                if capacity >= rays:
                    assert _same(frame, want).all(), (name, depth, mode, int((~_same(frame, want)).sum()))
                    assert (rec[1], rec[2]) == (st.secondary_rays, st.shades)
                    assert count[:depth + 1].sum() == rays
    finally:
        lib.emu_set_activemask(0, 1)
        device.rtc_scene_destroy(scene)


@pytest.mark.parametrize("mode", [1, 2, 3], ids=["minus2ulp", "plus2ulp", "random"])
def test_approximate_intrinsics_do_not_change_frames(mode, kern, emu_color, host, oracle):
    """rsqrtf and __fdividef anywhere in their documented envelopes: with the shadow filter on, the color_at cases and
    the lean and small-table frames are still the oracle's, bit for bit."""
    if TSAN:
        pytest.skip("not under ThreadSanitizer")
    device, lib = emu_color
    fp = lambda a: a.ctypes.data_as(FP)  # noqa: E731
    lib.emu_set_approx(mode, 99)
    kern[1].emu_set_approx(mode, 99)
    try:
        for name, (make, kw, small) in sorted(COLOR_CASES.items()):
            cam, world = make(host, **kw)
            ocam, oworld = make(oracle, **kw)
            n = 120
            o, d = _rays(oracle, ocam, n, seed=11)
            want = np.array([oracle.probe.color_at(oworld, o[i], d[i], 5) for i in range(n)], np.float32)
            scene = host.export_scene(cam, world)
            try:
                rgb = np.zeros((n, 3), np.float32)
                assert lib.emu_color_at(scene, n, fp(o), fp(d), 5, int(small), 1, fp(rgb), None, None) == 0
            finally:
                device.rtc_scene_destroy(scene)
            assert _same(rgb, want).all(), (name, mode)
        for make, lean in ((_soft_lean, 1), (_soft_table, 1), (_soft_table, 0)):
            ocam, oworld = make(oracle, 48, 24)
            want = np.asarray(ocam.render(oworld, 5).data, np.float32)
            scene = _scene(host, make, 48, 24)
            try:
                rgb, u8, _, _ = _render(kern, scene, 48, 24, lean=lean)
            finally:
                device.rtc_scene_destroy(scene)
            _check_frame(oracle, rgb, u8, want, (mode, lean))
    finally:
        lib.emu_set_approx(0, 1)
        kern[1].emu_set_approx(0, 1)


def _far_patterns(rt, width=40, height=24):
    """A floor of stripes, rings and checkers whose pattern space is the world scaled by 10^8: every hit lies at pattern
    coordinates far beyond 2^31, where __float2int_rz saturates."""
    from ray_tracer_challenge_b200.api import Material, PointLight
    from ray_tracer_challenge_b200.scenes import PI

    objs = []
    for i, pat in enumerate((rt.Stripes((1, 0.2, 0.2), (0.2, 0.2, 1)), rt.Rings((0.2, 1, 0.2), (1, 1, 0.2)),
                             rt.Checkers((0.9, 0.9, 0.9), (0.1, 0.1, 0.1)))):
        pat.set_transformation(rt.scaling(1e-8, 1e-8, 1e-8))
        objs.append(rt.Plane.build(rt.translation(0, 0, 0) * rt.rotation_z(0.3 * i) * rt.translation(0, -1.0 - i, 0),
                                   Material(pattern=pat, specular=0.0)))
    world = rt.World(objs, PointLight((-10, 10, -10), (1, 1, 1)))
    cam = rt.Camera(width, height, PI / 3.0, rt.view_transform((0, 1.5, -5), (0, 0, 0), (0, 1, 0)))
    return cam, world


def test_pattern_coordinates_beyond_int_range_match_oracle(emu_color, host, oracle):
    """Stripes, rings and checkers evaluated at pattern coordinates >= 2^31: the device's float-to-int conversion
    saturates (so does the oracle's sat_i32); a host shim that casts gives INT_MIN there and picks the other colour."""
    device, lib = emu_color
    cam, world = _far_patterns(host)
    ocam, oworld = _far_patterns(oracle)
    n = 200
    o, d = _rays(oracle, ocam, n, seed=3)
    o[n // 2:], d[n // 2:] = o[: n - n // 2], d[: n - n // 2]  # primary rays only: they all meet a floor
    want = np.array([oracle.probe.color_at(oworld, o[i], d[i], 5) for i in range(n)], np.float32)
    scene = host.export_scene(cam, world)
    try:
        rgb = np.zeros((n, 3), np.float32)
        fp = lambda a: a.ctypes.data_as(FP)  # noqa: E731
        assert lib.emu_color_at(scene, n, fp(o), fp(d), 5, 1, 1, fp(rgb), None, None) == 0
    finally:
        device.rtc_scene_destroy(scene)
    assert np.abs(want).sum() > 0
    same = _same(rgb, want)
    assert same.all(), (int((~same).sum()), rgb[~same][:2], want[~same][:2])


def test_every_variant_ran(kern):
    """The kernels this module ran are all the launch functions of the strict build can select (the frame, view and
    trace tests run before this one)."""
    if TSAN or not RAN:
        pytest.skip("needs the whole module")
    out = (C.c_int * 64)()
    n = kern[1].emu_variants(out)
    want = {(v >> 5, v & 31) for v in out[:n]}
    assert n == 11 + 8 + 3 + 3 and len(want) == n
    assert RAN == want, (sorted(want - RAN), sorted(RAN - want))


def _rerun(env_extra, preload, timeout):
    env = dict(os.environ, LD_PRELOAD=preload, **env_extra)
    # -s: a sanitizer report is written to the fd pytest would capture, and the run ends before pytest prints it
    proc = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-s", "-p", "no:cacheprovider"],
                          cwd=ROOT, env=env, capture_output=True, text=True, timeout=timeout)
    return proc, (proc.stdout + proc.stderr)[-4000:]


def test_kernels_under_address_sanitizer():
    """This module again with the harnesses built with -fsanitize=address,undefined: shared-memory carving (the lean
    build's dynamic block is poisoned past the kSmemOrg * 16 bytes its launch requests), frames, pools."""
    if os.environ.get("RTC_EMU_SANITIZE") or TSAN:
        pytest.skip("already inside a sanitized run")
    libasan = subprocess.run(["g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not libasan or not os.path.exists(libasan):
        pytest.skip("no libasan")
    proc, tail = _rerun(dict(RTC_EMU_SANITIZE="1", ASAN_OPTIONS="detect_leaks=0:abort_on_error=1",
                             UBSAN_OPTIONS="print_stacktrace=1:halt_on_error=1"), libasan, 1800)
    assert proc.returncode == 0, tail
    assert "passed" in proc.stdout and "AddressSanitizer" not in tail and "runtime error" not in tail, tail


def test_kernels_under_thread_sanitizer():
    """A subset of this module again with the harness built with -fsanitize=thread: no data race between the threads
    of a block (shared-memory staging, the warp-transposed epilogue, the origin cache) or between blocks (atomics,
    pixel streams, the wavefront pool)."""
    if os.environ.get("RTC_EMU_SANITIZE") or TSAN:
        pytest.skip("already inside a sanitized run")
    libtsan = subprocess.run(["g++", "-print-file-name=libtsan.so"], capture_output=True, text=True).stdout.strip()
    if not libtsan or not os.path.exists(libtsan):
        pytest.skip("no libtsan")
    proc, tail = _rerun(dict(RTC_EMU_TSAN="1", TSAN_OPTIONS="halt_on_error=1:report_signal_unsafe=0"), libtsan, 1800)
    assert proc.returncode == 0, tail
    assert "passed" in proc.stdout and "ThreadSanitizer" not in tail, tail
