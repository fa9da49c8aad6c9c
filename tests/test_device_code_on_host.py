"""The device code of the tree path, compiled for the HOST (tests/emu/emu_nearest.cpp: dev_math / dev_shapes / dev_bvh
.cuh behind a shim of the CUDA intrinsics they use) and run over the arrays the host half of rtc_scene_commit builds —
the primitive tests, the CSG programs, the group cull chains and the BVH walk checked against the oracle's
World::intersect + Intersection::hit (world.rs:52-60, intersection.rs:30-35) on a machine without a GPU.  Test
infrastructure only: nothing here is a render path, and the product never loads it."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from ray_tracer_challenge_b200 import scenes
from tests.wave_child import tight_glass_die

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA_INCLUDE = "/usr/local/cuda/include"


def _build(tmp_path_factory, source, defines=()):
    import ray_tracer_challenge_b200 as rt

    if shutil.which("g++") is None or not os.path.isdir(CUDA_INCLUDE):
        pytest.skip("needs g++ and the CUDA headers")
    out = tmp_path_factory.mktemp("emu") / ("lib" + source.replace(".cpp", ".so"))
    lib_dir = os.path.dirname(rt.LIB_DEVICE)
    # RTC_EMU_SANITIZE=1 (set by test_device_code_under_address_sanitizer, which re-runs this module in a process with
    # libasan preloaded): the device code's shared-memory carving, bounce stack, traversal stack and CSG hit buffers
    # under AddressSanitizer + UBSan — the memcheck pass a host can give CUDA code
    sanitize = ["-fsanitize=address,undefined", "-fno-omit-frame-pointer", "-fno-sanitize-recover=undefined"] \
        if os.environ.get("RTC_EMU_SANITIZE") else []
    # RTC_EMU_TSAN=1 (test_kernels_under_thread_sanitizer, libtsan preloaded): the host threads of emu_kernels.cpp's
    # blocks under ThreadSanitizer — the racecheck pass
    if os.environ.get("RTC_EMU_TSAN"):
        sanitize = ["-fsanitize=thread", "-fno-omit-frame-pointer"]
    subprocess.run(["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-fPIC", "-shared", "-pthread", *sanitize, *defines,
                    "-I", CUDA_INCLUDE,
                    "-I", os.path.join(ROOT, "ray_tracer_challenge_b200", "csrc"), os.path.join(ROOT, "tests", "emu", source),
                    "-o", str(out), "-L", lib_dir, "-lrtc_b200", f"-Wl,-rpath,{lib_dir}"], check=True)
    device = rt.device_library()  # the raw C ABI; RTLD_GLOBAL, so the harness binds rtc::flatten from it
    device.rtc_last_error.restype = C.c_char_p
    device.rtc_scene_destroy.argtypes = [C.c_void_p]
    return device, C.CDLL(str(out))


FP = C.POINTER(C.c_float)


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    device, lib = _build(tmp_path_factory, "emu_nearest.cpp")
    lib.emu_nearest.argtypes = [C.c_void_p, C.c_uint32, FP, FP, FP, C.POINTER(C.c_int32)]
    return device, lib


@pytest.fixture(scope="module")
def emu_color(tmp_path_factory):
    device, lib = _build(tmp_path_factory, "emu_color.cpp")
    lib.emu_color_at.argtypes = [C.c_void_p, C.c_uint32, FP, FP, C.c_int, C.c_int, C.c_int, FP, FP, C.POINTER(C.c_int32)]
    lib.emu_wave_chunk.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, FP, C.POINTER(C.c_int32),
                                   C.POINTER(C.c_ulonglong)]
    return device, lib


@pytest.fixture(scope="module")
def host():
    import ray_tracer_challenge_b200 as rt

    return rt.new_session()


class _Material(C.Structure):  # include/rtc_b200.h: RtcMaterial
    _fields_ = [("color", C.c_float * 3), ("v", C.c_float * 7), ("pattern", C.c_int32)]


def _raw_scene(device, host, world):
    """An RtcScene with the world's flattened geometry (materials are placeholders: a nearest-hit search reads none)."""
    prims, nodes, refs, _, _ = host.flatten(world)
    scene = C.c_void_p()
    assert device.rtc_scene_create(C.byref(scene)) == 0
    ident = (C.c_float * 16)(1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1)
    device.rtc_set_camera.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_float)]
    assert device.rtc_set_camera(scene, 8, 8, 1.0, 1.0, 0.25, ident) == 0
    assert device.rtc_set_point_light(scene, (C.c_float * 3)(-10, 10, -10), (C.c_float * 3)(1, 1, 1)) == 0
    import ray_tracer_challenge_b200 as rt

    parr = (rt.RtcPrim * max(len(prims), 1))(*prims)
    narr = (rt.RtcNode * max(len(nodes), 1))(*nodes)
    rarr = (C.c_int32 * max(len(refs), 1))(*refs)
    n_mat = max([p.material for p in prims] + [0]) + 1
    marr = (_Material * n_mat)()
    for m in marr:
        m.pattern = -1
    assert device.rtc_set_primitives(scene, len(prims), parr) == 0, device.rtc_last_error()
    assert device.rtc_set_nodes(scene, len(nodes), narr, len(refs), rarr) == 0, device.rtc_last_error()
    assert device.rtc_set_materials(scene, n_mat, marr) == 0, device.rtc_last_error()
    return scene


def _rays(camera_api, cam, n, seed):
    """Primary rays of random pixels plus rays between random points of the scene's volume (secondary-ray-like)."""
    rng = np.random.default_rng(seed)
    o = np.zeros((n, 3), np.float32)
    d = np.zeros((n, 3), np.float32)
    for i in range(n // 2):
        ro, rd = camera_api.probe.camera_ray(cam, int(rng.integers(0, cam.width_pixels - 1)), int(rng.integers(0, cam.height_pixels - 1)))
        o[i], d[i] = ro[:3], rd[:3]
    a = rng.uniform(-6, 6, (n - n // 2, 3)).astype(np.float32)
    b = rng.uniform(-6, 6, (n - n // 2, 3)).astype(np.float32)
    v = b - a
    o[n // 2:] = a
    d[n // 2:] = v / np.linalg.norm(v, axis=1, keepdims=True).astype(np.float32)
    return o, d


SCENES = {
    # tree over spheres, cylinders, cones, cubes and CSG roots (one primitive per leaf)
    "sphere_field": (scenes.stress, dict(width=64, height=36, n_spheres=1500, n_each=6, n_csg=6)),
    # triangle mesh in divided groups (four triangles per leaf, shared transform) + display case + pedestal
    "mesh": (scenes.dragon_element, dict(width=64, height=36, n_u=24, n_v=12)),
    # every CSG operator, nested, with transformed children
    "csg": (scenes.csg_gallery, dict(width=64, height=40)),
    # small scenes run through the same general functions here (linear list, no tree)
    "zoo": (scenes.shapes_zoo, dict(width=64, height=40)),
}


@pytest.mark.parametrize("name", sorted(SCENES))
def test_tree_path_nearest_hit_matches_oracle(name, emu, host, oracle):
    device, lib = emu
    make, kw = SCENES[name]
    cam, world = make(host, **kw)
    ocam, oworld = make(oracle, **kw)
    scene = _raw_scene(device, host, world)
    try:
        n = 600
        o, d = _rays(oracle, ocam, n, seed=7)
        t = np.zeros(n, np.float32)
        prim = np.zeros(n, np.int32)
        fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))  # noqa: E731
        rc = lib.emu_nearest(scene, n, fp(o), fp(d), fp(t), prim.ctypes.data_as(C.POINTER(C.c_int32)))
        assert rc == 0, device.rtc_last_error()
        hits = 0
        for i in range(n):
            ts, _ = oracle.probe.world_intersect(oworld, o[i], d[i], cap=256)
            h = oracle.probe.hit_index(ts)
            want = np.float32(ts[h]) if h >= 0 else np.float32(-1.0)
            assert t[i] == want, (name, i, float(t[i]), float(want), o[i], d[i])  # bit-exact: same IEEE expression order
            hits += h >= 0
        print(name, "hits", hits, "of", n)
        assert hits > n // 10, (name, hits)  # the rays do exercise the scene
    finally:
        device.rtc_scene_destroy.argtypes = [C.c_void_p]
        device.rtc_scene_destroy(scene)


# name -> (scene, arguments, take the small-scene path when the scene qualifies)
COLOR_CASES = {
    "sphere_field": (scenes.stress, dict(width=64, height=36, n_spheres=1500, n_each=6, n_csg=6), False),
    "mesh": (scenes.dragon_element, dict(width=64, height=36, n_u=24, n_v=12), False),
    "csg": (scenes.csg_gallery, dict(width=64, height=40), False),
    "zoo_general_path": (scenes.shapes_zoo, dict(width=64, height=40), False),
    "zoo": (scenes.shapes_zoo, dict(width=64, height=40), True),
    "zoo_area_light": (scenes.shapes_zoo, dict(width=64, height=40, area_light=True), True),
    "soft_shadows_table": (scenes.soft_shadows, dict(width=64, height=32, u_steps=4, v_steps=4), True),  # cell masks, plane cells
    "soft_shadows_100_cells": (scenes.soft_shadows, dict(width=64, height=32), True),
    "reflect_refract": (scenes.reflect_refract, dict(width=64, height=32), True),  # exact shadow test, n1 / n2, Schlick
    "reflect_refract_csg": (scenes.reflect_refract, dict(width=64, height=32, with_csg=True), True),
    "filter_zoo_table": (scenes.filter_zoo, dict(width=64, height=40, jitter="table"), True),
    "filter_zoo_point": (scenes.filter_zoo, dict(width=64, height=40, area_light=False), True),
    "textured": (scenes.textured, dict(width=64, height=40), True),
    "hexagons": (scenes.hexagons, dict(width=64, height=32), True),
}


@pytest.mark.parametrize("name", sorted(COLOR_CASES))
def test_color_at_of_the_device_code_matches_oracle_bit_for_bit(name, emu_color, host, oracle):
    """World::color_at (world.rs:88-101) with everything under it — hit record, patterns, Phong, shadow rays and area
    lights, reflect / refract stack — through the device code on the host: the tree path and the small-scene path, the
    latter with the shadow filter and the cell-mask loops on and off.  f32 results equal the oracle's bit for bit (host
    libm on both sides, IEEE expression order), so in particular the filter changes no value."""
    device, lib = emu_color
    make, kw, small = COLOR_CASES[name]
    cam, world = make(host, **kw)
    ocam, oworld = make(oracle, **kw)
    scene = host.export_scene(cam, world)
    try:
        n = 240
        o, d = _rays(oracle, ocam, n, seed=11)
        want = np.array([oracle.probe.color_at(oworld, o[i], d[i], 5) for i in range(n)], np.float32)
        assert np.abs(want).sum() > 0
        fp = lambda a: a.ctypes.data_as(FP)  # noqa: E731
        for use_filter, converge in (((0, 0), (1, 0), (1, 1)) if small else ((0, 0), (0, 1))):
            lib.emu_set_converge(converge)  # the converging build of color_at (single lane: the vote is the predicate)
            rgb = np.zeros((n, 3), np.float32)
            path = C.c_int32(-1)
            rc = lib.emu_color_at(scene, n, fp(o), fp(d), 5, int(small), use_filter, fp(rgb), None, C.byref(path))
            assert rc == 0, device.rtc_last_error()
            if small:
                assert path.value == 1, "the scene was meant to take the small-scene path"
            same = (rgb.view(np.uint32) == want.view(np.uint32)).all(axis=1)
            assert same.all(), (name, use_filter, converge, int((~same).sum()), rgb[~same][:3], want[~same][:3])
    finally:
        lib.emu_set_converge(0)
        device.rtc_scene_destroy(scene)


def test_empty_world_is_black_through_the_device_code(emu_color, host):
    """No objects at all, and only an empty group: every ray misses, color_at returns black (world.rs:98-100)."""
    device, lib = emu_color
    from ray_tracer_challenge_b200.scenes import PI

    for objects in ([], [host.GroupShape()]):
        cam = host.Camera(16, 8, PI / 2.0, host.view_transform((0, 0, -5), (0, 0, 0), (0, 1, 0)))
        world = host.World(objects, host.PointLight((-10, 10, -10), (1, 1, 1)))
        scene = host.export_scene(cam, world)
        try:
            o = np.zeros((8, 3), np.float32)
            o[:, 2] = -5
            d = np.tile(np.array([0, 0, 1], np.float32), (8, 1))
            rgb = np.ones((8, 3), np.float32)
            fp = lambda a: a.ctypes.data_as(FP)  # noqa: E731
            assert lib.emu_color_at(scene, 8, fp(o), fp(d), 5, 1, 1, fp(rgb), None, None) == 0, device.rtc_last_error()
            assert not rgb.any()
        finally:
            device.rtc_scene_destroy(scene)


@pytest.mark.parametrize("name,make,kw", [
    ("soft_shadows_as_shipped", scenes.soft_shadows, dict(width=40, height=16, u_steps=10, v_steps=10, jitter=None, seed=3)),
    ("filter_zoo_drawn", scenes.filter_zoo, dict(width=40, height=24)),
    ("first_textures_drawn", scenes.first_textures, dict(width=40, height=20, u_steps=4, v_steps=4)),
])
def test_counter_mode_jitter_frame_matches_oracle(name, make, kw, emu_color, host, oracle):
    """Area lights with `jitter_fn = None` draw their samples from the counter-based generator keyed by (seed, pixel,
    path, index): ray i of the harness is pixel i of the frame, so a whole small frame traced through the device code
    (drawn-sample cell masks where the scene is filter-eligible) equals the oracle's Camera::render bit for bit."""
    device, lib = emu_color
    cam, world = make(host, **kw)
    ocam, oworld = make(oracle, **kw)
    want = ocam.render(oworld, 5).data
    w, h = ocam.width_pixels, ocam.height_pixels
    o = np.zeros((w * h, 3), np.float32)
    d = np.zeros((w * h, 3), np.float32)
    o[:, 1], d[:, 1] = 1.0e6, 1.0
    for y in range(h - 1):
        for x in range(w - 1):
            ro, rd = oracle.probe.camera_ray(ocam, x, y)
            o[y * w + x], d[y * w + x] = ro[:3], rd[:3]
    scene = host.export_scene(cam, world)
    try:
        fp = lambda a: a.ctypes.data_as(FP)  # noqa: E731
        for use_filter in (0, 1):
            rgb = np.zeros((w * h, 3), np.float32)
            assert lib.emu_color_at(scene, w * h, fp(o), fp(d), 5, 1, use_filter, fp(rgb), None, None) == 0, device.rtc_last_error()
            got = rgb.reshape(h, w, 3)[: h - 1, : w - 1]
            ref = np.asarray(want, np.float32)[: h - 1, : w - 1]
            same = (got.view(np.uint32) == ref.view(np.uint32)).all(axis=2)
            assert same.all(), (name, use_filter, int((~same).sum()), got[~same][:2], ref[~same][:2])
            # the ray counters of the device code against the oracle's for the same frame (the never-rendered border
            # of the harness' w x h grid holds rays that start far above the scene and point away: they trace nothing)
            rays = (C.c_ulonglong * 4)()
            lib.emu_last_rays(rays)
            st = ocam.last_stats
            assert (rays[1], rays[2], rays[3]) == (st.secondary_rays, st.shadow_rays, st.shades), (list(rays), st.as_dict())
    finally:
        device.rtc_scene_destroy(scene)


def test_shadow_filter_fuzz_through_the_device_code(emu_color, host, oracle):
    """Random filter-eligible scenes (sheared / squashed spheres, tilted planes, boxes, touching and interpenetrating,
    area or point light, table or counter jitter): whole small frames through the device code with the filter and the
    cell-mask loops ON equal the oracle's render bit for bit — the CPU twin of test_gpu_parity's on-device fuzz, on other seeds."""
    device, lib = emu_color
    fp = lambda a: a.ctypes.data_as(FP)  # noqa: E731
    eligible = 0
    for seed in range(100, 116):
        kw = dict(width=28, height=18)
        cam, world = scenes.random_filter_scene(host, seed, **kw)
        ocam, oworld = scenes.random_filter_scene(oracle, seed, **kw)
        eligible += host.inspect(cam, world)["filter_ok"]
        want = np.asarray(ocam.render(oworld, 5).data, np.float32)
        w, h = ocam.width_pixels, ocam.height_pixels
        o = np.zeros((w * h, 3), np.float32)
        d = np.zeros((w * h, 3), np.float32)
        d[:, 2] = 1.0
        for y in range(h - 1):
            for x in range(w - 1):
                ro, rd = oracle.probe.camera_ray(ocam, x, y)
                o[y * w + x], d[y * w + x] = ro[:3], rd[:3]
        scene = host.export_scene(cam, world)
        try:
            rgb = np.zeros((w * h, 3), np.float32)
            assert lib.emu_color_at(scene, w * h, fp(o), fp(d), 5, 1, 1, fp(rgb), None, None) == 0, device.rtc_last_error()
            got = rgb.reshape(h, w, 3)[: h - 1, : w - 1]
            ref = want[: h - 1, : w - 1]
            same = (got.view(np.uint32) == ref.view(np.uint32)).all(axis=2)
            assert same.all(), (seed, int((~same).sum()), got[~same][:2], ref[~same][:2])
        finally:
            device.rtc_scene_destroy(scene)
    assert eligible >= 12, eligible


EXTREMES = ["millimetre", "kilometre", "far light", "tiny spheres", "stretched", "grazing"]


@pytest.mark.parametrize("extreme", EXTREMES)
def test_shadow_filter_at_scale_extremes_through_the_device_code(emu_color, host, oracle, extreme):
    """VERDICT r1 weak #1: the filter's bounds (sphere tolerance, 2^-18 plane / cube bounds, the 0.1 % ball padding, the
    2^-17 |w|^2 / R bundle padding) were only ever exercised in a +-10-unit world of unit-scale objects.  The same
    random scenes in millimetres and kilometres, with the light 10^4 units away, with radius-10^-3 spheres, with
    ellipsoids near the conditioning limit and with a light grazing the floor: whole frames through the device code
    with the filter ON are the oracle's frames, bit for bit."""
    device, lib = emu_color
    fp = lambda a: a.ctypes.data_as(FP)  # noqa: E731
    eligible = 0
    for seed in range(200, 206):
        kw = dict(width=28, height=18, extreme=extreme)
        cam, world = scenes.random_filter_scene(host, seed, **kw)
        ocam, oworld = scenes.random_filter_scene(oracle, seed, **kw)
        eligible += host.inspect(cam, world)["filter_ok"]
        want = np.asarray(ocam.render(oworld, 5).data, np.float32)
        w, h = ocam.width_pixels, ocam.height_pixels
        o = np.zeros((w * h, 3), np.float32)
        d = np.zeros((w * h, 3), np.float32)
        d[:, 2] = 1.0
        for y in range(h - 1):
            for x in range(w - 1):
                ro, rd = oracle.probe.camera_ray(ocam, x, y)
                o[y * w + x], d[y * w + x] = ro[:3], rd[:3]
        scene = host.export_scene(cam, world)
        try:
            rgb = np.zeros((w * h, 3), np.float32)
            assert lib.emu_color_at(scene, w * h, fp(o), fp(d), 5, 1, 1, fp(rgb), None, None) == 0, device.rtc_last_error()
            got = rgb.reshape(h, w, 3)[: h - 1, : w - 1]
            ref = want[: h - 1, : w - 1]
            same = (got.view(np.uint32) == ref.view(np.uint32)).all(axis=2)
            assert same.all(), (extreme, seed, int((~same).sum()), got[~same][:2], ref[~same][:2])
        finally:
            device.rtc_scene_destroy(scene)
    assert eligible >= (2 if extreme == "stretched" else 4), (extreme, eligible)


# ---- the wavefront renderer (dev_wave.cuh) through the device code ------------------------------------------------------
BAND_ROWS = 8                 # rtc_types.h: kBandRows
WAVE_LEVELS = 25              # rtc_types.h: kWaveLevels = kMaxFrames + 1
UNWRITTEN = 0x7FBADBAD        # a NaN no render writes: marks the pixels a chunk must leave alone

WAVE_SCENES = {
    "sphere_field": (scenes.stress, dict(width=64, height=36, n_spheres=1500, n_each=6, n_csg=6)),
    "mesh": (scenes.dragon_element, dict(width=64, height=36, n_u=24, n_v=12)),
    "csg": (scenes.csg_gallery, dict(width=64, height=40)),
    "csg_chain": (scenes.csg_chain, dict(width=61, height=37)),  # ragged last band and last 8-pixel column
    "reflect_refract_csg": (scenes.reflect_refract, dict(width=64, height=32, with_csg=True)),
    "tight_glass_die": (tight_glass_die, dict(width=40, height=26)),  # 26 rays per pixel at depth 5, 260 at depth 9
}


def _shard_bands(h, shard, n_shards):
    return [b for b in range((h + BAND_ROWS - 1) // BAND_ROWS) if b % n_shards == shard]


def _wave_chunk(emu_color, scene, w, h, depth, capacity, shard=0, n_shards=1, band_begin=0, n_bands=None):
    """One chunk through launch_wave's kernel sequence: (frame, base[L], count[L], (overflow, secondary, shades))."""
    device, lib = emu_color
    if n_bands is None:
        n_bands = len(_shard_bands(h, shard, n_shards)) - band_begin
    frame = np.full((h, w, 3), UNWRITTEN, np.uint32).view(np.float32)
    ints = np.zeros(4 * WAVE_LEVELS, np.int32)
    record = (C.c_ulonglong * 3)()
    rc = lib.emu_wave_chunk(scene, depth, shard, n_shards, band_begin, n_bands, capacity, frame.ctypes.data_as(FP),
                            ints.ctypes.data_as(C.POINTER(C.c_int32)), record)
    assert rc == 0, device.rtc_last_error()
    return frame, ints[:WAVE_LEVELS].astype(np.int64), ints[WAVE_LEVELS:2 * WAVE_LEVELS].astype(np.int64), tuple(record)


def _same_bits(a, b):
    return (a.view(np.uint32) == b.view(np.uint32)).all(axis=-1)


@pytest.mark.parametrize("depth", [0, 1, 5, 9])
@pytest.mark.parametrize("name", sorted(WAVE_SCENES))
def test_wavefront_of_the_device_code_matches_oracle_bit_for_bit(name, depth, emu_color, host, oracle):
    """The wavefront renderer's kernels (primary rays, per level the nearest-hit walk, hit record, shadow walk and shade,
    then the post-order combine) over the whole frame as one chunk with an ample pool: the frame is the oracle's
    Camera::render, bit for bit, black last row and column included; the chunk record counts the oracle's secondary rays
    and shades; and the levels lie end to end in the pool, holding exactly the primary plus secondary rays."""
    device, _ = emu_color
    make, kw = WAVE_SCENES[name]
    cam, world = make(host, **kw)
    ocam, oworld = make(oracle, **kw)
    want = np.asarray(ocam.render(oworld, depth).data, np.float32)
    st = ocam.last_stats
    rays = st.primary_rays + st.secondary_rays
    h, w = want.shape[:2]
    scene = host.export_scene(cam, world)
    try:
        frame, base, count, (overflow, secondary, shades) = _wave_chunk(emu_color, scene, w, h, depth, 2 * rays)
    finally:
        device.rtc_scene_destroy(scene)
    same = _same_bits(frame, want)
    assert same.all(), (name, depth, int((~same).sum()), np.argwhere(~same)[:3], frame[~same][:2], want[~same][:2])
    assert (overflow, secondary, shades) == (0, st.secondary_rays, st.shades), (name, depth, st.as_dict())
    assert base[0] == 0 and (base[1:depth + 2] == base[:depth + 1] + count[:depth + 1]).all(), (base, count)
    assert count[:depth + 1].sum() == rays and not count[depth + 1:].any(), (count, rays)
    assert count[0] == st.primary_rays


def test_wavefront_chunks_and_shards_of_the_device_code_match_oracle(emu_color, host, oracle):
    """A frame rendered as chunks of bands (band_begin, n_bands) and as three interleaved shards, one of them in two
    chunks: every part writes exactly the oracle's pixels of its bands and nothing outside them, and the parts' records
    add up to the oracle's secondary rays and shades."""
    device, _ = emu_color
    kw = dict(width=64, height=44, with_csg=True)  # six bands, the last of four rows
    cam, world = scenes.reflect_refract(host, **kw)
    ocam, oworld = scenes.reflect_refract(oracle, **kw)
    depth = 5
    want = np.asarray(ocam.render(oworld, depth).data, np.float32)
    st = ocam.last_stats
    h, w = want.shape[:2]
    partitions = {
        "chunks": [(0, 1, 0, 2), (0, 1, 2, 3), (0, 1, 5, 1)],               # (shard, n_shards, band_begin, n_bands)
        "shards": [(0, 3, 0, 2), (1, 3, 0, 1), (1, 3, 1, 1), (2, 3, 0, 2)],
    }
    scene = host.export_scene(cam, world)
    try:
        for label, parts in partitions.items():
            whole = np.full((h, w, 3), UNWRITTEN, np.uint32).view(np.float32)
            secondary = shades = 0
            for shard, n_shards, band_begin, n_bands in parts:
                frame, _, _, rec = _wave_chunk(emu_color, scene, w, h, depth, 6 * w * h, shard, n_shards, band_begin, n_bands)
                assert rec[0] == 0
                secondary, shades = secondary + rec[1], shades + rec[2]
                rows = np.zeros(h, bool)
                for band in _shard_bands(h, shard, n_shards)[band_begin:band_begin + n_bands]:
                    rows[band * BAND_ROWS:(band + 1) * BAND_ROWS] = True
                part = (label, shard, band_begin, n_bands)
                assert _same_bits(frame[rows], want[rows]).all(), part
                assert (frame[~rows].view(np.uint32) == UNWRITTEN).all(), part
                assert (whole[rows].view(np.uint32) == UNWRITTEN).all(), part  # the parts do not overlap ...
                whole[rows] = frame[rows]
            assert _same_bits(whole, want).all(), label  # ... and cover the frame
            assert (secondary, shades) == (st.secondary_rays, st.shades), label
    finally:
        device.rtc_scene_destroy(scene)


def test_overflowing_wavefront_pool_stays_in_bounds(emu_color, host, oracle):
    """A chunk whose rays do not fit the pool is rendered again by render_stream, but first its own kernels must stay
    inside the pool: every level keeps only the rays that were written (base + count <= capacity), the overflow record
    is non-zero exactly when the pool holds fewer than the chunk's primary plus secondary rays, and a pool of exactly
    that many renders the oracle's frame.  Under AddressSanitizer (test_device_code_under_address_sanitizer) the
    pool's arrays end in red zones, so a ray or node read or written past the end aborts the run."""
    device, _ = emu_color
    kw = dict(width=64, height=40)
    cam, world = tight_glass_die(host, **kw)
    ocam, oworld = tight_glass_die(oracle, **kw)
    depth = 5
    want = np.asarray(ocam.render(oworld, depth).data, np.float32)
    st = ocam.last_stats
    rays = st.primary_rays + st.secondary_rays
    h, w = want.shape[:2]
    chunk_px = len(_shard_bands(h, 0, 1)) * BAND_ROWS * ((w + 7) // 8 * 8)
    assert rays > 6 * chunk_px  # the product's first pool (kWaveRaysPerPixel = 6) overflows on this frame
    scene = host.export_scene(cam, world)
    try:
        for capacity in (rays, rays - 1, 6 * chunk_px, st.primary_rays - 1, 5):
            frame, base, count, (overflow, _, _) = _wave_chunk(emu_color, scene, w, h, depth, capacity)
            assert (base + count <= capacity).all(), (capacity, base[:depth + 2], count[:depth + 2])
            assert (base[1:depth + 2] == base[:depth + 1] + count[:depth + 1]).all(), (capacity, base, count)
            assert (overflow == 0) == (capacity >= rays), (capacity, overflow)
            assert count.sum() == min(capacity, rays), (capacity, count)
            if capacity >= rays:
                assert _same_bits(frame, want).all()
    finally:
        device.rtc_scene_destroy(scene)


def test_device_code_under_address_sanitizer():
    """compute-sanitizer is not available on the GPU pool, so the memcheck pass runs here: this module's tests again in
    a child process whose harness is built with -fsanitize=address,undefined (libasan preloaded into python).  The
    shared-memory block is a global array with red zones, the per-thread stacks are stack arrays: an out-of-bounds
    index in the table / samples / plane-cell / origin-cache carving, the bounce stack, the BVH stack or the CSG hit
    buffer aborts the child."""
    import sys

    if os.environ.get("RTC_EMU_SANITIZE"):
        pytest.skip("already inside the sanitized run")
    libasan = subprocess.run(["g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not libasan or not os.path.exists(libasan):
        pytest.skip("no libasan")
    env = dict(os.environ, RTC_EMU_SANITIZE="1", LD_PRELOAD=libasan, ASAN_OPTIONS="detect_leaks=0:abort_on_error=1",
               UBSAN_OPTIONS="print_stacktrace=1:halt_on_error=1")
    proc = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-p", "no:cacheprovider"],
                          cwd=ROOT, env=env, capture_output=True, text=True)
    tail = (proc.stdout + proc.stderr)[-3000:]
    assert proc.returncode == 0, tail
    assert "passed" in proc.stdout and "AddressSanitizer" not in tail and "runtime error" not in tail, tail
