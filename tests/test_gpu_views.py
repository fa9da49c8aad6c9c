"""Batches of camera views (rtc_render_views) on the GPU: every view of a batch is bit for bit the frame of a scene committed
with that camera, on every kernel path a batch can take, through every copy path; the reach rule, the isolation of
rtc_render's state, the stats and several devices.  Run on the B200 box: `pytest tests -m gpu`."""
import ctypes as C
import math

import numpy as np
import pytest

import ray_tracer_challenge_b200 as rt
from ray_tracer_challenge_b200 import scenes

pytestmark = pytest.mark.gpu

RTC_OPT_WAVEFRONT = 8

# name -> (builder, kwargs, inspect key that must hold, FMA settings to run)
SCENES = {
    "lean_table": (scenes.soft_shadows, dict(width=160, height=64, u_steps=4, v_steps=4), ("lean", 1), (False, True)),
    "lean_drawn": (scenes.soft_shadows, dict(width=160, height=64, u_steps=4, v_steps=4, jitter=None, seed=3), ("lean", 1), (False,)),
    "small_patterns": (scenes.first_patterns, dict(width=100, height=50), ("small_n", None), (False,)),
    "small_textured": (scenes.textured, dict(width=160, height=100), ("small_n", None), (False,)),
    "small_converging": (scenes.reflect_refract, dict(width=200, height=100), ("converge", 1), (False, True)),
    "tree_dragon": (scenes.dragon_element, dict(width=160, height=90, n_u=24, n_v=12), ("n_bvh_nodes", None), (False,)),
    "tree_stream": (scenes.stress, dict(width=192, height=108, n_spheres=3000, n_each=16, n_csg=4, extent=20.0), ("converge", 1),
                    (False,)),
    "sweep_csg_die": (scenes.csg_die, dict(width=160, height=100), (None, None), (False,)),
}


@pytest.fixture(scope="module")
def gpu():
    return rt.new_session()


def _views(gpu, cam):
    """About six views: four orbit positions, one with another field of view, and the committed camera itself."""
    orbit = scenes.orbit_cameras(gpu, cam, 4, degrees=60.0)
    wide = scenes.orbit_cameras(gpu, cam, 1, field_of_view=cam.field_of_view * 0.8)
    return orbit[1:] + [orbit[0]] + wide + [cam]


def _single(gpu, cam, world, fma, depth=5):
    p = cam.prepare(world)
    try:
        c = p.render(depth, fma=fma)
        return c.data.copy(), c.to_u8().copy()
    finally:
        p.release()


def _check_scene(gpu, name):
    build, kw, (key, val), fmas = SCENES[name]
    cam, world = build(gpu, **kw)
    info = gpu.inspect(cam, world)
    if key == "small_n":
        assert info["small_n"] > 0
    elif key == "n_bvh_nodes":
        assert info["n_bvh_nodes"] > 0
    elif key:
        assert info[key] == val, info
    views = _views(gpu, cam)
    # a tree scene takes views only within the committed reach: commit with the farthest camera
    far = views[gpu.farthest_camera(views)]
    p = far.prepare(world)
    try:
        for fma in fmas:
            got = p.render_views(views, 5, fma=fma)
            st = p.last_stats
            w, h = cam.width_pixels, cam.height_pixels
            assert st.primary_rays == len(views) * (w - 1) * (h - 1)
            for i, v in enumerate(views):
                rgb, u8 = _single(gpu, v, world, fma)
                assert np.array_equal(got[i].data.view(np.uint32), rgb.view(np.uint32)), (name, fma, i)
                assert np.array_equal(got[i].to_u8(), u8), (name, fma, i)
    finally:
        p.release()


@pytest.mark.parametrize("name", list(SCENES))
def test_views_equal_single_view_renders(gpu, name):
    _check_scene(gpu, name)


def test_views_match_the_oracle(gpu, oracle):
    from tests.parity import assert_parity, compare_frames

    # (scene, field of view, look-at point, three eyes): the scenes' own cameras and two turns about the look-at point
    cases = ((scenes.soft_shadows, dict(width=160, height=64, u_steps=4, v_steps=4), math.pi / 4.0, (0, 0.5, 0),
              ((-3, 1, 2.5), (-1.5, 1, 3.6), (2.0, 1, 3.3))),
             (scenes.first_patterns, dict(width=100, height=50), math.pi / 3.0, (0, 1, 0), ((0, 1.5, -5), (-2.5, 1.5, -4.3), (3.0, 1.5, -4.0))))
    for build, kw, fov, to, eyes in cases:
        cam, world = build(gpu, **kw)
        w, h = cam.width_pixels, cam.height_pixels
        views = [gpu.Camera(w, h, fov, gpu.view_transform(e, to, (0, 1, 0))) for e in eyes]
        p = cam.prepare(world)
        got = p.render_views(views, 5)
        p.release()
        _, oworld = build(oracle, **kw)
        for i, e in enumerate(eyes):
            want = oracle.Camera(w, h, fov, oracle.view_transform(e, to, (0, 1, 0))).render(oworld, 5)
            assert_parity(compare_frames(got[i].to_u8(), want.to_u8(), got[i].data, want.data), label=f"{build.__name__} view {i}")


def _planned_launches(w, h, n, bytes_per_px, chunk=None, slices=24, stream=False):
    """The launch plan rtc_render_views documents, for one device: one launch per chunk of views when the frames stay on
    the device (or the scene streams); copied to host memory, rtc_render's slice rule over the whole batch (one slice per
    MiB, at most RTC_OPT_RENDER_SLICES) as runs of whole views, or each view cut by bands when a view exceeds a slice."""
    chunk = chunk or n
    n_chunks = (n + chunk - 1) // chunk
    if bytes_per_px == 0 or stream:
        return n_chunks
    nb = (h + 7) // 8
    view_copy = w * 8 * nb * bytes_per_px
    want = max(1, min(slices, (view_copy * n) >> 20))
    if want > n:
        return n * max(1, min(slices, nb, view_copy >> 20))
    per_run = (n + want - 1) // want
    return sum((min(n, c0 + chunk) - c0 + per_run - 1) // per_run for c0 in range(0, n, chunk))


def _batch(p, views, **kw):
    got = p.render_views(views, 5, **kw)
    rgb = np.stack([c.data for c in got]) if kw.get("want_rgb", True) else None
    u8 = np.stack([c.to_u8() for c in got]) if kw.get("want_u8", True) else None
    return rgb, u8


def test_copy_paths_give_the_same_frames(gpu, monkeypatch):
    # 960x540 x 6 views: a batch of several MiB, cut into runs of views; the 8-bit plane alone is staged when pageable
    cam, world = scenes.soft_shadows(gpu, width=960, height=540, u_steps=4, v_steps=4)
    views = _views(gpu, cam)
    n, h, w = len(views), cam.height_pixels, cam.width_pixels
    p = cam.prepare(world)
    try:
        rgb, u8 = _batch(p, views)
        assert p.last_stats.launches == _planned_launches(w, h, n, 15) == 42  # each view cut into 7 band slices
        r2, _ = _batch(p, views, want_u8=False)
        _, u2 = _batch(p, views, want_rgb=False)
        assert np.array_equal(r2, rgb) and np.array_equal(u2, u8)
        lib = rt.device_library()
        lib.rtc_host_alloc.restype = C.c_void_p
        lib.rtc_host_free.argtypes = [C.c_void_p]
        nbytes = n * h * w * 3
        ptr_rgb, ptr_u8 = lib.rtc_host_alloc(C.c_size_t(nbytes * 4)), lib.rtc_host_alloc(C.c_size_t(nbytes))
        try:
            pin_rgb = np.ctypeslib.as_array((C.c_float * (nbytes)).from_address(ptr_rgb)).reshape(n, h, w, 3)
            pin_u8 = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(ptr_u8)).reshape(n, h, w, 3)
            pin_rgb[:] = -1.0
            pin_u8[:] = 7
            p.render_views(views, 5, out_rgb=pin_rgb, out_u8=pin_u8)
            assert np.array_equal(pin_rgb, rgb) and np.array_equal(pin_u8, u8)
        finally:
            lib.rtc_host_free(C.c_void_p(ptr_rgb))
            lib.rtc_host_free(C.c_void_p(ptr_u8))
        # several chunks through a small arena: two views' frames at a time, then one
        for per_chunk in (2, 1):
            monkeypatch.setenv("RTC_VIEW_ARENA_BYTES", str(per_chunk * h * w * 15))
            r3, u3 = _batch(p, views)
            assert np.array_equal(r3, rgb) and np.array_equal(u3, u8), per_chunk
            assert p.last_stats.launches == _planned_launches(w, h, n, 15, chunk=per_chunk) == 42
            assert p.last_stats.primary_rays == n * (w - 1) * (h - 1)
            p.render_views(views, 5, want_rgb=False, want_u8=False)  # left on the device: one launch per chunk
            assert p.last_stats.launches == _planned_launches(w, h, n, 0, chunk=per_chunk) == (n + per_chunk - 1) // per_chunk
        monkeypatch.delenv("RTC_VIEW_ARENA_BYTES")
        # a one-view batch of the committed camera is rtc_render's frame
        one = p.render_views([cam], 5)[0]
        ref = p.render(5)
        assert np.array_equal(one.data, ref.data) and np.array_equal(one.to_u8(), ref.to_u8())
    finally:
        p.release()


def test_reach_rule(gpu):
    cam, world = scenes.dragon_element(gpu, width=160, height=90, n_u=24, n_v=12)
    p = cam.prepare(world)
    far = gpu.Camera(cam.width_pixels, cam.height_pixels, cam.field_of_view,
                     gpu.view_transform((0.0, 2.5, -400.0), (0, 1, 0), (0, 1, 0)))
    try:
        with pytest.raises(rt.RtcError, match="reach"):
            p.render_views([cam, far], 5)
    finally:
        p.release()
    q = far.prepare(world)  # committed with the far camera: the batch renders, each view as its single-view frame
    try:
        got = q.render_views([cam, far], 5)
        for i, v in enumerate((cam, far)):
            rgb, u8 = _single(gpu, v, world, False)
            assert np.array_equal(got[i].data, rgb) and np.array_equal(got[i].to_u8(), u8)
    finally:
        q.release()
    # a small scene takes any finite view
    scam, sworld = scenes.soft_shadows(gpu, width=160, height=64, u_steps=4, v_steps=4)
    sfar = gpu.Camera(160, 64, scam.field_of_view, gpu.view_transform((0.0, 1.0, -1.0e4), (0, 1, 0), (0, 1, 0)))
    p = scam.prepare(sworld)
    try:
        got = p.render_views([sfar], 5)[0]
        rgb, u8 = _single(gpu, sfar, sworld, False)
        assert np.array_equal(got.data, rgb) and np.array_equal(got.to_u8(), u8)
    finally:
        p.release()


def test_staged_runs_of_whole_views(gpu, monkeypatch):
    """A turntable of small views into pageable memory: 36 views of 320x200 (0.92 MiB copied per view, 33 MiB in all) are
    rendered as 18 runs of two whole views, each run one launch, staged through pinned frames and copied on by the
    host's threads.  Pinned and pageable destinations, one chunk and several, and single-view renders agree."""
    cam, world = scenes.soft_shadows(gpu, width=320, height=200, u_steps=4, v_steps=4)
    views = scenes.orbit_cameras(gpu, cam, 36)
    n, h, w = len(views), cam.height_pixels, cam.width_pixels
    p = cam.prepare(world)
    try:
        rgb, u8 = _batch(p, views)  # numpy's own (pageable) arrays
        assert p.last_stats.launches == _planned_launches(w, h, n, 15) == 18
        assert p.last_stats.primary_rays == n * (w - 1) * (h - 1)
        lib = rt.device_library()
        lib.rtc_host_alloc.restype = C.c_void_p
        lib.rtc_host_free.argtypes = [C.c_void_p]
        nbytes = n * h * w * 3
        ptr_rgb, ptr_u8 = lib.rtc_host_alloc(C.c_size_t(nbytes * 4)), lib.rtc_host_alloc(C.c_size_t(nbytes))
        try:
            pin_rgb = np.ctypeslib.as_array((C.c_float * nbytes).from_address(ptr_rgb)).reshape(n, h, w, 3)
            pin_u8 = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(ptr_u8)).reshape(n, h, w, 3)
            p.render_views(views, 5, out_rgb=pin_rgb, out_u8=pin_u8)
            assert np.array_equal(pin_rgb, rgb) and np.array_equal(pin_u8, u8)
        finally:
            lib.rtc_host_free(C.c_void_p(ptr_rgb))
            lib.rtc_host_free(C.c_void_p(ptr_u8))
        # chunks of five views: runs of two, the last run of a chunk holding one
        monkeypatch.setenv("RTC_VIEW_ARENA_BYTES", str(5 * h * w * 15))
        r2, u2 = _batch(p, views)
        assert p.last_stats.launches == _planned_launches(w, h, n, 15, chunk=5) == 22
        assert np.array_equal(r2, rgb) and np.array_equal(u2, u8)
        monkeypatch.delenv("RTC_VIEW_ARENA_BYTES")
    finally:
        p.release()
    for i in (0, 7, 20, 35):
        srgb, su8 = _single(gpu, views[i], world, False)
        assert np.array_equal(rgb[i], srgb) and np.array_equal(u8[i], su8), i


def test_a_batch_leaves_render_state_alone(gpu, monkeypatch, tmp_path):
    """Two prepared scenes render the same sequence of frames, one with batches in between.  The frames agree, and the
    render that learns the adaptive tile order (the second one of a scene: it writes RTC_DUMP_TILE_COST) is the same call
    in both — a batch that counted as a render, or touched the learnt order's state, would move it."""
    cam, world = scenes.dragon_element(gpu, width=320, height=180, n_u=24, n_v=12)
    views = _views(gpu, cam)[:4]
    dump = tmp_path / "tile_cost.txt"
    monkeypatch.setenv("RTC_DUMP_TILE_COST", str(dump))

    def learnt():
        if dump.exists():
            dump.unlink()
            return True
        return False

    a, b = cam.prepare(world), cam.prepare(world)
    try:
        frames_a, frames_b, learn_a, learn_b = [], [], [], []
        for k in range(6):
            frames_a.append(a.render(5).to_u8().copy())
            learn_a.append(learnt())
            la = a.last_stats.launches
            if k % 2 == 0:
                b.render_views(views, 5)
                st = b.last_stats
                assert st.launches == _planned_launches(320, 180, len(views), 15) and st.primary_rays == len(views) * 319 * 179
                assert not learnt()
            frames_b.append(b.render(5).to_u8().copy())
            learn_b.append(learnt())
            assert b.last_stats.launches == la
        assert learn_a == learn_b == [k == 1 for k in range(6)], (learn_a, learn_b)
        for fa, fb in zip(frames_a, frames_b):
            assert np.array_equal(fa, fb)
    finally:
        a.release(), b.release()


def test_wavefront_option_does_not_change_a_batch(gpu):
    cam, world = scenes.stress(gpu, width=192, height=108, n_spheres=3000, n_each=16, n_csg=4, extent=20.0)
    views = _views(gpu, cam)[:3]
    far = views[gpu.farthest_camera(views)]
    p = far.prepare(world)
    try:
        p.set_option(RTC_OPT_WAVEFRONT, 1)
        got = p.render_views(views, 5)
        assert p.last_stats.launches == 1  # one persistent streaming launch for the whole batch
        for i, v in enumerate(views):
            rgb, u8 = _single(gpu, v, world, False)
            assert np.array_equal(got[i].data, rgb) and np.array_equal(got[i].to_u8(), u8)
    finally:
        p.release()


def test_one_shot_batch(gpu):
    cam, world = scenes.reflect_refract(gpu, width=200, height=100)
    views = _views(gpu, cam)
    got = gpu.render_views(world, views, 5)
    for i, v in enumerate(views):
        rgb, u8 = _single(gpu, v, world, False)
        assert np.array_equal(got[i].data, rgb) and np.array_equal(got[i].to_u8(), u8)


def test_two_devices_render_the_same_batch(gpu):
    if rt.device_library().rtc_device_count() < 2:
        pytest.skip("needs two devices")
    cam, world = scenes.dragon_element(gpu, width=320, height=180, n_u=24, n_v=12)
    views = _views(gpu, cam)
    far = views[gpu.farthest_camera(views)]
    out = []
    for n in (1, 2):
        gpu.set_render_options(n_devices=n)
        p = far.prepare(world)
        try:
            out.append(_batch(p, views))
        finally:
            p.release()
    gpu.set_render_options(n_devices=1)
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])


def test_bad_depth_is_refused_on_a_committed_scene(gpu):
    cam, world = scenes.soft_shadows(gpu, width=64, height=32, u_steps=2, v_steps=2)
    p = cam.prepare(world)
    try:
        with pytest.raises(rt.RtcError, match="reflection_recursion_depth"):
            p.render_views([cam], 30)
    finally:
        p.release()
