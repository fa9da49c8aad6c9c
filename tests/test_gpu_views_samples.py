"""Anti-aliased batches of views (rtc_render_views_samples, rtc_render_views_samples_ppm) on the GPU: view v of a batch is bit
for bit rtc_render_samples of a scene committed with that camera, in f32 and in 8 bits, on every kernel path a batch can
take and in each FP build, and n = 1 is rtc_render_views' batch; each view's text is the host writer's text of its 8-bit
plane.  Also the oracle at small sizes, c3 at full size, chunks and destinations with the documented launch counts, the
reach rule, argument checks on a committed scene, the isolation of rtc_render's state, the wavefront option, the stats, the
one-shot forms and two devices when present.  Run on the B200 box: `pytest tests -m gpu`."""
import ctypes as C

import numpy as np
import pytest

import ray_tracer_challenge_b200 as rt
from bench import WORKLOADS
from ray_tracer_challenge_b200 import scenes
from tests.test_gpu_samples import _scale_u8
from tests.test_gpu_views import SCENES, _planned_launches, _views
from tests.test_gpu_views_ppm import _pinned
from tests.test_kernels_on_host import _orbit
from tests.test_samples_on_host import box_filter

pytestmark = pytest.mark.gpu

RTC_OPT_WAVEFRONT = 8


@pytest.fixture(scope="module")
def gpu():
    return rt.new_session()


def _single(cam, world, n, fma, depth=5):
    """rtc_render_samples of the scene committed with `cam`"""
    p = cam.prepare(world)
    try:
        c = p.render_samples(n, depth, fma=fma)
        return c.data.copy(), c.to_u8().copy()
    finally:
        p.release()


def _batch(p, views, n, **kw):
    got = p.render_views_samples(views, n, 5, **kw)
    rgb = np.stack([c.data for c in got]) if kw.get("want_rgb", True) else None
    u8 = np.stack([c.to_u8() for c in got]) if kw.get("want_u8", True) else None
    return rgb, u8


def _texts(gpu, u8):
    """The host writer's text of each view's 8-bit plane"""
    return [rt.CanvasU8(v.shape[1], v.shape[0], np.ascontiguousarray(v), gpu).to_ppm() for v in u8]


@pytest.mark.parametrize("name", list(SCENES))
def test_views_equal_single_view_samples(gpu, name):
    """Every kernel path, each FP build the scene lists, n = 1, 2, 3: view v is rtc_render_samples of the scene committed with
    camera v; n = 1 is rtc_render_views' batch."""
    build, kw, _, fmas = SCENES[name]
    cam, world = build(gpu, **kw)
    views = _views(gpu, cam)
    far = views[gpu.farthest_camera(views)]
    w, h = cam.width_pixels, cam.height_pixels
    p = far.prepare(world)
    try:
        for fma in fmas:
            for n in (1, 2, 3):
                rgb, u8 = _batch(p, views, n, fma=fma)
                assert p.last_stats.primary_rays == n * n * len(views) * (w - 1) * (h - 1), (name, n)
                for i, v in enumerate(views):
                    srgb, su8 = _single(v, world, n, fma)
                    assert np.array_equal(rgb[i].view(np.uint32), srgb.view(np.uint32)), (name, fma, n, i)
                    assert np.array_equal(u8[i], su8), (name, fma, n, i)
                if n == 1:
                    got = p.render_views(views, 5, fma=fma)
                    assert np.array_equal(rgb.view(np.uint32), np.stack([c.data for c in got]).view(np.uint32)), (name, fma)
                    assert np.array_equal(u8, np.stack([c.to_u8() for c in got])), (name, fma)
    finally:
        p.release()


def test_views_samples_match_the_oracle(gpu, oracle):
    """Small batches against the box filter of the oracle's render of each view's camera at n times the size (strict
    build): bit for bit on the soft-shadow scene with generated jitter, within the parity bounds elsewhere."""
    from tests.parity import assert_parity, compare_frames

    cases = ((scenes.soft_shadows, dict(width=64, height=32, u_steps=4, v_steps=4, jitter=None, seed=3), 3, True),
             (scenes.reflect_refract, dict(width=80, height=40), 2, False),
             (scenes.dragon_element, dict(width=64, height=36, n_u=24, n_v=12), 2, False))
    for build, kw, n, exact in cases:
        w, h = kw["width"], kw["height"]
        cam, world = build(gpu, **kw)
        poses = _orbit(gpu, cam, 3, 60.0)
        views = [gpu.Camera(w, h, fov, gpu.view_transform(e, at, (0, 1, 0))) for e, at, fov in poses]
        far = views[gpu.farthest_camera(views)]
        p = far.prepare(world)
        try:
            rgb, u8 = _batch(p, views, n)
        finally:
            p.release()
        _, oworld = build(oracle, **dict(kw, width=n * w, height=n * h))
        for i, (e, at, fov) in enumerate(poses):
            ocam = oracle.Camera(n * w, n * h, fov, oracle.view_transform(e, at, (0, 1, 0)))
            want = box_filter(ocam.render(oworld, 5).data, w, h, n)
            assert_parity(compare_frames(u8[i], _scale_u8(want), rgb[i], want), label=f"{build.__name__} n={n} view {i}")
            if exact:
                assert np.array_equal(rgb[i].view(np.uint32), want.view(np.uint32)), (build.__name__, i)
                assert np.array_equal(u8[i], _scale_u8(want)), (build.__name__, i)


def test_full_size_c3_three_views(gpu):
    """c3 (3840x2160) at n = 2, a batch of three views: each view is rtc_render_samples of its own committed scene."""
    builder, kw, depth, _ = WORKLOADS["c3"]
    cam, world = getattr(scenes, builder)(gpu, **kw)
    views = scenes.orbit_cameras(gpu, cam, 3, degrees=30.0)
    p = cam.prepare(world)
    try:
        rgb, u8 = _batch(p, views, 2)
    finally:
        p.release()
    for i, v in enumerate(views):
        srgb, su8 = _single(v, world, 2, False)
        assert np.array_equal(rgb[i].view(np.uint32), srgb.view(np.uint32)), i
        assert np.array_equal(u8[i], su8), i


def test_chunks_and_copies(gpu, monkeypatch):
    """960x540 x 6 views at n = 2: pageable (staged), pinned, one plane at a time and NULL / NULL give the same frames, in one
    chunk and through a small arena, with rtc_render_views' launch plan."""
    cam, world = scenes.soft_shadows(gpu, width=960, height=540, u_steps=4, v_steps=4)
    views = _views(gpu, cam)
    n, h, w = len(views), cam.height_pixels, cam.width_pixels
    p = cam.prepare(world)
    try:
        rgb, u8 = _batch(p, views, 2)
        assert p.last_stats.launches == _planned_launches(w, h, n, 15) == 42
        r2, _ = _batch(p, views, 2, want_u8=False)
        _, u2 = _batch(p, views, 2, want_rgb=False)
        assert np.array_equal(r2, rgb) and np.array_equal(u2, u8)
        lib = rt.device_library()
        lib.rtc_host_alloc.restype = C.c_void_p
        lib.rtc_host_free.argtypes = [C.c_void_p]
        nbytes = n * h * w * 3
        ptr_rgb, ptr_u8 = lib.rtc_host_alloc(C.c_size_t(nbytes * 4)), lib.rtc_host_alloc(C.c_size_t(nbytes))
        try:
            pin_rgb = np.ctypeslib.as_array((C.c_float * nbytes).from_address(ptr_rgb)).reshape(n, h, w, 3)
            pin_u8 = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(ptr_u8)).reshape(n, h, w, 3)
            pin_rgb[:] = -1.0
            pin_u8[:] = 7
            p.render_views_samples(views, 2, 5, out_rgb=pin_rgb, out_u8=pin_u8)
            assert np.array_equal(pin_rgb, rgb) and np.array_equal(pin_u8, u8)
        finally:
            lib.rtc_host_free(C.c_void_p(ptr_rgb))
            lib.rtc_host_free(C.c_void_p(ptr_u8))
        p.render_views_samples(views, 2, 5, want_rgb=False, want_u8=False)
        assert p.last_stats.launches == 1 and p.last_stats.primary_rays == 4 * n * (w - 1) * (h - 1)
        for per_chunk in (2, 1):
            monkeypatch.setenv("RTC_VIEW_ARENA_BYTES", str(per_chunk * h * w * 15))
            r3, u3 = _batch(p, views, 2)
            assert np.array_equal(r3, rgb) and np.array_equal(u3, u8), per_chunk
            assert p.last_stats.launches == _planned_launches(w, h, n, 15, chunk=per_chunk) == 42
            p.render_views_samples(views, 2, 5, want_rgb=False, want_u8=False)
            assert p.last_stats.launches == (n + per_chunk - 1) // per_chunk
        monkeypatch.delenv("RTC_VIEW_ARENA_BYTES")
    finally:
        p.release()
    for i in (0, 5):
        srgb, su8 = _single(views[i], world, 2, False)
        assert np.array_equal(rgb[i], srgb) and np.array_equal(u8[i], su8), i


def test_staged_runs_of_whole_views(gpu, monkeypatch):
    """36 views of 320x200 at n = 2 into pageable memory: 18 runs of two whole views, staged; chunks of five: 22 runs."""
    cam, world = scenes.soft_shadows(gpu, width=320, height=200, u_steps=4, v_steps=4)
    views = scenes.orbit_cameras(gpu, cam, 36)
    n, h, w = len(views), cam.height_pixels, cam.width_pixels
    p = cam.prepare(world)
    try:
        rgb, u8 = _batch(p, views, 2)
        assert p.last_stats.launches == _planned_launches(w, h, n, 15) == 18
        monkeypatch.setenv("RTC_VIEW_ARENA_BYTES", str(5 * h * w * 15))
        r2, u2 = _batch(p, views, 2)
        assert p.last_stats.launches == _planned_launches(w, h, n, 15, chunk=5) == 22
        assert np.array_equal(r2, rgb) and np.array_equal(u2, u8)
        monkeypatch.delenv("RTC_VIEW_ARENA_BYTES")
    finally:
        p.release()
    for i in (0, 17, 35):
        srgb, su8 = _single(views[i], world, 2, False)
        assert np.array_equal(rgb[i], srgb) and np.array_equal(u8[i], su8), i


@pytest.mark.parametrize("name", ["lean_table", "small_converging", "tree_dragon", "tree_stream", "sweep_csg_die"])
def test_texts_are_the_host_writer_texts_of_the_planes(gpu, name):
    build, kw, _, _ = SCENES[name]
    cam, world = build(gpu, **kw)
    views = _views(gpu, cam)
    far = views[gpu.farthest_camera(views)]
    p = far.prepare(world)
    try:
        for n in (1, 2):
            _, u8 = _batch(p, views, n, want_rgb=False)
            texts = p.render_views_samples_ppm(views, n, 5)
            st = p.last_stats
            assert st.primary_rays == n * n * len(views) * (cam.width_pixels - 1) * (cam.height_pixels - 1)
            assert texts == _texts(gpu, u8), (name, n)
    finally:
        p.release()


def test_texts_through_chunks_and_destinations(gpu, monkeypatch):
    """960x540 x 6 views at n = 2: the texts into pageable memory (staged), through chunks of two and one views, and into
    pinned memory are the host writer's texts; render_samples_ppm is render_samples(...).to_ppm()."""
    cam, world = scenes.soft_shadows(gpu, width=960, height=540, u_steps=4, v_steps=4)
    views = _views(gpu, cam)
    n, h, w = len(views), cam.height_pixels, cam.width_pixels
    p = cam.prepare(world)
    try:
        _, u8 = _batch(p, views, 2, want_rgb=False)
        want = _texts(gpu, u8)
        assert p.render_views_samples_ppm(views, 2, 5) == want
        for per_chunk in (2, 1):
            monkeypatch.setenv("RTC_VIEW_ARENA_BYTES", str(per_chunk * h * w * 15))
            assert p.render_views_samples_ppm(views, 2, 5) == want, per_chunk
            assert p.last_stats.launches == (n + per_chunk - 1) // per_chunk
        monkeypatch.delenv("RTC_VIEW_ARENA_BYTES")
        bound = gpu.lib.rtc_ppm_bound(w, h)
        lib, ptr, buf = _pinned(n * bound)
        try:
            assert p.render_views_samples_ppm(views, 2, 5, out=buf) == want
        finally:
            lib.rtc_host_free(C.c_void_p(ptr))
        for k in (1, 3):
            assert p.render_samples_ppm(k, 5) == p.render_samples(k, 5).to_ppm(), k
    finally:
        p.release()


def test_reach_rule_and_bad_arguments_on_a_committed_scene(gpu):
    cam, world = scenes.dragon_element(gpu, width=160, height=90, n_u=24, n_v=12)
    far = gpu.Camera(cam.width_pixels, cam.height_pixels, cam.field_of_view,
                     gpu.view_transform((0.0, 2.5, -400.0), (0, 1, 0), (0, 1, 0)))
    p = cam.prepare(world)
    try:
        with pytest.raises(rt.RtcError, match="reach"):
            p.render_views_samples([cam, far], 2, 5)
        with pytest.raises(rt.RtcError, match="reach"):
            p.render_views_samples_ppm([cam, far], 2, 5)
        for call in (p.render_views_samples, p.render_views_samples_ppm):
            for n in (0, 17):
                with pytest.raises(rt.RtcError, match="samples_per_axis"):
                    call([cam], n, 5)
            with pytest.raises(rt.RtcError, match="reflection_recursion_depth"):
                call([cam], 2, 30)
    finally:
        p.release()
    q = far.prepare(world)  # committed with the far camera: the batch renders
    try:
        rgb, u8 = _batch(q, [cam, far], 2)
    finally:
        q.release()
    for i, v in enumerate((cam, far)):
        srgb, su8 = _single(v, world, 2, False)
        assert np.array_equal(rgb[i], srgb) and np.array_equal(u8[i], su8), i


def test_a_batch_leaves_render_state_alone(gpu, monkeypatch, tmp_path):
    """As rtc_render_views' test: the frames of rtc_render and the render that learns the tile order are the same with
    anti-aliased batches (frames and texts) in between."""
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
                b.render_views_samples(views, 2, 5)
                st = b.last_stats
                assert st.launches == _planned_launches(320, 180, len(views), 15)
                assert st.primary_rays == 4 * len(views) * 319 * 179
                b.render_views_samples_ppm(views, 2, 5)
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
        want = _batch(p, views, 2)
        p.set_option(RTC_OPT_WAVEFRONT, 1)
        got = _batch(p, views, 2)
        assert p.last_stats.launches == 1  # one persistent streaming launch for the whole batch
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    finally:
        p.release()


def test_one_shot_forms_equal_the_prepared_forms(gpu):
    cam, world = scenes.reflect_refract(gpu, width=200, height=100)
    views = _views(gpu, cam)
    far = views[gpu.farthest_camera(views)]
    p = far.prepare(world)
    try:
        rgb, u8 = _batch(p, views, 2)
        texts = p.render_views_samples_ppm(views, 2, 5)
    finally:
        p.release()
    got = gpu.render_views_samples(world, views, 2, 5)
    assert np.array_equal(np.stack([c.data for c in got]), rgb) and np.array_equal(np.stack([c.to_u8() for c in got]), u8)
    assert gpu.last_views_stats.primary_rays == 4 * len(views) * 199 * 99
    assert gpu.render_views_samples_ppm(world, views, 2, 5) == texts
    assert cam.render_b200_samples_ppm(world, 2, 5) == cam.render_b200_samples(world, 2, 5).to_ppm()


def test_two_devices_render_the_same_batch(gpu):
    if rt.device_library().rtc_device_count() < 2:
        pytest.skip("needs two devices")
    cam, world = scenes.dragon_element(gpu, width=320, height=180, n_u=24, n_v=12)
    views = _views(gpu, cam)
    far = views[gpu.farthest_camera(views)]
    out = []
    for n_dev in (1, 2):
        gpu.set_render_options(n_devices=n_dev)
        p = far.prepare(world)
        try:
            out.append(_batch(p, views, 2) + (p.render_views_samples_ppm(views, 2, 5),))
        finally:
            p.release()
    gpu.set_render_options(n_devices=1)
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1]) and out[0][2] == out[1][2]
