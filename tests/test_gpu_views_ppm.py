"""rtc_render_views_ppm on the GPU: each view's text of a batch is byte for byte rtc_render_ppm's text of a scene committed
with that camera, and the host writer's text (CanvasU8.to_ppm) of rtc_render_views' 8-bit plane, on every kernel path a
batch can take; the oracle; chunks, pinned and pageable (staged) destinations, a capacity exactly at the bound; two devices
when present; the reach rule, the isolation of rtc_render's state and the one-shot form.  Run on the B200 box:
`pytest tests -m gpu`."""
import ctypes as C
import math

import numpy as np
import pytest

import ray_tracer_challenge_b200 as rt
from ray_tracer_challenge_b200 import scenes
from tests.test_gpu_views import SCENES, _views

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu():
    return rt.new_session()


def _bound(gpu, cam):
    return gpu.lib.rtc_ppm_bound(cam.width_pixels, cam.height_pixels)


def _plane_texts(gpu, p, views, fma=False):
    """The host writer's text of each view of rtc_render_views' 8-bit planes."""
    got = p.render_views(views, 5, want_rgb=False, fma=fma)
    return [rt.CanvasU8(c.width, c.height, c.to_u8(), gpu).to_ppm() for c in got]


def _single_ppm(cam, world, fma=False):
    p = cam.prepare(world)
    try:
        return p.render_ppm(5, fma=fma)
    finally:
        p.release()


def _pinned(nbytes):
    lib = rt.device_library()
    lib.rtc_host_alloc.restype = C.c_void_p
    lib.rtc_host_alloc.argtypes = [C.c_size_t]
    lib.rtc_host_free.argtypes = [C.c_void_p]
    ptr = lib.rtc_host_alloc(nbytes)
    assert ptr
    return lib, ptr, np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(ptr))


@pytest.mark.parametrize("name", list(SCENES))
def test_views_equal_single_view_texts(gpu, name):
    build, kw, _, fmas = SCENES[name]
    cam, world = build(gpu, **kw)
    views = _views(gpu, cam)
    far = views[gpu.farthest_camera(views)]
    w, h = cam.width_pixels, cam.height_pixels
    p = far.prepare(world)
    try:
        for fma in fmas:
            texts = p.render_views_ppm(views, 5, fma=fma)
            st = p.last_stats
            assert len(texts) == len(views)
            assert st.primary_rays == len(views) * (w - 1) * (h - 1)
            assert st.launches == 1 and st.kernel_ms > 0.0 and st.total_ms >= st.kernel_ms
            assert texts == _plane_texts(gpu, p, views, fma), (name, fma)
            for i, v in enumerate(views):
                assert texts[i] == _single_ppm(v, world, fma), (name, fma, i)
    finally:
        p.release()


def _pixels(text, w, h):
    head = f"P3\n{w} {h}\n255\n"
    assert text.startswith(head) and text.endswith("\n") and max(len(line) for line in text.splitlines()) <= 70
    return np.array(text[len(head):].split(), np.int32).astype(np.uint8).reshape(h, w, 3)


def test_views_match_the_oracle(gpu, oracle):
    from tests.parity import assert_parity, compare_frames

    # the cases of test_gpu_views.test_views_match_the_oracle: the scenes' own cameras and two turns about the look-at point
    cases = ((scenes.soft_shadows, dict(width=160, height=64, u_steps=4, v_steps=4), math.pi / 4.0, (0, 0.5, 0),
              ((-3, 1, 2.5), (-1.5, 1, 3.6), (2.0, 1, 3.3))),
             (scenes.first_patterns, dict(width=100, height=50), math.pi / 3.0, (0, 1, 0), ((0, 1.5, -5), (-2.5, 1.5, -4.3), (3.0, 1.5, -4.0))))
    for build, kw, fov, to, eyes in cases:
        cam, world = build(gpu, **kw)
        w, h = cam.width_pixels, cam.height_pixels
        views = [gpu.Camera(w, h, fov, gpu.view_transform(e, to, (0, 1, 0))) for e in eyes]
        p = cam.prepare(world)
        texts = p.render_views_ppm(views, 5)
        p.release()
        _, oworld = build(oracle, **kw)
        for i, e in enumerate(eyes):
            want = oracle.Camera(w, h, fov, oracle.view_transform(e, to, (0, 1, 0))).render(oworld, 5).to_ppm()
            got_u8, want_u8 = _pixels(texts[i], w, h), _pixels(want, w, h)
            assert_parity(compare_frames(got_u8, want_u8), label=f"{build.__name__} view {i}")
            if np.array_equal(got_u8, want_u8):
                assert texts[i] == want, (build.__name__, i)


def test_chunks_and_destinations(gpu, monkeypatch):
    """960x540 x 6 views (37 MB of text bound; several MB of text per view): one chunk and chunks of two and one views,
    into pageable memory (staged: 4 MiB or more) and into pinned and pageable memory exactly n_views * rtc_ppm_bound long."""
    cam, world = scenes.soft_shadows(gpu, width=960, height=540, u_steps=4, v_steps=4)
    views = _views(gpu, cam)
    n, h, w = len(views), cam.height_pixels, cam.width_pixels
    p = cam.prepare(world)
    try:
        texts = p.render_views_ppm(views, 5)  # a new numpy array: pageable
        assert sum(map(len, texts)) >= 4 << 20
        assert p.last_stats.launches == 1 and p.last_stats.primary_rays == n * (w - 1) * (h - 1)
        assert texts == _plane_texts(gpu, p, views)
        cap = n * _bound(gpu, cam)
        lib, ptr, pinned = _pinned(cap)
        try:
            pinned[:] = 0x7F
            assert p.render_views_ppm(views, 5, out=pinned) == texts
            total = sum(map(len, texts))
            assert np.all(pinned[total:] == 0x7F)
            for per_chunk in (2, 1):
                monkeypatch.setenv("RTC_VIEW_ARENA_BYTES", str(per_chunk * h * w * 15))
                assert p.render_views_ppm(views, 5) == texts, per_chunk
                assert p.last_stats.launches == (n + per_chunk - 1) // per_chunk
                assert p.last_stats.primary_rays == n * (w - 1) * (h - 1)
                assert p.render_views_ppm(views, 5, out=pinned) == texts, per_chunk
                assert p.last_stats.launches == (n + per_chunk - 1) // per_chunk
            monkeypatch.delenv("RTC_VIEW_ARENA_BYTES")
        finally:
            lib.rtc_host_free(C.c_void_p(ptr))
        # a pageable destination of exactly the bound, caller-supplied
        exact = np.zeros(cap, np.uint8)
        assert p.render_views_ppm(views, 5, out=exact) == texts
    finally:
        p.release()


def test_a_long_turntable_into_pageable_memory(gpu, monkeypatch):
    """36 views of 320x200, staged piece by piece, in one chunk and in chunks of five; equal to the 8-bit planes' texts."""
    cam, world = scenes.soft_shadows(gpu, width=320, height=200, u_steps=4, v_steps=4)
    views = scenes.orbit_cameras(gpu, cam, 36)
    h, w = cam.height_pixels, cam.width_pixels
    p = cam.prepare(world)
    try:
        want = _plane_texts(gpu, p, views)
        assert p.render_views_ppm(views, 5) == want
        monkeypatch.setenv("RTC_VIEW_ARENA_BYTES", str(5 * h * w * 15))
        assert p.render_views_ppm(views, 5) == want
        assert p.last_stats.launches == 8
    finally:
        p.release()


def test_reach_rule(gpu):
    cam, world = scenes.dragon_element(gpu, width=160, height=90, n_u=24, n_v=12)
    far = gpu.Camera(cam.width_pixels, cam.height_pixels, cam.field_of_view,
                     gpu.view_transform((0.0, 2.5, -400.0), (0, 1, 0), (0, 1, 0)))
    p = cam.prepare(world)
    try:
        with pytest.raises(rt.RtcError, match="reach"):
            p.render_views_ppm([cam, far], 5)
    finally:
        p.release()
    q = far.prepare(world)
    try:
        texts = q.render_views_ppm([cam, far], 5)
        assert texts == [_single_ppm(cam, world), _single_ppm(far, world)]
    finally:
        q.release()


def test_a_batch_leaves_render_state_alone(gpu):
    """rtc_render_ppm and rtc_render of the committed camera return what they returned before a text batch."""
    cam, world = scenes.dragon_element(gpu, width=320, height=180, n_u=24, n_v=12)
    views = _views(gpu, cam)[:4]
    far = views[gpu.farthest_camera(views)]
    p = far.prepare(world)
    try:
        before_text = p.render_ppm(5)
        before = p.render(5)
        rgb, u8 = before.data.copy(), before.to_u8().copy()
        p.render_views_ppm(views, 5)
        assert p.render_ppm(5) == before_text
        after = p.render(5)
        assert np.array_equal(after.data, rgb) and np.array_equal(after.to_u8(), u8)
        p.render_views_ppm(views, 5)
        assert p.render_ppm(5) == before_text
    finally:
        p.release()


def test_one_shot_matches_the_prepared_form(gpu):
    cam, world = scenes.reflect_refract(gpu, width=200, height=100)
    views = _views(gpu, cam)
    texts = gpu.render_views_ppm(world, views, 5)
    far = views[gpu.farthest_camera(views)]
    p = far.prepare(world)
    try:
        assert texts == p.render_views_ppm(views, 5)
    finally:
        p.release()
    assert texts[-1] == cam.render_b200_ppm(world, 5)


def test_two_devices_write_the_same_texts(gpu):
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
            out.append(p.render_views_ppm(views, 5))
            out.append(p.render_views_ppm(views, 5, out=np.zeros(len(views) * _bound(gpu, cam), np.uint8)))
        finally:
            p.release()
    gpu.set_render_options(n_devices=1)
    assert out[0] == out[1] == out[2] == out[3]
