"""rtc_render_ppm on the GPU: the text written on the device is byte for byte the host writer's text of rtc_render's 8-bit
plane (CanvasU8.to_ppm) and the oracle's Canvas::to_ppm, for the parity scenes, full-size c1 and c3, both FP builds, pinned
and pageable destinations, the one-shot and prepared forms, a ragged size, a capacity exactly at the bound and two devices
when present.  Run on the B200 box: `pytest tests -m gpu`."""
import ctypes as C

import numpy as np
import pytest

import ray_tracer_challenge_b200 as rt
from ray_tracer_challenge_b200 import scenes
from tests.test_gpu_parity import SCENES

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def gpu():
    return rt.new_session()


def _bound(gpu, w, h):
    return gpu.lib.rtc_ppm_bound(w, h)


def _prepared_pair(gpu, cam, world, depth=5, fma=False, out=None):
    """(render_ppm's text, the host writer's text of rtc_render's 8-bit plane) of one prepared scene."""
    p = cam.prepare(world)
    try:
        u8 = p.render(depth, want_rgb=False, fma=fma).to_u8().copy()
        primary = p.last_stats.primary_rays
        text = p.render_ppm(depth, out=out, fma=fma)
        assert p.last_stats.primary_rays == primary and p.last_stats.n_devices >= 1
        return text, rt.CanvasU8(cam.width_pixels, cam.height_pixels, u8, gpu).to_ppm()
    finally:
        p.release()


@pytest.mark.parametrize("name", sorted(SCENES))
def test_parity_scenes(gpu, name):
    build, kw = SCENES[name]
    cam, world = build(gpu, **kw)
    got, want = _prepared_pair(gpu, cam, world)
    assert got == want, name


def test_equals_the_oracle(gpu, oracle):
    for build, kw in ((scenes.soft_shadows, dict(width=160, height=64, u_steps=4, v_steps=4)),
                      (scenes.default_world, dict(width=64, height=48))):
        cam, world = build(gpu, **kw)
        ocam, oworld = build(oracle, **kw)
        assert cam.render_b200_ppm(world, 5) == ocam.render(oworld, 5).to_ppm(), build.__name__


def test_both_fp_builds(gpu):
    for fma in (False, True):
        cam, world = scenes.reflect_refract(gpu, width=320, height=160)
        got, want = _prepared_pair(gpu, cam, world, fma=fma)
        assert got == want, fma


def _pinned(gpu, nbytes):
    lib = rt.device_library()
    lib.rtc_host_alloc.restype = C.c_void_p
    lib.rtc_host_alloc.argtypes = [C.c_size_t]
    lib.rtc_host_free.argtypes = [C.c_void_p]
    ptr = lib.rtc_host_alloc(nbytes)
    assert ptr
    return lib, ptr, np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(ptr))


@pytest.mark.parametrize("workload", ["c1", "c3"])
def test_full_size_one_shot_and_prepared_pinned_and_pageable(gpu, workload):
    """c3's 89 MB of text goes through the staged pieces into pageable memory; c1's 3.9 MB is below the staging threshold."""
    kw = dict(c1=dict(width=1000, height=400, u_steps=10, v_steps=10), c3=dict(width=3840, height=2160, u_steps=4, v_steps=4))[workload]
    cam, world = scenes.soft_shadows(gpu, **kw)
    want = cam.render_b200_u8(world, 5).to_ppm()
    assert cam.render_b200_ppm(world, 5) == want  # one-shot, pageable
    bound = _bound(gpu, cam.width_pixels, cam.height_pixels)
    lib, ptr, pinned = _pinned(gpu, bound)
    try:
        assert cam.render_b200_ppm(world, 5, out=pinned) == want  # one-shot, pinned
        got, host_text = _prepared_pair(gpu, cam, world, out=pinned)  # prepared, pinned
        assert got == host_text == want
        got, host_text = _prepared_pair(gpu, cam, world)  # prepared, pageable
        assert got == want
    finally:
        lib.rtc_host_free(ptr)


def test_ragged_size_and_capacity_exactly_at_the_bound(gpu):
    cam, world = scenes.soft_shadows(gpu, width=333, height=123, u_steps=3, v_steps=2, jitter="constant")
    want = cam.render_b200_u8(world, 5).to_ppm()
    bound = _bound(gpu, 333, 123)
    exact = np.full(bound, 0xAB, np.uint8)
    assert cam.render_b200_ppm(world, 5, out=exact) == want
    assert (exact[len(want):] == 0xAB).all()  # nothing written past the text
    with pytest.raises(ValueError):
        cam.render_b200_ppm(world, 5, out=np.zeros(bound - 1, np.uint8))
    p = cam.prepare(world)
    try:
        assert p.render_ppm(5, out=exact) == want
        for depth in (-1, 24):
            with pytest.raises(rt.RtcError):
                p.render_ppm(depth)
    finally:
        p.release()


def test_two_devices(gpu):
    n = rt.device_library().rtc_device_count()
    if n < 2:
        pytest.skip("one GPU visible")
    one = rt.new_session()
    one.set_render_options(device_ids=[0])
    for n_dev in sorted({2, min(n, 3)}):
        many = rt.new_session()
        many.set_render_options(device_ids=list(range(n_dev)))
        for kw in (dict(width=333, height=123, u_steps=4, v_steps=4), dict(width=3840, height=2160, u_steps=4, v_steps=4)):
            cam1, w1 = scenes.soft_shadows(one, **kw)
            camn, wn = scenes.soft_shadows(many, **kw)
            want = cam1.render_b200_u8(w1, 5).to_ppm()
            assert camn.render_b200_ppm(wn, 5) == want, (n_dev, kw["width"])
            assert camn.last_rtc_stats.n_devices == n_dev
            got, _ = _prepared_pair(many, camn, wn)
            assert got == want
