"""Anti-aliased frames (rtc_render_samples) on the GPU: n = 1 is rtc_render's frame bit for bit on every kernel path, and
n >= 2 is bit for bit the box filter of rtc_render's frame of the scene committed at n times the canvas size (device against
device), in f32 and in 8 bits; against the oracle at small sizes; through every destination and on several devices; and
without touching rtc_render's state.  Run on the B200 box: `pytest tests -m gpu`."""
import ctypes as C

import numpy as np
import pytest

import ray_tracer_challenge_b200 as rt
from bench import WORKLOADS
from ray_tracer_challenge_b200 import scenes
from tests.test_gpu_views import SCENES
from tests.test_samples_on_host import box_filter

pytestmark = pytest.mark.gpu

RTC_OPT_WAVEFRONT = 8


@pytest.fixture(scope="module")
def gpu():
    return rt.new_session()


def _scale_u8(rgb):
    """Canvas::scale_color (canvas.rs:39-43) of an f32 plane: clamp, then truncate; NaN -> 255"""
    s = np.where(np.isnan(rgb), np.float32(255.0), np.clip(rgb * np.float32(255.0), 0.0, 255.0)).astype(np.float32)
    return s.astype(np.uint8)


def _big_frame(gpu, build, kw, n, fma, depth=5):
    """rtc_render's f32 frame of the scene committed with the sample camera C_n: the builder at n times the canvas size"""
    big = dict(kw, width=n * kw["width"], height=n * kw["height"])
    cam, world = build(gpu, **big)
    p = cam.prepare(world)
    try:
        return p.render(depth, want_u8=False, fma=fma).data.copy()
    finally:
        p.release()


def _samples(gpu, build, kw, n, fma, depth=5):
    cam, world = build(gpu, **kw)
    p = cam.prepare(world)
    try:
        c = p.render_samples(n, depth, fma=fma)
        st = p.last_stats
        return c.data.copy(), c.to_u8().copy(), st
    finally:
        p.release()


def _check_box(gpu, build, kw, n, fma=False, label=""):
    w, h = kw["width"], kw["height"]
    rgb, u8, st = _samples(gpu, build, kw, n, fma)
    want = box_filter(_big_frame(gpu, build, kw, n, fma), w, h, n)
    same = rgb.view(np.uint32) == want.view(np.uint32)
    assert same.all(), (label, n, fma, int((~same).sum()), np.argwhere(~same)[:3])
    assert np.array_equal(u8, _scale_u8(want)), (label, n, fma)
    assert st.primary_rays == n * n * (w - 1) * (h - 1), (label, st.primary_rays)


@pytest.mark.parametrize("name", list(SCENES))
def test_one_sample_is_rtc_render(gpu, name):
    """n = 1: both of rtc_render's planes bit for bit, on every parity scene and kernel path, in each FP build listed."""
    build, kw, _, fmas = SCENES[name]
    cam, world = build(gpu, **kw)
    p = cam.prepare(world)
    try:
        for fma in (False, True):
            want = p.render(5, fma=fma)
            got = p.render_samples(1, 5, fma=fma)
            assert np.array_equal(got.data.view(np.uint32), want.data.view(np.uint32)), (name, fma)
            assert np.array_equal(got.to_u8(), want.to_u8()), (name, fma)
    finally:
        p.release()


# name -> (builder, kwargs at the output size, samples per axis, FMA settings)
BOX_CASES = {
    "lean_table": (scenes.soft_shadows, dict(width=160, height=64, u_steps=4, v_steps=4), (2, 3, 4), (False, True)),
    "lean_drawn": (scenes.soft_shadows, dict(width=160, height=64, u_steps=4, v_steps=4, jitter=None, seed=3), (2, 3, 4),
                   (False, True)),
    "small_converging": (scenes.reflect_refract, dict(width=200, height=100), (2, 3), (False, True)),
    "small_textured": (scenes.textured, dict(width=160, height=100), (2,), (False,)),
    "tree_mesh": (scenes.dragon_element, dict(width=160, height=90, n_u=24, n_v=12), (2, 3), (False, True)),
    "tree_stream": (scenes.stress, dict(width=192, height=108, n_spheres=3000, n_each=16, n_csg=4, extent=20.0), (2, 3),
                    (False,)),
    "sweep_csg_die": (scenes.csg_die, dict(width=160, height=100), (2, 3), (False, True)),
    "odd_width": (scenes.soft_shadows, dict(width=157, height=61, u_steps=4, v_steps=4, jitter=None, seed=5), (2, 3), (False,)),
}


@pytest.mark.parametrize("name", list(BOX_CASES))
def test_samples_are_the_box_filter_of_the_big_render(gpu, name):
    build, kw, ns, fmas = BOX_CASES[name]
    for n in ns:
        for fma in fmas:
            _check_box(gpu, build, kw, n, fma, name)


@pytest.mark.parametrize("workload", ["c1", "c3", "c3_counter"])
def test_full_size_two_by_two(gpu, workload):
    """c1 and c3 at full size (c3 also with generated jitter) at n = 2: the box filter of the 2x frame rendered on the device."""
    builder, kw, depth, _ = WORKLOADS[workload]
    _check_box(gpu, getattr(scenes, builder), kw, 2, False, workload)


def test_samples_match_the_oracle(gpu, oracle):
    """Small frames against the box filter of the oracle's render at n times the size (strict build): bit for bit on the
    soft-shadow scene with generated jitter, and within the parity bounds of the oracle frame tests elsewhere."""
    from tests.parity import assert_parity, compare_frames

    cases = ((scenes.soft_shadows, dict(width=64, height=32, u_steps=4, v_steps=4, jitter=None, seed=3), 3, True),
             (scenes.reflect_refract, dict(width=80, height=40), 2, False),
             (scenes.dragon_element, dict(width=64, height=36, n_u=24, n_v=12), 2, False))
    for build, kw, n, exact in cases:
        w, h = kw["width"], kw["height"]
        rgb, u8, _ = _samples(gpu, build, kw, n, False)
        ocam, oworld = build(oracle, **dict(kw, width=n * w, height=n * h))
        want = box_filter(ocam.render(oworld, 5).data, w, h, n)
        assert_parity(compare_frames(u8, _scale_u8(want), rgb, want), label=f"{build.__name__} n={n}")
        if exact:
            assert np.array_equal(rgb.view(np.uint32), want.view(np.uint32)), build.__name__
            assert np.array_equal(u8, _scale_u8(want)), build.__name__


def test_destinations_give_the_same_planes(gpu):
    """Pageable (staged: 960x540 planes of several MiB), pinned, one plane at a time, and NULL / NULL."""
    cam, world = scenes.soft_shadows(gpu, width=960, height=540, u_steps=4, v_steps=4)
    h, w = cam.height_pixels, cam.width_pixels
    p = cam.prepare(world)
    lib = rt.device_library()
    lib.rtc_host_alloc.restype = C.c_void_p
    lib.rtc_host_free.argtypes = [C.c_void_p]
    try:
        c = p.render_samples(2)
        rgb, u8 = c.data.copy(), c.to_u8().copy()
        assert np.array_equal(p.render_samples(2, want_u8=False).data, rgb)
        assert np.array_equal(p.render_samples(2, want_rgb=False).to_u8(), u8)
        p.render_samples(2, want_rgb=False, want_u8=False)
        assert p.last_stats.primary_rays == 4 * (w - 1) * (h - 1) and p.last_stats.launches >= 1
        nbytes = h * w * 3
        ptr_rgb, ptr_u8 = lib.rtc_host_alloc(C.c_size_t(nbytes * 4)), lib.rtc_host_alloc(C.c_size_t(nbytes))
        try:
            pin_rgb = np.ctypeslib.as_array((C.c_float * nbytes).from_address(ptr_rgb)).reshape(h, w, 3)
            pin_u8 = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(ptr_u8)).reshape(h, w, 3)
            pin_rgb[:], pin_u8[:] = -1.0, 7
            p.render_samples(2, out_rgb=pin_rgb, out_u8=pin_u8)
            assert np.array_equal(pin_rgb, rgb) and np.array_equal(pin_u8, u8)
        finally:
            lib.rtc_host_free(C.c_void_p(ptr_rgb))
            lib.rtc_host_free(C.c_void_p(ptr_u8))
    finally:
        p.release()


def test_two_devices_render_the_same_frame(gpu):
    if rt.device_library().rtc_device_count() < 2:
        pytest.skip("needs two devices")
    out = []
    for build, kw in ((scenes.dragon_element, dict(width=320, height=180, n_u=24, n_v=12)),
                      (scenes.stress, dict(width=192, height=108, n_spheres=3000, n_each=16, n_csg=4, extent=20.0))):
        for n_dev in (1, 2):
            gpu.set_render_options(n_devices=n_dev)
            cam, world = build(gpu, **kw)
            p = cam.prepare(world)
            try:
                c = p.render_samples(3)
                out.append((c.data.copy(), c.to_u8().copy()))
            finally:
                p.release()
        gpu.set_render_options(n_devices=1)
        assert np.array_equal(out[-2][0], out[-1][0]) and np.array_equal(out[-2][1], out[-1][1]), build.__name__


def test_samples_leave_render_state_alone(gpu, monkeypatch, tmp_path):
    """Two prepared scenes render the same sequence of frames, one with rtc_render_samples calls in between: the frames,
    launches and the render that learns the adaptive tile order (it writes RTC_DUMP_TILE_COST) agree."""
    cam, world = scenes.dragon_element(gpu, width=320, height=180, n_u=24, n_v=12)
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
            frames_a.append(a.render(5).data.copy())
            learn_a.append(learnt())
            sa = a.last_stats
            if k % 2 == 0:
                b.render_samples(2, 5)
                assert b.last_stats.primary_rays == 4 * 319 * 179
                assert not learnt()
            frames_b.append(b.render(5).data.copy())
            learn_b.append(learnt())
            sb = b.last_stats
            assert (sb.launches, sb.primary_rays, sb.secondary_rays, sb.shades) == \
                (sa.launches, sa.primary_rays, sa.secondary_rays, sa.shades)
        assert learn_a == learn_b == [k == 1 for k in range(6)], (learn_a, learn_b)
        for fa, fb in zip(frames_a, frames_b):
            assert np.array_equal(fa.view(np.uint32), fb.view(np.uint32))
    finally:
        a.release(), b.release()


def test_wavefront_option_does_not_change_samples(gpu):
    build, kw, _, _ = BOX_CASES["tree_stream"]
    cam, world = build(gpu, **kw)
    p = cam.prepare(world)
    try:
        want = p.render_samples(2).data.copy()
        p.set_option(RTC_OPT_WAVEFRONT, 1)
        got = p.render_samples(2)
        assert p.last_stats.launches == 1  # one persistent streaming launch
        assert np.array_equal(got.data.view(np.uint32), want.view(np.uint32))
    finally:
        p.release()


def test_one_shot_and_checks_on_a_committed_scene(gpu):
    cam, world = scenes.reflect_refract(gpu, width=200, height=100)
    p = cam.prepare(world)
    try:
        want = p.render_samples(2)
        for bad in (0, 17):
            with pytest.raises(rt.RtcError, match="samples_per_axis"):
                p.render_samples(bad)
        with pytest.raises(rt.RtcError, match="reflection_recursion_depth"):
            p.render_samples(2, 30)
        got = cam.render_b200_samples(world, 2)
        assert np.array_equal(got.data, want.data) and np.array_equal(got.to_u8(), want.to_u8())
    finally:
        p.release()
