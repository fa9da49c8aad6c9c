"""CSG trees beyond the whole-tree evaluator's limits on the GPU: frames of the die, the carved mesh and the sphere chain
against the CPU oracle, one-shot against prepared, shards, the wavefront renderer, and the scenes the whole-tree evaluator
accepts rendered again with every CSG sent to csg_sweep (RTC_CSG_SWEEP=1).  Run on the B200 box: `pytest tests -m gpu`."""
import numpy as np
import pytest

from ray_tracer_challenge_b200 import scenes
from tests.parity import assert_parity, assert_unrendered_border, compare_frames

pytestmark = pytest.mark.gpu
RTC_OPT_WAVEFRONT = 8

SCENES = {
    "die": (scenes.csg_die, dict(width=320, height=200)),
    "die_glass": (scenes.csg_die, dict(width=240, height=150, glassy=True)),
    "die_area": (scenes.csg_die, dict(width=200, height=120, area_light=True)),
    "die_glass_area": (scenes.csg_die, dict(width=160, height=100, glassy=True, area_light=True)),
    "die_surrounded": (scenes.csg_die, dict(width=240, height=150, surrounded=True)),
    "die_surrounded_glass": (scenes.csg_die, dict(width=240, height=150, glassy=True, surrounded=True)),
    "die_surrounded_glass_area": (scenes.csg_die, dict(width=160, height=100, glassy=True, area_light=True, surrounded=True)),
    "carved_mesh": (scenes.csg_carved_mesh, dict(width=240, height=150)),
    "chain": (scenes.csg_chain, dict(width=240, height=150)),
}


@pytest.fixture(scope="module")
def gpu():
    import ray_tracer_challenge_b200 as rt

    return rt.new_session()


@pytest.mark.parametrize("name", sorted(SCENES))
def test_frame_parity(name, gpu, oracle):
    build, kw = SCENES[name]
    oracle.probe.set_threads(oracle.probe.max_threads())
    ocam, oworld = build(oracle, **kw)
    want = ocam.render(oworld, 5)
    gcam, gworld = build(gpu, **kw)
    prepared = gcam.prepare(gworld)
    try:
        got = prepared.render(5)
        st = prepared.last_stats
        rep = compare_frames(got.to_u8(), want.to_u8(), got.data, want.data)
        rep["rays_gpu"], rep["rays_oracle"] = int(st.rays), int(ocam.last_stats.rays)
        assert_unrendered_border(got.to_u8(), got.data)
        assert rep["exact_u8"] == 1.0, rep                  # every 8-bit channel equal (IEEE build)
        assert rep["rays_gpu"] == rep["rays_oracle"], rep    # identical ray trees
        assert rep["bit_exact_f32"] >= 0.90, rep             # the rest differs only through powf / cosf / atan2f
        assert st.capacity_overflows == 0
        assert_parity(rep, min_within=0.9999, max_gross=0.0001, label=f"{name} (IEEE build)")
    finally:
        prepared.release()


def test_one_shot_render_b200_matches_prepared(gpu):
    cam, world = scenes.csg_die(gpu, width=160, height=100, glassy=True)
    a = cam.render_b200(world, 5)
    p = cam.prepare(world)
    b = p.render(5)
    p.release()
    assert np.array_equal(a.data.view(np.uint32), b.data.view(np.uint32))
    assert np.array_equal(a.to_u8(), b.to_u8())
    assert cam.last_rtc_stats.capacity_overflows == 0


@pytest.mark.parametrize("name", ["die_surrounded_glass", "carved_mesh"])
def test_two_shards_reassemble_bit_identical(name, gpu):
    build, kw = SCENES[name]
    cam, world = build(gpu, **kw)
    p = cam.prepare(world)
    try:
        full = p.render(5)
        rgb = np.full_like(full.data, np.nan)
        u8 = np.full_like(full.to_u8(), 7)
        for shard in range(2):
            p.render(5, out_rgb=rgb, out_u8=u8, shard=shard, n_shards=2)
        assert np.array_equal(rgb.view(np.uint32), full.data.view(np.uint32))
        assert np.array_equal(u8, full.to_u8())
    finally:
        p.release()


def test_wavefront_renders_the_same_frame(gpu):
    """The glass die among marbles is a tree scene with branching ray trees: what the wavefront renderer is for."""
    cam, world = scenes.csg_die(gpu, width=240, height=150, glassy=True, surrounded=True)
    assert gpu.inspect(cam, world)["converge"] == 1
    p = cam.prepare(world)
    try:
        p.set_option(RTC_OPT_WAVEFRONT, 0)
        stream = p.render(5)
        st_stream = p.last_stats
        p.set_option(RTC_OPT_WAVEFRONT, 1)
        wave = p.render(5)
        st_wave = p.last_stats
        assert st_wave.launches >= 8 and st_wave.wave_overflows == 0 and st_wave.capacity_overflows == 0
        assert (st_wave.secondary_rays, st_wave.shadow_rays, st_wave.shades) == \
               (st_stream.secondary_rays, st_stream.shadow_rays, st_stream.shades)
        assert np.array_equal(wave.data.view(np.uint32), stream.data.view(np.uint32))
        assert np.array_equal(wave.to_u8(), stream.to_u8())
    finally:
        p.release()


@pytest.mark.parametrize("name,build,kw", [
    ("csg_gallery", scenes.csg_gallery, dict(width=320, height=200)),
    ("reflect_refract_csg", scenes.reflect_refract, dict(width=240, height=120, with_csg=True)),
    ("stress_small", scenes.stress, dict(width=240, height=135, n_spheres=3000, n_each=8, n_csg=6)),
])
def test_sweep_renders_what_the_whole_tree_evaluator_renders(name, build, kw, gpu, monkeypatch):
    """RTC_CSG_SWEEP=1 sends every CSG to csg_sweep: the frame is the default path's, bit for bit."""
    frames = []
    for sweep in ("0", "1"):
        monkeypatch.setenv("RTC_CSG_SWEEP", sweep)
        cam, world = build(gpu, **kw)
        p = cam.prepare(world)
        try:
            for fma in (False, True):
                frames.append((p.render(5, fma=fma), p.last_stats))
        finally:
            p.release()
    for (a, sa), (b, sb) in ((frames[0], frames[2]), (frames[1], frames[3])):
        assert np.array_equal(a.data.view(np.uint32), b.data.view(np.uint32)), name
        assert np.array_equal(a.to_u8(), b.to_u8()), name
        assert sa.rays == sb.rays and sb.capacity_overflows == 0
