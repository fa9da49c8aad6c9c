"""The lean kernel build of small scenes on the GPU: a scene the commit marks lean (SmallScene::lean) renders the frame
the general small-scene build renders (RTC_LEAN=0), bit for bit — f32 and 8-bit canvases and ray counts, in both FMA
settings, whole or as two reassembled shards.  Run on the B200 box: `pytest tests -m gpu`."""
import numpy as np
import pytest

from ray_tracer_challenge_b200 import scenes

pytestmark = pytest.mark.gpu

SCENES = {
    "soft_shadows_table": (scenes.soft_shadows, dict(width=320, height=128, u_steps=4, v_steps=4)),
    "soft_shadows_100_cells": (scenes.soft_shadows, dict(width=250, height=100)),
    "soft_shadows_drawn": (scenes.soft_shadows, dict(width=250, height=100, jitter=None, seed=3)),
    "c3_reduced": (scenes.soft_shadows, dict(width=960, height=540, u_steps=4, v_steps=4)),
    "c3_counter_reduced": (scenes.soft_shadows, dict(width=960, height=540, u_steps=4, v_steps=4, jitter=None, seed=7)),
}


@pytest.fixture(scope="module")
def gpu():
    import ray_tracer_challenge_b200 as rt

    return rt.new_session()


def _frames(gpu, build, kw, lean, monkeypatch, shards=False):
    """{fma: (rgb, u8, (secondary, shadow, shades))} of the scene committed with RTC_LEAN unset or 0."""
    if lean:
        monkeypatch.delenv("RTC_LEAN", raising=False)
    else:
        monkeypatch.setenv("RTC_LEAN", "0")
    cam, world = build(gpu, **kw)
    assert gpu.inspect(cam, world)["lean"] == int(lean)
    p = cam.prepare(world)
    out = {}
    try:
        for fma in (False, True):
            f = p.render(5, fma=fma)
            st = p.last_stats
            rgb, u8 = f.data, f.to_u8()
            if shards:
                rgb = np.full_like(rgb, np.nan)
                u8 = np.full_like(u8, 7)
                for shard in range(2):
                    p.render(5, out_rgb=rgb, out_u8=u8, shard=shard, n_shards=2, fma=fma)
            out[fma] = (rgb, u8, (st.secondary_rays, st.shadow_rays, st.shades))
    finally:
        p.release()
    return out


def _assert_same(name, a, b):
    for fma in (False, True):
        (ra, ua, ca), (rb, ub, cb) = a[fma], b[fma]
        assert np.array_equal(ra.view(np.uint32), rb.view(np.uint32)), (name, fma)
        assert np.array_equal(ua, ub), (name, fma)
        assert ca == cb, (name, fma, ca, cb)


@pytest.mark.parametrize("name", sorted(SCENES))
def test_lean_build_renders_the_general_frame(name, gpu, monkeypatch):
    build, kw = SCENES[name]
    _assert_same(name, _frames(gpu, build, kw, True, monkeypatch), _frames(gpu, build, kw, False, monkeypatch))


@pytest.mark.parametrize("name", ["soft_shadows_table", "soft_shadows_drawn"])
def test_lean_shards_reassemble_the_general_frame(name, gpu, monkeypatch):
    build, kw = SCENES[name]
    _assert_same(name, _frames(gpu, build, kw, True, monkeypatch, shards=True), _frames(gpu, build, kw, False, monkeypatch))


def test_lean_build_on_random_scenes(gpu, monkeypatch):
    """Random filter-eligible scenes without patterns or transparency (table or counter jitter), at a tile-ragged size."""
    lean = 0
    for seed in range(300, 324):
        build = lambda rt, **kw: scenes.random_filter_scene(rt, seed, **kw)  # noqa: E731
        kw = dict(width=150, height=90)
        monkeypatch.delenv("RTC_LEAN", raising=False)
        cam, world = build(gpu, **kw)
        if not gpu.inspect(cam, world)["lean"]:
            continue
        lean += 1
        _assert_same(seed, _frames(gpu, build, kw, True, monkeypatch), _frames(gpu, build, kw, False, monkeypatch))
    assert lean >= 8, lean
