"""RTC_OPT_EXACT_GROUPS on the GPU: with the option on, frames the reference's group culls decide are the oracle's,
100 % in 8 bits with equal ray counts; on the sphere fields the option makes no pixel differ that did not differ before;
and the renderers agree with each other."""
import numpy as np
import pytest

from bench import build_scene
from ray_tracer_challenge_b200 import scenes
from tests import exact_groups_scenes as eg
from tests.parity import assert_parity, compare_frames

pytestmark = pytest.mark.gpu

RTC_OPT_WAVEFRONT = 8


@pytest.fixture
def gpu():
    import ray_tracer_challenge_b200 as rt

    api = rt.new_session()
    api.set_exact_groups(True)
    return api


def _identical(gpu, oracle, make, kw):
    gcam, gworld = make(gpu, **kw)[:2]
    ocam, oworld = make(oracle, **kw)[:2]
    got = gcam.render_b200(gworld, 5)
    want = ocam.render(oworld, 5)
    rep = compare_frames(got.to_u8(), want.to_u8(), got.data, want.data)
    assert rep["exact_u8"] == 1.0, rep
    assert gcam.last_rtc_stats.rays == ocam.last_stats.rays, (gcam.last_rtc_stats.rays, ocam.last_stats.rays)
    return rep


@pytest.mark.parametrize("case", ["stale_box", "csg_tree", "csg_tree_glass", "csg_small", "csg_small_glass"])
def test_group_cull_scenes_match_oracle(case, gpu, oracle):
    if case == "stale_box":
        _identical(gpu, oracle, eg.stale_box, dict())
    else:
        _identical(gpu, oracle, eg.csg_in_group, dict(n_spheres=60 if "tree" in case else 3, glass="glass" in case))


def _closer(gpu, oracle, make, kw, rows=None):
    """Option on against option off, both against the oracle: the option removes differences and adds none.  Frames of
    fields of far, small spheres keep a few pixels that no group cull decides: the reference reports hits outside the
    hit primitive's own bounding box (phantom hits of its f32 tests), beyond the tree's padding (DESIGN.md §7)."""
    import ray_tracer_challenge_b200 as rt

    reps = []
    for exact in (False, True):
        api = rt.new_session()
        api.set_exact_groups(exact)
        gcam, gworld = make(api, **kw)[:2]
        got = gcam.render_b200(gworld, 5)
        reps.append((got.to_u8(), got.data))
    ocam, oworld = make(oracle, **kw)[:2]
    if rows is None:
        want = ocam.render(oworld, 5)
        want_u8, want_f32 = want.to_u8(), want.data
    else:
        want_f32, want_u8, _ = oracle.probe.render_rows(ocam, oworld, 5, rows[0], ocam.height_pixels, rows[1] - rows[0],
                                                        want_u8=True)
        sel = np.arange(rows[0], ocam.height_pixels - 1, rows[1] - rows[0])
        reps = [(u8[sel], f32[sel]) for u8, f32 in reps]
        want_u8, want_f32 = want_u8[sel], want_f32[sel]
    bad = [(u8 != want_u8).any(axis=2) for u8, _ in reps]
    assert not (bad[1] & ~bad[0]).any(), "the option made a pixel differ"
    rep = compare_frames(reps[1][0], want_u8, reps[1][1], want_f32)
    print("off", int(bad[0].sum()), "on", int(bad[1].sum()), rep)
    assert_parity(rep, min_within=0.99995, max_gross=0.00005)
    return bad


def test_sphere_field_against_oracle(oracle):
    """test_sphere_field_parity_at_scale's 20 k field."""
    oracle.probe.set_threads(oracle.probe.max_threads())
    _closer(None, oracle, scenes.stress, dict(width=640, height=360, n_spheres=20_000, n_each=16, n_csg=8))


def test_c5_full_size_rows_against_oracle(oracle):
    oracle.probe.set_threads(oracle.probe.max_threads())
    _closer(None, oracle, lambda api: build_scene(api, "c5")[:2], dict(), rows=(24, 72))


def _frame(p, **kw):
    out = p.render(5, **kw)
    return out.data.copy(), out.to_u8().copy(), p.last_stats.rays


@pytest.mark.parametrize("case", ["stale_box", "csg_tree_glass", "stress"])
def test_renderers_agree(case, gpu, monkeypatch):
    """Streaming and wavefront, one shard and two, csg_eval and csg_sweep: the same frame with the option on."""
    make, kw = {"stale_box": (eg.stale_box, dict()),
                "csg_tree_glass": (eg.csg_in_group, dict(glass=True)),
                "stress": (scenes.stress, dict(width=320, height=180, n_spheres=5000, n_each=8, n_csg=6))}[case]
    cam, world = make(gpu, **kw)[:2]
    p = cam.prepare(world)
    try:
        ref, ref_u8, rays = _frame(p)
        p.set_option(RTC_OPT_WAVEFRONT, 1)
        wave, _, wave_rays = _frame(p)
        p.set_option(RTC_OPT_WAVEFRONT, 0)
        assert (wave.view(np.uint32) == ref.view(np.uint32)).all() and wave_rays == rays
        h, w = ref.shape[:2]
        rgb, u8 = np.zeros((h, w, 3), np.float32), np.zeros((h, w, 3), np.uint8)
        for shard in (0, 1):
            p.render(5, out_rgb=rgb, out_u8=u8, shard=shard, n_shards=2)
        assert (rgb.view(np.uint32) == ref.view(np.uint32)).all() and (u8 == ref_u8).all()
    finally:
        p.release()
    monkeypatch.setenv("RTC_CSG_SWEEP", "1")
    p = cam.prepare(world)
    try:
        swept, _, swept_rays = _frame(p)
        assert (swept.view(np.uint32) == ref.view(np.uint32)).all() and swept_rays == rays
    finally:
        p.release()


def test_silhouette_rays_trace_to_oracle(gpu, oracle):
    """rtc_trace_rays on rays whose answer the group boxes decide: the oracle's distance and sphere."""
    cam, world, centres, handles = eg.far_field(gpu)
    _, grouped, _, ohandles = eg.far_field(oracle)
    _, ungrouped, _, _ = eg.far_field(oracle, grouped=False)
    o, d = eg.far_field_rays(centres, 2000, spread_radii=1.5)
    want = eg.oracle_nearest(oracle, grouped, o, d)
    decided = want != eg.oracle_nearest(oracle, ungrouped, o, d)
    assert decided.sum() >= 50
    p = cam.prepare(world)
    try:
        _, t, shape = p.trace_rays(o, d, 5)
    finally:
        p.release()
    assert (t.view(np.uint32) == np.where(want >= 0, want, np.float32(-1)).view(np.uint32)).all(), int((t != want).sum())
    index = {h: i for i, h in enumerate(handles)}
    oindex = {h: i for i, h in enumerate(ohandles)}
    for i in range(len(o)):
        if want[i] < 0:
            assert shape[i] < 0
            continue
        ts, objs = oracle.probe.world_intersect(grouped, o[i], d[i], cap=4096)
        assert index[int(shape[i])] == oindex[int(objs[oracle.probe.hit_index(ts)])], i
