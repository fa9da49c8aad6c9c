"""The wavefront renderer (csrc/dev_wave.cuh, RTC_OPT_WAVEFRONT = 8): rays as work items, one queue per bounce level, tree
walks / shading / post-order combine in kernels of their own.  It must render what the streaming kernel renders, bit
for bit, with the same ray counts — and a chunk whose ray pool overflows is rendered again by the streaming kernel, so
the frame is complete either way."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from ray_tracer_challenge_b200 import scenes
from tests.parity import compare_frames
from tests.wave_child import RTC_OPT_WAVEFRONT, tight_glass_die

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def gpu():
    import ray_tracer_challenge_b200 as rt

    return rt.new_session()


@pytest.mark.parametrize("kw", [dict(width=384, height=216, n_spheres=5000, n_each=8, n_csg=4),
                                dict(width=163, height=67, n_spheres=1500, n_each=4, n_csg=2)])  # ragged edges too
def test_wavefront_frame_equals_streaming_frame(gpu, oracle, kw):
    cam, world = scenes.stress(gpu, **kw)
    assert gpu.inspect(cam, world)["converge"] == 1  # branching ray trees: the scene class both renderers are for
    p = cam.prepare(world)
    try:
        for depth in (5, 1, 0):
            p.set_option(RTC_OPT_WAVEFRONT, 0)
            stream = p.render(depth)
            st_stream = p.last_stats
            p.set_option(RTC_OPT_WAVEFRONT, 1)
            wave = p.render(depth)
            st_wave = p.last_stats
            assert st_wave.launches >= 8 and st_wave.wave_overflows == 0, (st_wave.launches, st_wave.wave_overflows)
            assert (st_wave.primary_rays, st_wave.secondary_rays, st_wave.shadow_rays, st_wave.shades) == \
                   (st_stream.primary_rays, st_stream.secondary_rays, st_stream.shadow_rays, st_stream.shades), depth
            assert np.array_equal(wave.data.view(np.uint32), stream.data.view(np.uint32)), depth
            assert np.array_equal(wave.to_u8(), stream.to_u8())
    finally:
        p.release()
    ocam, oworld = scenes.stress(oracle, **kw)
    want = ocam.render(oworld, 0)
    rep = compare_frames(wave.to_u8(), want.to_u8(), wave.data, want.data)
    assert rep["exact_u8"] >= 0.9995, rep


@pytest.mark.parametrize("name,make,kw,branching", [
    # the glass case refracts but does not reflect: its ray trees do not branch, so RTC_STREAM=1 sends it to the
    # streaming kernel, and with RTC_OPT_WAVEFRONT to the wavefront renderer
    ("mesh_in_glass_case", scenes.dragon_element, dict(width=320, height=180, n_u=24, n_v=12), False),
    ("glass_die_with_marbles", scenes.csg_die, dict(width=240, height=150, glassy=True, surrounded=True), True),
    ("tight_glass_die", tight_glass_die, dict(width=320, height=200), True),  # 26 rays per pixel: the first pools overflow
])
def test_wavefront_equals_streaming_on_glass_scenes(gpu, monkeypatch, name, make, kw, branching):
    """A mesh in a glass case, CSG glass and glass that fills the frame: the wavefront frame is the streaming frame, bit
    for bit, with the same ray counts — also while the pool overflows, until it has grown to hold the chunk."""
    cam, world = make(gpu, **kw)
    info = gpu.inspect(cam, world)
    assert info["small_n"] == 0 and info["converge"] == int(branching), info  # a tree scene
    if not branching:
        monkeypatch.setenv("RTC_STREAM", "1")  # read when the scene is created
    p = cam.prepare(world)
    try:
        p.set_option(RTC_OPT_WAVEFRONT, 0)
        stream = p.render(5)
        st_stream = p.last_stats
        p.set_option(RTC_OPT_WAVEFRONT, 1)
        for _ in range(5):  # the pool doubles after every render that overflowed, from 6 to 64 rays per pixel
            wave = p.render(5)
            st_wave = p.last_stats
            assert st_wave.launches == _launches(1, 5, st_wave.wave_overflows), st_wave.launches  # one chunk, wavefront
            assert (st_wave.primary_rays, st_wave.secondary_rays, st_wave.shadow_rays, st_wave.shades) == \
                   (st_stream.primary_rays, st_stream.secondary_rays, st_stream.shadow_rays, st_stream.shades)
            assert np.array_equal(wave.data.view(np.uint32), stream.data.view(np.uint32))
            assert np.array_equal(wave.to_u8(), stream.to_u8())
            if st_wave.wave_overflows == 0:
                break
        assert st_wave.wave_overflows == 0, name
    finally:
        p.release()


def _child(case):
    """tests/wave_child.py in a fresh process: a pool of known size (it lives as long as the process)."""
    proc = subprocess.run([sys.executable, "-m", "tests.wave_child", case], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert proc.returncode == 0, (proc.stdout + proc.stderr)[-3000:]
    out = json.loads(proc.stdout.strip().splitlines()[-1])
    print(case, out)
    assert out["small_n"] == 0 and out["converge"] == 1, out
    return out


def _launches(n_chunks, depth, overflows):
    """rtc_api.cu: render_impl — a chunk's launch_wave, plus one render_stream per chunk that overflowed."""
    return n_chunks * (2 + 6 * (depth + 1)) + overflows


def test_wavefront_pool_overflow_falls_back_and_grows():
    """A fresh pool holds 6 rays per pixel of the chunk and doubles after every render that overflowed, up to 64.  The
    tight glass die needs 26: renders 0, 1 and 2 overflow (6, 12 and 24 rays per pixel), and their chunk is rendered
    again by the streaming kernel; render 3 (48) and later fit.  Every frame is the streaming frame, bit for bit."""
    out = _child("grow")
    rays, chunk_px = out["rays"], out["chunk_px"]
    assert out["n_chunks"] == 1
    overflowed = [r["overflows"] for r in out["renders"]]
    assert overflowed == [int(rays > chunk_px * min(64, 6 * 2 ** i)) for i in range(len(overflowed))], (rays, chunk_px, overflowed)
    assert overflowed == [1, 1, 1, 0, 0], (rays / chunk_px, overflowed)
    for i, r in enumerate(out["renders"]):
        assert r["same"] and r["same_stats"], (i, r)
        assert r["launches"] == _launches(1, 5, r["overflows"]), (i, r)


def test_wavefront_chunks_shards_and_staged_canvases_while_the_pool_overflows():
    """A frame of more than 2^20 pixels is rendered in chunks through one pool; into NumPy (pageable) canvases of more
    than 4 MiB, which are filled through the pinned staging frame.  At about 9 rays per pixel the first render overflows
    (6 per pixel), its overflowing chunks are rendered again by the streaming kernel at their band offset, and the pool
    settles at 12 per pixel.  Both renders, and three shards of the frame, are the streaming frame bit for bit."""
    out = _child("chunks")
    assert out["n_chunks"] >= 2, out
    first, second = out["whole"]
    assert first["overflows"] >= 1 and second["overflows"] == 0, out
    for r in out["whole"]:
        assert r["same"] and r["same_stats"], out
        assert r["launches"] == _launches(out["n_chunks"], 5, r["overflows"]), out
    for s in out["shards"]:
        assert s["overflows"] == 0 and s["launches"] == _launches(s["n_chunks"], 5, 0), out
    assert out["reassembled"] and out["shard_stats"], out


def test_wavefront_shards_reassemble(gpu):
    kw = dict(width=200, height=120, n_spheres=2000, n_each=4, n_csg=2)
    cam, world = scenes.stress(gpu, **kw)
    p = cam.prepare(world)
    try:
        p.set_option(RTC_OPT_WAVEFRONT, 1)
        whole = p.render(5)
        parts = np.zeros_like(whole.data)
        for shard in range(3):
            p.render(5, out_rgb=parts, shard=shard, n_shards=3)
        assert np.array_equal(parts.view(np.uint32), whole.data.view(np.uint32))
    finally:
        p.release()
