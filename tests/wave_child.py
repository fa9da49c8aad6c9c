"""The tight glass die, and the wavefront renders that need a process of their own.

The wavefront renderer's ray pool lives on the device slot, which is pooled for the life of the process: it starts at
kWaveRaysPerPixel = 6 rays per pixel of a chunk and doubles after every render in which a chunk overflowed, up to 64.
Only a fresh process has a known pool, so tests/test_gpu_wavefront.py runs `python -m tests.wave_child <case>` and
asserts on the JSON line it prints."""
import json
import sys

import numpy as np

from ray_tracer_challenge_b200 import scenes

RTC_OPT_WAVEFRONT = 8
KBAND_ROWS = 8          # rtc_types.h: kBandRows
KWAVE_MAX_CHUNKS = 64   # rtc_types.h: kWaveMaxChunks


def tight_glass_die(rt, width, height, fov=scenes.PI / 10.0):
    """The glass die among its marbles (a tree scene with branching ray trees), framed so that glass fills the frame:
    at a tenth of pi the oracle counts 26 rays per pixel, primary plus secondary, at depth 5."""
    _, world = scenes.csg_die(rt, width=width, height=height, glassy=True, surrounded=True)
    return rt.Camera(width, height, fov, rt.view_transform((1.0, 3.5, -5.5), (0.0, 1.0, 0.0), (0, 1, 0))), world


def wave_chunk_bands(width, nb):
    """rtc_api.cu: wave_chunk_bands — about 2^20 pixels of the shard per chunk, whole bands, at most 64 chunks."""
    per_band = max(1, width) * KBAND_ROWS
    bands = max(1, (1 << 20) // per_band)
    while (nb + bands - 1) // bands > KWAVE_MAX_CHUNKS:
        bands *= 2
    return min(bands, max(nb, 1))


def _stats(st):
    return [st.primary_rays, st.secondary_rays, st.shadow_rays, st.shades]


def _render(p, wavefront, depth, **kw):
    p.set_option(RTC_OPT_WAVEFRONT, wavefront)
    frame = p.render(depth, **kw)
    return frame, p.last_stats


def _path(gpu, cam, world):
    # the wavefront renders tree scenes (small_n == 0) whose ray trees branch (converge == 1)
    info = gpu.inspect(cam, world)
    return dict(small_n=info["small_n"], converge=info["converge"])


def _same(a, b):
    return bool(np.array_equal(a.data.view(np.uint32), b.data.view(np.uint32)) and np.array_equal(a.to_u8(), b.to_u8()))


def grow(gpu, depth=5, n_renders=5):
    """The tight glass die in one chunk, rendered by the wavefront renderer again and again from a fresh pool."""
    width, height = 320, 200
    cam, world = tight_glass_die(gpu, width, height)
    nb = (height + KBAND_ROWS - 1) // KBAND_ROWS
    p = cam.prepare(world)
    try:
        stream, st_stream = _render(p, 0, depth)
        renders = []
        for _ in range(n_renders):
            wave, st = _render(p, 1, depth)
            renders.append(dict(overflows=st.wave_overflows, launches=st.launches, same=_same(wave, stream),
                                same_stats=_stats(st) == _stats(st_stream)))
    finally:
        p.release()
    return dict(rays=st_stream.primary_rays + st_stream.secondary_rays, chunk_px=wave_chunk_bands(width, nb) * KBAND_ROWS * ((width + 7) // 8 * 8),
                n_chunks=-(-nb // wave_chunk_bands(width, nb)), renders=renders, **_path(gpu, cam, world))


def chunks(gpu, depth=5):
    """A frame of more than 2^20 pixels (two chunks) into plain NumPy canvases, whole and as three shards."""
    width, height = 1280, 832  # at a quarter of pi the oracle counts about 9 rays per pixel
    cam, world = tight_glass_die(gpu, width, height, fov=scenes.PI / 4.0)
    nb = (height + KBAND_ROWS - 1) // KBAND_ROWS
    p = cam.prepare(world)
    try:
        stream, st_stream = _render(p, 0, depth)
        whole = []
        for _ in range(2):
            wave, st = _render(p, 1, depth)
            whole.append(dict(overflows=st.wave_overflows, launches=st.launches, same=_same(wave, stream),
                              same_stats=_stats(st) == _stats(st_stream)))
        rgb, u8 = np.zeros((height, width, 3), np.float32), np.zeros((height, width, 3), np.uint8)
        shards, totals = [], np.zeros(4, np.int64)
        for k in range(3):
            _, st = _render(p, 1, depth, out_rgb=rgb, out_u8=u8, shard=k, n_shards=3)
            shard_nb = len(range(k, nb, 3))
            shards.append(dict(overflows=st.wave_overflows, launches=st.launches,
                               n_chunks=-(-shard_nb // wave_chunk_bands(width, shard_nb))))
            totals += _stats(st)
        reassembled = bool(np.array_equal(rgb.view(np.uint32), stream.data.view(np.uint32)) and np.array_equal(u8, stream.to_u8()))
    finally:
        p.release()
    return dict(n_chunks=-(-nb // wave_chunk_bands(width, nb)), whole=whole, shards=shards, reassembled=reassembled,
                shard_stats=[int(x) for x in totals] == _stats(st_stream), **_path(gpu, cam, world))


if __name__ == "__main__":
    import ray_tracer_challenge_b200 as rt

    session = rt.new_session()
    print(json.dumps({"grow": grow, "chunks": chunks}[sys.argv[1]](session), default=int))
