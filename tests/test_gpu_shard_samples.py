"""Anti-aliased frames shared by several processes, one shard each, on the GPU (rtc_render_shard_samples,
rtc_render_shard_samples_ppm_rows + rtc_write_shard_ppm).  The union of shards 0..N-1 is rtc_render_samples' frame bit for bit
in f32 and 8 bits, on every kernel path and in each FP build the scene lists, for N = 1, 2, 3, 8 and n = 1..4, and each
shard's writes stay inside its bands; pinned and pageable destinations, a ragged frame and full-size c3 at n = 2 (a pageable
plane big enough to be staged).  The union of the shards' phase-2 writes is render_samples_ppm's text.  Also the phase state
through the raw C ABI, the one-device rule, and 2 and 3 processes through multi.SharedCanvas and multi.SharedText.  Run on the
B200 box: `pytest tests -m gpu`."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import ray_tracer_challenge_b200 as rt
from bench import WORKLOADS
from ray_tracer_challenge_b200 import scenes
from tests.test_gpu_shard_ppm import _own_mask, _pinned
from tests.test_gpu_views import SCENES

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BAND_ROWS = 8
SENTINEL = 0x7F  # DEL: no byte of a PPM text
UNWRITTEN = 0x7FBADBAD  # a NaN no render writes
U8_UNWRITTEN = 0xAB
RTC_ERR_INVALID, RTC_ERR_STATE = -1, -4
RAGGED = dict(width=333, height=123, u_steps=3, v_steps=2, jitter="constant")


@pytest.fixture(scope="module")
def gpu():
    api = rt.new_session()
    api.set_render_options(n_devices=1)  # a shard's scene is committed on one device
    return api


def _mine(h, shard, n_shards):
    return np.array([y // BAND_ROWS % n_shards == shard for y in range(h)])


def _planes(h, w):
    return np.full((h, w, 3), UNWRITTEN, np.uint32).view(np.float32), np.full((h, w, 3), U8_UNWRITTEN, np.uint8)


def _whole(p, n, fma=False):
    c = p.render_samples(n, 5, fma=fma)
    return c.data.copy(), c.to_u8().copy()


def _shard_rows_below_last(h, shard, n_shards):
    return int(_mine(h, shard, n_shards)[:h - 1].sum())


def _union(p, n, n_shards, fma=False, out_rgb=None, out_u8=None):
    """Shards 0..n_shards-1 of one prepared scene, each into sentinel-filled planes: its own pageable pair (checked to hold the
    sentinel outside its bands) or, given out_rgb / out_u8, the caller's shared pair.  Returns the union."""
    h, w = p.camera.height_pixels, p.camera.width_pixels
    rgb, u8 = _planes(h, w)
    if out_rgb is not None:
        out_rgb.view(np.uint32)[:] = UNWRITTEN
        out_u8[:] = U8_UNWRITTEN
    for s in range(n_shards):
        if out_rgb is not None:
            p.render_samples(n, 5, out_rgb=out_rgb, out_u8=out_u8, fma=fma, shard=s, n_shards=n_shards)
            continue
        srgb, su8 = _planes(h, w)
        p.render_samples(n, 5, out_rgb=srgb, out_u8=su8, fma=fma, shard=s, n_shards=n_shards)
        st = p.last_stats
        mine = _mine(h, s, n_shards)
        assert st.n_devices == 1 and (st.launches >= 1) == mine.any(), (s, n_shards, st.launches)  # a shard may own no band
        assert st.primary_rays == n * n * (w - 1) * _shard_rows_below_last(h, s, n_shards), (s, n_shards)
        assert (srgb[~mine].view(np.uint32) == UNWRITTEN).all(), (s, n_shards, "f32 row outside the shard")
        assert (su8[~mine] == U8_UNWRITTEN).all(), (s, n_shards, "8-bit row outside the shard")
        rgb[mine], u8[mine] = srgb[mine], su8[mine]
    if out_rgb is not None:
        return out_rgb, out_u8
    return rgb, u8


def _same(a, b):
    return np.array_equal(np.ascontiguousarray(a).view(np.uint32), np.ascontiguousarray(b).view(np.uint32))


@pytest.mark.parametrize("name", list(SCENES))
def test_shards_make_up_render_samples_on_every_kernel_path(gpu, name):
    """Lean table, lean drawn, general small, converging small, tree tiles, tree stream, sweep CSG; each FP build the scene
    lists; n = 1..4; N = 1, 2, 3, 8."""
    build, kw, _, fmas = SCENES[name]
    cam, world = build(gpu, **kw)
    p = cam.prepare(world)
    try:
        for fma in fmas:
            for n in (1, 2, 3, 4):
                want_rgb, want_u8 = _whole(p, n, fma)
                for n_shards in (1, 2, 3, 8):
                    rgb, u8 = _union(p, n, n_shards, fma)
                    assert _same(rgb, want_rgb), (name, fma, n, n_shards)
                    assert np.array_equal(u8, want_u8), (name, fma, n, n_shards)
    finally:
        p.release()


@pytest.mark.parametrize("size", ["ragged", "c3"])
def test_ragged_and_full_size_pinned_and_pageable(gpu, size):
    """A ragged frame at n = 3, and c3 (3840x2160) at n = 2, whose 100 MB pageable f32 plane is staged through pinned frames:
    every shard into its own pageable planes, and all of them into one pair of registered (pinned) planes."""
    if size == "c3":
        builder, kw, _, _ = WORKLOADS["c3"]
        cam, world = getattr(scenes, builder)(gpu, **kw)
        n = 2
    else:
        cam, world = scenes.soft_shadows(gpu, **RAGGED)
        n = 3
    h, w = cam.height_pixels, cam.width_pixels
    p = cam.prepare(world)
    lib, pin_rgb = _pinned(h * w * 12)
    _, pin_u8 = _pinned(h * w * 3)
    try:
        want_rgb, want_u8 = _whole(p, n)
        for n_shards in (2, 3, 8):
            rgb, u8 = _union(p, n, n_shards)
            assert _same(rgb, want_rgb) and np.array_equal(u8, want_u8), (size, n_shards, "pageable")
            rgb, u8 = _union(p, n, n_shards, out_rgb=pin_rgb.view(np.float32).reshape(h, w, 3), out_u8=pin_u8.reshape(h, w, 3))
            assert _same(rgb, want_rgb) and np.array_equal(u8, want_u8), (size, n_shards, "pinned")
        # one plane at a time, and the shard left on the device
        s_u8 = np.full((h, w, 3), U8_UNWRITTEN, np.uint8)
        p.render_samples(n, 5, want_rgb=False, out_u8=s_u8, shard=1, n_shards=3)
        mine = _mine(h, 1, 3)
        assert np.array_equal(s_u8[mine], want_u8[mine]) and (s_u8[~mine] == U8_UNWRITTEN).all()
        p.render_samples(n, 5, want_rgb=False, want_u8=False, shard=1, n_shards=3)
        assert p.last_stats.primary_rays == n * n * (w - 1) * _shard_rows_below_last(h, 1, 3)
    finally:
        lib.rtc_host_unregister(pin_rgb.ctypes.data)
        lib.rtc_host_unregister(pin_u8.ctypes.data)
        p.release()


def _sharded_text(gpu, cam, world, n, n_shards, fma=False, out=None):
    """The text n_shards shards write into one sentinel-filled buffer, each from its own prepared scene on device 0: every
    anti-aliased phase 1 into one row-length array, then every phase 2."""
    w, h = cam.width_pixels, cam.height_pixels
    bound = gpu.lib.rtc_ppm_bound(w, h)
    buf = np.empty(bound, np.uint8) if out is None else out
    buf[:] = SENTINEL
    row_bytes = np.zeros(h, np.uint64)
    shards = [cam.prepare(world) for _ in range(n_shards)]
    try:
        for s, p in enumerate(shards):
            p.render_shard_ppm_rows(s, n_shards, row_bytes, 5, fma=fma, samples=n)
            assert p.last_stats.primary_rays == n * n * (w - 1) * _shard_rows_below_last(h, s, n_shards)
        lengths = {p.write_shard_ppm(s, n_shards, row_bytes, buf) for s, p in enumerate(shards)}
        assert len(lengths) == 1, lengths
        length = lengths.pop()
        assert not (buf[:length] == SENTINEL).any() and (buf[length:] == SENTINEL).all()
        return buf[:length].tobytes().decode("ascii")
    finally:
        for p in shards:
            p.release()


@pytest.mark.parametrize("name", ["lean_table", "small_converging", "tree_stream"])
def test_shard_texts_make_up_render_samples_ppm(gpu, name):
    build, kw, _, fmas = SCENES[name]
    cam, world = build(gpu, **kw)
    p = cam.prepare(world)
    try:
        for fma in fmas:
            for n in (1, 2, 3):
                want = p.render_samples_ppm(n, 5, fma=fma)
                assert want == p.render_samples(n, 5, fma=fma).to_ppm()
                for n_shards in (1, 2, 3, 8):
                    assert _sharded_text(gpu, cam, world, n, n_shards, fma) == want, (name, fma, n, n_shards)
    finally:
        p.release()


def test_shard_texts_ragged_and_c3_pinned_and_pageable(gpu):
    """c3's 78 MB text at n = 2 reaches a pageable destination through the staging frame; the ragged frame's directly."""
    builder, kw, _, _ = WORKLOADS["c3"]
    for cam, world, n in ((*scenes.soft_shadows(gpu, **RAGGED), 3), (*getattr(scenes, builder)(gpu, **kw), 2)):
        p = cam.prepare(world)
        try:
            want = p.render_samples_ppm(n, 5)
        finally:
            p.release()
        lib, pinned = _pinned(gpu.lib.rtc_ppm_bound(cam.width_pixels, cam.height_pixels))
        try:
            for n_shards in (2, 8):
                assert _sharded_text(gpu, cam, world, n, n_shards) == want, (cam.width_pixels, n_shards, "pageable")
                assert _sharded_text(gpu, cam, world, n, n_shards, out=pinned) == want, (cam.width_pixels, n_shards, "pinned")
        finally:
            lib.rtc_host_unregister(pinned.ctypes.data)


def _abi():
    lib = rt.device_library()
    lib.rtc_last_error.restype = C.c_char_p
    lib.rtc_ppm_bound.restype = C.c_size_t
    lib.rtc_ppm_bound.argtypes = [C.c_uint32, C.c_uint32]
    lib.rtc_render_shard_samples.argtypes = [C.c_void_p, C.c_int32, C.c_uint32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                             C.c_void_p]
    lib.rtc_render_shard_samples_ppm_rows.argtypes = [C.c_void_p, C.c_int32, C.c_uint32, C.c_int32, C.c_int32, C.c_void_p,
                                                      C.c_void_p]
    lib.rtc_render_shard_ppm_rows.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    lib.rtc_write_shard_ppm.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t,
                                        C.POINTER(C.c_size_t)]
    lib.rtc_render.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.rtc_render_shard.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.rtc_render_samples.argtypes = [C.c_void_p, C.c_int32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.rtc_scene_commit.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
    lib.rtc_scene_destroy.argtypes = [C.c_void_p]
    return lib


def test_phase_state(gpu):
    """Phase 2 encodes the plane of the last phase 1, samples or plain; a plain rtc_render_shard or rtc_render_samples in
    between voids it; a wrong own-row entry is refused; a repeated phase 2 writes the same bytes."""
    lib = _abi()
    w, h, n = 96, 40, 3
    cam, world = scenes.soft_shadows(gpu, width=w, height=h, u_steps=2, v_steps=2)
    p = cam.prepare(world)
    try:
        want_aa, want_plain = p.render_samples_ppm(n, 5), p.render_ppm(5)
    finally:
        p.release()
    assert want_aa != want_plain
    scene = gpu.export_scene(cam, world)
    bound = lib.rtc_ppm_bound(w, h)
    buf = np.full(bound, SENTINEL, np.uint8)
    got = C.c_size_t(0)
    shard, n_shards = 1, 3
    own = [y for y in range(h) if y // BAND_ROWS % n_shards == shard]
    header = len(f"P3\n{w} {h}\n255\n")

    def aa_rows(s, rows):
        return lib.rtc_render_shard_samples_ppm_rows(scene, 5, n, s, n_shards, rows.ctypes.data, None)

    def plain_rows(s, rows):
        return lib.rtc_render_shard_ppm_rows(scene, 5, s, n_shards, rows.ctypes.data, None)

    def exchanged(phase1):
        """every shard's phase 1 into one array, shard `shard`'s last (its phase 1 is then the scene's)"""
        rows = np.zeros(h, np.uint64)
        for s in [x for x in range(n_shards) if x != shard] + [shard]:
            assert phase1(s, rows) == 0, lib.rtc_last_error()
        return rows

    def phase2(rows):
        buf[:] = SENTINEL
        return lib.rtc_write_shard_ppm(scene, shard, n_shards, rows.ctypes.data, buf.ctypes.data, bound, C.byref(got))

    def written_is(want, rows):
        mine = _own_mask(rows, header, shard, n_shards, bound)
        return got.value == len(want) and np.array_equal(buf != SENTINEL, mine) and \
            buf[mine].tobytes() == np.frombuffer(want.encode(), np.uint8)[mine[:len(want)]].tobytes()

    def refused(code, text, rc):
        assert rc == code, (rc, lib.rtc_last_error())
        assert text.encode() in lib.rtc_last_error(), lib.rtc_last_error()

    try:
        assert lib.rtc_scene_commit(scene, 1, (C.c_int32 * 1)(0)) == 0
        assert lib.rtc_render(scene, 5, None, None, None) == 0  # rtc_render's frame on the device: not what phase 2 encodes
        rows_aa = exchanged(aa_rows)
        assert (rows_aa >= 6 * w).all()
        for _ in range(2):  # repeated: the same bytes
            assert phase2(rows_aa) == 0, lib.rtc_last_error()
            assert written_is(want_aa, rows_aa)
        # a plain phase 1 after it: phase 2 encodes rtc_render_shard's plane again, and back
        rows_plain = exchanged(plain_rows)
        assert phase2(rows_plain) == 0 and written_is(want_plain, rows_plain)
        assert aa_rows(shard, rows_aa) == 0
        assert phase2(rows_aa) == 0 and written_is(want_aa, rows_aa)
        # a wrong own-row entry: a broken exchange
        for y in (own[0], own[-1]):
            bad = rows_aa.copy()
            bad[y] += np.uint64(1)
            refused(RTC_ERR_INVALID, f"row_bytes[{y}] = {int(bad[y])}", phase2(bad))
            assert (buf == SENTINEL).all()
        # a render of another kind in between voids the samples phase 1
        for between in (lambda: lib.rtc_render_shard(scene, 5, shard, n_shards, None, None, None),
                        lambda: lib.rtc_render_samples(scene, 5, n, None, None, None),
                        lambda: lib.rtc_render_shard_samples(scene, 5, n, shard, n_shards, None, None, None)):
            assert aa_rows(shard, rows_aa) == 0
            assert between() == 0, lib.rtc_last_error()
            refused(RTC_ERR_STATE, "needs rtc_render_shard_ppm_rows", phase2(rows_aa))
        # another shard's or shard count's phase 1
        assert aa_rows(0, np.zeros(h, np.uint64)) == 0
        refused(RTC_ERR_STATE, "needs rtc_render_shard_ppm_rows", phase2(rows_aa))
    finally:
        lib.rtc_scene_destroy(scene)


def test_a_scene_on_two_devices_is_refused(gpu):
    lib = _abi()
    if lib.rtc_device_count() < 2:
        pytest.skip("one GPU visible")
    cam, world = scenes.soft_shadows(gpu, width=64, height=32, u_steps=2, v_steps=2)
    scene = gpu.export_scene(cam, world)
    rows = np.zeros(32, np.uint64)
    try:
        assert lib.rtc_scene_commit(scene, 2, (C.c_int32 * 2)(0, 1)) == 0
        assert lib.rtc_render_shard_samples(scene, 5, 2, 0, 2, None, None, None) == RTC_ERR_STATE
        assert b"exactly one device" in lib.rtc_last_error()
        assert lib.rtc_render_shard_samples_ppm_rows(scene, 5, 2, 0, 2, rows.ctypes.data, None) == RTC_ERR_STATE
        assert b"exactly one device" in lib.rtc_last_error()
    finally:
        lib.rtc_scene_destroy(scene)


def _rank(rank, world_size, port, size, n, result_path):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world_size))
    import torch.distributed as dist

    import ray_tracer_challenge_b200 as rt
    from bench import WORKLOADS
    from ray_tracer_challenge_b200 import multi, scenes

    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    api = rt.new_session()
    lib = rt.device_library()
    lib.rtc_host_register.argtypes = [C.c_void_p, C.c_size_t]
    lib.rtc_host_unregister.argtypes = [C.c_void_p]
    api.set_render_options(device_ids=[rank % lib.rtc_device_count()])
    if size == "c3":
        builder, kw, _, _ = WORKLOADS["c3"]
        cam, world = getattr(scenes, builder)(api, **kw)
    else:
        cam, world = scenes.soft_shadows(api, **RAGGED)
    w, h = cam.width_pixels, cam.height_pixels
    prepared = cam.prepare(world)
    canvas = multi.open_shared_canvas(dist, rank, f"rtc_test_aa_canvas_{port}", w, h)
    text = multi.open_shared_text(dist, rank, f"rtc_test_aa_text_{port}", w, h)
    results = []
    try:
        for registered in (False, True):
            if registered:
                assert lib.rtc_host_register(canvas.address, canvas.nbytes) == 0
                assert lib.rtc_host_register(text.address, text.nbytes) == 0
            if rank == 0:
                canvas.rgb.view(np.uint32)[:] = UNWRITTEN
                canvas.u8[:] = U8_UNWRITTEN
                text.buf[:] = SENTINEL
            dist.barrier()
            multi.render_samples_shared(dist, rank, world_size, prepared, canvas, n, 5)
            length = multi.render_ppm_shared(dist, rank, world_size, prepared, text, 5, samples=n)
            lengths = [None] * world_size
            dist.all_gather_object(lengths, length)
            if rank == 0:
                want = prepared.render_samples(n, 5)
                frame_ok = np.array_equal(canvas.rgb.view(np.uint32), want.data.view(np.uint32)) and \
                    np.array_equal(canvas.u8, want.to_u8())
                text_ok = len(set(lengths)) == 1 and text.text(length) == prepared.render_samples_ppm(n, 5) and \
                    (text.buf[length:] == SENTINEL).all()
                results.append(f"{'registered' if registered else 'unregistered'}:frame {'ok' if frame_ok else 'mismatch'}:"
                               f"text {'ok' if text_ok else 'mismatch'}")
            dist.barrier()
            if registered:
                lib.rtc_host_unregister(canvas.address)
                lib.rtc_host_unregister(text.address)
        if rank == 0:
            with open(result_path, "w") as fh:
                fh.write(" ".join(results))
    finally:
        prepared.release()
        canvas.close()
        text.close()
        dist.destroy_process_group()


@pytest.mark.timeout(900)
@pytest.mark.parametrize("world_size", [2, 3])
def test_processes_through_shared_canvas_and_text(world_size, tmp_path):
    """world_size processes (gloo; each commits device rank % device_count, so on one GPU they share it) write one anti-aliased
    frame through multi.SharedCanvas and its text through multi.SharedText, registered with rtc_host_register and not; rank 0
    compares them with the single-process render_samples and render_samples_ppm."""
    import torch.multiprocessing as mp

    for size, n in (("ragged", 3), ("c3", 2)):
        port = 29500 + (os.getpid() + 11 * world_size + len(size)) % 2000
        result = tmp_path / f"result_{size}.txt"
        mp.spawn(_rank, args=(world_size, port, size, n, str(result)), nprocs=world_size, join=True)
        want = "unregistered:frame ok:text ok registered:frame ok:text ok"
        assert result.read_text() == want, (world_size, size)
