"""One frame's PPM text written by several processes, one shard each, on the GPU (rtc_render_shard_ppm_rows, then the callers'
exchange of row lengths, then rtc_write_shard_ppm).  The union of the shards' writes is byte for byte rtc_render_ppm's text of
the same scene: in one process with one prepared scene per shard (the parity scenes, the oracle, both FP builds, a ragged frame
and full-size c3, pinned and pageable destinations), and in 2 and 3 processes through multi.SharedText and
multi.render_ppm_shared.  Each shard writes exactly its bands (shard 0 also the header).  Also the phase state, the own-row
check and the one-device rule, through the raw C ABI.  Run on the B200 box: `pytest tests -m gpu`."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import ray_tracer_challenge_b200 as rt
from ray_tracer_challenge_b200 import scenes
from tests.test_gpu_parity import SCENES

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BAND_ROWS = 8
SENTINEL = 0x7F  # DEL: no byte of a PPM text
RTC_ERR_INVALID, RTC_ERR_STATE = -1, -4
C3 = dict(width=3840, height=2160, u_steps=4, v_steps=4)


@pytest.fixture(scope="module")
def gpu():
    api = rt.new_session()
    api.set_render_options(n_devices=1)  # a shard's scene is committed on one device
    return api


def _bound(gpu, cam):
    return gpu.lib.rtc_ppm_bound(cam.width_pixels, cam.height_pixels)


def _single(cam, world, fma=False):
    p = cam.prepare(world)
    try:
        return p.render_ppm(5, fma=fma)
    finally:
        p.release()


def _pinned(nbytes):
    """A NumPy buffer page-locked with rtc_host_register (it stays valid after rtc_host_unregister, unlike freed pinned memory
    a failing assertion's traceback could still show)."""
    lib = rt.device_library()
    lib.rtc_host_register.argtypes = [C.c_void_p, C.c_size_t]
    lib.rtc_host_unregister.argtypes = [C.c_void_p]
    buf = np.empty(nbytes, np.uint8)
    assert lib.rtc_host_register(buf.ctypes.data, nbytes) == 0
    return lib, buf


def _own_mask(row_bytes, header, shard, n_shards, size):
    """The bytes shard `shard` may write: its rows' texts (placed by every row's length) and, for shard 0, the header."""
    mine = np.zeros(size, bool)
    at = header + np.concatenate([[0], np.cumsum(row_bytes.astype(np.int64))])
    if shard == 0:
        mine[:header] = True
    for y in range(len(row_bytes)):
        if y // BAND_ROWS % n_shards == shard:
            mine[at[y]:at[y + 1]] = True
    return mine


def _sharded(gpu, cam, world, n_shards, out=None, fma=False, regions=False):
    """The text n_shards shards write into one buffer (out, or a new pageable one), each from its own prepared scene on device 0:
    every phase 1 into one row-length array, then every phase 2.  regions: each shard also writes alone into a buffer of the
    sentinel, which must then differ from it exactly on that shard's bytes."""
    w, h = cam.width_pixels, cam.height_pixels
    bound = gpu.lib.rtc_ppm_bound(w, h)
    buf = np.empty(bound, np.uint8) if out is None else out
    buf[:] = SENTINEL
    row_bytes = np.zeros(h, np.uint64)
    shards = [cam.prepare(world) for _ in range(n_shards)]
    try:
        for s, p in enumerate(shards):
            p.render_shard_ppm_rows(s, n_shards, row_bytes, 5, fma=fma)
            assert p.last_stats.n_devices == 1
        assert (row_bytes >= 6 * w).all() and (row_bytes <= 12 * w).all()
        lengths = {p.write_shard_ppm(s, n_shards, row_bytes, buf) for s, p in enumerate(shards)}
        assert len(lengths) == 1, lengths
        n = lengths.pop()
        header = len(f"P3\n{w} {h}\n255\n")
        assert n == header + int(row_bytes.sum())
        assert not (buf[:n] == SENTINEL).any() and (buf[n:] == SENTINEL).all()
        if regions:
            for s, p in enumerate(shards):  # phase 2 again, alone, into a fresh buffer
                alone = np.full(bound, SENTINEL, np.uint8)
                assert p.write_shard_ppm(s, n_shards, row_bytes, alone) == n
                mine = _own_mask(row_bytes, header, s, n_shards, bound)
                assert np.array_equal(alone != SENTINEL, mine), (s, n_shards)
                assert np.array_equal(alone[mine], buf[mine])
        return buf[:n].tobytes().decode("ascii")
    finally:
        for p in shards:
            p.release()


@pytest.mark.parametrize("name", sorted(SCENES))
def test_parity_scenes(gpu, name):
    build, kw = SCENES[name]
    cam, world = build(gpu, **kw)
    want = _single(cam, world)
    for n_shards in (1, 2, 3, 8):
        assert _sharded(gpu, cam, world, n_shards, regions=n_shards in (3, 8)) == want, (name, n_shards)


def test_equals_the_oracle(gpu, oracle):
    kw = dict(width=160, height=64, u_steps=4, v_steps=4)
    cam, world = scenes.soft_shadows(gpu, **kw)
    ocam, oworld = scenes.soft_shadows(oracle, **kw)
    want = ocam.render(oworld, 5).to_ppm()
    for n_shards in (2, 3):
        assert _sharded(gpu, cam, world, n_shards) == want, n_shards


def test_both_fp_builds(gpu):
    cam, world = scenes.reflect_refract(gpu, width=320, height=160)
    for fma in (False, True):
        want = _single(cam, world, fma=fma)
        for n_shards in (2, 3):
            assert _sharded(gpu, cam, world, n_shards, fma=fma) == want, (fma, n_shards)


@pytest.mark.parametrize("size", ["ragged", "c3"])
def test_ragged_and_full_size_pinned_and_pageable(gpu, size):
    """c3's 78 MB text is staged into a pageable destination piece by piece; the ragged frame's 0.5 MB is copied directly."""
    kw = dict(ragged=dict(width=333, height=123, u_steps=3, v_steps=2, jitter="constant"), c3=C3)[size]
    cam, world = scenes.soft_shadows(gpu, **kw)
    want = _single(cam, world)
    lib, pinned = _pinned(_bound(gpu, cam))
    try:
        for n_shards in (2, 3, 8):
            assert _sharded(gpu, cam, world, n_shards, out=pinned, regions=size == "ragged") == want, (size, n_shards, "pinned")
            assert _sharded(gpu, cam, world, n_shards) == want, (size, n_shards, "pageable")
    finally:
        lib.rtc_host_unregister(pinned.ctypes.data)


def _abi():
    lib = rt.device_library()
    lib.rtc_last_error.restype = C.c_char_p
    lib.rtc_ppm_bound.restype = C.c_size_t
    lib.rtc_ppm_bound.argtypes = [C.c_uint32, C.c_uint32]
    lib.rtc_render_shard_ppm_rows.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    lib.rtc_write_shard_ppm.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t,
                                        C.POINTER(C.c_size_t)]
    lib.rtc_render_ppm.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t), C.c_void_p]
    lib.rtc_render.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.rtc_render_shard.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.rtc_set_option.argtypes = [C.c_void_p, C.c_int32, C.c_int64]
    lib.rtc_scene_commit.argtypes = [C.c_void_p, C.c_int32, C.c_void_p]
    lib.rtc_scene_destroy.argtypes = [C.c_void_p]
    return lib


def test_phase_state_and_the_own_row_check(gpu):
    lib = _abi()
    cam, world = scenes.soft_shadows(gpu, width=96, height=40, u_steps=2, v_steps=2)
    w, h = 96, 40
    want = _single(cam, world)
    scene = gpu.export_scene(cam, world)
    bound = lib.rtc_ppm_bound(w, h)
    buf = np.full(bound, SENTINEL, np.uint8)
    n = C.c_size_t(0)
    shard, n_shards = 1, 3  # rows 8-15 (band 1) and 32-39 (band 4)
    own = [y for y in range(h) if y // BAND_ROWS % n_shards == shard]
    header = len(f"P3\n{w} {h}\n255\n")

    def phase1(s=shard, k=n_shards, rows=None):
        return lib.rtc_render_shard_ppm_rows(scene, 5, s, k, (rows if rows is not None else row_bytes).ctypes.data, None)

    def phase2(s=shard, k=n_shards, rows=None):
        return lib.rtc_write_shard_ppm(scene, s, k, (rows if rows is not None else row_bytes).ctypes.data, buf.ctypes.data, bound,
                                       C.byref(n))

    def refused(code, text, rc):
        assert rc == code, (rc, lib.rtc_last_error())
        assert text.encode() in lib.rtc_last_error(), lib.rtc_last_error()

    try:
        assert lib.rtc_scene_commit(scene, 1, (C.c_int32 * 1)(0)) == 0
        # every row's length, as the exchange would gather it: shards 0 and 2 from their own phase 1
        row_bytes = np.zeros(h, np.uint64)
        refused(RTC_ERR_STATE, "needs rtc_render_shard_ppm_rows", phase2(rows=np.full(h, 9 * w, np.uint64)))  # no phase 1
        assert phase1() == 0, lib.rtc_last_error()
        assert (row_bytes[[y for y in range(h) if y not in own]] == 0).all()  # other shards' entries untouched
        for other in (0, 2):
            rows = np.zeros(h, np.uint64)
            assert phase1(s=other, rows=rows) == 0
            row_bytes[[y for y in range(h) if y // BAND_ROWS % n_shards == other]] = \
                rows[[y for y in range(h) if y // BAND_ROWS % n_shards == other]]
        # the scene now holds shard 2's phase 1
        refused(RTC_ERR_STATE, "needs rtc_render_shard_ppm_rows", phase2())
        refused(RTC_ERR_STATE, "needs rtc_render_shard_ppm_rows", phase2(k=4))
        assert phase1() == 0
        refused(RTC_ERR_STATE, "needs rtc_render_shard_ppm_rows", phase2(s=2))
        refused(RTC_ERR_STATE, "needs rtc_render_shard_ppm_rows", phase2(k=2, s=1))
        # an altered own-row entry: a broken exchange, refused and nothing written
        for y in (own[0], own[-1]):  # (the last row is never rendered: 6 * width, the least a row can take)
            bad = row_bytes.copy()
            bad[y] += np.uint64(1)
            refused(RTC_ERR_INVALID, f"row_bytes[{y}] = {int(bad[y])}", phase2(rows=bad))
            assert b"exchange" in lib.rtc_last_error()
        assert (buf == SENTINEL).all()
        # a failed phase 2 changes nothing: the right one still works, and may be repeated
        for _ in range(2):
            assert phase2() == 0, lib.rtc_last_error()
            assert n.value == len(want)
            mine = _own_mask(row_bytes, header, shard, n_shards, bound)
            assert np.array_equal(buf != SENTINEL, mine)
            assert buf[mine].tobytes() == np.frombuffer(want.encode(), np.uint8)[mine[:len(want)]].tobytes()
        # a render, an option or a commit in between voids the pending phase 2
        for between in (lambda: lib.rtc_render(scene, 5, None, None, None),
                        lambda: lib.rtc_render_shard(scene, 5, shard, n_shards, None, None, None),
                        lambda: lib.rtc_set_option(scene, 1, 0),
                        lambda: lib.rtc_scene_commit(scene, 1, (C.c_int32 * 1)(0))):
            assert phase1() == 0
            assert between() == 0, lib.rtc_last_error()
            refused(RTC_ERR_STATE, "needs rtc_render_shard_ppm_rows", phase2())
        # the frame stays renderable: the whole text and a fresh pair of phases
        text = np.zeros(bound, np.uint8)
        assert lib.rtc_render_ppm(scene, 5, text.ctypes.data, bound, C.byref(n), None) == 0
        assert text[:n.value].tobytes().decode("ascii") == want
        assert phase1() == 0 and phase2() == 0
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
        assert lib.rtc_render_shard_ppm_rows(scene, 5, 0, 2, rows.ctypes.data, None) == RTC_ERR_STATE
        assert b"exactly one device" in lib.rtc_last_error()
    finally:
        lib.rtc_scene_destroy(scene)


def _rank(rank, world_size, port, kw, result_path):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world_size))
    import torch.distributed as dist

    import ray_tracer_challenge_b200 as rt
    from ray_tracer_challenge_b200 import multi, scenes

    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    api = rt.new_session()
    lib = rt.device_library()
    api.set_render_options(device_ids=[rank % lib.rtc_device_count()])
    cam, world = scenes.soft_shadows(api, **kw)
    prepared = cam.prepare(world)
    text = multi.open_shared_text(dist, rank, f"rtc_test_text_{port}", cam.width_pixels, cam.height_pixels)
    results = []
    try:
        for registered in (False, True):
            if registered:
                lib.rtc_host_register.argtypes = [C.c_void_p, C.c_size_t]
                assert lib.rtc_host_register(text.address, text.nbytes) == 0
            if rank == 0:
                text.buf[:] = SENTINEL
            dist.barrier()
            length = multi.render_ppm_shared(dist, rank, world_size, prepared, text, 5)
            lengths = [None] * world_size
            dist.all_gather_object(lengths, length)
            if rank == 0:
                want = prepared.render_ppm(5)
                ok = (len(set(lengths)) == 1 and text.text(length) == want and (text.buf[length:] == SENTINEL).all())
                results.append(f"{'registered' if registered else 'unregistered'}:{'ok' if ok else 'mismatch'}")
            dist.barrier()
            if registered:
                lib.rtc_host_unregister.argtypes = [C.c_void_p]
                lib.rtc_host_unregister(text.address)
        if rank == 0:
            with open(result_path, "w") as fh:
                fh.write(" ".join(results))
    finally:
        prepared.release()
        text.close()
        dist.destroy_process_group()


@pytest.mark.timeout(600)
@pytest.mark.parametrize("world_size", [2, 3])
def test_processes_through_shared_text(world_size, tmp_path):
    """world_size processes (gloo; each commits device rank % device_count, so on one GPU they share it) write one frame's
    text through multi.SharedText, registered with rtc_host_register and not; rank 0 compares it with render_ppm."""
    import torch.multiprocessing as mp

    for size, kw in (("small", dict(width=333, height=123, u_steps=3, v_steps=2)), ("c3", C3)):
        port = 29500 + (os.getpid() + 7 * world_size + len(size)) % 2000
        result = tmp_path / f"result_{size}.txt"
        mp.spawn(_rank, args=(world_size, port, kw, str(result)), nprocs=world_size, join=True)
        assert result.read_text() == "unregistered:ok registered:ok", (world_size, size)
