"""The lean kernel build of small scenes (SmallScene::lean: an area light on the cell-mask loops, no pattern and no
transparency on any table item) without a GPU: which scenes the commit marks lean, and World::color_at through the lean
build (tests/emu/emu_lean.cpp: the device code compiled for the host) against the oracle, bit for bit."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from ray_tracer_challenge_b200 import scenes
from tests.test_device_code_on_host import FP, _build


@pytest.fixture(scope="module")
def host():
    import ray_tracer_challenge_b200 as rt

    return rt.new_session()


@pytest.fixture(scope="module")
def emu_lean(tmp_path_factory):
    device, lib = _build(tmp_path_factory, "emu_lean.cpp")
    lib.emu_lean_color_at.argtypes = [C.c_void_p, C.c_uint32, FP, FP, C.c_int, FP]
    return device, lib


def test_commit_marks_lean_scenes(host, monkeypatch):
    from bench import build_scene

    for workload in ("c1", "c3", "c3_counter"):
        cam, world, _, _ = build_scene(host, workload)
        p = host.inspect(cam, world)
        assert (p["cell_masks"], p["lean"]) == (1, 1), (workload, p)
    # c2: cylinder, cone, glass and a striped floor
    cam, world, _, _ = build_scene(host, "c2")
    assert host.inspect(cam, world)["lean"] == 0
    # filter_zoo: cell masks, but a checkered floor and a transparent ghost sphere
    for jitter in ("table", None):
        cam, world = scenes.filter_zoo(host, width=64, height=40, jitter=jitter)
        p = host.inspect(cam, world)
        assert (p["cell_masks"], p["lean"]) == (1, 0), (jitter, p)
    # a point light never takes the cell-mask loops
    cam, world = scenes.filter_zoo(host, width=64, height=40, area_light=False)
    assert host.inspect(cam, world)["lean"] == 0
    # RTC_LEAN=0 (read on every commit) keeps a lean scene on the general build
    monkeypatch.setenv("RTC_LEAN", "0")
    cam, world, _, _ = build_scene(host, "c3")
    p = host.inspect(cam, world)
    assert (p["cell_masks"], p["lean"]) == (1, 0), p


def _frame_rays(oracle, ocam):
    """Camera rays of every rendered pixel; ray i is pixel i (the never-rendered border traces nothing)."""
    w, h = ocam.width_pixels, ocam.height_pixels
    o = np.zeros((w * h, 3), np.float32)
    d = np.zeros((w * h, 3), np.float32)
    o[:, 1], d[:, 1] = 1.0e6, 1.0
    for y in range(h - 1):
        for x in range(w - 1):
            ro, rd = oracle.probe.camera_ray(ocam, x, y)
            o[y * w + x], d[y * w + x] = ro[:3], rd[:3]
    return o, d


def _check_frame(label, make, kw, emu_lean, host, oracle):
    device, lib = emu_lean
    cam, world = make(host, **kw)
    if not host.inspect(cam, world)["lean"]:
        return False
    ocam, oworld = make(oracle, **kw)
    want = np.asarray(ocam.render(oworld, 5).data, np.float32)
    w, h = ocam.width_pixels, ocam.height_pixels
    o, d = _frame_rays(oracle, ocam)
    scene = host.export_scene(cam, world)
    try:
        rgb = np.zeros((w * h, 3), np.float32)
        rc = lib.emu_lean_color_at(scene, w * h, o.ctypes.data_as(FP), d.ctypes.data_as(FP), 5, rgb.ctypes.data_as(FP))
        assert rc == 0, device.rtc_last_error()
        got = rgb.reshape(h, w, 3)[: h - 1, : w - 1]
        ref = want[: h - 1, : w - 1]
        same = (got.view(np.uint32) == ref.view(np.uint32)).all(axis=2)
        assert same.all(), (label, int((~same).sum()), got[~same][:2], ref[~same][:2])
        rays = (C.c_ulonglong * 4)()
        lib.emu_last_rays(rays)
        st = ocam.last_stats
        assert (rays[1], rays[2], rays[3]) == (st.secondary_rays, st.shadow_rays, st.shades), (label, list(rays), st.as_dict())
    finally:
        device.rtc_scene_destroy(scene)
    return True


@pytest.mark.parametrize("name,kw", [
    ("table_16_cells", dict(width=48, height=24, u_steps=4, v_steps=4)),
    ("table_100_cells", dict(width=40, height=16)),
    ("drawn_as_shipped", dict(width=40, height=16, jitter=None, seed=3)),
    ("drawn_16_cells", dict(width=48, height=24, u_steps=4, v_steps=4, jitter=None, seed=7)),
])
def test_lean_color_at_of_soft_shadows_matches_oracle(name, kw, emu_lean, host, oracle):
    """Whole small frames of the soft-shadow scene (c1 / c3 / c3_counter in miniature) through the lean build: f32 equal
    to the oracle's Camera::render bit for bit, and the same secondary rays, shadow rays and shades."""
    assert _check_frame(name, scenes.soft_shadows, kw, emu_lean, host, oracle), "soft_shadows was meant to be lean"


def test_lean_color_at_of_random_scenes_matches_oracle(emu_lean, host, oracle):
    """Random filter-eligible scenes (sheared / squashed spheres, tilted planes, boxes, non-casters, table or counter
    jitter): those the commit marks lean, through the lean build, equal the oracle's frames bit for bit."""
    lean = sum(_check_frame(seed, lambda rt, **kw: scenes.random_filter_scene(rt, seed, **kw), dict(width=28, height=18),
                            emu_lean, host, oracle) for seed in range(100, 124))
    assert lean >= 8, lean


def test_lean_build_under_address_sanitizer():
    """This module again in a child process whose harness is built with -fsanitize=address,undefined: the lean bounce
    stack and the shared-memory carving under AddressSanitizer + UBSan (see test_device_code_under_address_sanitizer)."""
    if os.environ.get("RTC_EMU_SANITIZE"):
        pytest.skip("already inside the sanitized run")
    libasan = subprocess.run(["g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not libasan or not os.path.exists(libasan):
        pytest.skip("no libasan")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, RTC_EMU_SANITIZE="1", LD_PRELOAD=libasan, ASAN_OPTIONS="detect_leaks=0:abort_on_error=1",
               UBSAN_OPTIONS="print_stacktrace=1:halt_on_error=1")
    proc = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-p", "no:cacheprovider"],
                          cwd=root, env=env, capture_output=True, text=True)
    tail = (proc.stdout + proc.stderr)[-3000:]
    assert proc.returncode == 0, tail
    assert "passed" in proc.stdout and "AddressSanitizer" not in tail and "runtime error" not in tail, tail
