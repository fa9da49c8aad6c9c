"""CSG trees beyond the whole-tree evaluator's limits (more than 32 worst-case hits, more than 5 nesting levels) are
evaluated by csg_sweep (dev_bvh.cuh), whose memory does not depend on the size of the tree.  On the host: the commit
accepts the book's die, a carved mesh and a 40-sphere union chain and refuses what is beyond the sweep's own caps; the
device code, compiled for the host (tests/emu), gives the oracle's nearest hits and colours bit for bit on those scenes,
and with RTC_CSG_SWEEP=1 (every CSG through the sweep) on the CSG scenes the whole-tree evaluator handles."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import ray_tracer_challenge_b200 as rt_pkg
from ray_tracer_challenge_b200 import scenes
from ray_tracer_challenge_b200.scenes import CSG_UNION, Material
from tests.test_device_code_on_host import FP, ROOT, _build, _raw_scene, _rays

RTC_ERR_CAPACITY = -3


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    device, lib = _build(tmp_path_factory, "emu_nearest.cpp")
    lib.emu_nearest.argtypes = [C.c_void_p, C.c_uint32, FP, FP, FP, C.POINTER(C.c_int32)]
    return device, lib


@pytest.fixture(scope="module")
def emu_color(tmp_path_factory):
    device, lib = _build(tmp_path_factory, "emu_color.cpp")
    lib.emu_color_at.argtypes = [C.c_void_p, C.c_uint32, FP, FP, C.c_int, C.c_int, C.c_int, FP, FP, C.POINTER(C.c_int32)]
    return device, lib


def _build_small_pass(tmp_path_factory, source, hits_per_pass):
    """The harness with csg_sweep taking `hits_per_pass` hits per pass instead of 32: every ray that meets a swept CSG
    then needs several passes, so the cursor, the state carried across passes and the early stops are all exercised."""
    device, _ = _build(tmp_path_factory, source)  # checks the toolchain and loads the device library
    out = tmp_path_factory.mktemp("emu_pass") / ("lib" + source.replace(".cpp", ".so"))
    lib_dir = os.path.dirname(rt_pkg.LIB_DEVICE)
    sanitize = ["-fsanitize=address,undefined", "-fno-omit-frame-pointer", "-fno-sanitize-recover=undefined"] \
        if os.environ.get("RTC_EMU_SANITIZE") else []
    subprocess.run(["g++", "-std=c++17", "-O1", "-ffp-contract=off", "-fPIC", "-shared", *sanitize, f"-DRTC_CSG_SWEEP_PASS={hits_per_pass}",
                    "-I", "/usr/local/cuda/include", "-I", os.path.join(ROOT, "ray_tracer_challenge_b200", "csrc"),
                    os.path.join(ROOT, "tests", "emu", source), "-o", str(out), "-L", lib_dir, "-lrtc_b200",
                    f"-Wl,-rpath,{lib_dir}"], check=True)
    return device, C.CDLL(str(out))


@pytest.fixture(scope="module")
def emu_pass3(tmp_path_factory):
    device, lib = _build_small_pass(tmp_path_factory, "emu_nearest.cpp", 3)
    lib.emu_nearest.argtypes = [C.c_void_p, C.c_uint32, FP, FP, FP, C.POINTER(C.c_int32)]
    return device, lib


@pytest.fixture(scope="module")
def emu_color_pass3(tmp_path_factory):
    device, lib = _build_small_pass(tmp_path_factory, "emu_color.cpp", 3)
    lib.emu_color_at.argtypes = [C.c_void_p, C.c_uint32, FP, FP, C.c_int, C.c_int, C.c_int, FP, FP, C.POINTER(C.c_int32)]
    return device, lib


@pytest.fixture(scope="module")
def host():
    return rt_pkg.new_session()


NEW_SCENES = {
    "die": (scenes.csg_die, dict(width=64, height=40)),
    "die_glass_area": (scenes.csg_die, dict(width=64, height=40, glassy=True, area_light=True)),
    "die_surrounded_glass": (scenes.csg_die, dict(width=64, height=40, glassy=True, surrounded=True)),
    "die_surrounded_area": (scenes.csg_die, dict(width=64, height=40, area_light=True, surrounded=True)),
    "carved_mesh": (scenes.csg_carved_mesh, dict(width=64, height=40)),
    "chain": (scenes.csg_chain, dict(width=64, height=40)),
}
# scenes the whole-tree evaluator accepts, rendered with every CSG sent to the sweep
SWEPT_SCENES = {
    "csg_gallery": (scenes.csg_gallery, dict(width=64, height=40)),
    "reflect_refract_csg": (scenes.reflect_refract, dict(width=64, height=32, with_csg=True)),
    "stress": (scenes.stress, dict(width=64, height=36, n_spheres=1500, n_each=6, n_csg=6)),
}


def _inspect_rc(device, host, cam, world):
    scene = host.export_scene(cam, world)
    try:
        rc = device.rtc_scene_inspect(scene, C.byref(rt_pkg.RtcCommitInfo()))
        return rc, device.rtc_last_error().decode()
    finally:
        device.rtc_scene_destroy(scene)


def _spheres(host, n):
    return [host.Sphere.build(host.translation(0.1 * i, 0.0, 0.0), Material()) for i in range(n)]


def _world(host, objects):
    cam = host.Camera(16, 8, scenes.PI / 2.0, host.view_transform((0, 0, -5), (0, 0, 0), (0, 1, 0)))
    return cam, host.World(objects, host.PointLight((-10, 10, -10), (1, 1, 1)))


@pytest.mark.parametrize("name", sorted(NEW_SCENES))
def test_commit_accepts_scenes_beyond_the_whole_tree_limits(name, host):
    make, kw = NEW_SCENES[name]
    info = host.inspect(*make(host, **kw))
    assert info["n_positions"] > 0
    # the surrounded die is a tree scene; the others are small scenes
    assert (info["small_n"] == 0) == name.startswith("die_surrounded"), info


def test_commit_refuses_beyond_the_sweep_caps(emu, host):
    device, _ = emu
    # nesting: a union chain of 64 spheres nests 63 levels (accepted), of 65 spheres 64 levels
    rc, _ = _inspect_rc(device, host, *_world(host, [scenes._union_chain(host, _spheres(host, 64))]))
    assert rc == 0
    rc, msg = _inspect_rc(device, host, *_world(host, [scenes._union_chain(host, _spheres(host, 65))]))
    assert rc == RTC_ERR_CAPACITY and "CSG nesting depth 64 exceeds 63" in msg, (rc, msg)

    # size: a balanced tree of 1025 CSG nodes (1026 leaves, nesting 11) is refused, 1024 nodes are accepted
    def balanced(shapes):
        while len(shapes) > 1:
            shapes = [host.CSG(CSG_UNION, shapes[i], shapes[i + 1]) if i + 1 < len(shapes) else shapes[i]
                      for i in range(0, len(shapes), 2)]
        return shapes[0]

    rc, msg = _inspect_rc(device, host, *_world(host, [balanced(_spheres(host, 1025))]))
    assert rc == 0, msg
    rc, msg = _inspect_rc(device, host, *_world(host, [balanced(_spheres(host, 1026))]))
    assert rc == RTC_ERR_CAPACITY and "1025 CSG nodes" in msg and "1024" in msg, (rc, msg)


def _nearest_matches_oracle(device, lib, host, oracle, make, kw, n=600):
    cam, world = make(host, **kw)
    ocam, oworld = make(oracle, **kw)
    scene = _raw_scene(device, host, world)
    try:
        o, d = _rays(oracle, ocam, n, seed=7)
        t = np.zeros(n, np.float32)
        prim = np.zeros(n, np.int32)
        rc = lib.emu_nearest(scene, n, o.ctypes.data_as(FP), d.ctypes.data_as(FP), t.ctypes.data_as(FP),
                             prim.ctypes.data_as(C.POINTER(C.c_int32)))
        assert rc == 0, device.rtc_last_error()
        hits = 0
        for i in range(n):
            ts, _ = oracle.probe.world_intersect(oworld, o[i], d[i], cap=4096)
            h = oracle.probe.hit_index(ts)
            want = np.float32(ts[h]) if h >= 0 else np.float32(-1.0)
            assert t[i] == want, (i, float(t[i]), float(want), o[i], d[i])  # bit-exact: same IEEE expression order
            hits += h >= 0
        assert hits > n // 10, hits
        return t, prim
    finally:
        device.rtc_scene_destroy(scene)


@pytest.mark.parametrize("name", sorted(NEW_SCENES))
def test_nearest_hit_matches_oracle(name, emu, host, oracle):
    device, lib = emu
    make, kw = NEW_SCENES[name]
    _nearest_matches_oracle(device, lib, host, oracle, make, kw)


@pytest.mark.parametrize("name", sorted(SWEPT_SCENES))
def test_nearest_hit_through_the_sweep_matches_oracle(name, emu, host, oracle, monkeypatch):
    device, lib = emu
    make, kw = SWEPT_SCENES[name]
    t0, p0 = _nearest_matches_oracle(device, lib, host, oracle, make, kw)
    monkeypatch.setenv("RTC_CSG_SWEEP", "1")
    t1, p1 = _nearest_matches_oracle(device, lib, host, oracle, make, kw)
    assert (t0.view(np.uint32) == t1.view(np.uint32)).all() and (p0 == p1).all()


def _color_matches_oracle(device, lib, host, oracle, make, kw, small, n=240):
    cam, world = make(host, **kw)
    ocam, oworld = make(oracle, **kw)
    scene = host.export_scene(cam, world)
    try:
        o, d = _rays(oracle, ocam, n, seed=11)
        want = np.array([oracle.probe.color_at(oworld, o[i], d[i], 5) for i in range(n)], np.float32)
        assert np.abs(want).sum() > 0
        for use_filter, converge in (((0, 0), (1, 1)) if small else ((0, 0), (0, 1))):
            lib.emu_set_converge(converge)
            rgb = np.zeros((n, 3), np.float32)
            path = C.c_int32(-1)
            rc = lib.emu_color_at(scene, n, o.ctypes.data_as(FP), d.ctypes.data_as(FP), 5, int(small), use_filter,
                                  rgb.ctypes.data_as(FP), None, C.byref(path))
            assert rc == 0, device.rtc_last_error()
            assert path.value == (1 if small else 0) or not small
            same = (rgb.view(np.uint32) == want.view(np.uint32)).all(axis=1)
            assert same.all(), (use_filter, converge, int((~same).sum()), rgb[~same][:3], want[~same][:3])
    finally:
        lib.emu_set_converge(0)
        device.rtc_scene_destroy(scene)


@pytest.mark.parametrize("small", [True, False], ids=["small_path", "tree_path"])
@pytest.mark.parametrize("name", sorted(NEW_SCENES))
def test_color_at_matches_oracle_bit_for_bit(name, small, emu_color, host, oracle):
    """World::color_at through the device code, including the glass variants' n1 / n2 container walk over swept CSGs."""
    device, lib = emu_color
    make, kw = NEW_SCENES[name]
    if small and name.startswith("die_surrounded"):
        pytest.skip("a tree scene: there is no small path to take")
    _color_matches_oracle(device, lib, host, oracle, make, kw, small)


@pytest.mark.parametrize("name", sorted(SWEPT_SCENES))
def test_color_at_through_the_sweep_matches_oracle(name, emu_color, host, oracle, monkeypatch):
    device, lib = emu_color
    make, kw = SWEPT_SCENES[name]
    monkeypatch.setenv("RTC_CSG_SWEEP", "1")
    small = host.inspect(*make(host, **kw))["small_n"] > 0
    _color_matches_oracle(device, lib, host, oracle, make, kw, small)


@pytest.mark.parametrize("name", sorted(NEW_SCENES) + ["sweep_" + k for k in sorted(SWEPT_SCENES)])
def test_several_passes_per_ray_match_oracle(name, emu_pass3, emu_color_pass3, host, oracle, monkeypatch):
    """Three hits per pass: nearest hits and colours are still the oracle's, bit for bit."""
    if name.startswith("sweep_"):
        monkeypatch.setenv("RTC_CSG_SWEEP", "1")
        make, kw = SWEPT_SCENES[name[len("sweep_"):]]
    else:
        make, kw = NEW_SCENES[name]
    _nearest_matches_oracle(*emu_pass3, host, oracle, make, kw, n=300)
    small = host.inspect(*make(host, **kw))["small_n"] > 0
    _color_matches_oracle(*emu_color_pass3, host, oracle, make, kw, small, n=120)


def test_sweep_ends_on_nan_and_infinite_rays(emu, host):
    """A NaN distance is never delivered and the cursor always moves forward: rays with NaN or infinite components
    through swept CSGs come back (a miss or some hit), they do not loop."""
    device, lib = emu
    for make, kw in (NEW_SCENES["chain"], NEW_SCENES["carved_mesh"], NEW_SCENES["die_surrounded_glass"]):
        cam, world = make(host, **kw)
        scene = _raw_scene(device, host, world)
        try:
            nan, inf = np.float32(np.nan), np.float32(np.inf)
            o = np.array([[0, 1, -6], [nan, 1, -6], [0, 1, -6], [inf, 1, -6], [0, 1, -6], [0, 1, -6]], np.float32)
            d = np.array([[0, 0, 1], [0, 0, 1], [nan, 0, 1], [0, 0, 1], [inf, 0, 1], [0, 1e-30, 1]], np.float32)
            t = np.zeros(len(o), np.float32)
            prim = np.zeros(len(o), np.int32)
            rc = lib.emu_nearest(scene, len(o), o.ctypes.data_as(FP), d.ctypes.data_as(FP), t.ctypes.data_as(FP),
                                 prim.ctypes.data_as(C.POINTER(C.c_int32)))
            assert rc == 0, device.rtc_last_error()
        finally:
            device.rtc_scene_destroy(scene)


def test_sweep_under_address_sanitizer():
    """The memcheck pass for the sweep's local arrays (ray stack, state bits, hit buffer, open-solid list): this module
    again in a child process whose harness is built with -fsanitize=address,undefined."""
    if os.environ.get("RTC_EMU_SANITIZE"):
        pytest.skip("already inside the sanitized run")
    libasan = subprocess.run(["g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not libasan or not os.path.exists(libasan):
        pytest.skip("no libasan")
    env = dict(os.environ, RTC_EMU_SANITIZE="1", LD_PRELOAD=libasan, ASAN_OPTIONS="detect_leaks=0:abort_on_error=1",
               UBSAN_OPTIONS="print_stacktrace=1:halt_on_error=1")
    proc = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-x", "-q", "-p", "no:cacheprovider"],
                          cwd=ROOT, env=env, capture_output=True, text=True)
    tail = (proc.stdout + proc.stderr)[-3000:]
    assert proc.returncode == 0, tail
    assert "passed" in proc.stdout and "AddressSanitizer" not in tail and "runtime error" not in tail, tail
