"""RTC_OPT_EXACT_GROUPS on the host: the option and what the commit reports, and the device code compiled for the host
(tests/emu) against the oracle bit for bit with the option on — scenes whose group boxes are stale, rays whose answer
the group boxes decide (phantom hits of the reference's f32 sphere test), CSGs inside groups through csg_eval and
csg_sweep, and the existing device-code scene sets."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import ray_tracer_challenge_b200 as rt_pkg
from ray_tracer_challenge_b200 import scenes
from tests import exact_groups_scenes as eg
from tests.test_device_code_on_host import COLOR_CASES, FP, ROOT, SCENES, _build, _raw_scene, _rays

RTC_ERR_INVALID = -1

# what the commit reported before the option existed (digest: FNV-1a over heads, records, transforms and tree), which is
# what it must still report with the option off
PARENT_DIGESTS = {
    "stress": 13607633653662890957,
    "dragon": 3922214089963511966,
    "csg_gallery": 14162644651228271131,
    "shapes_zoo": 3032382358964346441,
    "stale_box": 11403924040457885577,
    "csg_in_group": 4143820165434737740,
    "csg_in_group_small": 8356033128687377374,
}
INSPECT_CASES = {
    "stress": (scenes.stress, dict(width=64, height=36, n_spheres=1500, n_each=6, n_csg=6)),
    "dragon": (scenes.dragon_element, dict(width=64, height=36, n_u=24, n_v=12)),
    "csg_gallery": (scenes.csg_gallery, dict(width=64, height=40)),
    "shapes_zoo": (scenes.shapes_zoo, dict(width=64, height=40)),
    "stale_box": (eg.stale_box, dict()),
    "csg_in_group": (eg.csg_in_group, dict()),
    "csg_in_group_small": (eg.csg_in_group, dict(n_spheres=3)),
}
# scenes whose heads carry a chain only with the option on: grouped tree primitives, or a CSG root inside a group
# (csg_gallery: a small scene with a grouped CSG)
CHANGED_BY_OPTION = {"stress", "dragon", "csg_gallery", "stale_box", "csg_in_group", "csg_in_group_small"}


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    device, lib = _build(tmp_path_factory, "emu_nearest.cpp")
    lib.emu_nearest.argtypes = [C.c_void_p, C.c_uint32, FP, FP, FP, C.POINTER(C.c_int32)]
    device.rtc_set_option.argtypes = [C.c_void_p, C.c_int32, C.c_int64]
    return device, lib


@pytest.fixture(scope="module")
def emu_color(tmp_path_factory):
    device, lib = _build(tmp_path_factory, "emu_color.cpp")
    lib.emu_color_at.argtypes = [C.c_void_p, C.c_uint32, FP, FP, C.c_int, C.c_int, C.c_int, FP, FP, C.POINTER(C.c_int32)]
    device.rtc_set_option.argtypes = [C.c_void_p, C.c_int32, C.c_int64]
    return device, lib


@pytest.fixture
def host():
    return rt_pkg.new_session()


def _inspect(host, name, exact=None):
    make, kw = INSPECT_CASES[name]
    if exact is not None:
        host.set_exact_groups(exact)
    return host.inspect(*make(host, **kw)[:2])


@pytest.mark.parametrize("name", sorted(INSPECT_CASES))
def test_option_off_commits_what_the_parent_committed(name, host):
    default = _inspect(host, name)
    off = _inspect(host, name, exact=False)
    assert default["digest"] == off["digest"] == PARENT_DIGESTS[name], (default, off)
    for k in default:
        if k not in ("host_ms", "flatten_ms"):
            assert default[k] == off[k], k
    assert default["exact_groups"] == 0


@pytest.mark.parametrize("name", sorted(INSPECT_CASES))
def test_option_on_changes_only_scenes_with_chains_to_add(name, host):
    off = _inspect(host, name, exact=False)
    on = _inspect(host, name, exact=True)
    assert on["exact_groups"] == 1
    assert (on["digest"] != off["digest"]) == (name in CHANGED_BY_OPTION), (on["digest"], off["digest"])
    for k in ("n_positions", "n_bvh_nodes", "n_linear", "bvh_depth", "small_n", "loose_group_boxes"):
        assert on[k] == off[k], k  # the same tree and the same table: only the heads' flags differ


def test_loose_group_boxes(host):
    assert _inspect(host, "stale_box")["loose_group_boxes"] > 0
    assert _inspect(host, "csg_in_group")["loose_group_boxes"] > 0
    # the same world with the transform applied before divide(): every cached box is current
    assert host.inspect(*eg.stale_box(host, stale=False)[:2])["loose_group_boxes"] == 0
    # divide() leaves the parent's box around its new subgroups: the stress field and the divided mesh are tight
    assert _inspect(host, "stress")["loose_group_boxes"] == 0
    assert _inspect(host, "dragon")["loose_group_boxes"] == 0
    assert host.inspect(*scenes.here_be_dragons(host, width=64, height=32, n_u=16, n_v=8))["loose_group_boxes"] == 0


def test_bad_values_are_rejected(emu, host):
    device, _ = emu
    cam, world, _ = eg.stale_box(host)
    scene = host.export_scene(cam, world)
    try:
        for bad in (-1, 2, 9):
            assert device.rtc_set_option(scene, eg.RTC_OPT_EXACT_GROUPS, bad) == RTC_ERR_INVALID
        for good in (0, 1):
            assert device.rtc_set_option(scene, eg.RTC_OPT_EXACT_GROUPS, good) == 0
    finally:
        device.rtc_scene_destroy(scene)
    assert host.lib.sg_set_exact_groups(host.ctx, 2) != 0
    assert host.lib.sg_set_exact_groups(host.ctx, 1) == 0


def _emu_nearest(device, lib, host, world, o, d, exact):
    scene = _raw_scene(device, host, world)
    try:
        assert device.rtc_set_option(scene, eg.RTC_OPT_EXACT_GROUPS, exact) == 0
        t = np.zeros(len(o), np.float32)
        prim = np.zeros(len(o), np.int32)
        rc = lib.emu_nearest(scene, len(o), o.ctypes.data_as(FP), d.ctypes.data_as(FP), t.ctypes.data_as(FP),
                             prim.ctypes.data_as(C.POINTER(C.c_int32)))
        assert rc == 0, device.rtc_last_error()
        return t, prim
    finally:
        device.rtc_scene_destroy(scene)


def _camera_rays(oracle, ocam):
    """Ray i = pixel i of the frame (the never-rendered last row and column: rays that start far above and miss)."""
    w, h = ocam.width_pixels, ocam.height_pixels
    o = np.zeros((w * h, 3), np.float32)
    d = np.zeros((w * h, 3), np.float32)
    o[:, 1], d[:, 1] = 1.0e6, 1.0
    for y in range(h - 1):
        for x in range(w - 1):
            ro, rd = oracle.probe.camera_ray(ocam, x, y)
            o[y * w + x], d[y * w + x] = ro[:3], rd[:3]
    return o, d


def _emu_frame(device, lib, scene, ocam, oracle, exact, small):
    o, d = _camera_rays(oracle, ocam)
    w, h = ocam.width_pixels, ocam.height_pixels
    assert device.rtc_set_option(scene, eg.RTC_OPT_EXACT_GROUPS, exact) == 0
    rgb = np.zeros((w * h, 3), np.float32)
    path = C.c_int32(-1)
    assert lib.emu_color_at(scene, w * h, o.ctypes.data_as(FP), d.ctypes.data_as(FP), 5, int(small), 1, rgb.ctypes.data_as(FP),
                            None, C.byref(path)) == 0, device.rtc_last_error()
    assert path.value == int(small)
    rays = (C.c_ulonglong * 4)()
    lib.emu_last_rays(rays)
    return rgb.reshape(h, w, 3)[: h - 1, : w - 1], rays


def _frame_matches(device, lib, host, oracle, make, kw, small):
    """The frame through the device code with the option on equals the oracle's render bit for bit (pixels and ray
    counts); with it off it does not."""
    cam, world = make(host, **kw)[:2]
    ocam, oworld = make(oracle, **kw)[:2]
    want = np.asarray(ocam.render(oworld, 5).data, np.float32)[: ocam.height_pixels - 1, : ocam.width_pixels - 1]
    st = ocam.last_stats
    scene = host.export_scene(cam, world)
    try:
        got, rays = _emu_frame(device, lib, scene, ocam, oracle, 1, small)
        same = (got.view(np.uint32) == want.view(np.uint32)).all(axis=2)
        assert same.all(), (int((~same).sum()), got[~same][:2], want[~same][:2])
        assert (rays[1], rays[2], rays[3]) == (st.secondary_rays, st.shadow_rays, st.shades), (list(rays), st.as_dict())
        off, _ = _emu_frame(device, lib, scene, ocam, oracle, 0, small)
        assert not (off.view(np.uint32) == want.view(np.uint32)).all()
    finally:
        device.rtc_scene_destroy(scene)


def test_stale_box_nearest_hits(emu, host, oracle):
    """Every primary ray of the stale-box scene: the option on gives World::intersect's distance and sphere; off it
    does not."""
    device, lib = emu
    _, world, handles = eg.stale_box(host)
    ocam, oworld, ohandles = eg.stale_box(oracle)
    o, d = _camera_rays(oracle, ocam)
    want, shapes = eg.oracle_nearest(oracle, oworld, o, d, with_shapes=True)
    assert (want >= 0).sum() > 1000
    on, prim = _emu_nearest(device, lib, host, world, o, d, 1)
    assert (on == want).all(), int((on != want).sum())
    assert eg.same_spheres(host, world, prim, handles, shapes, ohandles).all()
    off, _ = _emu_nearest(device, lib, host, world, o, d, 0)
    assert (off != want).sum() > 500  # the stale boxes clip whole spheres


def test_stale_box_frame(emu_color, host, oracle):
    _frame_matches(*emu_color, host, oracle, eg.stale_box, dict(), small=False)


def test_silhouette_rays_decided_by_group_boxes(emu, host, oracle):
    """Rays grazing tiny, far spheres, where the reference's sphere test reports phantom hits: at least 50 of them get
    a different answer from the oracle with the spheres grouped than ungrouped.  With the option on the device code
    gives the grouped answer (distance and sphere) on every ray; off, it keeps some phantom hits the group boxes cull."""
    device, lib = emu
    _, world, centres, handles = eg.far_field(host)
    _, grouped, _, ohandles = eg.far_field(oracle)
    _, ungrouped, _, _ = eg.far_field(oracle, grouped=False)
    o, d = eg.far_field_rays(centres, 2000, spread_radii=1.5)
    want, shapes = eg.oracle_nearest(oracle, grouped, o, d, with_shapes=True)
    decided = want != eg.oracle_nearest(oracle, ungrouped, o, d)
    assert decided.sum() >= 50, int(decided.sum())
    on, prim = _emu_nearest(device, lib, host, world, o, d, 1)
    assert (on == want).all(), (int((on != want).sum()), int((on[decided] != want[decided]).sum()))
    assert eg.same_spheres(host, world, prim, handles, shapes, ohandles).all()
    off, _ = _emu_nearest(device, lib, host, world, o, d, 0)
    assert (off[decided] != want[decided]).any()


def test_silhouette_rays_of_the_stress_field(emu, host, oracle):
    """Rays from the stress scene's camera grazing its field spheres (1e-4 of a radius around the silhouette), the
    structure behind c5.  Its divided groups hold up to 8 spheres each, so their boxes rarely decide such a ray (the
    same rays against the undivided field: `decided`); whatever they decide, the option on gives the oracle's answer."""
    from ray_tracer_challenge_b200.scenes import _xorshift64star

    device, lib = emu
    kw = dict(width=64, height=36, n_spheres=1500, n_each=6, n_csg=6)
    _, world = scenes.stress(host, **kw)
    _, oworld = scenes.stress(oracle, **kw)
    _, undivided = scenes.stress(oracle, divide=0, **kw)
    rnd = _xorshift64star(1)
    spheres = []
    for _ in range(kw["n_spheres"]):
        c = np.array([(rnd() * 2 - 1) * 50.0 for _ in range(3)])
        spheres.append((c, 0.2 + 0.4 * rnd()))  # scenes.stress: centre, then radius
    rng = np.random.default_rng(5)
    eye = np.array([0.0, 50.0 * 0.4, -50.0 * 2.2])
    n = 1500
    o = np.tile(eye.astype(np.float32), (n, 1))
    d = np.zeros((n, 3), np.float32)
    for i in range(n):
        c, r = spheres[rng.integers(len(spheres))]
        v = c - eye
        side = np.cross(v, rng.normal(size=3))
        target = c + side / np.linalg.norm(side) * r * (1.0 + rng.normal() * 1e-4)
        d[i] = (target - eye) / np.linalg.norm(target - eye)
    want = eg.oracle_nearest(oracle, oworld, o, d)
    decided = want != eg.oracle_nearest(oracle, undivided, o, d)
    print("stress silhouette rays decided by the divided groups' boxes:", int(decided.sum()), "of", n)
    on, _ = _emu_nearest(device, lib, host, world, o, d, 1)
    assert (on.view(np.uint32) == want.view(np.uint32)).all(), int((on != want).sum())
    assert (want >= 0).sum() > n // 4


# Primary rays of test_sphere_field_parity_at_scale's 20 k field (640 x 360) whose nearest hit still differs from the
# oracle's with the option on: the reference reports hits outside the hit shape's own bounding box, beyond the tree's
# padding (DESIGN.md §7, deviation (1)).  Pinned here to show that no group cull decides them.
FIELD_20K = dict(width=640, height=360, n_spheres=20_000, n_each=16, n_csg=8)
FIELD_20K_PIXELS = [(583, 85), (120, 86), (118, 90), (588, 195)]


def test_remaining_field_differences_involve_no_group(emu, host, oracle):
    device, lib = emu
    _, world = scenes.stress(host, **FIELD_20K)
    ocam, oworld = scenes.stress(oracle, **FIELD_20K)
    _, undivided = scenes.stress(oracle, divide=0, **FIELD_20K)
    o = np.zeros((len(FIELD_20K_PIXELS), 3), np.float32)
    d = np.zeros_like(o)
    for i, (x, y) in enumerate(FIELD_20K_PIXELS):
        ro, rd = oracle.probe.camera_ray(ocam, x, y)
        o[i], d[i] = ro[:3], rd[:3]
    want = eg.oracle_nearest(oracle, oworld, o, d)
    on, prim_on = _emu_nearest(device, lib, host, world, o, d, 1)
    off, prim_off = _emu_nearest(device, lib, host, world, o, d, 0)
    assert (on != want).all(), (on, want)  # the known deviation: if this fails, the tree now finds these hits
    # the option changes nothing on these rays, and the reference's divided group boxes decide none of them
    assert (on.view(np.uint32) == off.view(np.uint32)).all() and (prim_on == prim_off).all()
    assert (want.view(np.uint32) == eg.oracle_nearest(oracle, undivided, o, d).view(np.uint32)).all()


@pytest.mark.parametrize("sweep", ["0", "1"], ids=["csg_eval", "csg_sweep"])
@pytest.mark.parametrize("n_spheres", [60, 3], ids=["tree", "small"])
def test_csg_in_a_stale_group(n_spheres, sweep, emu, emu_color, host, oracle, monkeypatch):
    """CSGs inside a group whose box is stale: nearest hits, and frames of opaque and glass CSGs (the n1 / n2 walk),
    through csg_eval and csg_sweep, in a tree scene and a small one."""
    monkeypatch.setenv("RTC_CSG_SWEEP", sweep)
    device, lib = emu
    _, world = eg.csg_in_group(host, n_spheres=n_spheres)
    ocam, oworld = eg.csg_in_group(oracle, n_spheres=n_spheres)
    assert (host.inspect(*eg.csg_in_group(host, n_spheres=n_spheres))["small_n"] > 0) == (n_spheres < 10)
    o, d = _camera_rays(oracle, ocam)
    want = eg.oracle_nearest(oracle, oworld, o, d)
    on, _ = _emu_nearest(device, lib, host, world, o, d, 1)
    assert (on == want).all(), int((on != want).sum())
    assert (_emu_nearest(device, lib, host, world, o, d, 0)[0] != want).any()
    for glass in (False, True):
        _frame_matches(*emu_color, host, oracle, eg.csg_in_group, dict(n_spheres=n_spheres, glass=glass), small=n_spheres < 10)


@pytest.mark.parametrize("name", sorted(SCENES))
def test_scene_set_nearest_hits_with_the_option_on(name, emu, host, oracle):
    device, lib = emu
    make, kw = SCENES[name]
    _, world = make(host, **kw)
    ocam, oworld = make(oracle, **kw)
    o, d = _rays(oracle, ocam, 600, seed=7)
    want = eg.oracle_nearest(oracle, oworld, o, d)
    got, _ = _emu_nearest(device, lib, host, world, o, d, 1)
    assert (got.view(np.uint32) == want.view(np.uint32)).all(), int((got != want).sum())


@pytest.mark.parametrize("name", sorted(COLOR_CASES))
def test_color_cases_with_the_option_on(name, emu_color, host, oracle):
    device, lib = emu_color
    make, kw, small = COLOR_CASES[name]
    cam, world = make(host, **kw)
    ocam, oworld = make(oracle, **kw)
    scene = host.export_scene(cam, world)
    try:
        assert device.rtc_set_option(scene, eg.RTC_OPT_EXACT_GROUPS, 1) == 0
        n = 240
        o, d = _rays(oracle, ocam, n, seed=11)
        want = np.array([oracle.probe.color_at(oworld, o[i], d[i], 5) for i in range(n)], np.float32)
        for use_filter in ((0, 1) if small else (0,)):
            rgb = np.zeros((n, 3), np.float32)
            rc = lib.emu_color_at(scene, n, o.ctypes.data_as(FP), d.ctypes.data_as(FP), 5, int(small), use_filter,
                                  rgb.ctypes.data_as(FP), None, None)
            assert rc == 0, device.rtc_last_error()
            same = (rgb.view(np.uint32) == want.view(np.uint32)).all(axis=1)
            assert same.all(), (name, use_filter, int((~same).sum()))
    finally:
        device.rtc_scene_destroy(scene)


F32 = np.float32


def _certified(mn, mx, o, d, t):
    """dev_bvh.cuh: axis_certified on all three axes, in f32 with the strict build's operation order."""
    ok = np.ones(len(t), bool)
    with np.errstate(invalid="ignore", over="ignore"):
        for k in range(3):
            p = o[:, k] + t * d[:, k]
            m = F32(2.0 ** -21) * (np.maximum(np.abs(mn[:, k]), np.abs(mx[:, k])) + np.abs(o[:, k]) + np.abs(p)) + F32(2.0 ** -100)
            ok &= (np.abs(d[:, k]) >= F32(2.0 ** -60)) & (m <= F32(1e30)) & (mn[:, k] + m <= p) & (p + m <= mx[:, k])
    return ok


def _aabb_ref(o, d, mn, mx):
    """dev_shapes.cuh: aabb_ref, the reference's aabb_intersection (cube.rs:90-129), in f32."""
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        inv = F32(1.0) / d
        a, b = (mn - o) * inv, (mx - o) * inv
        lo, hi = np.fmin(a[:, 0], b[:, 0]), np.fmax(a[:, 0], b[:, 0])
        for k in (1, 2):
            lo, hi = np.fmax(lo, np.fmin(a[:, k], b[:, k])), np.fmin(hi, np.fmax(a[:, k], b[:, k]))
        return hi >= np.fmax(F32(0.0), lo)


@pytest.mark.parametrize("scale", [1e-3, 1.0, 1e3, 1e5], ids=["millimetre", "unit", "kilometre", "far"])
def test_certificate_never_passes_a_box_the_reference_rejects(scale):
    """The one-box certificate at the shipped margin against aabb_intersection: hit points on and near the faces of an
    innermost box, enclosing boxes that share some of its faces, origins 1 to 1000 box-scales away, a few ulps of
    jitter on t, and some zero direction components.  Wherever the certificate passes, the reference passes the
    innermost box and the enclosing one."""
    rng = np.random.default_rng(int(np.log10(scale)) + 10)
    n = 400_000
    c = rng.uniform(-10, 10, (n, 3)) * scale
    h = scale * np.exp(rng.uniform(np.log(1e-4), 0, (n, 3)))
    mn, mx = (c - h).astype(F32), (c + h).astype(F32)
    grow = lambda: np.where(rng.random((n, 3)) < 0.5, 0.0, scale * 10 ** rng.uniform(-7, 0, (n, 3)))  # noqa: E731
    amn, amx = np.minimum((mn - grow()).astype(F32), mn), np.maximum((mx + grow()).astype(F32), mx)
    u = rng.normal(size=(n, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    o = (c + u * scale * 10 ** rng.uniform(0, 3, (n, 1))).astype(F32)
    near_face = np.where(rng.random((n, 3)) < 0.5, 1.0, 1 - 10 ** rng.uniform(-8, -5, (n, 3)))
    q = c + h * rng.uniform(-1.0000005, 1.0000005, (n, 3)) * near_face
    v = np.where(rng.random((n, 3)) < 0.01, 0.0, q - o)
    v[~(np.abs(v) > 0).any(axis=1)] = 1.0
    d = (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(F32)
    t = np.einsum("ij,ij->i", q - o, d.astype(np.float64)).astype(F32)
    t = np.abs((t.view(np.int32) + rng.integers(-4, 5, n).astype(np.int32)).view(F32))
    cert = _certified(mn, mx, o, d, t)
    assert cert.mean() > 0.5  # the certificate does answer for most hits
    assert not (cert & ~_aabb_ref(o, d, mn, mx)).any()
    assert not (cert & ~_aabb_ref(o, d, amn, amx)).any()


def test_exact_groups_under_address_sanitizer():
    """This module again in a child process whose harnesses are built with -fsanitize=address,undefined."""
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
