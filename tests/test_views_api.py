"""rtc_render_views without a device: argument validation ahead of the state check, the ctypes layout of RtcView, the host
library's camera -> RtcView conversion and the camera its one-shot batch commits with."""
import ctypes as C
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RTC_ERR_INVALID, RTC_ERR_STATE = -1, -4


def _scene(lib):
    ident = (C.c_float * 16)(1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1)
    lib.rtc_last_error.restype = C.c_char_p
    lib.rtc_set_camera.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_float)]
    scene = C.c_void_p()
    assert lib.rtc_scene_create(C.byref(scene)) == 0
    assert lib.rtc_set_camera(scene, 64, 32, 1.0, 0.5, 2.0 / 64, ident) == 0
    return scene, ident


def test_render_views_validates_arguments_before_the_state():
    import ray_tracer_challenge_b200 as rt

    lib = C.CDLL(rt.LIB_DEVICE)
    lib.rtc_render_views.argtypes = [C.c_void_p, C.c_int32, C.c_uint32, C.POINTER(rt.RtcView), C.c_void_p, C.c_void_p, C.c_void_p]
    scene, ident = _scene(lib)
    views = (rt.RtcView * 2)()
    for v in views:
        v.half_width, v.half_height, v.pixel_size = 1.0, 0.5, 2.0 / 64
        v.transform_inverse[:] = list(ident)

    def call(n=2, vs=views, depth=5):
        rc = lib.rtc_render_views(scene, depth, n, vs, None, None, None)
        return rc, lib.rtc_last_error()

    assert call(n=0)[0] == RTC_ERR_INVALID
    assert call(vs=None)[0] == RTC_ERR_INVALID
    for field, bad in (("pixel_size", math.nan), ("half_width", math.inf), ("pixel_size", 0.0), ("pixel_size", -1.0)):
        old = getattr(views[1], field)
        setattr(views[1], field, bad)
        rc, msg = call()
        assert rc == RTC_ERR_INVALID and b"view 1" in msg, (field, bad, msg)
        setattr(views[1], field, old)
    views[0].transform_inverse[7] = math.nan
    assert call()[0] == RTC_ERR_INVALID
    views[0].transform_inverse[7] = 0.0
    for depth in (-1, 24):
        rc, msg = call(depth=depth)
        assert rc == RTC_ERR_INVALID and b"reflection_recursion_depth" in msg
    # a valid batch of an uncommitted scene: the state error
    rc, msg = call()
    assert rc == RTC_ERR_STATE and b"before rtc_scene_commit" in msg
    lib.rtc_scene_destroy(scene)


def test_rtc_view_ctypes_layout_matches_the_header(tmp_path):
    import ray_tracer_challenge_b200 as rt

    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    src = tmp_path / "view.c"
    fields = [f for f, _ in rt.RtcView._fields_]
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "rtc_b200.h"\nint main(void) {\nprintf("%zu", sizeof(RtcView));\n'
                   + "".join(f'printf(" %zu", offsetof(RtcView, {f}));\n' for f in fields) + "return 0;\n}\n")
    exe = tmp_path / "view"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    size, *offsets = map(int, subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split())
    assert size == C.sizeof(rt.RtcView) == 76
    assert offsets == [getattr(rt.RtcView, f).offset for f in fields]


def test_camera_view_carries_the_fields_rtc_set_camera_receives():
    """The host library builds a batch's RtcView with the helper that fill_scene hands rtc_set_camera its fields from; here
    those fields are held to Camera::new (camera.rs:23-56) restated in f32."""
    import ray_tracer_challenge_b200 as rt

    s = rt.new_session()
    for w, h, fov, eye in ((160, 64, math.pi / 4.0, (-3, 1, 2.5)), (50, 100, 1.2, (0.3, 2.0, -7.0)), (64, 64, math.pi / 2, (0, 0, -5))):
        t = s.view_transform(eye, (0, 0.5, 0), (0, 1, 0))
        cam = s.Camera(w, h, fov, t)
        v = s.camera_view(cam)
        inv = np.zeros(16, np.float32)
        s.lib.sg_inverse(rt._api.fptr(np.ascontiguousarray(np.asarray(t.m, np.float32).reshape(16))), rt._api.fptr(inv))
        assert np.array_equal(np.asarray(v.transform_inverse, np.float32).view(np.uint32), inv.view(np.uint32))
        f = np.float32
        half_view = f(v.half_width) if w >= h else f(v.half_height)
        assert abs(float(half_view) - math.tan(fov / 2)) <= 2 * np.spacing(half_view)
        aspect = f(w) / f(h)
        if aspect >= 1:
            assert f(v.half_height) == half_view / aspect
        else:
            assert f(v.half_width) == half_view * aspect
        assert f(v.pixel_size) == (f(v.half_width) * f(2.0)) / f(w)


def test_one_shot_batch_commits_with_the_farthest_camera():
    import ray_tracer_challenge_b200 as rt

    s = rt.new_session()
    eyes = [(0, 1.5, -5), (0, 1.5, -40), (12, 1, 3), (-3, 50.5, 0), (0, 1, 49)]
    cams = [s.Camera(32, 16, 1.0, s.view_transform(e, (0, 1, 0), (0, 1, 0))) for e in eyes]
    assert s.farthest_camera(cams) == 3
    assert s.farthest_camera(cams[:3]) == 1
    assert s.farthest_camera([cams[0]]) == 0
    assert s.farthest_camera(cams[2:3] + cams[:2]) == 2
    other = s.Camera(16, 16, 1.0, s.identity_4x4())
    world = s.World.default()
    with pytest.raises(rt.RtcError, match="canvas size"):
        s.render_views(world, [cams[0], other])
