"""ray_tracer_challenge_b200 — B200 (sm_100a) implementation of the reference's `Camera::render` hot path.

    import ray_tracer_challenge_b200 as rt
    world = rt.World([rt.Sphere()], rt.PointLight((-10, 10, -10), (1, 1, 1)))
    camera = rt.Camera(400, 200, math.pi / 3, rt.view_transform((0, 1.5, -5), (0, 1, 0), (0, 1, 0)))
    canvas = camera.render_b200(world, 5)          # drop-in sibling of Camera::render (camera.rs:76-91)

The names mirror the Rust reference's `lib` crate (see api.py).  All work is done by two native libraries
built in-tree by `python -m ray_tracer_challenge_b200.build` (or `__graft_entry__.build()`):
librtc_host.so (C++ host mirror + scene flattener) and librtc_b200.so (the C ABI of include/rtc_b200.h and
the CUDA kernels).  There is no CPU fallback: importing without the libraries, or rendering without a CUDA
device, raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import api as _api
from .api import (DEFAULT_RAY_RECURSION_DEPTH, REFRACTION_AIR, REFRACTION_DIAMOND, REFRACTION_GLASS,  # noqa: F401
                  REFRACTION_VACCUM, REFRACTION_WATER, Canvas, Material, PointLight, RectangleLight, RtcError, SgStats,
                  color_from_hex, constant_jitter, glass, hardcoded_jitter, metal)

_PKG = os.path.dirname(os.path.abspath(__file__))
# RTC_LIB_DIR: load another build of the two libraries (A/B timing of kernel variants on one GPU box)
_LIB_DIR = os.environ.get("RTC_LIB_DIR", _PKG)
LIB_HOST = os.path.join(_LIB_DIR, "librtc_host.so")
LIB_DEVICE = os.path.join(_LIB_DIR, "librtc_b200.so")


class RtcStats(C.Structure):
    """include/rtc_b200.h: RtcStats"""

    _fields_ = [
        ("primary_rays", C.c_uint64), ("secondary_rays", C.c_uint64), ("shadow_rays", C.c_uint64),
        ("shades", C.c_uint64), ("node_visits", C.c_uint64), ("prim_tests", C.c_uint64 * 8), ("xforms", C.c_uint64),
        ("patterns", C.c_uint64), ("cells", C.c_uint64), ("schlicks", C.c_uint64), ("refr_dirs", C.c_uint64),
        ("capacity_overflows", C.c_uint64), ("flops", C.c_double), ("kernel_ms", C.c_double), ("total_ms", C.c_double),
        ("n_devices", C.c_int32), ("detailed", C.c_int32), ("launches", C.c_int32), ("wave_overflows", C.c_int32),
    ]

    @property
    def rays(self) -> int:
        return self.primary_rays + self.secondary_rays + self.shadow_rays

    def as_dict(self) -> dict:
        d = {}
        for name, _ in self._fields_:
            v = getattr(self, name)
            d[name] = list(v) if name == "prim_tests" else v
        d["rays"] = self.rays
        return d


class RtcCommitInfo(C.Structure):
    """include/rtc_b200.h: RtcCommitInfo"""

    _fields_ = [
        ("n_positions", C.c_int32), ("n_bvh_nodes", C.c_int32), ("n_linear", C.c_int32), ("n_xforms", C.c_int32),
        ("bvh_leaf_size", C.c_int32), ("small_n", C.c_int32), ("filter_ok", C.c_int32), ("cell_masks", C.c_int32),
        ("plane_cells", C.c_int32), ("converge", C.c_int32), ("tol_sphere", C.c_float), ("light_ball", C.c_float * 4),
        ("bvh_depth", C.c_int32), ("host_ms", C.c_double), ("digest", C.c_uint64), ("lean", C.c_int32),
        ("exact_groups", C.c_int32), ("loose_group_boxes", C.c_int32),
    ]

    def as_dict(self) -> dict:
        return {name: (list(getattr(self, name)) if name == "light_ball" else getattr(self, name)) for name, _ in self._fields_}


class RtcPrim(C.Structure):
    _fields_ = [("type", C.c_int32), ("material", C.c_int32), ("casts_shadow", C.c_int32), ("parent", C.c_int32),
                ("inv", C.c_float * 16), ("params", C.c_float * 12), ("bbox_min", C.c_float * 3),
                ("bbox_max", C.c_float * 3)]


class RtcNode(C.Structure):
    _fields_ = [("kind", C.c_int32), ("parent", C.c_int32), ("op", C.c_int32), ("child_begin", C.c_int32),
                ("child_count", C.c_int32), ("inv", C.c_float * 16), ("bbox_min", C.c_float * 3),
                ("bbox_max", C.c_float * 3), ("world_bbox_min", C.c_float * 3), ("world_bbox_max", C.c_float * 3)]


class RtcView(C.Structure):
    """include/rtc_b200.h: RtcView — one camera of rtc_render_views (Camera::new's derived fields)"""

    _fields_ = [("half_width", C.c_float), ("half_height", C.c_float), ("pixel_size", C.c_float),
                ("transform_inverse", C.c_float * 16)]


_V, _I, _FP, _IP, _U8P = C.c_void_p, C.c_int, _api.FP, _api.IP, _api.U8P
_HOST_EXTRAS = {
    "sg_set_render_options": (_I, [_V, _I, _IP, _I, _I]),
    "sg_last_rtc_stats": (_I, [_V, C.POINTER(RtcStats)]),
    "sg_set_bvh_builder": (_I, [_V, _I]),
    "sg_set_exact_groups": (_I, [_V, _I]),
    "sg_ppm_from_u8": (C.c_int64, [_V, _I, _I, _U8P, C.c_char_p, C.c_int64]),
    "sg_prepare": (_I, [_V, _I, _I]),
    "sg_camera_render_shard": (_I, [_V, _I, _I, _I, _I, _I, _FP, _U8P, C.POINTER(SgStats)]),
    "sg_inspect": (_I, [_V, _I, _I, C.c_void_p, C.POINTER(C.c_double)]),
    "sg_export_scene": (_I, [_V, _I, _I, C.POINTER(C.c_void_p)]),
    "sg_release_prepared": (_I, [_V, _I]),
    "sg_render_prepared": (_I, [_V, _I, _I, _I, _I, _I, _I, _FP, _U8P, C.POINTER(SgStats)]),
    "sg_flush_l2": (_I, [_V, _I]),
    "sg_set_prepared_option": (_I, [_V, _I, _I, C.c_int64]),
    "sg_trace_rays": (_I, [_V, _I, C.c_uint32, _FP, _FP, _I, _I, _FP, _FP, _IP]),
    "sg_flatten": (_I, [_V, _I, _IP, C.POINTER(RtcPrim), C.POINTER(RtcNode), C.POINTER(C.c_int32), _IP]),
    "sg_render_prepared_views": (_I, [_V, _I, _I, _I, _IP, _I, _FP, _U8P, C.POINTER(SgStats)]),
    "sg_camera_render_views": (_I, [_V, _IP, _I, _I, _I, _FP, _U8P, C.POINTER(SgStats)]),
    "sg_camera_view": (_I, [_V, _I, C.POINTER(RtcView)]),
    "sg_farthest_camera": (_I, [_V, _IP, _I]),
}


def _handles(cameras):
    return (C.c_int * len(cameras))(*[c.handle for c in cameras])


def _view_planes(n, h, w, want_rgb, want_u8, out_rgb, out_u8):
    """The (n, h, w, 3) planes of a batch: the caller's (checked) or new ones; None where not wanted."""
    rgb = u8 = None
    if want_rgb:
        rgb = out_rgb if out_rgb is not None else np.zeros((n, h, w, 3), np.float32)
        if rgb.shape != (n, h, w, 3) or rgb.dtype != np.float32 or not rgb.flags.c_contiguous:
            raise ValueError(f"out_rgb must be a C-contiguous float32 array of shape {(n, h, w, 3)}")
    if want_u8:
        u8 = out_u8 if out_u8 is not None else np.zeros((n, h, w, 3), np.uint8)
        if u8.shape != (n, h, w, 3) or u8.dtype != np.uint8 or not u8.flags.c_contiguous:
            raise ValueError(f"out_u8 must be a C-contiguous uint8 array of shape {(n, h, w, 3)}")
    return rgb, u8


def _canvases(api, n, h, w, rgb, u8):
    return [Canvas(w, h, rgb[i] if rgb is not None else None, u8[i] if u8 is not None else None, api=api) for i in range(n)]


class PreparedScene:
    """A world + camera committed to the device(s) and kept resident for repeated renders."""

    def __init__(self, api, camera, world):
        self.api, self.camera, self.world = api, camera, world
        self.handle = api.check(api.lib.sg_prepare(api.ctx, camera.handle, world.handle))
        self.last_stats = None

    def render(self, depth=DEFAULT_RAY_RECURSION_DEPTH, out_rgb=None, out_u8=None, want_rgb=True, want_u8=True,
               shard=0, n_shards=0, detailed=False, fma=False):
        """rtc_render / rtc_render_shard.  Buffers may be caller-supplied (e.g. pinned); want_* = False leaves the
        frame on the device (kernel timing)."""
        w, h = self.camera.width_pixels, self.camera.height_pixels
        if want_rgb and out_rgb is None:
            out_rgb = np.zeros((h, w, 3), np.float32)
        if want_u8 and out_u8 is None:
            out_u8 = np.zeros((h, w, 3), np.uint8)
        stats = SgStats()
        api = self.api
        api.check(api.lib.sg_render_prepared(
            api.ctx, self.handle, int(depth), int(shard), int(n_shards), int(detailed), int(fma),
            _api.fptr(out_rgb) if want_rgb else None, out_u8.ctypes.data_as(_U8P) if want_u8 else None,
            C.byref(stats)))
        self.last_stats = api.last_rtc_stats()
        return Canvas(w, h, out_rgb if want_rgb else None, out_u8 if want_u8 else None, api=api)

    def render_views(self, cameras, depth=DEFAULT_RAY_RECURSION_DEPTH, want_rgb=True, want_u8=True, out_rgb=None, out_u8=None,
                     fma=False):
        """rtc_render_views: every camera (of this scene's canvas size) rendered from the committed scene in one batch.
        Returns one Canvas per camera, views into one (n, h, w, 3) array per plane; want_* = False leaves the frames on the
        device.  In a scene with a tree a camera farther out than the committed one is refused (commit with the farthest)."""
        cameras = list(cameras)
        n, w, h = len(cameras), self.camera.width_pixels, self.camera.height_pixels
        rgb, u8 = _view_planes(n, h, w, want_rgb, want_u8, out_rgb, out_u8)
        stats = SgStats()
        api = self.api
        api.check(api.lib.sg_render_prepared_views(
            api.ctx, self.handle, int(depth), n, _handles(cameras), int(fma), _api.fptr(rgb) if rgb is not None else None,
            u8.ctypes.data_as(_U8P) if u8 is not None else None, C.byref(stats)))
        self.last_stats = api.last_rtc_stats()
        return _canvases(api, n, h, w, rgb, u8)

    def trace_rays(self, origins, directions, depth=DEFAULT_RAY_RECURSION_DEPTH, fma=False):
        """World::color_at (world.rs:88-101) for arbitrary rays: returns (rgb[n,3], t[n], shape_handle[n])."""
        o, d = _api.f32(origins).reshape(-1, 3), _api.f32(directions).reshape(-1, 3)
        n = o.shape[0]
        rgb, t, shape = np.zeros((n, 3), np.float32), np.zeros(n, np.float32), np.zeros(n, np.int32)
        api = self.api
        api.check(api.lib.sg_trace_rays(api.ctx, self.handle, n, _api.fptr(o), _api.fptr(d), int(depth), int(fma),
                                        _api.fptr(rgb), _api.fptr(t), shape.ctypes.data_as(_IP)))
        return rgb, t, shape

    def set_option(self, option: int, value: int):
        """rtc_set_option: RTC_OPT_RENDER_SLICES = 4, RTC_OPT_ADAPTIVE_ORDER = 5, ..."""
        self.api.check(self.api.lib.sg_set_prepared_option(self.api.ctx, self.handle, int(option), int(value)))

    def flush_l2(self):
        self.api.check(self.api.lib.sg_flush_l2(self.api.ctx, self.handle))

    def release(self):
        if self.handle is not None:
            self.api.lib.sg_release_prepared(self.api.ctx, self.handle)
            self.handle = None


class CanvasU8:
    """What `Canvas::to_ppm` (canvas.rs:58-96) needs and nothing more: the frame's 8-bit plane — every channel through
    `scale_color` (canvas.rs:39-43) on the device.  Returned by Camera.render_b200_u8 (the Rust glue's `CanvasU8`)."""

    def __init__(self, width: int, height: int, u8: np.ndarray, api):
        self.width, self.height, self._u8, self.api = width, height, u8, api

    def to_u8(self) -> np.ndarray:
        return self._u8

    def to_ppm(self) -> str:
        api = self.api
        u8 = np.ascontiguousarray(self._u8)
        n = api.check(api.lib.sg_ppm_from_u8(api.ctx, self.width, self.height, u8.ctypes.data_as(_U8P), None, 0))
        buf = C.create_string_buffer(int(n))
        api.check(api.lib.sg_ppm_from_u8(api.ctx, self.width, self.height, u8.ctypes.data_as(_U8P), buf, n))
        return buf.raw[:n].decode("ascii")


class HostApi(_api.Api):
    """api.Api bound to librtc_host.so, plus the device-side controls that only the product has."""

    def __init__(self, lib_path=LIB_HOST):
        if not os.path.exists(lib_path) or not os.path.exists(LIB_DEVICE):
            raise ImportError(
                f"{lib_path} / {LIB_DEVICE} not built: run `python -m ray_tracer_challenge_b200.build` "
                "(there is no pure-Python or CPU fallback)")
        super().__init__(lib_path, _HOST_EXTRAS)
        api = self
        base_render = self.Camera.render

        def render_b200(camera, world, reflection_recursion_depth=DEFAULT_RAY_RECURSION_DEPTH, want_u8=True):
            """Camera::render_b200 — same signature and result as Camera::render (camera.rs:76-91)."""
            canvas = base_render(camera, world, reflection_recursion_depth, want_u8)
            camera.last_rtc_stats = api.last_rtc_stats()
            return canvas

        def render_b200_u8(camera, world, reflection_recursion_depth=DEFAULT_RAY_RECURSION_DEPTH, out_u8=None):
            """The demos' flow, `camera.render(world, depth).to_ppm()`, without the f32 plane ever leaving the device:
            one-shot (flatten, commit, render), 3 bytes per pixel over PCIe instead of 15."""
            w, h = camera.width_pixels, camera.height_pixels
            u8 = out_u8 if out_u8 is not None else np.zeros((h, w, 3), np.uint8)
            stats = SgStats()
            api.check(api.lib.sg_camera_render_shard(api.ctx, camera.handle, world.handle, int(reflection_recursion_depth), 0, 1,
                                                     None, u8.ctypes.data_as(_U8P), C.byref(stats)))
            camera.last_stats = stats
            camera.last_rtc_stats = api.last_rtc_stats()
            return CanvasU8(w, h, u8, api)

        self.Camera.render_b200 = render_b200
        self.Camera.render_b200_u8 = render_b200_u8
        self.Camera.render = render_b200
        self.Camera.prepare = lambda camera, world: PreparedScene(api, camera, world)

    def set_render_options(self, n_devices=1, device_ids=None, fma=False, detailed=False):
        ids = None
        if device_ids is not None:
            ids = (C.c_int * len(device_ids))(*device_ids)
            n_devices = len(device_ids)
        self.check(self.lib.sg_set_render_options(self.ctx, int(n_devices), ids, int(fma), int(detailed)))

    def set_bvh_builder(self, mode: int = -1):
        """RTC_OPT_BVH_BUILDER policy of this session: -1 automatic (device LBVH for one-shot renders of >= 10 000
        primitives, the host's binned SAH for prepared scenes), 0 always host, 1 always device."""
        self.check(self.lib.sg_set_bvh_builder(self.ctx, int(mode)))

    def set_exact_groups(self, on: bool = True):
        """RTC_OPT_EXACT_GROUPS for every later render, prepare and inspect of this session: grouped primitives and CSGs
        of tree scenes honour the reference's group box culls exactly (default off)."""
        self.check(self.lib.sg_set_exact_groups(self.ctx, 1 if on else 0))

    def last_rtc_stats(self) -> RtcStats:
        st = RtcStats()
        self.lib.sg_last_rtc_stats(self.ctx, C.byref(st))
        return st

    def render_views(self, world, cameras, depth=DEFAULT_RAY_RECURSION_DEPTH, want_u8=True):
        """The one-shot batch (Camera::render_b200 for several cameras of one canvas size): flatten the world once, commit it
        with the camera farthest out, render every view, release.  Returns one Canvas per camera."""
        cameras = list(cameras)
        if not cameras:
            raise ValueError("render_views needs at least one camera")
        n, w, h = len(cameras), cameras[0].width_pixels, cameras[0].height_pixels
        rgb, u8 = _view_planes(n, h, w, True, want_u8, None, None)
        stats = SgStats()
        self.check(self.lib.sg_camera_render_views(self.ctx, _handles(cameras), n, world.handle, int(depth), _api.fptr(rgb),
                                                   u8.ctypes.data_as(_U8P) if u8 is not None else None, C.byref(stats)))
        self.last_views_stats = self.last_rtc_stats()
        return _canvases(self, n, h, w, rgb, u8)

    def camera_view(self, camera) -> RtcView:
        """The RtcView a batch hands the device library for `camera` (the fields rtc_set_camera receives for it)."""
        v = RtcView()
        self.check(self.lib.sg_camera_view(self.ctx, camera.handle, C.byref(v)))
        return v

    def farthest_camera(self, cameras) -> int:
        """Index of the camera the one-shot batch commits with: the origin farthest out."""
        cameras = list(cameras)
        return self.check(self.lib.sg_farthest_camera(self.ctx, _handles(cameras), len(cameras)))

    def inspect(self, camera, world) -> dict:
        """rtc_scene_inspect: what a commit of (camera, world) would build — tree size, leaf size, small-scene path and
        shadow-filter eligibility, host time — without touching a device."""
        info, flatten_ms = RtcCommitInfo(), C.c_double()
        self.check(self.lib.sg_inspect(self.ctx, camera.handle, world.handle, C.byref(info), C.byref(flatten_ms)))
        out = info.as_dict()
        out["flatten_ms"] = flatten_ms.value
        return out

    def export_scene(self, camera, world) -> C.c_void_p:
        """The flattened (camera, world) as a raw RtcScene handle of include/rtc_b200.h; the caller destroys it with
        rtc_scene_destroy of device_library()."""
        scene = C.c_void_p()
        self.check(self.lib.sg_export_scene(self.ctx, camera.handle, world.handle, C.byref(scene)))
        return scene

    def flatten(self, world):
        """The flattener's output (no device needed): (prims, nodes, refs, prim_shape_handles, counts)."""
        counts = (C.c_int * 6)()
        self.check(self.lib.sg_flatten(self.ctx, world.handle, counts, None, None, None, None))
        prims = (RtcPrim * max(counts[0], 1))()
        nodes = (RtcNode * max(counts[1], 1))()
        refs = (C.c_int32 * max(counts[2], 1))()
        shapes = (C.c_int * max(counts[0], 1))()
        self.check(self.lib.sg_flatten(self.ctx, world.handle, counts, prims, nodes, refs, shapes))
        return (list(prims)[:counts[0]], list(nodes)[:counts[1]], list(refs)[:counts[2]], list(shapes)[:counts[0]],
                list(counts))


def new_session() -> HostApi:
    """A fresh scene context bound to the product libraries."""
    return HostApi()


def device_library() -> C.CDLL:
    """librtc_b200.so loaded directly (the raw C ABI of include/rtc_b200.h)."""
    return C.CDLL(LIB_DEVICE, mode=C.RTLD_GLOBAL)


_default: HostApi | None = None


def __getattr__(name):
    """Module-level access to a default session: `rt.Sphere()`, `rt.translation(...)`, `rt.Camera(...)`."""
    global _default
    if name.startswith("__"):
        raise AttributeError(name)
    if name in ("build", "scenes", "sharding", "multi"):  # submodules: `from ray_tracer_challenge_b200 import build`
        import importlib  # works before the libraries exist (build is how they come to exist)

        return importlib.import_module(f"{__name__}.{name}")
    if _default is None:
        _default = HostApi()
    return getattr(_default, name)
