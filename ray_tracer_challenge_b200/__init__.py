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
    "sg_render_prepared_samples": (_I, [_V, _I, _I, _I, _I, _I, _I, _FP, _U8P, C.POINTER(SgStats)]),
    "sg_camera_render_views": (_I, [_V, _IP, _I, _I, _I, _FP, _U8P, C.POINTER(SgStats)]),
    "sg_camera_view": (_I, [_V, _I, C.POINTER(RtcView)]),
    "sg_farthest_camera": (_I, [_V, _IP, _I]),
    "sg_camera_render_ppm": (C.c_int64, [_V, _I, _I, _I, C.c_void_p, C.c_int64, C.POINTER(SgStats)]),
    "sg_render_prepared_ppm": (C.c_int64, [_V, _I, _I, _I, C.c_void_p, C.c_int64, C.POINTER(SgStats)]),
    "sg_render_prepared_shard_ppm_rows": (_I, [_V, _I, _I, _I, _I, _I, C.c_void_p, C.POINTER(SgStats)]),
    "sg_render_prepared_shard_samples_ppm_rows": (_I, [_V, _I, _I, _I, _I, _I, _I, C.c_void_p, C.POINTER(SgStats)]),
    "sg_write_prepared_shard_ppm": (C.c_int64, [_V, _I, _I, _I, C.c_void_p, C.c_void_p, C.c_int64]),
    "sg_render_prepared_views_ppm": (C.c_int64, [_V, _I, _I, _I, _IP, _I, C.c_void_p, C.c_int64, C.POINTER(C.c_size_t),
                                                 C.POINTER(SgStats)]),
    "sg_camera_render_views_ppm": (C.c_int64, [_V, _IP, _I, _I, _I, C.c_void_p, C.c_int64, C.POINTER(C.c_size_t),
                                               C.POINTER(SgStats)]),
    "sg_render_prepared_views_samples": (_I, [_V, _I, _I, _I, _IP, _I, _I, _FP, _U8P, C.POINTER(SgStats)]),
    "sg_render_prepared_views_samples_ppm": (C.c_int64, [_V, _I, _I, _I, _IP, _I, _I, C.c_void_p, C.c_int64, C.POINTER(C.c_size_t),
                                                         C.POINTER(SgStats)]),
    "sg_camera_render_views_samples": (_I, [_V, _IP, _I, _I, _I, _I, _FP, _U8P, C.POINTER(SgStats)]),
    "sg_camera_render_views_samples_ppm": (C.c_int64, [_V, _IP, _I, _I, _I, _I, C.c_void_p, C.c_int64, C.POINTER(C.c_size_t),
                                                       C.POINTER(SgStats)]),
    "rtc_ppm_bound": (C.c_size_t, [C.c_uint32, C.c_uint32]),  # librtc_b200.so, reached through the host library
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


def _ppm_buffer(api, w, h, out, n=1):
    """The bytes rtc_render_ppm (n = 1) or rtc_render_views_ppm (n views) writes into: the caller's C-contiguous uint8 array
    (e.g. over pinned memory) or a new one, at least n * rtc_ppm_bound bytes."""
    bound = api.lib.rtc_ppm_bound(w, h)
    buf = out if out is not None else np.empty(n * bound, np.uint8)
    if not isinstance(buf, np.ndarray) or buf.dtype != np.uint8 or not buf.flags.c_contiguous or not buf.flags.writeable \
            or buf.nbytes < n * bound:
        need = f"rtc_ppm_bound = {bound}" if n == 1 else f"{n} * rtc_ppm_bound = {n * bound}"
        raise ValueError(f"out must be a writable C-contiguous uint8 array of at least {need} bytes")
    return buf


def _row_bytes(row_bytes, h):
    """The row lengths of a shard's text (rtc_render_shard_ppm_rows / rtc_write_shard_ppm): a writable C-contiguous uint64
    array of one entry per frame row."""
    if not isinstance(row_bytes, np.ndarray) or row_bytes.dtype != np.uint64 or row_bytes.shape != (h,) \
            or not row_bytes.flags.c_contiguous or not row_bytes.flags.writeable:
        raise ValueError(f"row_bytes must be a writable C-contiguous uint64 array of shape ({h},)")
    return row_bytes


def _ppm_texts(buf, offsets):
    """The views' texts of rtc_render_views_ppm: view i's is buf[offsets[i]:offsets[i + 1]]."""
    return [buf[offsets[i]:offsets[i + 1]].tobytes().decode("ascii") for i in range(len(offsets) - 1)]


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

    def render_samples(self, samples, depth=DEFAULT_RAY_RECURSION_DEPTH, want_rgb=True, want_u8=True, out_rgb=None, out_u8=None,
                       fma=False, shard=0, n_shards=0):
        """rtc_render_samples: the committed scene anti-aliased with samples x samples samples per pixel, each sample a pixel
        of the reference's render at samples times the canvas size, box-filtered on the device (samples = 1 is render()'s
        frame).  Buffers may be caller-supplied (e.g. pinned); want_* = False leaves the frame on the device.  shard /
        n_shards as render's: n_shards >= 1 renders and writes only that shard's bands (rtc_render_shard_samples; a scene
        committed on one device), the other rows of the buffers untouched."""
        w, h = self.camera.width_pixels, self.camera.height_pixels
        rgb, u8 = _view_planes(1, h, w, want_rgb, want_u8, None if out_rgb is None else out_rgb[None],
                               None if out_u8 is None else out_u8[None])
        stats = SgStats()
        api = self.api
        api.check(api.lib.sg_render_prepared_samples(
            api.ctx, self.handle, int(depth), int(samples), int(shard), int(n_shards), int(fma),
            _api.fptr(rgb) if rgb is not None else None, u8.ctypes.data_as(_U8P) if u8 is not None else None, C.byref(stats)))
        self.last_stats = api.last_rtc_stats()
        return Canvas(w, h, rgb[0] if rgb is not None else None, u8[0] if u8 is not None else None, api=api)

    def render_views_samples(self, cameras, samples, depth=DEFAULT_RAY_RECURSION_DEPTH, want_rgb=True, want_u8=True, out_rgb=None,
                             out_u8=None, fma=False):
        """rtc_render_views_samples: render_views' batch anti-aliased as render_samples does it — view i is
        render_samples(samples) of this scene committed with cameras[i].  Returns one Canvas per camera, views into one
        (n, h, w, 3) array per plane; want_* = False leaves the frames on the device.  The reach rule is render_views'."""
        cameras = list(cameras)
        n, w, h = len(cameras), self.camera.width_pixels, self.camera.height_pixels
        rgb, u8 = _view_planes(n, h, w, want_rgb, want_u8, out_rgb, out_u8)
        stats = SgStats()
        api = self.api
        api.check(api.lib.sg_render_prepared_views_samples(
            api.ctx, self.handle, int(depth), n, _handles(cameras), int(samples), int(fma),
            _api.fptr(rgb) if rgb is not None else None, u8.ctypes.data_as(_U8P) if u8 is not None else None, C.byref(stats)))
        self.last_stats = api.last_rtc_stats()
        return _canvases(api, n, h, w, rgb, u8)

    def render_views_samples_ppm(self, cameras, samples, depth=DEFAULT_RAY_RECURSION_DEPTH, out=None, fma=False) -> list:
        """rtc_render_views_samples_ppm: render_views_samples' batch with each view's `Canvas::to_ppm` text written on the
        device.  Returns one str per camera; `out` as render_views_ppm's."""
        cameras = list(cameras)
        n, w, h = len(cameras), self.camera.width_pixels, self.camera.height_pixels
        api = self.api
        buf = _ppm_buffer(api, w, h, out, max(n, 1))
        offsets = (C.c_size_t * (n + 1))()
        stats = SgStats()
        api.check(api.lib.sg_render_prepared_views_samples_ppm(api.ctx, self.handle, int(depth), n, _handles(cameras), int(samples),
                                                               int(fma), buf.ctypes.data, buf.nbytes, offsets, C.byref(stats)))
        self.last_stats = api.last_rtc_stats()
        return _ppm_texts(buf, list(offsets))

    def render_samples_ppm(self, samples, depth=DEFAULT_RAY_RECURSION_DEPTH, out=None, fma=False) -> str:
        """`render_samples(samples).to_ppm()` with the text written on the device: the committed camera rendered as a one-view
        rtc_render_views_samples_ppm batch.  `out` as render_ppm's."""
        return self.render_views_samples_ppm([self.camera], samples, depth, out, fma)[0]

    def render_ppm(self, depth=DEFAULT_RAY_RECURSION_DEPTH, out=None, fma=False) -> str:
        """rtc_render_ppm: the committed scene rendered and its frame's `Canvas::to_ppm` text (canvas.rs:58-96) written on the
        device.  `out`: where the bytes land (a writable uint8 array of at least rtc_ppm_bound bytes, e.g. over pinned memory);
        a new pageable one by default."""
        w, h = self.camera.width_pixels, self.camera.height_pixels
        api = self.api
        buf = _ppm_buffer(api, w, h, out)
        stats = SgStats()
        n = api.check(api.lib.sg_render_prepared_ppm(api.ctx, self.handle, int(depth), int(fma), buf.ctypes.data, buf.nbytes,
                                                     C.byref(stats)))
        self.last_stats = api.last_rtc_stats()
        return buf[:n].tobytes().decode("ascii")

    def render_shard_ppm_rows(self, shard, n_shards, row_bytes, depth=DEFAULT_RAY_RECURSION_DEPTH, fma=False, samples=0):
        """rtc_render_shard_ppm_rows, the first phase of one shard's text of a frame shared by several processes: renders the
        shard's bands (rtc_render_shard, the frame left on the device) and writes the byte length of each of their rows'
        text into `row_bytes` (a uint64 array of one entry per frame row; the other shards' entries are not touched).  The
        callers then exchange the entries (multi.render_ppm_shared does it through shared memory) and call write_shard_ppm.
        samples >= 1 renders the shard anti-aliased instead (rtc_render_shard_samples_ppm_rows): the texts then make up
        render_samples_ppm(samples)'s."""
        h = self.camera.height_pixels
        api = self.api
        row_bytes = _row_bytes(row_bytes, h)
        stats = SgStats()
        if samples:
            api.check(api.lib.sg_render_prepared_shard_samples_ppm_rows(api.ctx, self.handle, int(depth), int(samples), int(shard),
                                                                        int(n_shards), int(fma), row_bytes.ctypes.data,
                                                                        C.byref(stats)))
        else:
            api.check(api.lib.sg_render_prepared_shard_ppm_rows(api.ctx, self.handle, int(depth), int(shard), int(n_shards),
                                                                int(fma), row_bytes.ctypes.data, C.byref(stats)))
        self.last_stats = api.last_rtc_stats()

    def write_shard_ppm(self, shard, n_shards, row_bytes, out) -> int:
        """rtc_write_shard_ppm, the second phase: given every row's length (all shards' entries of `row_bytes`), writes the
        text of this shard's bands at their offsets in `out` (a writable uint8 array of at least rtc_ppm_bound bytes, shared
        by the ranks); shard 0 also writes the header.  Returns the whole text's length; once every shard has written,
        out[:length] is render_ppm's text."""
        w, h = self.camera.width_pixels, self.camera.height_pixels
        api = self.api
        row_bytes = _row_bytes(row_bytes, h)
        if out is None:
            raise ValueError("write_shard_ppm needs out: the buffer every shard writes its bands into")
        buf = _ppm_buffer(api, w, h, out)
        return api.check(api.lib.sg_write_prepared_shard_ppm(api.ctx, self.handle, int(shard), int(n_shards), row_bytes.ctypes.data,
                                                             buf.ctypes.data, buf.nbytes))

    def render_views_ppm(self, cameras, depth=DEFAULT_RAY_RECURSION_DEPTH, out=None, fma=False) -> list:
        """rtc_render_views_ppm: every camera (of this scene's canvas size) rendered from the committed scene in one batch,
        and each view's `Canvas::to_ppm` text written on the device.  Returns one str per camera.  `out`: where the bytes
        land (a writable uint8 array of at least len(cameras) * rtc_ppm_bound bytes, e.g. over pinned memory); a new
        pageable one by default.  The reach rule is render_views'."""
        cameras = list(cameras)
        n, w, h = len(cameras), self.camera.width_pixels, self.camera.height_pixels
        api = self.api
        buf = _ppm_buffer(api, w, h, out, max(n, 1))
        offsets = (C.c_size_t * (n + 1))()
        stats = SgStats()
        api.check(api.lib.sg_render_prepared_views_ppm(api.ctx, self.handle, int(depth), n, _handles(cameras), int(fma),
                                                       buf.ctypes.data, buf.nbytes, offsets, C.byref(stats)))
        self.last_stats = api.last_rtc_stats()
        return _ppm_texts(buf, list(offsets))

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

        def render_b200_ppm(camera, world, reflection_recursion_depth=DEFAULT_RAY_RECURSION_DEPTH, out=None) -> str:
            """The demos' flow, `camera.render(world, depth).to_ppm()`, in one call: flatten, commit, render, and the frame's
            PPM text written on the device (rtc_render_ppm).  `out` as PreparedScene.render_ppm's."""
            w, h = camera.width_pixels, camera.height_pixels
            buf = _ppm_buffer(api, w, h, out)
            stats = SgStats()
            n = api.check(api.lib.sg_camera_render_ppm(api.ctx, camera.handle, world.handle, int(reflection_recursion_depth),
                                                       buf.ctypes.data, buf.nbytes, C.byref(stats)))
            camera.last_stats = stats
            camera.last_rtc_stats = api.last_rtc_stats()
            return buf[:n].tobytes().decode("ascii")

        def render_b200_samples(camera, world, samples, reflection_recursion_depth=DEFAULT_RAY_RECURSION_DEPTH, want_u8=True):
            """Camera::render_b200_samples — render_b200 anti-aliased with samples x samples samples per pixel
            (rtc_render_samples): flatten, commit, render, release."""
            prepared = PreparedScene(api, camera, world)
            try:
                canvas = prepared.render_samples(samples, reflection_recursion_depth, want_u8=want_u8)
            finally:
                prepared.release()
            camera.last_rtc_stats = prepared.last_stats
            return canvas

        def render_b200_samples_ppm(camera, world, samples, reflection_recursion_depth=DEFAULT_RAY_RECURSION_DEPTH, out=None) -> str:
            """The anti-aliased demo flow, `camera.render_b200_samples(world, samples).to_ppm()`, in one call: flatten,
            commit, render with samples x samples samples per pixel and write the PPM text on the device
            (rtc_render_views_samples_ppm of one view), release.  `out` as PreparedScene.render_ppm's."""
            prepared = PreparedScene(api, camera, world)
            try:
                text = prepared.render_samples_ppm(samples, reflection_recursion_depth, out)
            finally:
                prepared.release()
            camera.last_rtc_stats = prepared.last_stats
            return text

        self.Camera.render_b200 = render_b200
        self.Camera.render_b200_samples = render_b200_samples
        self.Camera.render_b200_samples_ppm = render_b200_samples_ppm
        self.Camera.render_b200_u8 = render_b200_u8
        self.Camera.render_b200_ppm = render_b200_ppm
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

    def render_views_ppm(self, world, cameras, depth=DEFAULT_RAY_RECURSION_DEPTH, out=None) -> list:
        """The one-shot batch in text: render_views' flatten and commit, then rtc_render_views_ppm.  Returns
        `camera.render(world, depth).to_ppm()` for each camera; `out` as PreparedScene.render_views_ppm's."""
        cameras = list(cameras)
        if not cameras:
            raise ValueError("render_views_ppm needs at least one camera")
        n, w, h = len(cameras), cameras[0].width_pixels, cameras[0].height_pixels
        buf = _ppm_buffer(self, w, h, out, n)
        offsets = (C.c_size_t * (n + 1))()
        stats = SgStats()
        self.check(self.lib.sg_camera_render_views_ppm(self.ctx, _handles(cameras), n, world.handle, int(depth), buf.ctypes.data,
                                                       buf.nbytes, offsets, C.byref(stats)))
        self.last_views_stats = self.last_rtc_stats()
        return _ppm_texts(buf, list(offsets))

    def render_views_samples(self, world, cameras, samples, depth=DEFAULT_RAY_RECURSION_DEPTH, want_u8=True):
        """The one-shot anti-aliased batch: render_views' flatten and commit, then rtc_render_views_samples.  Canvas i is
        `cameras[i].render_b200_samples(world, samples, depth)`."""
        cameras = list(cameras)
        if not cameras:
            raise ValueError("render_views_samples needs at least one camera")
        n, w, h = len(cameras), cameras[0].width_pixels, cameras[0].height_pixels
        rgb, u8 = _view_planes(n, h, w, True, want_u8, None, None)
        stats = SgStats()
        self.check(self.lib.sg_camera_render_views_samples(self.ctx, _handles(cameras), n, world.handle, int(depth), int(samples),
                                                           _api.fptr(rgb), u8.ctypes.data_as(_U8P) if u8 is not None else None,
                                                           C.byref(stats)))
        self.last_views_stats = self.last_rtc_stats()
        return _canvases(self, n, h, w, rgb, u8)

    def render_views_samples_ppm(self, world, cameras, samples, depth=DEFAULT_RAY_RECURSION_DEPTH, out=None) -> list:
        """The one-shot anti-aliased batch in text: render_views' flatten and commit, then rtc_render_views_samples_ppm.
        Returns `cameras[i].render_b200_samples(world, samples, depth).to_ppm()` for each camera; `out` as
        PreparedScene.render_views_ppm's."""
        cameras = list(cameras)
        if not cameras:
            raise ValueError("render_views_samples_ppm needs at least one camera")
        n, w, h = len(cameras), cameras[0].width_pixels, cameras[0].height_pixels
        buf = _ppm_buffer(self, w, h, out, n)
        offsets = (C.c_size_t * (n + 1))()
        stats = SgStats()
        self.check(self.lib.sg_camera_render_views_samples_ppm(self.ctx, _handles(cameras), n, world.handle, int(depth), int(samples),
                                                               buf.ctypes.data, buf.nbytes, offsets, C.byref(stats)))
        self.last_views_stats = self.last_rtc_stats()
        return _ppm_texts(buf, list(offsets))

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
