"""Loader and Python side of tests/emu/tree_probe.cpp (the tree builders of a commit, exposed for exact checks), and the
input families the device tree builder is checked on.  Test infrastructure only."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

from tests.lbvh_reference import lbvh_reference

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA = "/usr/local/cuda"

I32P = C.POINTER(C.c_int32)
U8P = C.POINTER(C.c_uint8)
FP = C.POINTER(C.c_float)
BUILDER_CALLBACK = C.CFUNCTYPE(C.c_int, FP, U8P, C.c_int, C.c_int, I32P, C.c_void_p, I32P, I32P)


def ptr(a, kind):
    return a.ctypes.data_as(kind)


class Probe:
    def __init__(self, device, lib):
        self.device, self.lib = device, lib
        lib.probe_flatten.argtypes = [C.c_void_p, C.c_int, C.c_void_p, I32P]
        lib.probe_copy_flat.argtypes = [C.c_void_p, C.c_void_p, I32P]
        lib.probe_copy_input.argtypes = [FP, U8P]
        lib.probe_positions.argtypes = [C.c_void_p, FP, U8P, U8P]
        lib.probe_lbvh.argtypes = [FP, U8P, C.c_int, C.c_int, I32P, C.c_void_p, I32P, I32P]
        lib.probe_release.argtypes = []

    def lbvh(self, boxes, closed, leaf_size):
        """rtc::lbvh_build: (rc, order, nodes as (n - 1) x 16 int32 words, root, depth)."""
        boxes = np.ascontiguousarray(boxes, np.float32).reshape(-1, 6)
        closed = np.ascontiguousarray(closed, np.uint8)
        n = len(boxes)
        order = np.full(max(n, 1), -7, np.int32)
        nodes = np.zeros((max(n - 1, 1), 16), np.int32)
        root, depth = C.c_int32(-7), C.c_int32(-7)
        rc = self.lib.probe_lbvh(ptr(boxes, FP), ptr(closed, U8P), n, leaf_size, ptr(order, I32P), nodes.ctypes.data,
                                 C.byref(root), C.byref(depth))
        return rc, order[:n], nodes[: max(n - 1, 0)], root.value, depth.value

    def flatten(self, scene, mode, callback=None):
        """rtc::flatten of the scene with builder `mode` (0 host SAH, 1 `callback`, 2 device): a dict of the result."""
        info = np.zeros(9, np.int32)
        rc = self.lib.probe_flatten(scene, mode, C.cast(callback, C.c_void_p) if callback else None, ptr(info, I32P))
        assert rc == 0, self.device.rtc_last_error()
        m, root, depth, leaf, n_pos, on_device, n_linear, calls, n_in = (int(v) for v in info)
        nodes = np.zeros((max(m, 1), 16), np.int32)
        head = np.zeros((max(2 * n_pos, 1), 4), np.int32)
        linear = np.zeros(max(n_linear, 1), np.int32)
        self.lib.probe_copy_flat(nodes.ctypes.data, head.ctypes.data, ptr(linear, I32P))
        boxes = np.zeros((max(n_in, 1), 6), np.float32)
        closed = np.zeros(max(n_in, 1), np.uint8)
        self.lib.probe_copy_input(ptr(boxes, FP), ptr(closed, U8P))
        pos_box = np.zeros((max(n_pos, 1), 6), np.float32)
        pos_closed = np.zeros(max(n_pos, 1), np.uint8)
        in_csg = np.zeros(max(n_pos, 1), np.uint8)
        self.lib.probe_positions(scene, ptr(pos_box, FP), ptr(pos_closed, U8P), ptr(in_csg, U8P))
        # the tree's items are the positions that are neither inside a CSG nor in the linear list: they come first
        item = in_csg[:n_pos] == 0
        item[linear[:n_linear]] = False
        n_tree = int(item.sum())
        assert item[:n_tree].all(), "the tree's items are not the first positions"
        return dict(nodes=nodes[:m], root=root, depth=depth, leaf_size=leaf, n_pos=n_pos, built_on_device=on_device,
                    calls=calls, head=head, n_tree=n_tree, input_boxes=boxes[:n_in], input_closed=closed[:n_in],
                    pos_box=pos_box[:n_tree], pos_closed=pos_closed[:n_tree].astype(bool))


def load_probe(tmp_path_factory):
    import ray_tracer_challenge_b200 as rt

    if shutil.which("g++") is None or not all(os.path.isdir(os.path.join(CUDA, d)) for d in ("include", "lib64")):
        pytest.skip("needs g++, the CUDA headers and libcudart")
    out = tmp_path_factory.mktemp("probe") / "libtree_probe.so"
    lib_dir = os.path.dirname(rt.LIB_DEVICE)
    cuda_lib = os.path.join(CUDA, "lib64")
    subprocess.run(["g++", "-std=c++17", "-O1", "-fPIC", "-shared", "-I", os.path.join(CUDA, "include"),
                    "-I", os.path.join(ROOT, "ray_tracer_challenge_b200", "csrc"), os.path.join(ROOT, "tests", "emu", "tree_probe.cpp"),
                    "-o", str(out), "-L", lib_dir, "-lrtc_b200", f"-Wl,-rpath,{lib_dir}", "-L", cuda_lib, "-lcudart",
                    f"-Wl,-rpath,{cuda_lib}"], check=True)
    device = rt.device_library()  # the raw C ABI; RTLD_GLOBAL, so the harness binds rtc::flatten and rtc::lbvh_build from it
    device.rtc_last_error.restype = C.c_char_p
    device.rtc_scene_destroy.argtypes = [C.c_void_p]
    return Probe(device, C.CDLL(str(out)))


def reference_callback(log=None):
    """A TreeBuilderFn body for probe_flatten mode 1: lbvh_reference in place of the device builder."""

    def build(boxes, closed, n, leaf_size, order, nodes, root, depth):
        b = np.ctypeslib.as_array(boxes, (n, 6)).copy()
        c = np.ctypeslib.as_array(closed, (n,)).copy()
        o, w, r, d = lbvh_reference(b, c, leaf_size)
        C.memmove(order, o.ctypes.data, o.nbytes)
        C.memmove(nodes, w.ctypes.data, w.nbytes)
        root[0], depth[0] = r, d
        if log is not None:
            log.append((n, leaf_size))
        return 0

    return BUILDER_CALLBACK(build)


def assert_same_tree(got, want):
    """(order, nodes, root, depth) equal bit for bit; box words compared as floats (+0 == -0)."""
    order, nodes, root, depth = got
    w_order, w_nodes, w_root, w_depth = want
    assert root == w_root, (root, w_root)
    assert depth == w_depth, (depth, w_depth)
    bad = np.flatnonzero(order != w_order)
    assert not len(bad), f"order differs at {len(bad)} positions, first {bad[0]}: {order[bad[0]]} != {w_order[bad[0]]}"
    links_bad = np.flatnonzero((nodes[:, 12:] != w_nodes[:, 12:]).any(axis=1))
    assert not len(links_bad), f"links / closed bits of {len(links_bad)} nodes differ, first {links_bad[0]}: " \
                               f"{nodes[links_bad[0], 12:]} != {w_nodes[links_bad[0], 12:]}"
    fb, wb = nodes[:, :12].view(np.float32), w_nodes[:, :12].view(np.float32)
    boxes_bad = np.flatnonzero(((fb != wb) & ~(np.isnan(fb) & np.isnan(wb))).any(axis=1))
    assert not len(boxes_bad), f"boxes of {len(boxes_bad)} nodes differ, first {boxes_bad[0]}: {fb[boxes_bad[0]]} != {wb[boxes_bad[0]]}"


# ---- input families of the device tree builder: n x 6 boxes (lo.xyz, hi.xyz) and n closed flags
def _boxes(centre, half):
    centre, half = np.asarray(centre, np.float32), np.asarray(half, np.float32)
    return np.concatenate([centre - half, centre + half], axis=1).astype(np.float32)


def family(name, n, seed=0):
    rng = np.random.default_rng(seed)
    closed = np.ones(n, np.uint8)
    if name == "uniform":
        lo = rng.uniform(-100, 100, (n, 3)).astype(np.float32)
        boxes = np.concatenate([lo, lo + rng.uniform(0, 3, (n, 3)).astype(np.float32)], axis=1)
        closed = (rng.random(n) < 0.5).astype(np.uint8)
    elif name == "clusters":  # tight clusters of coincident centroids (dyadic centres and half-extents: exact sums)
        centres = rng.integers(-64, 64, (max(1, n // 40), 3)) * 0.5
        boxes = _boxes(centres[rng.integers(0, len(centres), n)], rng.choice([0.125, 0.25, 1.0], (n, 3)))
    elif name == "all_equal":  # one centroid for every item: the position tie-break builds the whole tree
        boxes = _boxes(np.tile([1.5, -2.0, 3.25], (n, 1)), rng.choice([0.25, 0.5, 2.0], (n, 3)))
    elif name == "collinear":  # two axes of zero extent: their scale is 0
        c = np.zeros((n, 3))
        c[:, 0] = rng.uniform(-50, 50, n)
        c[:, 1], c[:, 2] = 2.0, -1.0
        boxes = _boxes(c, np.full((n, 3), 0.5))
    elif name == "geometric":  # spacing halves from item to item: most codes equal at the dense end
        x = np.cumsum(2.0 ** -np.arange(n, dtype=np.float64).clip(max=100)) * 1e3
        c = np.stack([x, np.zeros(n), np.zeros(n)], axis=1)
        boxes = _boxes(c, np.full((n, 3), 1e-3))
    elif name == "huge":  # x near +-1e37; y: some centres overflow to +-inf (range inf, scale 0, (c - lo) * 0 NaN)
        c = np.zeros((n, 3), np.float32)
        c[:, 0] = rng.uniform(-1e37, 1e37, n)
        c[:, 1] = rng.choice([-3e38, -1e37, 0.0, 1e37, 3e38], n)
        c[:, 2] = rng.uniform(-1.6e38, 1.6e38, n)
        boxes = np.concatenate([c, c], axis=1)  # lo + hi of a box at +-3e38 overflows: its centroid is +-inf
    elif name == "tiny":  # centroid range near 1e-40 (denormal): cells / range = inf, (c - lo) * inf NaN at lo, inf above
        c = np.zeros((n, 3), np.float32)
        c[:, 0] = (rng.integers(0, 8, n) * 2.0 ** -133).astype(np.float32)
        c[:, 1] = rng.uniform(-1, 1, n)
        c[:, 2] = (rng.integers(-3, 3, n) * 2.0 ** -140).astype(np.float32)
        boxes = np.concatenate([c, c], axis=1)
    elif name == "mixed_closed":  # most items closed: whole subtrees are, their ancestors are not
        lo = rng.uniform(-10, 10, (n, 3)).astype(np.float32)
        boxes = np.concatenate([lo, lo + np.float32(0.1)], axis=1)
        closed = (rng.random(n) < 0.97).astype(np.uint8)
    else:
        raise ValueError(name)
    return np.ascontiguousarray(boxes, np.float32), closed


FAMILIES = ["uniform", "clusters", "all_equal", "collinear", "geometric", "huge", "tiny", "mixed_closed"]
