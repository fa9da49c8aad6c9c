"""The trees of a commit, checked whole and without a GPU.

- The NumPy reference of the device tree builder (tests/lbvh_reference.py) builds Karras' example tree and passes the
  structural checker (tests/bvh_check.py) on every input family the device builder is checked on.
- The host's binned-SAH trees pass the checker on the parity scenes and on degenerate layouts of 10^5 spheres.
- rtc::flatten, given the reference as its tree builder through tests/emu/tree_probe.cpp, takes a builder's tree from
  1 024 bounded items on, and reorders the items by the builder's `order`.
The device builder itself is compared with the reference bit for bit in test_gpu_lbvh_exact.py."""
import ctypes as C

import numpy as np
import pytest

from ray_tracer_challenge_b200 import scenes
from tests.bvh_check import check_tree
from tests.lbvh_reference import code_bits, lbvh_reference, topology
from tests.tree_probe import FAMILIES, assert_same_tree, family, load_probe, reference_callback


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    return load_probe(tmp_path_factory)


@pytest.fixture(scope="module")
def host():
    import ray_tracer_challenge_b200 as rt

    return rt.new_session()


def test_reference_topology_is_karras_figure_3():
    """Karras 2012, Fig. 3: eight sorted keys; internal node i has i at one end of its range."""
    codes = np.array([0b00001, 0b00010, 0b00100, 0b00101, 0b10011, 0b11000, 0b11001, 0b11110], np.uint64)
    first, last, split, left, right, _ = topology(codes)
    want = {  # node: (first, last, split, left, right); ~k is leaf k
        0: (0, 7, 3, 3, 4),
        1: (0, 1, 0, ~0, ~1),
        2: (2, 3, 2, ~2, ~3),
        3: (0, 3, 1, 1, 2),
        4: (4, 7, 4, ~4, 5),
        5: (5, 7, 6, 6, ~7),
        6: (5, 6, 5, ~5, ~6),
    }
    for i, (f, l, g, a, b) in want.items():
        assert (first[i], last[i], split[i], left[i], right[i]) == (f, l, g, a, b), i


def test_reference_splits_equal_codes_by_position():
    """Equal codes: the split falls at the highest differing bit of the first and last positions."""
    first, last, split, left, right, _ = topology(np.zeros(6, np.uint64))
    # [0, 5]: bit 2 -> split 3; [0, 3]: bit 1 -> 1; [4, 5]: 4; [0, 1]: 0; [2, 3]: 2
    assert list(split) == [3, 0, 2, 1, 4]
    assert (first[0], last[0], left[0], right[0]) == (0, 5, 3, 4)


def test_code_widths():
    """3 * bits + ceil(log2 n) <= kBvhStack - 4: 11 bits per axis at 1 024 items, 9 at 10^5, 8 above 2^17 (the sizes
    test_gpu_lbvh_exact builds), never more than 21."""
    assert [code_bits(n) for n in (2, 1024, 1025, 100_000, 131_072, 131_073)] == [14, 11, 11, 9, 9, 8]


@pytest.mark.parametrize("fam", FAMILIES)
@pytest.mark.parametrize("n", [2, 3, 16, 17, 1024, 1025, 4097])
def test_reference_trees_pass_the_checker(fam, n):
    boxes, closed = family(fam, n, seed=n)
    for leaf in (1, 4, 16):
        order, nodes, root, depth = lbvh_reference(boxes, closed, leaf)
        assert sorted(order) == list(range(n))
        check_tree(nodes, root, leaf, n, boxes[order], closed[order], depth)


def test_checker_rejects_broken_trees():
    """Each invariant the checker states, broken once in a valid tree, is caught."""
    boxes, closed = family("mixed_closed", 300, seed=5)
    order, nodes, root, depth = lbvh_reference(boxes, closed, 4)
    args = (4, 300, boxes[order], closed[order])
    check_tree(nodes, root, *args, depth)

    def broken(edit):
        bad = nodes.copy()
        edit(bad, bad.view(np.float32))
        return bad

    # nodes the tree links to (subtrees of at most leaf_size items are leaves: their nodes are never reached)
    reached = np.zeros(len(nodes), bool)
    reached[root] = True
    reached[nodes[:, 12:14][nodes[:, 12:14] >= 0]] = True
    inner = int(np.flatnonzero(reached & (nodes[:, 12] >= 0) & (nodes[:, 13] >= 0))[0])
    leafy = int(np.flatnonzero(reached & (nodes[:, 12] < 0))[0])
    cases = {
        "node reached twice": broken(lambda w, f: w.__setitem__((inner, 13), w[inner, 12])),
        "leaf moved by one position": broken(lambda w, f: w.__setitem__((leafy, 12), ~(~w[leafy, 12] + 16))),
        "leaf of 5 items": broken(lambda w, f: w.__setitem__((leafy, 12), ~((~w[leafy, 12] >> 4 << 4) | 4))),
        "box wider than the union": broken(lambda w, f: f.__setitem__((inner, 0), f[inner, 0] - 1.0)),
        "item outside its leaf's box": broken(lambda w, f: f.__setitem__((leafy, 3), f[leafy, 0])),
        "closed bit flipped": broken(lambda w, f: w.__setitem__((0, 14), w[0, 14] ^ 1)),
    }
    for what, bad in cases.items():
        try:
            check_tree(bad, root, *args, depth)
        except AssertionError:
            continue
        raise AssertionError(f"not caught: {what}")
    with pytest.raises(AssertionError, match="reported"):
        check_tree(nodes, root, *args, depth + 1)


def _check_flat(flat):
    check_tree(flat["nodes"], flat["root"], flat["leaf_size"], flat["n_tree"], flat["pos_box"], flat["pos_closed"], flat["depth"])


PARITY_SCENES = {
    "stress": (scenes.stress, dict(width=64, height=36, n_spheres=1500, n_each=6, n_csg=6)),
    "dragon_element": (scenes.dragon_element, dict(width=64, height=36, n_u=48, n_v=24)),
    "here_be_dragons": (scenes.here_be_dragons, dict(width=64, height=32, n_u=16, n_v=8)),
    "csg_gallery": (scenes.csg_gallery, dict(width=64, height=40)),
}


@pytest.mark.parametrize("name", sorted(PARITY_SCENES))
def test_host_trees_of_the_parity_scenes_pass_the_checker(name, probe, host):
    make, kw = PARITY_SCENES[name]
    cam, world = make(host, **kw)[:2]
    scene = host.export_scene(cam, world)
    try:
        if name == "csg_gallery":  # a small scene: give it a tree (every CSG root is one item)
            probe.device.rtc_set_option.argtypes = [C.c_void_p, C.c_int32, C.c_int64]
            assert probe.device.rtc_set_option(scene, 3, 1) == 0  # RTC_OPT_BVH_MIN_PRIMS
        flat = probe.flatten(scene, 0)
        assert flat["built_on_device"] == 0 and flat["calls"] == 0 and flat["n_tree"] > 2
        _check_flat(flat)
    finally:
        probe.device.rtc_scene_destroy(scene)


def _sphere_scene(probe, centres, radius=1.0):
    """A raw scene of spheres at `centres` (one API primitive, one tree item each, in this order)."""
    import ray_tracer_challenge_b200 as rt

    lib = probe.device
    scene = C.c_void_p()
    assert lib.rtc_scene_create(C.byref(scene)) == 0
    ident = (C.c_float * 16)(1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1)
    lib.rtc_set_camera.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_float)]
    assert lib.rtc_set_camera(scene, 16, 8, 1.0, 0.5, 2.0 / 16, ident) == 0
    assert lib.rtc_set_point_light(scene, (C.c_float * 3)(-10, 10, -10), (C.c_float * 3)(1, 1, 1)) == 0

    class Material(C.Structure):  # include/rtc_b200.h: RtcMaterial
        _fields_ = [("color", C.c_float * 3), ("v", C.c_float * 7), ("pattern", C.c_int32)]

    mat = Material()
    mat.color[:], mat.v[:], mat.pattern = [1, 1, 1], [0.1, 0.9, 0.9, 200.0, 0.0, 0.0, 1.0], -1
    assert lib.rtc_set_materials(scene, 1, C.byref(mat)) == 0
    n = len(centres)
    base = rt.RtcPrim()
    base.type, base.material, base.casts_shadow, base.parent = 0, 0, 1, -1
    base.inv[:] = list(ident)
    raw = np.frombuffer(bytes(base), np.uint8)
    prims = (rt.RtcPrim * n)()
    words = np.ctypeslib.as_array(C.cast(prims, C.POINTER(C.c_uint8)), (n, C.sizeof(rt.RtcPrim)))
    words[:] = raw
    f = words.view(np.float32)
    inv, lo, hi = rt.RtcPrim.inv.offset // 4, rt.RtcPrim.bbox_min.offset // 4, rt.RtcPrim.bbox_max.offset // 4
    c = np.asarray(centres, np.float32)
    for a in range(3):
        f[:, inv + 4 * a + 3] = -c[:, a] / radius
        f[:, inv + 5 * a] = 1.0 / radius
        f[:, lo + a] = c[:, a] - radius
        f[:, hi + a] = c[:, a] + radius
    assert lib.rtc_set_primitives(scene, n, prims) == 0, lib.rtc_last_error()
    return scene


@pytest.mark.parametrize("layout", ["coincident", "geometric", "line"])
def test_host_trees_of_degenerate_layouts_pass_the_checker(layout, probe):
    """test_c_abi's 10^5 spheres with one centre, geometrically shrinking spacing (SAH peels one sphere per level) and on
    a line: the balanced fallback of the host builder keeps every item and every box."""
    n = 100_000
    c = np.zeros((n, 3))
    if layout == "geometric":
        c[:, 0] = np.cumsum(2.0 ** -np.arange(n, dtype=np.float64).clip(max=100)) * 1e3
    elif layout == "line":
        c[:, 0] = np.arange(n) * 2.5
    scene = _sphere_scene(probe, c)
    try:
        flat = probe.flatten(scene, 0)
        assert flat["n_tree"] == n and flat["built_on_device"] == 0
        assert 17 <= flat["depth"] <= 46
        _check_flat(flat)
    finally:
        probe.device.rtc_scene_destroy(scene)


@pytest.mark.parametrize("n", [1023, 1024, 3000])
def test_flatten_takes_the_builders_tree_from_1024_items(n, probe):
    """rtc::flatten hands a tree builder the padded boxes of 1 024 or more bounded items, and only then; with the
    reference standing in for the device builder, the committed tree is the reference's tree, its depth is the
    reference's depth, and position p holds the item order[p] (its API primitive, whose box its leaf contains)."""
    rng = np.random.default_rng(n)
    centres = rng.uniform(-40, 40, (n, 3))
    centres[: n // 8] = centres[0]  # some coincident centres too
    scene = _sphere_scene(probe, centres, radius=0.75)
    log = []
    callback = reference_callback(log)
    try:
        flat = probe.flatten(scene, 1, callback)
        assert flat["n_tree"] == n and flat["leaf_size"] == 1
        if n < 1024:
            assert flat["built_on_device"] == 0 and flat["calls"] == 0 and not log
            _check_flat(flat)
            return
        assert flat["built_on_device"] == 1 and flat["calls"] == 1 and log == [(n, 1)]
        boxes, closed = flat["input_boxes"], flat["input_closed"]
        assert len(boxes) == n and closed.all()
        order, nodes, root, depth = lbvh_reference(boxes, closed, 1)
        assert_same_tree((order, flat["nodes"], flat["root"], flat["depth"]), (order, nodes, root, depth))
        # the reorder: position p is API primitive order[p] (the item index is the primitive index in this scene)
        prim_of_pos = flat["head"][flat["n_pos"]:, 1][:n]
        assert (prim_of_pos == order).all()
        # and its world box lies inside its padded box, which is the box its leaf was built from
        b, pb = flat["pos_box"], boxes[order]
        assert ((b[:, :3] >= pb[:, :3]) & (b[:, 3:] <= pb[:, 3:])).all()
        check_tree(flat["nodes"], flat["root"], 1, n, pb, closed[order], flat["depth"])
        _check_flat(flat)
    finally:
        probe.device.rtc_scene_destroy(scene)
