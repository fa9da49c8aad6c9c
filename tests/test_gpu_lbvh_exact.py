"""The device tree builder K3 (csrc/rtc_lbvh.cu: lbvh_build) equals its NumPy restatement (tests/lbvh_reference.py)
bit for bit: the item order, the root link, the depth and every one of the n - 1 nodes (box words compared as floats).

Frames cannot show most ways K3 could be wrong: a sort with another tie-break, a merge step skipped, a leaf one item
smaller, a code one bit wider, closed bits OR-ed instead of AND-ed all still give a valid tree, and a valid tree renders
the same pixels.  The exact comparison sees each of them.  The sizes cover the three sort paths (padded to 1 024: global
passes only; 1 025-2 048: one shared-memory block; above: global merge steps alternating with shared-memory finishes)
and the code widths they imply (11 bits per axis at 1 024 items, 9 at 10^5, 8 above 2^17); the inputs cover coincident
centroids, zero-extent axes, a centroid range that overflows to inf and one so small that its scale is inf."""
import pytest

from ray_tracer_challenge_b200 import scenes
from tests.bvh_check import check_tree
from tests.lbvh_reference import lbvh_reference
from tests.tree_probe import FAMILIES, assert_same_tree, family, load_probe

pytestmark = pytest.mark.gpu

SIZES = [2, 3, 16, 17, 1023, 1024, 1025, 2047, 2048, 2049, 4096, 4097, 65_537, 100_000, 131_073]
LEAF_SIZES = [1, 4, 16]


@pytest.fixture(scope="module")
def probe(tmp_path_factory):
    p = load_probe(tmp_path_factory)
    yield p
    p.lib.probe_release()


def _exact(probe, boxes, closed, leaf):
    rc, *got = probe.lbvh(boxes, closed, leaf)
    assert rc == 0, probe.device.rtc_last_error()
    want = lbvh_reference(boxes, closed, leaf)
    assert_same_tree(got, want)
    order, nodes, root, depth = got
    n = len(boxes)
    check_tree(nodes, root, leaf, n, boxes[order], closed[order], depth)


@pytest.mark.parametrize("n", [0, 1])
def test_fewer_than_two_items_are_refused(probe, n):
    boxes, closed = family("uniform", max(n, 1), seed=1)
    rc, *_ = probe.lbvh(boxes[:n], closed[:n], 1)
    assert rc != 0


@pytest.mark.parametrize("fam", FAMILIES)
@pytest.mark.parametrize("n", SIZES)
def test_device_tree_equals_the_reference(probe, n, fam):
    boxes, closed = family(fam, n, seed=n)
    for leaf in LEAF_SIZES:
        _exact(probe, boxes, closed, leaf)


def test_scratch_reused_while_growing_and_shrinking(probe):
    """One context, grow-only buffers: a big build, then a small one and a middle one over the stale scratch."""
    for n, fam in ((260_000, "mixed_closed"), (1025, "clusters"), (100_000, "uniform")):
        boxes, closed = family(fam, n, seed=n + 1)
        _exact(probe, boxes, closed, 4)


COMMITS = {
    "dragon_element_25k": (scenes.dragon_element, dict(width=160, height=90, n_u=160, n_v=80)),  # 25 k triangles, leaf 4
    "stress_c5": (scenes.stress, dict(width=64, height=36, n_spheres=100_000)),  # c5's scene: 10^5 spheres, CSG, leaf 1
}


@pytest.mark.parametrize("name", sorted(COMMITS))
def test_commit_through_the_device_builder(probe, name):
    """rtc::flatten with the real device builder: the committed tree is the reference's tree of the recorded builder
    input, position p holds item order[p], and the flattened tree passes the structural checker."""
    import ray_tracer_challenge_b200 as rt

    host = rt.new_session()
    make, kw = COMMITS[name]
    cam, world = make(host, **kw)[:2]
    scene = host.export_scene(cam, world)
    try:
        flat = probe.flatten(scene, 2)
        assert flat["built_on_device"] == 1 and flat["calls"] == 1
        boxes, closed = flat["input_boxes"], flat["input_closed"]
        n = len(boxes)
        assert n == flat["n_tree"] and n >= 25_000
        order, nodes, root, depth = lbvh_reference(boxes, closed, flat["leaf_size"])
        assert_same_tree((order, flat["nodes"], flat["root"], flat["depth"]), (order, nodes, root, depth))
        # the reorder: each position's own world box lies inside the padded box of the item the builder put there
        b, pb = flat["pos_box"], boxes[order]
        assert ((b[:, :3] >= pb[:, :3]) & (b[:, 3:] <= pb[:, 3:])).all()
        assert (flat["pos_closed"] == closed[order].astype(bool)).all()
        check_tree(flat["nodes"], flat["root"], flat["leaf_size"], n, pb, closed[order], flat["depth"])
        check_tree(flat["nodes"], flat["root"], flat["leaf_size"], n, b, flat["pos_closed"], flat["depth"])
    finally:
        probe.device.rtc_scene_destroy(scene)
