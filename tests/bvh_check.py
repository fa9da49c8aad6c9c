"""Structural invariants of a flattened BVH (rtc_types.h: DevBvhNode), whichever builder made it.

A tree that renders correctly on a sample of rays can still miss a primitive, link a node twice or carry a box that is
too small: such a tree changes pixels only where some ray needs the missing piece.  `check_tree` walks the whole tree
and requires, for every node and every item:
  - every internal node is reached at most once (no node shared, no cycle), every position of [0, n) lies in exactly
    one reachable leaf, and no leaf holds more than `leaf_size` items;
  - each child box of an inner node equals the union of that child's two child boxes (exact f32 compare: both builders
    refit with min / max);
  - every item's box lies inside every box on its path from the root;
  - bit i of `d.z` is set exactly when every item under child i is closed (a sphere or a cube);
  - the measured depth (inner nodes on the longest root-to-leaf path) equals the reported one and stays below
    kBvhStack - 1.
A tree that is one leaf comes wrapped in one node whose second child has a NaN box (rtc_commit.cu: flatten); that form is
accepted.  Levels are processed whole, so 2.6 * 10^5 items take well under a second.
"""
import numpy as np

from tests.lbvh_reference import K_BVH_STACK

_EVERYWHERE = np.array([-np.inf] * 3 + [np.inf] * 3, np.float32)


def _leaf(link):
    code = ~link
    return code >> 4, (code & 15) + 1


def check_tree(nodes, root, leaf_size, n, item_boxes, closed, depth=None):
    """nodes: (m, 16) int32 words of DevBvhNode; root: the root link; item_boxes: (n, 6) float32, the box of the item at
    each leaf position (lo.xyz, hi.xyz); closed: (n,) flags per leaf position; depth: the builder's reported depth (None:
    not checked).  Returns the measured depth."""
    nodes = np.ascontiguousarray(nodes, np.int32).reshape(-1, 16)
    boxes = nodes.view(np.float32)[:, :12].reshape(-1, 2, 6)  # [node, child, lo.xyz hi.xyz]
    links = nodes[:, 12:14].astype(np.int64)
    bits = nodes[:, 14]
    m = len(nodes)
    item_boxes = np.asarray(item_boxes, np.float32).reshape(n, 6)
    closed = np.asarray(closed).astype(bool).reshape(n)

    # the wrapped single leaf: both links name the same leaf, the second box is NaN
    wrapped = 0 <= root < m and links[root, 0] < 0 and links[root, 0] == links[root, 1] and np.isnan(boxes[root, 1]).all()
    n_sides = lambda level: 1 if wrapped and level == 0 else 2  # noqa: E731

    # ---- top-down: reachability, each internal node once
    levels = []
    frontier = np.array([root] if root >= 0 else [], np.int64)
    visits = np.zeros(m, np.int64)
    while len(frontier):
        assert ((frontier >= 0) & (frontier < m)).all(), "a link outside the node array"
        np.add.at(visits, frontier, 1)
        assert (visits[frontier] == 1).all(), f"an internal node reached twice (shared, or a cycle) at level {len(levels)}"
        levels.append(frontier)
        child = links[frontier, :n_sides(len(levels) - 1)].ravel()
        frontier = child[child >= 0]

    # ---- bottom-up: the positions under every child, which must be one contiguous range
    node_lo = np.zeros(m, np.int64)
    node_hi = np.zeros(m, np.int64)
    node_cnt = np.zeros(m, np.int64)
    child_range = {}
    for level in range(len(levels) - 1, -1, -1):
        idx = levels[level]
        for side in range(n_sides(level)):
            link = links[idx, side]
            f, c = _leaf(link)
            k = np.where(link >= 0, link, 0)
            lo = np.where(link >= 0, node_lo[k], f)
            hi = np.where(link >= 0, node_hi[k], f + c)
            cnt = np.where(link >= 0, node_cnt[k], c)
            assert (cnt == hi - lo).all(), "the leaves under a child do not cover one contiguous range of positions"
            child_range[level, side] = lo, hi
            node_lo[idx] = lo if side == 0 else np.minimum(node_lo[idx], lo)
            node_hi[idx] = hi if side == 0 else np.maximum(node_hi[idx], hi)
            node_cnt[idx] = cnt if side == 0 else node_cnt[idx] + cnt

    # ---- top-down again: boxes, closed bits, leaves, depth
    not_closed = np.concatenate([[0], np.cumsum(~closed)])
    leaf_first, leaf_count, leaf_level, leaf_bound = [], [], [], []
    if root < 0:  # a bare leaf root (lbvh_build when n <= leaf_size): no box above it
        f, c = _leaf(np.array([root], np.int64))
        leaf_first.append(f), leaf_count.append(c), leaf_level.append(np.zeros(1, np.int64)), leaf_bound.append(_EVERYWHERE[None])
    path_box = np.tile(_EVERYWHERE, (m, 1))  # intersection of the boxes on the way down to each internal node
    for level, idx in enumerate(levels):
        for side in range(n_sides(level)):
            link = links[idx, side]
            box = boxes[idx, side]
            below = np.concatenate([np.maximum(path_box[idx, :3], box[:, :3]), np.minimum(path_box[idx, 3:], box[:, 3:])], axis=1)
            lo, hi = child_range[level, side]
            want = not_closed[hi] - not_closed[lo] == 0
            assert (((bits[idx] >> side) & 1).astype(bool) == want).all(), f"closed bit of child {side} wrong at level {level}"
            internal = link >= 0
            k = link[internal]
            union = np.concatenate([np.minimum(boxes[k, 0, :3], boxes[k, 1, :3]), np.maximum(boxes[k, 0, 3:], boxes[k, 1, 3:])], axis=1)
            tight = (box[internal] == union).all(axis=1)
            assert tight.all(), f"child {side} box of node {int(idx[internal][~tight][0])} is not the union of its children's boxes"
            path_box[k] = below[internal]
            f, c = _leaf(link[~internal])
            leaf_first.append(f), leaf_count.append(c), leaf_level.append(np.full(len(f), level + 1)), leaf_bound.append(below[~internal])

    first = np.concatenate(leaf_first)
    count = np.concatenate(leaf_count)
    bound = np.concatenate(leaf_bound)
    assert (count <= leaf_size).all(), "a leaf holds more than leaf_size items"
    assert (first >= 0).all() and (first + count <= n).all(), "a leaf outside [0, n)"
    owner = np.repeat(np.arange(len(first)), count)
    pos = np.repeat(first, count) + (np.arange(count.sum()) - np.repeat(np.cumsum(count) - count, count))
    hits = np.bincount(pos, minlength=n)
    assert (hits == 1).all(), f"{int((hits == 0).sum())} positions in no leaf, {int((hits > 1).sum())} in several"
    # containment: every item inside the intersection of the boxes on its path
    ib, pb = item_boxes[pos], bound[owner]
    inside = (ib[:, :3] >= pb[:, :3]).all(axis=1) & (ib[:, 3:] <= pb[:, 3:]).all(axis=1)
    assert inside.all(), f"{int((~inside).sum())} items outside a box on their path, e.g. position {int(pos[~inside][0])}"
    measured = int(np.concatenate(leaf_level).max())
    if depth is not None:
        assert measured == depth, f"measured depth {measured}, reported {depth}"
    assert measured < K_BVH_STACK - 1, measured
    return measured
