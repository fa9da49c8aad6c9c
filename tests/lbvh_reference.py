"""A plain NumPy restatement of the device tree builder, K3 (ray_tracer_challenge_b200/csrc/rtc_lbvh.cu: lbvh_build).

K3's output is a function of its input alone: the sort is a total order on (code, item), Karras' construction yields the
binary radix tree of the sorted keys extended by their positions, the refit is a min / max of the input boxes, and the
links, "closed" bits and depth are integer functions of the topology.  So this reference must match the device's
`order`, all n - 1 nodes, `root` and `depth` bit for bit (box words compared as floats: the sign of a zero that fminf
picks is not part of the result).

The topology is built top-down as a radix tree, not by porting Karras' bottom-up search, so that it checks that search
rather than repeats it.  Every step is vectorised over one level of the tree at a time, so 2.6 * 10^5 items take about a
second.  Test infrastructure only: the product never imports this.
"""
import numpy as np

K_BVH_STACK = 48  # rtc_types.h: kBvhStack


def code_bits(n):
    """Bits per axis: 3 * bits + ceil(log2 n) <= kBvhStack - 4, clamped to [1, 21]."""
    log2n = max(0, int(n - 1).bit_length())
    return max(1, min(21, (K_BVH_STACK - 4 - log2n) // 3))


def _spread21(v):
    x = v.astype(np.uint64) & np.uint64(0x1FFFFF)
    for shift, mask in ((32, 0x1F00000000FFFF), (16, 0x1F0000FF0000FF), (8, 0x100F00F00F00F00F), (4, 0x10C30C30C30C30C3),
                        (2, 0x1249249249249249)):
        x = (x | (x << np.uint64(shift))) & np.uint64(mask)
    return x


def morton_codes(boxes):
    """The 63-bit Morton code of every box centre, quantised inside the centroid bounds as lbvh_build does."""
    n = len(boxes)
    with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
        c = np.float32(0.5) * (boxes[:, :3] + boxes[:, 3:])
        # the host's centroid bounds: std::min / std::max from +-FLT_MAX
        fmax = np.float32(np.finfo(np.float32).max)
        lo = np.minimum(fmax, c.min(axis=0))
        hi = np.maximum(-fmax, c.max(axis=0))
        cells = np.float32(1 << code_bits(n))
        scale = np.where(hi > lo, cells / (hi - lo), np.float32(0)).astype(np.float32)
        # fmax / fmin return the non-NaN operand, as CUDA's fmaxf / fminf do: NaN -> 0
        q = np.fmin(np.fmax((c - lo) * scale, np.float32(0)), cells - np.float32(1)).astype(np.uint32)
    return _spread21(q[:, 0]) << np.uint64(2) | _spread21(q[:, 1]) << np.uint64(1) | _spread21(q[:, 2])


def _bit_length(x):
    """Vectorised int.bit_length of non-negative uint64 values (exact: each 32-bit half converts to float64 exactly)."""
    x = x.astype(np.uint64)
    hi = (x >> np.uint64(32)).astype(np.float64)
    lo = (x & np.uint64(0xFFFFFFFF)).astype(np.float64)
    return np.where(hi > 0, np.frexp(hi)[1] + 32, np.frexp(lo)[1]).astype(np.int64)


def topology(codes):
    """The binary radix tree of the sorted keys (code, position), numbered as Karras 2012 numbers it.

    Returns per internal node: first, last, split (gamma), the child references (>= 0 internal node, < 0 ~position of a
    leaf) and the level of every node (root 0), plus the list of levels, each an array of node indices."""
    n = len(codes)
    m = n - 1
    first = np.full(m, -1, np.int64)
    last = np.full(m, -1, np.int64)
    split = np.full(m, -1, np.int64)
    left = np.zeros(m, np.int64)
    right = np.zeros(m, np.int64)
    seen = np.zeros(m, np.int64)
    levels = []
    f, l, idx = np.array([0]), np.array([n - 1]), np.array([0])
    while len(idx):
        cf, cl = codes[f], codes[l]
        differ = cf != cl
        # codes differ: split before the first key with the highest differing bit set (the keys of [f, l] share every
        # bit above it, so a search of the whole sorted array lands inside the range)
        b = np.maximum(_bit_length(cf ^ cl) - 1, 0).astype(np.uint64)
        threshold = ((cf >> b) | np.uint64(1)) << b
        g_code = np.searchsorted(codes, threshold, side="left").astype(np.int64) - 1
        # equal codes: split at the highest differing bit of the positions
        bp = np.maximum(_bit_length((f ^ l).astype(np.uint64)) - 1, 0)
        g_pos = ((l >> bp) << bp) - 1
        g = np.where(differ, g_code, g_pos)
        assert ((g >= f) & (g < l)).all(), "a split outside its range"
        np.add.at(seen, idx, 1)
        first[idx], last[idx], split[idx] = f, l, g
        left[idx] = np.where(g == f, ~g, g)
        right[idx] = np.where(g + 1 == l, ~(g + 1), g + 1)
        levels.append(idx)
        li, ri = g > f, g + 1 < l
        f, l, idx = np.concatenate([f[li], g[ri] + 1]), np.concatenate([g[li], l[ri]]), np.concatenate([g[li], g[ri] + 1])
    assert (seen == 1).all(), "the internal node indices are not a permutation of 0..n-2"
    return first, last, split, left, right, levels


def lbvh_reference(boxes, closed, leaf_size):
    """lbvh_build of `boxes` (n x 6 float32: lo.xyz, hi.xyz), `closed` (n flags) and `leaf_size`.

    Returns (order, nodes, root, depth): the items in leaf order, the n - 1 nodes as an (n - 1) x 16 int32 array of the
    words of DevBvhNode (rtc_types.h: a, b, c = child 0 box lo.xyz hi.xyz, child 1 box lo.xyz hi.xyz; d = link 0,
    link 1, closed bits, 0), the root link and the depth.  n >= 2 (lbvh_build refuses fewer)."""
    boxes = np.ascontiguousarray(boxes, np.float32).reshape(-1, 6)
    n = len(boxes)
    assert n >= 2
    closed = np.asarray(closed).astype(bool).reshape(n)
    items = np.arange(n, dtype=np.int64)
    codes = morton_codes(boxes)
    order = np.lexsort((items, codes))
    codes = codes[order]
    first, last, _, left, right, levels = topology(codes)
    m = n - 1
    count = last - first + 1

    sorted_boxes = boxes[order]
    not_closed = np.concatenate([[0], np.cumsum(~closed[order])])

    def range_closed(f, l):
        return not_closed[l + 1] - not_closed[f] == 0

    def link(child):  # link_of: a subtree of at most leaf_size items is one leaf
        leaf = child < 0
        pos = np.where(leaf, ~child, 0)
        c = np.where(leaf, 0, child)
        cnt = np.where(leaf, 1, count[c])
        fst = np.where(leaf, pos, first[c])
        return np.where(cnt <= leaf_size, ~((fst << 4) | (cnt - 1)), child)

    def child_range(child):
        leaf = child < 0
        c = np.where(leaf, 0, child)
        return np.where(leaf, ~child, first[c]), np.where(leaf, ~child, last[c])

    node_box = np.zeros((m, 6), np.float32)
    words = np.zeros((m, 16), np.int32)
    fwords = words.view(np.float32)
    for idx in reversed(levels):  # deepest level first: an internal child's box is ready before its parent needs it
        cbox = []
        for side, child in enumerate((left[idx], right[idx])):
            leaf = child < 0
            box = np.where(leaf[:, None], sorted_boxes[np.where(leaf, ~child, 0)], node_box[np.where(leaf, 0, child)])
            cbox.append(box)
            fwords[idx, 6 * side:6 * side + 6] = box
            words[idx, 12 + side] = link(child)
            f, l = child_range(child)
            words[idx, 14] |= np.where(range_closed(f, l), 1 << side, 0).astype(np.int32)
        node_box[idx, :3] = np.minimum(cbox[0][:, :3], cbox[1][:, :3])
        node_box[idx, 3:] = np.maximum(cbox[0][:, 3:], cbox[1][:, 3:])

    # depth: the most ancestors of a leaf whose range holds more than leaf_size items
    # (every node has a leaf below it, so the maximum over the internal nodes, each counting itself, is the same)
    depth_of = np.zeros(m, np.int64)
    depth_of[0] = count[0] > leaf_size
    for idx in levels:
        for child in (left[idx], right[idx]):
            c = child[child >= 0]
            depth_of[c] = depth_of[idx[child >= 0]] + (count[c] > leaf_size)
    depth = int(depth_of.max())
    root = 0 if n > leaf_size else ~((0 << 4) | (n - 1))
    return order.astype(np.int32), words, root, depth
