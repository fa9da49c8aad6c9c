// tree_probe.cpp — TEST INFRASTRUCTURE ONLY (built and loaded by tests/test_tree_structure.py and
// tests/test_gpu_lbvh_exact.py, never by the product): the two tree builders of a commit, exposed for exact checks.
//
//   probe_flatten  runs rtc::flatten (the host half of rtc_scene_commit) with one of three tree builders and keeps the
//                  result for probe_copy_*:
//                    mode 0  none: the host's binned-SAH builder
//                    mode 1  a TreeBuilderFn that hands the TreeBuildInput to a callback (a reference in Python can
//                            stand in for the device builder on a machine without a GPU)
//                    mode 2  the device builder, rtc::lbvh_build, with its input recorded
//   probe_lbvh     calls rtc::lbvh_build directly, through one LbvhContext whose grow-only buffers live between calls
//   probe_release  frees those buffers
#include <cstring>
#include <vector>

#include "rtc_internal.h"  // Flattened, RtcScene, rtc::flatten, rtc::lbvh_build (exported by librtc_b200.so)

namespace {

using BuilderCallback = int (*)(const float* boxes, const unsigned char* closed, int n, int leaf_size, int* order,
                                rtc::DevBvhNode* nodes, int* root, int* depth);

rtc::Flattened g_flat;
std::vector<float> g_boxes;  // the last TreeBuildInput seen by probe_flatten
std::vector<unsigned char> g_closed;
int g_calls = 0;  // builder calls of the last probe_flatten

char* g_scratch = nullptr;
size_t g_scratch_bytes = 0;
char* g_pinned = nullptr;
size_t g_pinned_bytes = 0;

rtc::LbvhContext context() { return rtc::LbvhContext{nullptr, &g_scratch, &g_scratch_bytes, &g_pinned, &g_pinned_bytes}; }

void record(const rtc::TreeBuildInput& in) {
    g_calls++;
    g_boxes.assign(in.boxes, in.boxes + 6 * (size_t)in.n);
    g_closed.assign(in.closed, in.closed + in.n);
}

int forward_to_callback(void* cb, const rtc::TreeBuildInput& in, rtc::TreeBuildOutput& out) {
    record(in);
    out.order.resize(in.n);
    out.nodes.resize(in.n > 1 ? in.n - 1 : 0);
    return reinterpret_cast<BuilderCallback>(cb)(in.boxes, in.closed, in.n, in.leaf_size, out.order.data(), out.nodes.data(),
                                                 &out.root, &out.depth);
}

int record_then_device(void* ctx, const rtc::TreeBuildInput& in, rtc::TreeBuildOutput& out) {
    record(in);
    return rtc::lbvh_build(ctx, in, out);
}

}  // namespace

// info: [0] bvh nodes, [1] bvh_root, [2] bvh_depth, [3] leaf_size, [4] n_pos, [5] built_on_device, [6] linear entries,
// [7] builder calls, [8] n of the recorded builder input
extern "C" int probe_flatten(RtcScene* s, int mode, void* callback, int* info) {
    g_flat = rtc::Flattened{};
    g_calls = 0;
    g_boxes.clear(), g_closed.clear();
    rtc::LbvhContext ctx = context();
    int rc;
    if (mode == 0)
        rc = rtc::flatten(s, g_flat);
    else if (mode == 1)
        rc = rtc::flatten(s, g_flat, forward_to_callback, callback);
    else
        rc = rtc::flatten(s, g_flat, record_then_device, &ctx);
    if (rc) return rc;
    info[0] = (int)g_flat.bvh.size(), info[1] = g_flat.bvh_root, info[2] = g_flat.bvh_depth, info[3] = g_flat.leaf_size;
    info[4] = g_flat.n_pos, info[5] = s->built_on_device, info[6] = (int)g_flat.linear.size(), info[7] = g_calls;
    info[8] = (int)g_closed.size();
    return 0;
}

// the tree, the heads (2 * n_pos int4) and the linear list of the last probe_flatten
extern "C" void probe_copy_flat(rtc::DevBvhNode* bvh, int4* head, int* linear) {
    memcpy(bvh, g_flat.bvh.data(), g_flat.bvh.size() * sizeof(rtc::DevBvhNode));
    memcpy(head, g_flat.head.data(), g_flat.head.size() * sizeof(int4));
    memcpy(linear, g_flat.linear.data(), g_flat.linear.size() * sizeof(int));
}

// the builder input the last probe_flatten recorded: n x 6 padded boxes and n closed flags
extern "C" void probe_copy_input(float* boxes, unsigned char* closed) {
    memcpy(boxes, g_boxes.data(), g_boxes.size() * sizeof(float));
    memcpy(closed, g_closed.data(), g_closed.size());
}

// per device position of the last flattened scene `s`: the primitive's world box as the scene holds it (before the
// tree's padding; a CSG pseudo-primitive gets an empty box, which every box contains), its "closed" flag (a sphere or a
// cube, as rtc_commit.cu defines it), and whether it lies inside a CSG (then it is no item of the tree or the linear list)
extern "C" void probe_positions(const RtcScene* s, float* box, unsigned char* closed, unsigned char* in_csg) {
    const int n_pos = g_flat.n_pos;
    for (int p = 0; p < n_pos; p++) {
        const int prim = g_flat.head[(size_t)n_pos + p].y;  // API primitive, -1 for a CSG pseudo-primitive
        closed[p] = prim >= 0 && (s->prims[prim].type == RTC_SPHERE || s->prims[prim].type == RTC_CUBE);
        in_csg[p] = 0;
        for (int k = prim >= 0 ? s->prims[prim].parent : -1; k >= 0; k = s->nodes[k].parent)
            if (s->nodes[k].kind == RTC_NODE_CSG) in_csg[p] = 1;
        for (int a = 0; a < 3; a++) {
            box[6 * p + a] = prim >= 0 ? s->prims[prim].bbox_min[a] : INFINITY;
            box[6 * p + 3 + a] = prim >= 0 ? s->prims[prim].bbox_max[a] : -INFINITY;
        }
    }
}

// lbvh_build on the given input; order: n ints, nodes: n - 1 DevBvhNode.  Returns lbvh_build's result.
extern "C" int probe_lbvh(const float* boxes, const unsigned char* closed, int n, int leaf_size, int* order, rtc::DevBvhNode* nodes,
                          int* root, int* depth) {
    rtc::LbvhContext ctx = context();
    rtc::TreeBuildOutput out;
    const int rc = rtc::lbvh_build(&ctx, rtc::TreeBuildInput{boxes, closed, n, leaf_size}, out);
    if (rc) return rc;
    memcpy(order, out.order.data(), (size_t)n * sizeof(int));
    memcpy(nodes, out.nodes.data(), out.nodes.size() * sizeof(rtc::DevBvhNode));
    *root = out.root, *depth = out.depth;
    return 0;
}

extern "C" void probe_release() {
    if (g_scratch) cudaFree(g_scratch);
    if (g_pinned) cudaFreeHost(g_pinned);
    g_scratch = g_pinned = nullptr;
    g_scratch_bytes = g_pinned_bytes = 0;
}
