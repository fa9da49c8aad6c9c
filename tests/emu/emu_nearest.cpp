// emu_nearest.cpp — TEST INFRASTRUCTURE ONLY (built and loaded by tests/test_device_code_on_host.py, never by the
// product): the device code of the tree path — dev_math / dev_shapes / dev_bvh .cuh: every primitive test, the CSG
// programs, the group cull chain, the while-while BVH walk — compiled for the HOST behind a shim of the few CUDA
// intrinsics it uses, and run over the arrays rtc::flatten() (the host half of rtc_scene_commit) would upload.
// With -ffp-contract=off the host evaluates the same IEEE expression order as the strict kernel build, so the nearest
// hit of a ray can be compared with the oracle's World::intersect + Intersection::hit without a GPU.
#include <cmath>
#include <cstring>

#include "rtc_internal.h"  // Flattened, RtcScene, rtc::flatten (exported by librtc_b200.so)

#include "shim.h"

#define RTC_NS emu
#include "dev_math.cuh"
#include "dev_shapes.cuh"
#include "dev_bvh.cuh"

extern "C" int emu_nearest(RtcScene* s, uint32_t n, const float* origins, const float* directions, float* out_t,
                           int32_t* out_prim) {
    using namespace rtc;
    Flattened f;
    if (int rc = flatten(s, f)) return rc;
    DevScene S;
    memset(&S, 0, sizeof(S));
    S.head = f.head.data(), S.rec = f.rec.data(), S.xform = f.xform.data(), S.tri = f.tri.data(), S.bound = f.bound.data();
    S.bvh = f.bvh.data(), S.linear = f.linear.data(), S.n_linear = (int)f.linear.size(), S.bvh_root = f.bvh_root;
    S.n_prims = f.n_pos, S.nodes = f.nodes.data(), S.csg_ops = f.ops.data(), S.materials = f.materials.data();
    for (uint32_t i = 0; i < n; i++) {
        emu::V3 o = emu::ld3(origins + 3 * (size_t)i), d = emu::ld3(directions + 3 * (size_t)i);
        emu::Hit best{emu::kInfF, -1, -1};
        emu::Ctr<false> k;
        emu::nearest_hit<false, false>(S, o, d, best, k);
        out_t[i] = best.pos >= 0 ? best.t : -1.0f;
        out_prim[i] = best.pos >= 0 ? f.head[(size_t)f.n_pos + best.pos].y : -1;
    }
    return 0;
}
