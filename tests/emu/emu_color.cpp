// emu_color.cpp — TEST INFRASTRUCTURE ONLY (built and loaded by tests/test_device_code_on_host.py, never by the
// product): the WHOLE device code of the render path (rtc_device.cuh: shapes, tree, CSG, patterns, small-scene loops,
// shadow filter and cell masks, color_at) compiled for the HOST behind a shim of the CUDA intrinsics it uses, one
// "thread" per "block".  It runs World::color_at for caller-supplied rays over the arrays rtc::flatten() — the host half
// of rtc_scene_commit — would upload, so kernel logic can be compared with the oracle on a machine without a GPU.
// With -ffp-contract=off the host evaluates the strict build's IEEE expression order; libm is glibc's on both sides.
// It also runs the wavefront renderer's kernel sequence (dev_wave.cuh) over one chunk of a frame, one lane per "warp".
#include <vector>

// one lane per "warp": wave_trace refills as soon as that lane is idle (with the default of 8 idle lanes it never
// would); of the rest of the device code only PixelStream reads this, and it is compiled here but never run
#define RTC_REFILL_LANES 1
#include "rtc_internal.h"  // Flattened, RtcScene, rtc::flatten (exported by librtc_b200.so)

#include "shim.h"
#undef __shared__
#define __shared__

namespace {
struct EmuDim {
    unsigned x = 0, y = 0, z = 0;
};
}  // namespace
static EmuDim threadIdx, blockIdx;
static EmuDim blockDim{1, 1, 1}, gridDim{1, 1, 1};

static inline int __any_sync(unsigned, int p) { return p; }
// PixelStream (dev_shade.cuh) is compiled but never run here: one lane per "warp" (simt.h runs it with 32)
static inline unsigned __ballot_sync(unsigned, int p) { return p ? 1u : 0u; }
static inline unsigned __shfl_sync(unsigned, unsigned v, int) { return v; }
static inline unsigned __activemask() { return 1u; }
static inline unsigned __reduce_add_sync(unsigned, unsigned v) { return v; }
template <typename T>
static inline T atomicAdd(T* p, T v) {  // unsigned, int, unsigned long long
    T old = *p;
    *p += v;
    return old;
}
static inline void __syncthreads() {}

namespace rtc {
namespace emu {
float4 rtc_smem[kSmallSmemBytes / sizeof(float4) + 64];  // the block's dynamic shared memory
}
}  // namespace rtc

#define RTC_NS emu
#include "dev_math.cuh"
#include "dev_shapes.cuh"
#include "dev_bvh.cuh"
#include "dev_patterns.cuh"
#include "dev_small.cuh"
#include "dev_shadow.cuh"
#include "dev_shade.cuh"
#include "dev_wave.cuh"

#include "host_scene.h"

static unsigned long long g_rays[4];  // primary, secondary, shadow rays and shades of the last emu_color_at call
extern "C" void emu_last_rays(unsigned long long out[4]) { memcpy(out, g_rays, sizeof(g_rays)); }
static int g_converge = 0;
// 1: the converging build of color_at (a warp vote before every ray; here a warp of one lane)
extern "C" void emu_set_converge(int on) { g_converge = on; }

// World::color_at for n rays.  use_small: take the small-scene path when the scene qualifies (as the kernels do);
// use_filter: with the shadow filter and the cell-mask loops where eligible.  out_path: 0 tree / linear path, 1 small.
extern "C" int emu_color_at(RtcScene* s, uint32_t n, const float* origins, const float* directions, int depth, int use_small,
                            int use_filter, float* out_rgb, float* out_t, int32_t* out_path) {
    using namespace rtc;
    Flattened f;
    if (int rc = flatten(s, f)) return rc;
    DevScene S;
    host_scene(s, f, S);
    SmallScene SS = f.small;
    if (!use_small) SS.n = 0;
    if (!use_filter) SS.filter_ok = SS.cell_masks = SS.plane_cells = 0;
    const bool small = SS.n > 0;
    const bool drawn = small && SS.cell_masks && S.jitter_len == 0;
    if (out_path) *out_path = small ? 1 : 0;
    const emu::Env E{S, SS};
    memset(g_rays, 0, sizeof(g_rays));
    for (uint32_t i = 0; i < n; i++) {
        if (small) emu::stage_small_scene(S, SS);  // one thread per block: it stages the whole table
        emu::V3 o = emu::ld3(origins + 3 * (size_t)i), d = emu::ld3(directions + 3 * (size_t)i);
        emu::Ctr<false> k;
        emu::Rays r;
        float t = -1.0f;
        int pos = -1;
        emu::V3 c;
        if (drawn)
            c = g_converge ? emu::color_at<false, true, true, true>(E, true, o, d, depth, i, r, k, &t, &pos)
                           : emu::color_at<false, true, false, true>(E, true, o, d, depth, i, r, k, &t, &pos);
        else if (small)
            c = g_converge ? emu::color_at<false, true, true, false>(E, true, o, d, depth, i, r, k, &t, &pos)
                           : emu::color_at<false, true, false, false>(E, true, o, d, depth, i, r, k, &t, &pos);
        else
            c = g_converge ? emu::color_at<false, false, true, false>(E, true, o, d, depth, i, r, k, &t, &pos)
                           : emu::color_at<false, false, false, false>(E, true, o, d, depth, i, r, k, &t, &pos);
        emu::finish_rays(S, r);
        g_rays[0] += r.primary, g_rays[1] += r.secondary, g_rays[2] += r.shadow, g_rays[3] += r.shades;
        out_rgb[3 * (size_t)i] = c.x, out_rgb[3 * (size_t)i + 1] = c.y, out_rgb[3 * (size_t)i + 2] = c.z;
        if (out_t) out_t[i] = t;
    }
    return 0;
}

// The detailed pass's work counters of every ray, one lane at a time: color_at<STATS = true> in the converging build, as
// render_tiles<true, ...> runs it.  out: n x kRayCounts, in the order of the fields below.
constexpr int kRayCounts = 19;
extern "C" int emu_color_at_counts(RtcScene* s, uint32_t n, const float* origins, const float* directions, int depth,
                                   unsigned* out) {
    using namespace rtc;
    Flattened f;
    if (int rc = flatten(s, f)) return rc;
    DevScene S;
    host_scene(s, f, S);
    const SmallScene SS = f.small;
    const bool small = SS.n > 0, drawn = small && SS.cell_masks && S.jitter_len == 0;
    const emu::Env E{S, SS};
    for (uint32_t i = 0; i < n; i++) {
        if (small) emu::stage_small_scene(S, SS);
        const emu::V3 o = emu::ld3(origins + 3 * (size_t)i), d = emu::ld3(directions + 3 * (size_t)i);
        emu::Ctr<true> k;
        emu::Rays r;
        if (drawn)
            emu::color_at<true, true, true, true>(E, true, o, d, depth, i, r, k, nullptr, nullptr);
        else if (small)
            emu::color_at<true, true, true, false>(E, true, o, d, depth, i, r, k, nullptr, nullptr);
        else
            emu::color_at<true, false, true, false>(E, true, o, d, depth, i, r, k, nullptr, nullptr);
        unsigned* c = out + (size_t)i * kRayCounts;
        c[0] = k.nodes;
        for (int j = 0; j < 8; j++) c[1 + j] = k.prims[j];
        c[9] = k.xforms, c[10] = k.patterns, c[11] = k.cells, c[12] = k.schlicks, c[13] = k.refr_dirs, c[14] = k.overflows;
        c[15] = k.refilters, c[16] = r.secondary, c[17] = r.shades, c[18] = r.primary;
    }
    return 0;
}

// One chunk of a frame through the wavefront renderer: launch_wave's kernel sequence (rtc_kernels.cu) over bands
// [band_begin, band_begin + n_bands) of the shard, into the caller's w x h x 3 f32 frame.  The pool holds exactly
// `capacity` rays and nodes (heap arrays: AddressSanitizer guards their ends).  out_ints: base[L], count[L] and the two
// cursors of every level after the render (4 * kWaveLevels); out_record: {rays that did not fit, secondary rays, shades}.
extern "C" int emu_wave_chunk(RtcScene* s, int depth, int shard, int n_shards, int band_begin, int n_bands, int capacity,
                              float* out_rgb, int32_t* out_ints, unsigned long long* out_record) {
    using namespace rtc;
    if (s->light_is_rect) return fail(RTC_ERR_INVALID, "the wavefront renderer takes point lights only");
    if (depth < 0 || depth > kMaxFrames - 1 || capacity < 1 || n_shards < 1 || shard < 0 || shard >= n_shards)
        return fail(RTC_ERR_INVALID, "bad wavefront chunk");
    Flattened f;
    if (int rc = flatten(s, f)) return rc;
    DevScene S;
    host_scene(s, f, S);
    std::vector<emu::WaveRay> rays((size_t)capacity);
    std::vector<emu::WaveNode> nodes((size_t)capacity);
    std::vector<int> ints(kWaveInts, 0);
    std::vector<unsigned long long> record(3, 0ull);
    const DevFrame F{out_rgb, nullptr, shard, n_shards, depth, n_bands, band_begin, nullptr, nullptr, 1, nullptr, 0};
    const emu::WavePool P = emu::wave_pool(WavePoolRaw{rays.data(), nodes.data(), capacity, ints.data(), record.data()});
    emu::wave_primary(S, F, P);
    for (int level = 0; level <= depth; level++) {
        emu::wave_next_level(P, level);
        emu::wave_trace<false>(S, P, level);
        emu::wave_hit(S, P, level);
        emu::wave_trace<true>(S, P, level);
        emu::wave_shade(S, P, level, depth);
    }
    for (int level = depth; level >= 0; level--) emu::wave_combine(S, F, P, level);
    memcpy(out_ints, ints.data(), ints.size() * sizeof(int));
    memcpy(out_record, record.data(), record.size() * sizeof(unsigned long long));
    return 0;
}
