// emu_kernels.cpp — TEST INFRASTRUCTURE ONLY (built and loaded by tests/test_kernels_on_host.py, never by the product):
// the kernels themselves (dev_kernels.cuh: render_tiles, render_tiles_views, render_stream, render_stream_views,
// trace_rays, the wavefront renderer's kernels) run on the HOST in blocks of 128 threads and warps of 32 lanes
// (simt.h), over the arrays rtc::flatten() — the host half of rtc_scene_commit — would upload.  The kernel a call runs is
// the one the launch functions of rtc_kernels.cu pick for the same inputs (rtc_launch.h: frame_variant, trace_variant),
// from the decisions rtc_api.cu takes for the scene (rtc_internal.h: streams_pixels, frame_converge, stream_blocks).
// With -ffp-contract=off the host evaluates the strict build's IEEE expression order; with -DRTC_CSG_SWEEP_BUILD it is
// the strict_sweep build.
#include <vector>

#include "rtc_internal.h"  // Flattened, RtcScene, rtc::flatten (exported by librtc_b200.so)
#include "rtc_launch.h"
#include "simt.h"

namespace rtc {
namespace emu {
float4 rtc_smem[kSmallSmemBytes / sizeof(float4)];  // the block's dynamic shared memory
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
#include "dev_kernels.cuh"
#include "host_scene.h"

namespace {
using rtc::DevCounters;
constexpr int kThreads = rtc::kBlockThreads;
constexpr int kConcurrent = 3;  // blocks at once of the kernels without shared memory
// an SM count for stream_blocks(): a persistent grid of 6 blocks, 3 at a time
constexpr int kEmuSms = 1;

// the kernel kinds of a variant id: kind * 32 + variant_code
enum Kind { kTiles, kViews, kTrace, kStream, kStreamViews, kWave };

struct Scene {
    rtc::Flattened f;
    rtc::DevScene S;
    rtc::SmallScene SS;
};
int load(RtcScene* s, Scene& sc) {
    if (int rc = rtc::flatten(s, sc.f)) return rc;
    host_scene(s, sc.f, sc.S);
    sc.SS = sc.f.small;
    simt::g_smem = rtc::emu::rtc_smem, simt::g_smem_cap = sizeof(rtc::emu::rtc_smem);
    return 0;
}
simt::Dim dim(unsigned x, unsigned y = 1, unsigned z = 1) { return simt::Dim{x, y, z}; }
}  // namespace

// __activemask's mode (simt.h) and the timeout after which a rendezvous that has not completed aborts
extern "C" void emu_set_activemask(int mode, unsigned seed) { simt::g_activemask_mode = mode, simt::g_activemask_seed = seed ? seed : 1; }
extern "C" void emu_set_timeout(double seconds) { simt::g_timeout_s = seconds; }

// Every variant the launch functions of this build can select: out[i] = kind * 32 + variant_code; returns the count
extern "C" int emu_variants(int* out) {
    int n = 0;
#define RTC_EMU_TILES(ST, SM, CV, DR, LE) out[n++] = kTiles * 32 + rtc::variant_code(ST, SM, CV, DR, LE);
#define RTC_EMU_VIEWS(ST, SM, CV, DR, LE) \
    if (!ST) out[n++] = kViews * 32 + rtc::variant_code(ST, SM, CV, DR, LE);
#define RTC_EMU_TRACE(SM, DR) out[n++] = kTrace * 32 + rtc::variant_code(false, SM, true, DR, false);
    RTC_TILE_VARIANTS(RTC_EMU_TILES)
    RTC_TILE_VARIANTS(RTC_EMU_VIEWS)
    RTC_TRACE_VARIANTS(RTC_EMU_TRACE)
#undef RTC_EMU_TILES
#undef RTC_EMU_VIEWS
#undef RTC_EMU_TRACE
    out[n++] = kStream * 32 + rtc::variant_code(true, false, true, false, false);
    out[n++] = kStream * 32 + rtc::variant_code(false, false, true, false, false);
    out[n++] = kStreamViews * 32 + rtc::variant_code(false, false, true, false, false);
    return n;
}

// launch_render over the bands [band_begin, band_begin + n_bands) of a shard.  converge / stream: -1 the scene's decision
// (frame_converge, streams_pixels), 0 / 1 forced.  tile_order / tile_cost as DevFrame's (may be null).  rgb / u8: the
// caller's full frames (either may be null); counters: the DevCounters the launch accumulated; variant: what ran.
extern "C" int emu_render(RtcScene* s, int depth, int shard, int n_shards, int band_begin, int n_bands, const int* tile_order,
                          unsigned* tile_cost, int detailed, int converge, int stream, float* rgb, unsigned char* u8,
                          DevCounters* counters, int* variant) {
    using namespace rtc;
    Scene sc;
    if (int rc = load(s, sc)) return rc;
    const DevScene& S = sc.S;
    const SmallScene& SS = sc.SS;
    unsigned stream_counter = 0;
    const bool streams = stream < 0 ? streams_pixels(s, SS) : (SS.n == 0 && stream != 0);
    DevFrame F{rgb, u8, shard, n_shards, depth, n_bands, band_begin, tile_order, tile_cost,
               converge < 0 ? frame_converge(s) : converge, streams ? &stream_counter : nullptr, stream_blocks(kEmuSms)};
    memset(counters, 0, sizeof(DevCounters));
    const unsigned tiles_x = (unsigned)(S.width + kTileW - 1) / kTileW;
    if (tiles_x == 0 || n_bands <= 0) return 0;
    const KernelVariant v = frame_variant(S, SS, F, detailed != 0, emu::kHasLean);
    if (v.stream) {
        *variant = kStream * 32 + variant_code(v);
        if (v.stats)
            simt::launch(dim(F.stream_blocks), kThreads, 0, kConcurrent, [&] { emu::render_stream<true>(S, SS, F, counters); });
        else
            simt::launch(dim(F.stream_blocks), kThreads, 0, kConcurrent, [&] { emu::render_stream<false>(S, SS, F, counters); });
        return 0;
    }
    *variant = kTiles * 32 + variant_code(v);
    switch (variant_code(v)) {
#define RTC_EMU_TILES(ST, SM, CV, DR, LE)                                                                                   \
    case variant_code(ST, SM, CV, DR, LE):                                                                                  \
        simt::launch(dim(tiles_x, (unsigned)n_bands), kThreads, (size_t)dynamic_smem(v), 1,                                 \
                     [&] { emu::render_tiles<ST, SM, CV, DR, LE>(S, SS, F, counters); });                                   \
        return 0;
        RTC_TILE_VARIANTS(RTC_EMU_TILES)
#undef RTC_EMU_TILES
    }
    return fail(RTC_ERR_INVALID, "no kernel for the variant");
}

// launch_views for n_views views whose cameras are those of the scenes cams[v] (the DevView table rtc_render_views
// builds): view v's frame at rgb / u8 + v * width * height * 3
extern "C" int emu_render_views(RtcScene* s, int depth, int shard, int n_shards, int band_begin, int n_bands, RtcScene* const* cams,
                                int n_views, int converge, int stream, float* rgb, unsigned char* u8, DevCounters* counters,
                                int* variant) {
    using namespace rtc;
    Scene sc;
    if (int rc = load(s, sc)) return rc;
    std::vector<DevView> table((size_t)(n_views > 0 ? n_views : 0));
    for (int i = 0; i < n_views; i++) {
        rows3(cams[i]->cam_inv, table[(size_t)i].cam_inv);
        table[(size_t)i].half_w = cams[i]->half_w, table[(size_t)i].half_h = cams[i]->half_h;
        table[(size_t)i].pixel_size = cams[i]->pixel_size, table[(size_t)i].pad = 0.f;
    }
    const DevView* views = table.data();
    const DevScene& S = sc.S;
    const SmallScene& SS = sc.SS;
    unsigned stream_counter = 0;
    const bool streams = stream < 0 ? streams_pixels(s, SS) : (SS.n == 0 && stream != 0);
    DevFrame F{rgb, u8, shard, n_shards, depth, n_bands, band_begin, nullptr, nullptr,
               converge < 0 ? frame_converge(s) : converge, streams ? &stream_counter : nullptr, stream_blocks(kEmuSms)};
    memset(counters, 0, sizeof(DevCounters));
    const unsigned tiles_x = (unsigned)(S.width + kTileW - 1) / kTileW;
    if (tiles_x == 0 || n_bands <= 0 || n_views <= 0) return 0;
    const KernelVariant v = frame_variant(S, SS, F, false, emu::kHasLean);
    if (v.stream) {
        *variant = kStreamViews * 32 + variant_code(v);
        simt::launch(dim(F.stream_blocks), kThreads, 0, kConcurrent,
                     [&] { emu::render_stream_views(S, SS, F, counters, views, n_views); });
        return 0;
    }
    *variant = kViews * 32 + variant_code(v);
    const simt::Dim grid = dim(tiles_x, (unsigned)n_bands, (unsigned)n_views);
    switch (variant_code(v)) {
#define RTC_EMU_VIEWS(ST, SM, CV, DR, LE) RTC_EMU_VIEWS_##ST(SM, CV, DR, LE)
#define RTC_EMU_VIEWS_true(SM, CV, DR, LE)
#define RTC_EMU_VIEWS_false(SM, CV, DR, LE)                                                                              \
    case variant_code(false, SM, CV, DR, LE):                                                                            \
        simt::launch(grid, kThreads, (size_t)dynamic_smem(v), 1,                                                          \
                     [&] { emu::render_tiles_views<SM, CV, DR, LE>(S, SS, F, counters, views); });                       \
        return 0;
        RTC_TILE_VARIANTS(RTC_EMU_VIEWS)
#undef RTC_EMU_VIEWS
#undef RTC_EMU_VIEWS_true
#undef RTC_EMU_VIEWS_false
    }
    return fail(RTC_ERR_INVALID, "no kernel for the variant");
}

// launch_trace for n caller rays
extern "C" int emu_trace(RtcScene* s, int n, const float* origins, const float* directions, int depth, float* out_rgb, float* out_t,
                         int* out_pos, DevCounters* counters, int* variant) {
    using namespace rtc;
    Scene sc;
    if (int rc = load(s, sc)) return rc;
    const DevScene& S = sc.S;
    const SmallScene& SS = sc.SS;
    memset(counters, 0, sizeof(DevCounters));
    if (n <= 0) return 0;
    const KernelVariant v = trace_variant(S, SS);
    *variant = kTrace * 32 + variant_code(v);
    const unsigned blocks = (unsigned)(n + kThreads - 1) / kThreads;
    switch (variant_code(v)) {
#define RTC_EMU_TRACE(SM, DR)                                                                                             \
    case variant_code(false, SM, true, DR, false):                                                                        \
        simt::launch(dim(blocks), kThreads, (size_t)dynamic_smem(v), 1, [&] {                                             \
            emu::trace_rays<SM, DR>(S, SS, n, origins, directions, depth, out_rgb, out_t, out_pos, counters);           \
        });                                                                                                               \
        return 0;
        RTC_TRACE_VARIANTS(RTC_EMU_TRACE)
#undef RTC_EMU_TRACE
    }
    return fail(RTC_ERR_INVALID, "no kernel for the variant");
}

// One chunk of a frame through launch_wave's kernel sequence (rtc_kernels.cu) with 32-lane warps and the product's
// refill threshold (RTC_REFILL_LANES): `blocks` blocks of the persistent tree walks, twice as many of the per-ray kernels,
// a few at a time.  The pool holds exactly `capacity` rays and nodes (heap arrays: AddressSanitizer guards their ends).
// out_ints / out_record as emu_color.cpp's emu_wave_chunk.
extern "C" int emu_wave_chunk32(RtcScene* s, int depth, int shard, int n_shards, int band_begin, int n_bands, int capacity, int blocks,
                                float* out_rgb, int32_t* out_ints, unsigned long long* out_record) {
    using namespace rtc;
    if (s->light_is_rect) return fail(RTC_ERR_INVALID, "the wavefront renderer takes point lights only");
    if (depth < 0 || depth > kMaxFrames - 1 || capacity < 1 || blocks < 1 || n_shards < 1 || shard < 0 || shard >= n_shards)
        return fail(RTC_ERR_INVALID, "bad wavefront chunk");
    Scene sc;
    if (int rc = load(s, sc)) return rc;
    const DevScene& S = sc.S;
    std::vector<emu::WaveRay> rays((size_t)capacity);
    std::vector<emu::WaveNode> nodes((size_t)capacity);
    std::vector<int> ints(kWaveInts, 0);
    std::vector<unsigned long long> record(3, 0ull);
    DevCounters counters{};
    const DevFrame F{out_rgb, nullptr, shard, n_shards, depth, n_bands, band_begin, nullptr, nullptr, 1, nullptr, 0};
    const WavePoolRaw pool{rays.data(), nodes.data(), capacity, ints.data(), record.data()};
    const unsigned wide = (unsigned)blocks * 2;
    simt::launch(dim(wide), 128, 0, kConcurrent, [&] { emu::wave_primary_kernel(S, F, pool, &counters); });
    for (int level = 0; level <= depth; level++) {
        simt::launch(dim(1), 1, 0, 1, [&] { emu::wave_next_level_kernel(pool, level); });
        simt::launch(dim((unsigned)blocks), 128, 0, kConcurrent, [&] { emu::wave_trace_kernel<false>(S, pool, &counters, level); });
        simt::launch(dim(wide), 128, 0, kConcurrent, [&] { emu::wave_hit_kernel(S, pool, &counters, level); });
        simt::launch(dim((unsigned)blocks), 128, 0, kConcurrent, [&] { emu::wave_trace_kernel<true>(S, pool, &counters, level); });
        simt::launch(dim(wide), 128, 0, kConcurrent, [&] { emu::wave_shade_kernel(S, pool, &counters, level, depth); });
    }
    for (int level = depth; level >= 0; level--)
        simt::launch(dim(wide), 128, 0, kConcurrent, [&] { emu::wave_combine_kernel(S, F, pool, &counters, level); });
    memcpy(out_ints, ints.data(), ints.size() * sizeof(int));
    memcpy(out_record, record.data(), record.size() * sizeof(unsigned long long));
    return 0;
}
