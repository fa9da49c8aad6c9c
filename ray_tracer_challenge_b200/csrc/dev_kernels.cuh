// dev_kernels.cuh — the kernels of rtc_kernels.cu and their device helpers, apart from the launch functions, so that
// the host harness of the kernels (tests/emu/emu_kernels.cpp) compiles the same bodies.  Included after rtc_device.cuh;
// like the other device parts it opens namespace rtc::RTC_NS itself.
#pragma once

// resident 128-thread blocks per SM the compiler must make room for (register budget = 65536 / (128 * blocks))
#ifndef RTC_SMALL_MINBLOCKS
#define RTC_SMALL_MINBLOCKS 4
#endif
#ifndef RTC_SMALL_LEAN_MINBLOCKS
#define RTC_SMALL_LEAN_MINBLOCKS 8  // the lean build: 8 blocks (64 regs, 36 / 8 B spill) beat 7 on c3_counter, 6 on both
#endif
#ifndef RTC_SMALL_CONVERGE_MINBLOCKS
#define RTC_SMALL_CONVERGE_MINBLOCKS 3  // the converging small-scene build keeps more state live: 3 blocks (168 regs) win
#endif
#ifndef RTC_BVH_CONVERGE_MINBLOCKS
#define RTC_BVH_CONVERGE_MINBLOCKS 6  // the converging BVH build (branching ray trees) gains from more warps (80 regs)
#endif
#ifndef RTC_BVH_MINBLOCKS
#define RTC_BVH_MINBLOCKS 5
#endif

namespace rtc {
namespace RTC_NS {

template <bool STATS>
__device__ __forceinline__ void flush_counters(const Rays& r, const Ctr<STATS>& k, DevCounters* out);

__device__ __forceinline__ void warp_add(unsigned long long* dst, unsigned v) {
    unsigned s = __reduce_add_sync(0xffffffffu, v);
    if ((threadIdx.x & 31) == 0 && s) atomicAdd(dst, (unsigned long long)s);
}
// primary and shadow are not accumulated: the host knows how many pixels a launch renders, and every shade casts
// exactly cells-of-the-light shadow rays (rtc_api.cu: add_counters)
__device__ __forceinline__ void flush_rays(const Rays& r, DevCounters* out) {
    warp_add(&out->secondary, r.secondary);
    warp_add(&out->shades, r.shades);
}
__device__ __forceinline__ void warp_add_u32(unsigned* dst, unsigned v) {
    unsigned s = __reduce_add_sync(0xffffffffu, v);
    if ((threadIdx.x & 31) == 0 && s) atomicAdd(dst, s);
}
template <>
__device__ __forceinline__ void flush_counters<false>(const Rays& r, const Ctr<false>&, DevCounters* out) {
    flush_rays(r, out);
}
template <>
__device__ __forceinline__ void flush_counters<true>(const Rays& r, const Ctr<true>& k, DevCounters* out) {
    flush_rays(r, out);
    warp_add(&out->node_visits, k.nodes);
    for (int i = 0; i < 8; i++) warp_add(&out->prim_tests[i], k.prims[i]);
    warp_add(&out->xforms, k.xforms);
    warp_add(&out->patterns, k.patterns);
    warp_add(&out->cells, k.cells);
    warp_add(&out->schlicks, k.schlicks);
    warp_add(&out->refr_dirs, k.refr_dirs);
    warp_add(&out->overflows, k.overflows);
    warp_add(&out->prim_tests[7], k.refilters);  // shadow-filter fallbacks to the exact test
}

// the RTC_*_MINBLOCKS figures are resident blocks of 128 threads: the same warps per SM for any tile width
constexpr int min_blocks(int of_128_threads) { return of_128_threads * 128 / kBlockThreads > 0 ? of_128_threads * 128 / kBlockThreads : 1; }

// Block -> tile of 16x8 pixels: natural order = (tile column bx, band `shard + by * n_shards`), or the learnt
// longest-first list.
__device__ __forceinline__ void tile_of(const DevFrame& F, int& band, int& bx) {
    band = F.shard + (F.band_begin + blockIdx.y) * F.n_shards, bx = blockIdx.x;
    if (F.tile_order) {
        const int id = F.tile_order[blockIdx.y * gridDim.x + blockIdx.x];
        band = id / (int)gridDim.x;
        bx = id - band * (int)gridDim.x;
    }
}

// LEAN: the build for small scenes marked SmallScene::lean (dev_shade.cuh: color_at), with its own occupancy target.
// It holds nothing of the epilogue across color_at — the tile coordinates are evaluated again after it (one more
// tile_order load per thread) and the tile-cost probe's start is one shared word per warp — which lets it run more
// resident blocks.  The other builds keep both in registers: the same change made c4 1 % and c2 0.5 % slower
// (profiles/README.md).
constexpr int tile_min_blocks(bool SMALL, bool CONVERGE, bool LEAN) {
    return min_blocks(LEAN ? RTC_SMALL_LEAN_MINBLOCKS
                           : SMALL ? (CONVERGE ? RTC_SMALL_CONVERGE_MINBLOCKS : RTC_SMALL_MINBLOCKS)
                                   : (CONVERGE ? RTC_BVH_CONVERGE_MINBLOCKS : RTC_BVH_MINBLOCKS));
}
template <bool STATS, bool SMALL, bool CONVERGE, bool DRAWN, bool LEAN = false>
__global__ void __launch_bounds__(kBlockThreads, tile_min_blocks(SMALL, CONVERGE, LEAN))
    render_tiles(const __grid_constant__ DevScene S, const __grid_constant__ SmallScene SS,
                                                    const DevFrame F, DevCounters* counters) {
    // small scenes: primitive table + per-thread shadow-origin cache in dynamic shared memory (kSmallSmemBytes)
    if (SMALL) stage_small_scene(S, SS);
    const Env E{S, SS};
    const long long t_start = !LEAN && F.tile_cost ? clock64() : 0;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __shared__ long long s_t_start[LEAN ? kBlockThreads / 32 : 1];
    if (LEAN && F.tile_cost && lane == 0) s_t_start[warp] = clock64();
    // warp w -> 8x4 sub-tile
    int band, bx;
    tile_of(F, band, bx);
    int x = bx * kTileW + (warp % kWarpsX) * 8 + (lane & 7);
    int y = band * kBandRows + (warp / kWarpsX) * 4 + (lane >> 3);
    Ctr<STATS> k;
    Rays r;
    V3 c = mk(0.f, 0.f, 0.f);
    bool inside = x < S.width && y < S.height;
    // camera.rs:80-81 — the last row and the last column are never rendered and stay black (canvas.rs:23)
    const bool rendered = inside && x < S.width - 1 && y < S.height - 1;
    V3 o = mk(0.f, 0.f, 0.f), d = mk(0.f, 0.f, 1.f);
    if (rendered) ray_for_pixel(S, x, y, o, d);
    if (CONVERGE || rendered)
        c = color_at<STATS, SMALL, CONVERGE, DRAWN, LEAN>(E, rendered, o, d, F.depth, (unsigned)(y * S.width + x), r, k, nullptr, nullptr);
    if (LEAN) {
        tile_of(F, band, bx);
        x = bx * kTileW + (warp % kWarpsX) * 8 + (lane & 7);
        y = band * kBandRows + (warp / kWarpsX) * 4 + (lane >> 3);
        inside = x < S.width && y < S.height;
    }
    // Canvas::write_pixel + scale_color (canvas.rs:26-43).  A warp owns 8x4 pixels: four canvas rows of 96 B (f32) and
    // 24 B (8-bit).  When the frame's width is a multiple of 8 those row pieces are 16- / 8-byte aligned in global memory,
    // so the warp transposes its colours through shared memory and writes them as 24 STG.128 + 12 STG.64 streaming
    // stores instead of six scalar stores per thread at 12- / 3-byte strides.  Warp-private staging: no block barrier,
    // a warp that has finished its pixels leaves.  Ragged right / bottom edges and odd widths keep the per-pixel stores.
    __shared__ __align__(16) float s_rgb[kBlockThreads * 3];
    __shared__ __align__(16) unsigned char s_u8[kBlockThreads * 3];
    const int wx0 = bx * kTileW + (warp % kWarpsX) * 8, wy0 = band * kBandRows + (warp / kWarpsX) * 4;  // warp-uniform
    if ((S.width & 7) == 0 && wx0 + 8 <= S.width && wy0 + 4 <= S.height) {
        float* w_rgb = s_rgb + warp * 96;          // [row 0..3][8 px][rgb]
        unsigned char* w_u8 = s_u8 + warp * 96;
        w_rgb[lane * 3] = c.x, w_rgb[lane * 3 + 1] = c.y, w_rgb[lane * 3 + 2] = c.z;
        w_u8[lane * 3] = scale_color(c.x), w_u8[lane * 3 + 1] = scale_color(c.y), w_u8[lane * 3 + 2] = scale_color(c.z);
        __syncwarp();
        const size_t px0 = (size_t)wy0 * S.width + wx0;  // the warp's first pixel
        if (F.rgb && lane < 24) {  // 6 float4 per row
            const int row = lane / 6, q = lane - row * 6;
            __stcs(reinterpret_cast<float4*>(F.rgb + (px0 + (size_t)row * S.width) * 3) + q, reinterpret_cast<const float4*>(w_rgb)[lane]);
        }
        if (F.u8 && lane >= 20) {  // 3 uint2 per row: lanes 20..31
            const int u = lane - 20, row = u / 3, q = u - row * 3;
            __stcs(reinterpret_cast<uint2*>(F.u8 + (px0 + (size_t)row * S.width) * 3) + q, reinterpret_cast<const uint2*>(w_u8)[u]);
        }
    } else if (inside) {
        size_t idx = ((size_t)y * S.width + x) * 3;
        if (F.rgb) {
            F.rgb[idx] = c.x;
            F.rgb[idx + 1] = c.y;
            F.rgb[idx + 2] = c.z;
        }
        if (F.u8) {
            F.u8[idx] = scale_color(c.x);
            F.u8[idx + 1] = scale_color(c.y);
            F.u8[idx + 2] = scale_color(c.z);
        }
    }
    flush_counters<STATS>(r, k, counters);
    if (F.tile_cost && lane == 0)  // a block lasts as long as its slowest warp
        atomicMax(&F.tile_cost[band * gridDim.x + bx], (unsigned)min(clock64() - (LEAN ? s_t_start[warp] : t_start), 0xffffffffLL));
}

// K1c render_tiles_views: render_tiles for a batch of views of the committed scene (rtc_render_views).  blockIdx.z is a view
// of the launch: the block takes its camera from the view table instead of DevScene and writes view z's frame, which
// follows view z - 1's in the frame planes.  There is no learnt tile order and no tile-cost probe.  The body restates
// render_tiles' instead of sharing it: with render_tiles made a wrapper over a shared inlined body, ptxas allocated the
// existing builds differently (4 B more spill in the lean and the tree builds).
template <bool SMALL, bool CONVERGE, bool DRAWN, bool LEAN>
__global__ void __launch_bounds__(kBlockThreads, tile_min_blocks(SMALL, CONVERGE, LEAN))
    render_tiles_views(const __grid_constant__ DevScene S, const __grid_constant__ SmallScene SS, const DevFrame F,
                       DevCounters* counters, const DevView* views) {
    if (SMALL) stage_small_scene(S, SS);
    const Env E{S, SS};
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int band = F.shard + (F.band_begin + (int)blockIdx.y) * F.n_shards, bx = blockIdx.x;
    // warp w -> 8x4 sub-tile (the lean build evaluates these again after color_at, as render_tiles does)
    auto px_x = [&] { return bx * kTileW + (warp % kWarpsX) * 8 + (lane & 7); };
    auto px_y = [&] { return band * kBandRows + (warp / kWarpsX) * 4 + (lane >> 3); };
    int x = px_x(), y = px_y();
    Ctr<false> k;
    Rays r;
    V3 c = mk(0.f, 0.f, 0.f);
    const bool rendered = x < S.width - 1 && y < S.height - 1;  // camera.rs:80-81
    V3 o = mk(0.f, 0.f, 0.f), d = mk(0.f, 0.f, 1.f);
    {
        const DevView& V = views[blockIdx.z];  // warp-uniform
        if (rendered) ray_for_pixel(V, x, y, o, d);
    }
    if (CONVERGE || rendered)
        c = color_at<false, SMALL, CONVERGE, DRAWN, LEAN>(E, rendered, o, d, F.depth, (unsigned)(y * S.width + x), r, k, nullptr, nullptr);
    if (LEAN) x = px_x(), y = px_y();
    // Canvas::write_pixel + scale_color as in render_tiles: warp-transposed streaming stores where the rows allow them
    const size_t view0 = (size_t)blockIdx.z * ((size_t)S.width * S.height * 3);
    __shared__ __align__(16) float s_rgb[kBlockThreads * 3];
    __shared__ __align__(16) unsigned char s_u8[kBlockThreads * 3];
    const int wx0 = bx * kTileW + (warp % kWarpsX) * 8, wy0 = band * kBandRows + (warp / kWarpsX) * 4;  // warp-uniform
    if ((S.width & 7) == 0 && wx0 + 8 <= S.width && wy0 + 4 <= S.height) {
        float* w_rgb = s_rgb + warp * 96;
        unsigned char* w_u8 = s_u8 + warp * 96;
        w_rgb[lane * 3] = c.x, w_rgb[lane * 3 + 1] = c.y, w_rgb[lane * 3 + 2] = c.z;
        w_u8[lane * 3] = scale_color(c.x), w_u8[lane * 3 + 1] = scale_color(c.y), w_u8[lane * 3 + 2] = scale_color(c.z);
        __syncwarp();
        const size_t px0 = (size_t)wy0 * S.width + wx0;
        if (F.rgb && lane < 24) {
            const int row = lane / 6, q = lane - row * 6;
            __stcs(reinterpret_cast<float4*>(F.rgb + view0 + (px0 + (size_t)row * S.width) * 3) + q, reinterpret_cast<const float4*>(w_rgb)[lane]);
        }
        if (F.u8 && lane >= 20) {
            const int u = lane - 20, row = u / 3, q = u - row * 3;
            __stcs(reinterpret_cast<uint2*>(F.u8 + view0 + (px0 + (size_t)row * S.width) * 3) + q, reinterpret_cast<const uint2*>(w_u8)[u]);
        }
    } else if (x < S.width && y < S.height) {
        const size_t idx = view0 + ((size_t)y * S.width + x) * 3;
        if (F.rgb) F.rgb[idx] = c.x, F.rgb[idx + 1] = c.y, F.rgb[idx + 2] = c.z;
        if (F.u8) F.u8[idx] = scale_color(c.x), F.u8[idx + 1] = scale_color(c.y), F.u8[idx + 2] = scale_color(c.z);
    }
    flush_counters<false>(r, k, counters);
}

// K1b render_stream: Camera::render for tree scenes with branching ray trees — a persistent grid whose lanes draw
// pixels from a counter as their ray trees finish (dev_shade.cuh: PixelStream) instead of owning one pixel each.
#ifndef RTC_STREAM_MINBLOCKS
#define RTC_STREAM_MINBLOCKS 6
#endif
template <bool STATS>
__global__ void __launch_bounds__(kBlockThreads, min_blocks(RTC_STREAM_MINBLOCKS))
    render_stream(const __grid_constant__ DevScene S, const __grid_constant__ SmallScene SS, const DevFrame F, DevCounters* counters) {
    const Env E{S, SS};
    const int blocks_x = (S.width + 7) / 8;
    PixelStream src{S, F, F.stream_counter, (unsigned)F.n_bands * (unsigned)blocks_x * 2u * 32u, blocks_x};
    Ctr<STATS> k;
    Rays r;
    color_at<STATS, false, true, false, false, PixelStream>(E, false, mk(0.f, 0.f, 0.f), mk(0.f, 0.f, 1.f), F.depth, 0u, r, k, nullptr, nullptr, src);
    flush_counters<STATS>(r, k, counters);
}

// The same for a batch of views: the stream covers views x bands x 8x4 blocks, the view outermost
__global__ void __launch_bounds__(kBlockThreads, min_blocks(RTC_STREAM_MINBLOCKS))
    render_stream_views(const __grid_constant__ DevScene S, const __grid_constant__ SmallScene SS, const DevFrame F, DevCounters* counters,
                        const DevView* views, int n_views) {
    const Env E{S, SS};
    const int blocks_x = (S.width + 7) / 8;
    const unsigned view_blocks = (unsigned)F.n_bands * (unsigned)blocks_x * 2u;
    ViewPixelStream src{S, F, F.stream_counter, (unsigned)n_views * view_blocks * 32u, blocks_x, views, view_blocks};
    Ctr<false> k;
    Rays r;
    color_at<false, false, true, false, false, ViewPixelStream>(E, false, mk(0.f, 0.f, 0.f), mk(0.f, 0.f, 1.f), F.depth, 0u, r, k, nullptr,
                                                                    nullptr, src);
    flush_counters<false>(r, k, counters);
}

// K1d render_tiles_samples: rtc_render_samples, n x n samples per pixel.  The samples of output pixel (x, y) are the pixels
// (n x + i, n y + j) of the reference's Camera::render at n W x n H (camera C: Camera::new at that size), each with the jitter
// key that frame gives it; the output is their box filter, summed in f32 from sample (0, 0) with j outer and i inner, then
// divided by n * n.  A lane owns one output pixel of the 8x4 warp tile and traces its n * n samples one after the other, the
// running sum in registers: lanes at the same (i, j) trace rays as coherent as render_tiles', and the n W x n H frame is
// never stored.  Natural tile order, no tile-cost probe.  The lean build keeps the sum, the sample index and the pixel live
// across color_at, so it has its own occupancy target.
#ifndef RTC_SAMPLES_LEAN_MINBLOCKS
#define RTC_SAMPLES_LEAN_MINBLOCKS 8
#endif
constexpr int samples_min_blocks(bool SMALL, bool CONVERGE, bool LEAN) {
    return LEAN ? min_blocks(RTC_SAMPLES_LEAN_MINBLOCKS) : tile_min_blocks(SMALL, CONVERGE, false);
}
// The mean of the n * n samples' sum (rtc_render_samples' last step)
__device__ __forceinline__ V3 sample_mean(V3 sum, int n) {
    const float nn = (float)(n * n);
    return mk(sum.x / nn, sum.y / nn, sum.z / nn);
}
template <bool SMALL, bool CONVERGE, bool DRAWN, bool LEAN>
__global__ void __launch_bounds__(kBlockThreads, samples_min_blocks(SMALL, CONVERGE, LEAN))
    render_tiles_samples(const __grid_constant__ DevScene S, const __grid_constant__ SmallScene SS, const DevFrame F,
                         DevCounters* counters, const __grid_constant__ DevView C, int n) {
    if (SMALL) stage_small_scene(S, SS);
    const Env E{S, SS};
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int band = F.shard + (F.band_begin + (int)blockIdx.y) * F.n_shards, bx = blockIdx.x;
    const int x = bx * kTileW + (warp % kWarpsX) * 8 + (lane & 7);
    const int y = band * kBandRows + (warp / kWarpsX) * 4 + (lane >> 3);
    Ctr<false> k;
    Rays r;
    const bool rendered = x < S.width - 1 && y < S.height - 1;  // camera.rs:80-81
    const unsigned big_w = (unsigned)n * (unsigned)S.width;      // the sample frame's width: the jitter key's row stride
    V3 sum = mk(0.f, 0.f, 0.f);
    for (int s = 0; s < n * n; s++) {  // warp-uniform trip count: the converging build votes in every color_at
        const int j = s / n, i = s - j * n;
        const int sx = n * x + i, sy = n * y + j;
        V3 o = mk(0.f, 0.f, 0.f), d = mk(0.f, 0.f, 1.f);
        if (rendered) ray_for_pixel(C, sx, sy, o, d);
        V3 c = mk(0.f, 0.f, 0.f);
        if (CONVERGE || rendered)
            c = color_at<false, SMALL, CONVERGE, DRAWN, LEAN>(E, rendered, o, d, F.depth, (unsigned)sy * big_w + (unsigned)sx, r, k,
                                                             nullptr, nullptr);
        sum = s == 0 ? c : sum + c;
    }
    const V3 c = rendered ? sample_mean(sum, n) : mk(0.f, 0.f, 0.f);
    // Canvas::write_pixel + scale_color as in render_tiles: warp-transposed streaming stores where the rows allow them
    __shared__ __align__(16) float s_rgb[kBlockThreads * 3];
    __shared__ __align__(16) unsigned char s_u8[kBlockThreads * 3];
    const int wx0 = bx * kTileW + (warp % kWarpsX) * 8, wy0 = band * kBandRows + (warp / kWarpsX) * 4;  // warp-uniform
    if ((S.width & 7) == 0 && wx0 + 8 <= S.width && wy0 + 4 <= S.height) {
        float* w_rgb = s_rgb + warp * 96;
        unsigned char* w_u8 = s_u8 + warp * 96;
        w_rgb[lane * 3] = c.x, w_rgb[lane * 3 + 1] = c.y, w_rgb[lane * 3 + 2] = c.z;
        w_u8[lane * 3] = scale_color(c.x), w_u8[lane * 3 + 1] = scale_color(c.y), w_u8[lane * 3 + 2] = scale_color(c.z);
        __syncwarp();
        const size_t px0 = (size_t)wy0 * S.width + wx0;
        if (F.rgb && lane < 24) {
            const int row = lane / 6, q = lane - row * 6;
            __stcs(reinterpret_cast<float4*>(F.rgb + (px0 + (size_t)row * S.width) * 3) + q, reinterpret_cast<const float4*>(w_rgb)[lane]);
        }
        if (F.u8 && lane >= 20) {
            const int u = lane - 20, row = u / 3, q = u - row * 3;
            __stcs(reinterpret_cast<uint2*>(F.u8 + (px0 + (size_t)row * S.width) * 3) + q, reinterpret_cast<const uint2*>(w_u8)[u]);
        }
    } else if (x < S.width && y < S.height) {
        const size_t idx = ((size_t)y * S.width + x) * 3;
        if (F.rgb) F.rgb[idx] = c.x, F.rgb[idx + 1] = c.y, F.rgb[idx + 2] = c.z;
        if (F.u8) F.u8[idx] = scale_color(c.x), F.u8[idx + 1] = scale_color(c.y), F.u8[idx + 2] = scale_color(c.z);
    }
    flush_counters<false>(r, k, counters);
}

// The pixel stream of rtc_render_samples: a lane claims an output pixel in PixelStream's order and is handed its n * n
// sample rays one after the other — the next sample starts at the first converged top of the loop after the previous one
// finished, before the warp draws new pixels — and finish() keeps the running sum; the last sample stores the mean.
struct SamplePixelStream {
    static constexpr bool kStream = true;
    const DevScene& S;
    const DevFrame& F;
    const DevView& C;       // the sample camera
    unsigned* counter;      // next unclaimed stream index of this launch
    unsigned total;         // stream indices of this launch
    int blocks_x;           // 8-pixel blocks across the frame
    int n;                  // samples per axis
    bool done = false;      // warp-uniform: the counter has run past the end
    bool pending = false;   // the claimed pixel has samples left to trace
    int x = 0, y = 0;       // the claimed pixel
    int next = 0;           // its sample in flight (finish) or to start (refill)
    V3 sum = mk(0.f, 0.f, 0.f);
    __device__ __forceinline__ bool exhausted() const { return done; }
    __device__ __forceinline__ void start(V3& ro, V3& rd, unsigned& pixel) {
        const int j = next / n, i = next - j * n;
        const int sx = n * x + i, sy = n * y + j;
        pixel = (unsigned)sy * ((unsigned)n * (unsigned)S.width) + (unsigned)sx;  // the sample frame's jitter key
        ray_for_pixel(C, sx, sy, ro, rd);
    }
    __device__ __forceinline__ void store(int px, int py, V3 c) {  // Canvas::write_pixel + scale_color (canvas.rs:26-43)
        const size_t i = ((size_t)py * S.width + px) * 3;
        if (F.rgb) F.rgb[i] = c.x, F.rgb[i + 1] = c.y, F.rgb[i + 2] = c.z;
        if (F.u8) F.u8[i] = scale_color(c.x), F.u8[i + 1] = scale_color(c.y), F.u8[i + 2] = scale_color(c.z);
    }
    __device__ __forceinline__ bool refill(bool& running, V3& ro, V3& rd, unsigned& pixel) {
        bool started = false;
        if (!running && pending) start(ro, rd, pixel), running = started = true;
        const unsigned idle = __ballot_sync(0xffffffffu, !running);
        if (done || (__popc(idle) < kRefillLanes && idle != 0xffffffffu)) return started;
        const int lane = threadIdx.x & 31, leader = __ffs(idle) - 1;
        unsigned base = 0;
        if (lane == leader) base = atomicAdd(counter, (unsigned)__popc(idle));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (base + (unsigned)__popc(idle) >= total) done = true;
        if (running) return started;
        const unsigned idx = base + (unsigned)__popc(idle & ((1u << lane) - 1u));
        if (idx >= total) return false;
        const unsigned block = idx >> 5, within = idx & 31u;
        const unsigned per_band = (unsigned)blocks_x * 2u;
        const unsigned band_i = block / per_band, b = block - band_i * per_band;
        const int band = F.shard + (F.band_begin + (int)band_i) * F.n_shards;
        const int px = (int)(b >> 1) * 8 + (int)(within & 7u), py = band * kBandRows + (int)(b & 1u) * 4 + (int)(within >> 3);
        if (px >= S.width || py >= S.height) return false;
        if (px >= S.width - 1 || py >= S.height - 1) {  // camera.rs:80-81: never rendered, stays black (canvas.rs:23)
            store(px, py, mk(0.f, 0.f, 0.f));
            return false;
        }
        x = px, y = py, next = 0, pending = true;
        start(ro, rd, pixel);
        running = true;
        return true;
    }
    __device__ __forceinline__ void finish(unsigned, V3 c) {
        sum = next == 0 ? c : sum + c;
        if (++next == n * n) {
            pending = false;
            store(x, y, sample_mean(sum, n));
        }
    }
};

__global__ void __launch_bounds__(kBlockThreads, min_blocks(RTC_STREAM_MINBLOCKS))
    render_stream_samples(const __grid_constant__ DevScene S, const __grid_constant__ SmallScene SS, const DevFrame F,
                          DevCounters* counters, const __grid_constant__ DevView C, int n) {
    const Env E{S, SS};
    const int blocks_x = (S.width + 7) / 8;
    SamplePixelStream src{S, F, C, F.stream_counter, (unsigned)F.n_bands * (unsigned)blocks_x * 2u * 32u, blocks_x, n};
    Ctr<false> k;
    Rays r;
    color_at<false, false, true, false, false, SamplePixelStream>(E, false, mk(0.f, 0.f, 0.f), mk(0.f, 0.f, 1.f), F.depth, 0u, r, k,
                                                                  nullptr, nullptr, src);
    flush_counters<false>(r, k, counters);
}

// K1e render_tiles_views_samples: rtc_render_views_samples, render_tiles_samples for a batch of views.  blockIdx.z is a
// view of the launch: the block reads its sample camera from the view table (one warp-uniform load per sample) and writes
// view z's frame, which follows view z - 1's.  A sample's jitter key is its index in its own view's n W x n H frame.  The
// body restates render_tiles_samples' rather than sharing it, for the reason render_tiles_views gives: a shared inlined
// body lets ptxas allocate the existing kernels differently.
template <bool SMALL, bool CONVERGE, bool DRAWN, bool LEAN>
__global__ void __launch_bounds__(kBlockThreads, samples_min_blocks(SMALL, CONVERGE, LEAN))
    render_tiles_views_samples(const __grid_constant__ DevScene S, const __grid_constant__ SmallScene SS, const DevFrame F,
                               DevCounters* counters, const DevView* views, int n) {
    if (SMALL) stage_small_scene(S, SS);
    const Env E{S, SS};
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int band = F.shard + (F.band_begin + (int)blockIdx.y) * F.n_shards, bx = blockIdx.x;
    const int x = bx * kTileW + (warp % kWarpsX) * 8 + (lane & 7);
    const int y = band * kBandRows + (warp / kWarpsX) * 4 + (lane >> 3);
    const DevView* C = views + blockIdx.z;  // warp-uniform
    Ctr<false> k;
    Rays r;
    const bool rendered = x < S.width - 1 && y < S.height - 1;  // camera.rs:80-81
    const unsigned big_w = (unsigned)n * (unsigned)S.width;      // the sample frame's width: the jitter key's row stride
    V3 sum = mk(0.f, 0.f, 0.f);
    for (int s = 0; s < n * n; s++) {  // warp-uniform trip count: the converging build votes in every color_at
        const int j = s / n, i = s - j * n;
        const int sx = n * x + i, sy = n * y + j;
        V3 o = mk(0.f, 0.f, 0.f), d = mk(0.f, 0.f, 1.f);
        if (rendered) ray_for_pixel(*C, sx, sy, o, d);
        V3 c = mk(0.f, 0.f, 0.f);
        if (CONVERGE || rendered)
            c = color_at<false, SMALL, CONVERGE, DRAWN, LEAN>(E, rendered, o, d, F.depth, (unsigned)sy * big_w + (unsigned)sx, r, k,
                                                             nullptr, nullptr);
        sum = s == 0 ? c : sum + c;
    }
    const V3 c = rendered ? sample_mean(sum, n) : mk(0.f, 0.f, 0.f);
    // Canvas::write_pixel + scale_color as in render_tiles: warp-transposed streaming stores where the rows allow them
    const size_t view0 = (size_t)blockIdx.z * ((size_t)S.width * S.height * 3);
    __shared__ __align__(16) float s_rgb[kBlockThreads * 3];
    __shared__ __align__(16) unsigned char s_u8[kBlockThreads * 3];
    const int wx0 = bx * kTileW + (warp % kWarpsX) * 8, wy0 = band * kBandRows + (warp / kWarpsX) * 4;  // warp-uniform
    if ((S.width & 7) == 0 && wx0 + 8 <= S.width && wy0 + 4 <= S.height) {
        float* w_rgb = s_rgb + warp * 96;
        unsigned char* w_u8 = s_u8 + warp * 96;
        w_rgb[lane * 3] = c.x, w_rgb[lane * 3 + 1] = c.y, w_rgb[lane * 3 + 2] = c.z;
        w_u8[lane * 3] = scale_color(c.x), w_u8[lane * 3 + 1] = scale_color(c.y), w_u8[lane * 3 + 2] = scale_color(c.z);
        __syncwarp();
        const size_t px0 = (size_t)wy0 * S.width + wx0;
        if (F.rgb && lane < 24) {
            const int row = lane / 6, q = lane - row * 6;
            __stcs(reinterpret_cast<float4*>(F.rgb + view0 + (px0 + (size_t)row * S.width) * 3) + q, reinterpret_cast<const float4*>(w_rgb)[lane]);
        }
        if (F.u8 && lane >= 20) {
            const int u = lane - 20, row = u / 3, q = u - row * 3;
            __stcs(reinterpret_cast<uint2*>(F.u8 + view0 + (px0 + (size_t)row * S.width) * 3) + q, reinterpret_cast<const uint2*>(w_u8)[u]);
        }
    } else if (x < S.width && y < S.height) {
        const size_t idx = view0 + ((size_t)y * S.width + x) * 3;
        if (F.rgb) F.rgb[idx] = c.x, F.rgb[idx + 1] = c.y, F.rgb[idx + 2] = c.z;
        if (F.u8) F.u8[idx] = scale_color(c.x), F.u8[idx + 1] = scale_color(c.y), F.u8[idx + 2] = scale_color(c.z);
    }
    flush_counters<false>(r, k, counters);
}

// The pixel stream of rtc_render_views_samples: SamplePixelStream over views x bands x 8x4 blocks, the view outermost as in
// ViewPixelStream.  A lane keeps its pixel's view (its sample camera and its frame's offset) until the pixel's last sample.
struct ViewSamplePixelStream {
    static constexpr bool kStream = true;
    const DevScene& S;
    const DevFrame& F;
    unsigned* counter;      // next unclaimed stream index of this launch
    unsigned total;         // stream indices of this launch
    int blocks_x;           // 8-pixel blocks across the frame
    const DevView* views;   // the launch's sample cameras
    unsigned view_blocks;   // 8x4 blocks of one view in this launch
    int n;                  // samples per axis
    bool done = false;      // warp-uniform: the counter has run past the end
    bool pending = false;   // the claimed pixel has samples left to trace
    int x = 0, y = 0;       // the claimed pixel
    int next = 0;           // its sample in flight (finish) or to start (refill)
    const DevView* cam = nullptr;  // its view's sample camera
    size_t out = 0;         // where its view starts in the frame planes (elements)
    V3 sum = mk(0.f, 0.f, 0.f);
    __device__ __forceinline__ bool exhausted() const { return done; }
    __device__ __forceinline__ void start(V3& ro, V3& rd, unsigned& pixel) {
        const int j = next / n, i = next - j * n;
        const int sx = n * x + i, sy = n * y + j;
        pixel = (unsigned)sy * ((unsigned)n * (unsigned)S.width) + (unsigned)sx;  // the view's sample frame's jitter key
        ray_for_pixel(*cam, sx, sy, ro, rd);
    }
    __device__ __forceinline__ void store(int px, int py, V3 c) {  // Canvas::write_pixel + scale_color (canvas.rs:26-43)
        const size_t i = out + ((size_t)py * S.width + px) * 3;
        if (F.rgb) F.rgb[i] = c.x, F.rgb[i + 1] = c.y, F.rgb[i + 2] = c.z;
        if (F.u8) F.u8[i] = scale_color(c.x), F.u8[i + 1] = scale_color(c.y), F.u8[i + 2] = scale_color(c.z);
    }
    __device__ __forceinline__ bool refill(bool& running, V3& ro, V3& rd, unsigned& pixel) {
        bool started = false;
        if (!running && pending) start(ro, rd, pixel), running = started = true;
        const unsigned idle = __ballot_sync(0xffffffffu, !running);
        if (done || (__popc(idle) < kRefillLanes && idle != 0xffffffffu)) return started;
        const int lane = threadIdx.x & 31, leader = __ffs(idle) - 1;
        unsigned base = 0;
        if (lane == leader) base = atomicAdd(counter, (unsigned)__popc(idle));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (base + (unsigned)__popc(idle) >= total) done = true;
        if (running) return started;
        const unsigned idx = base + (unsigned)__popc(idle & ((1u << lane) - 1u));
        if (idx >= total) return false;
        const unsigned within = idx & 31u, view = (idx >> 5) / view_blocks, block = (idx >> 5) - view * view_blocks;
        const unsigned per_band = (unsigned)blocks_x * 2u;
        const unsigned band_i = block / per_band, b = block - band_i * per_band;
        const int band = F.shard + (F.band_begin + (int)band_i) * F.n_shards;
        const int px = (int)(b >> 1) * 8 + (int)(within & 7u), py = band * kBandRows + (int)(b & 1u) * 4 + (int)(within >> 3);
        if (px >= S.width || py >= S.height) return false;
        out = (size_t)view * ((size_t)S.width * S.height * 3);
        if (px >= S.width - 1 || py >= S.height - 1) {  // camera.rs:80-81: never rendered, stays black (canvas.rs:23)
            store(px, py, mk(0.f, 0.f, 0.f));
            return false;
        }
        x = px, y = py, next = 0, pending = true, cam = views + view;
        start(ro, rd, pixel);
        running = true;
        return true;
    }
    __device__ __forceinline__ void finish(unsigned, V3 c) {
        sum = next == 0 ? c : sum + c;
        if (++next == n * n) {
            pending = false;
            store(x, y, sample_mean(sum, n));
        }
    }
};

__global__ void __launch_bounds__(kBlockThreads, min_blocks(RTC_STREAM_MINBLOCKS))
    render_stream_views_samples(const __grid_constant__ DevScene S, const __grid_constant__ SmallScene SS, const DevFrame F,
                                DevCounters* counters, const DevView* views, int n_views, int n) {
    const Env E{S, SS};
    const int blocks_x = (S.width + 7) / 8;
    const unsigned view_blocks = (unsigned)F.n_bands * (unsigned)blocks_x * 2u;
    ViewSamplePixelStream src{S, F, F.stream_counter, (unsigned)n_views * view_blocks * 32u, blocks_x, views, view_blocks, n};
    Ctr<false> k;
    Rays r;
    color_at<false, false, true, false, false, ViewSamplePixelStream>(E, false, mk(0.f, 0.f, 0.f), mk(0.f, 0.f, 1.f), F.depth, 0u, r,
                                                                      k, nullptr, nullptr, src);
    flush_counters<false>(r, k, counters);
}

// ---- the wavefront renderer's kernels (dev_wave.cuh) --------------------------------------------------------------------
#ifndef RTC_WAVE_TRACE_MINBLOCKS
#define RTC_WAVE_TRACE_MINBLOCKS 8
#endif
__global__ void __launch_bounds__(128) wave_primary_kernel(const __grid_constant__ DevScene S, const DevFrame F, const WavePoolRaw raw,
                                                          DevCounters* counters) {
    wave_primary(S, F, wave_pool(raw));
}
__global__ void wave_next_level_kernel(const WavePoolRaw raw, int level) { wave_next_level(wave_pool(raw), level); }
template <bool SHADOW>
__global__ void __launch_bounds__(128, RTC_WAVE_TRACE_MINBLOCKS) wave_trace_kernel(const __grid_constant__ DevScene S, const WavePoolRaw raw,
                                                                                 DevCounters* counters, int level) {
    wave_trace<SHADOW>(S, wave_pool(raw), level);
}
__global__ void __launch_bounds__(128) wave_hit_kernel(const __grid_constant__ DevScene S, const WavePoolRaw raw, DevCounters* counters,
                                                      int level) {
    wave_hit(S, wave_pool(raw), level);
}
__global__ void __launch_bounds__(128) wave_shade_kernel(const __grid_constant__ DevScene S, const WavePoolRaw raw, DevCounters* counters,
                                                        int level, int depth) {
    wave_shade(S, wave_pool(raw), level, depth);
}
__global__ void __launch_bounds__(128) wave_combine_kernel(const __grid_constant__ DevScene S, const DevFrame F, const WavePoolRaw raw,
                                                          DevCounters* counters, int level) {
    wave_combine(S, F, wave_pool(raw), level);
}
// DRAWN: as in render_tiles — a small scene whose area light draws its jitter (`jitter_fn = None`) takes the
// drawn-sample cell loop; without it intensity_cells would read light samples nobody staged.
template <bool SMALL, bool DRAWN>
__global__ void __launch_bounds__(kBlockThreads) trace_rays(const __grid_constant__ DevScene S, const __grid_constant__ SmallScene SS, int n,
                                                  const float* origins, const float* directions, int depth, float* out_rgb,
                                                  float* out_t, int* out_pos, DevCounters* counters) {
    if (SMALL) stage_small_scene(S, SS);
    const Env E{S, SS};
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    Ctr<false> k;
    Rays r;
    const bool active = i < n;
    V3 o = mk(0.f, 0.f, 0.f), d = mk(0.f, 0.f, 1.f);
    if (active) o = ld3(origins + 3 * (size_t)i), d = ld3(directions + 3 * (size_t)i);
    float t = -1.0f;
    int pos = -1;
    const V3 c = color_at<false, SMALL, true, DRAWN>(E, active, o, d, depth, (unsigned)i, r, k, &t, &pos);
    if (active) {
        out_rgb[3 * (size_t)i] = c.x;
        out_rgb[3 * (size_t)i + 1] = c.y;
        out_rgb[3 * (size_t)i + 2] = c.z;
        if (out_t) out_t[i] = t;
        if (out_pos) out_pos[i] = pos;
    }
    flush_counters<false>(r, k, counters);
}

// The instantiations frame_variant (rtc_launch.h) can select, X(STATS, SMALL, CONVERGE, DRAWN, LEAN): render_tiles takes all
// of them, render_tiles_views, render_tiles_samples and render_tiles_views_samples those without STATS.  The *_sweep builds have no lean kernel.
#ifndef RTC_CSG_SWEEP_BUILD
constexpr bool kHasLean = true;
#define RTC_LEAN_TILE_VARIANTS(X) X(false, true, false, true, true) X(false, true, false, false, true)
#else
constexpr bool kHasLean = false;
#define RTC_LEAN_TILE_VARIANTS(X)
#endif
#define RTC_TILE_VARIANTS(X)                                                                                                 \
    RTC_LEAN_TILE_VARIANTS(X)                                                                                                \
    X(true, true, true, true, false) X(false, true, true, true, false) X(false, true, false, true, false)                    \
    X(true, true, true, false, false) X(true, false, true, false, false)                                                     \
    X(false, true, true, false, false) X(false, true, false, false, false)                                                   \
    X(false, false, true, false, false) X(false, false, false, false, false)
// trace_variant's choices, X(SMALL, DRAWN)
#define RTC_TRACE_VARIANTS(X) X(true, true) X(true, false) X(false, false)

}  // namespace RTC_NS
}  // namespace rtc
