// rtc_kernels.cu — the sm_100a kernels.  Compiled twice into the library: as namespace `fast` (FMA
// contraction on) and, with -DRTC_STRICT -fmad=false, as namespace `strict` (the Rust / IEEE evaluation
// order bit for bit).  rtc_api.cu picks one per scene (RTC_OPT_STRICT_FP).
//
// K1 render_tiles : Camera::render (camera.rs:76-91) — one thread per pixel, 128-thread blocks covering a
//                   16x8 pixel tile as four 8x4 warps so that a warp's rays stay coherent; writes the f32
//                   RGB canvas and the 8-bit canvas (canvas.rs:39-43) in the same pass.
// K4 trace_rays   : World::color_at for caller-supplied rays (the unit-test probe).
// K5 fma_peak     : dependent-FMA micro-benchmark for the measured FP32 roofline denominator.
// Each is compiled once more with -DRTC_CSG_SWEEP_BUILD, as `fast_sweep` / `strict_sweep`: the builds that evaluate CSGs
// beyond csg_eval's limits with csg_sweep (dev_bvh.cuh), used only for scenes that hold one.
#if defined(RTC_STRICT) && defined(RTC_CSG_SWEEP_BUILD)
#define RTC_NS strict_sweep
#elif defined(RTC_STRICT)
#define RTC_NS strict
#elif defined(RTC_CSG_SWEEP_BUILD)
#define RTC_NS fast_sweep
#else
#define RTC_NS fast
#endif

#include "rtc_device.cuh"
#include "rtc_launch.h"

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

// ---- the wavefront renderer's kernels (dev_wave.cuh) --------------------------------------------------------------------
#ifndef RTC_WAVE_TRACE_MINBLOCKS
#define RTC_WAVE_TRACE_MINBLOCKS 8
#endif
__device__ __forceinline__ WavePool wave_pool(const WavePoolRaw& raw, DevCounters* counters) {
    WavePool P;
    P.rays = static_cast<WaveRay*>(raw.rays), P.nodes = static_cast<WaveNode*>(raw.nodes), P.capacity = raw.capacity;
    P.base = raw.ints, P.count = raw.ints + kWaveLevels, P.cursor = raw.ints + 2 * kWaveLevels;
    P.overflow = raw.record, P.secondary = raw.record + 1, P.shades = raw.record + 2;
    (void)counters;
    return P;
}
__global__ void __launch_bounds__(128) wave_primary_kernel(const __grid_constant__ DevScene S, const DevFrame F, const WavePoolRaw raw,
                                                          DevCounters* counters) {
    wave_primary(S, F, wave_pool(raw, counters));
}
// the next level starts where this one ends
__global__ void wave_next_level_kernel(const WavePoolRaw raw, int level) {
    int* base = raw.ints;
    int* count = raw.ints + kWaveLevels;
    base[level + 1] = min(base[level] + count[level], raw.capacity);
}
template <bool SHADOW>
__global__ void __launch_bounds__(128, RTC_WAVE_TRACE_MINBLOCKS) wave_trace_kernel(const __grid_constant__ DevScene S, const WavePoolRaw raw,
                                                                                 DevCounters* counters, int level) {
    wave_trace<SHADOW>(S, wave_pool(raw, counters), level);
}
__global__ void __launch_bounds__(128) wave_hit_kernel(const __grid_constant__ DevScene S, const WavePoolRaw raw, DevCounters* counters,
                                                      int level) {
    wave_hit(S, wave_pool(raw, counters), level);
}
__global__ void __launch_bounds__(128) wave_shade_kernel(const __grid_constant__ DevScene S, const WavePoolRaw raw, DevCounters* counters,
                                                        int level, int depth) {
    wave_shade(S, wave_pool(raw, counters), level, depth);
}
__global__ void __launch_bounds__(128) wave_combine_kernel(const __grid_constant__ DevScene S, const DevFrame F, const WavePoolRaw raw,
                                                          DevCounters* counters, int level) {
    wave_combine(S, F, wave_pool(raw, counters), level);
}

void launch_wave(const DevScene& S, const SmallScene&, const DevFrame& F, const WavePoolRaw& pool, DevCounters* counters, int blocks,
                 cudaStream_t stream) {
    cudaMemsetAsync(pool.ints, 0, kWaveInts * sizeof(int), stream);
    cudaMemsetAsync(pool.record, 0, 3 * sizeof(unsigned long long), stream);
    const int wide = blocks * 2;  // the one-thread-per-ray kernels: a grid-stride loop over a count only the device knows
    wave_primary_kernel<<<wide, 128, 0, stream>>>(S, F, pool, counters);
    for (int level = 0; level <= F.depth; level++) {
        wave_next_level_kernel<<<1, 1, 0, stream>>>(pool, level);
        wave_trace_kernel<false><<<blocks, 128, 0, stream>>>(S, pool, counters, level);
        wave_hit_kernel<<<wide, 128, 0, stream>>>(S, pool, counters, level);
        wave_trace_kernel<true><<<blocks, 128, 0, stream>>>(S, pool, counters, level);
        wave_shade_kernel<<<wide, 128, 0, stream>>>(S, pool, counters, level, F.depth);
    }
    for (int level = F.depth; level >= 0; level--) wave_combine_kernel<<<wide, 128, 0, stream>>>(S, F, pool, counters, level);
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

void launch_render(const DevScene& S, const SmallScene& SS, const DevFrame& F, DevCounters* counters, bool detailed,
                   cudaStream_t stream) {
    dim3 grid((S.width + kTileW - 1) / kTileW, F.n_bands);
    if (grid.x == 0 || grid.y == 0) return;
    const bool small = SS.n > 0;
    if (!small && F.stream_counter) {  // the host zeroed the counter on this stream
        if (detailed)
            render_stream<true><<<F.stream_blocks, kBlockThreads, 0, stream>>>(S, SS, F, counters);
        else
            render_stream<false><<<F.stream_blocks, kBlockThreads, 0, stream>>>(S, SS, F, counters);
        return;
    }
    // small scenes whose area light draws its samples (jitter None) need the build with the drawn-sample cell loop
    const bool drawn = small && SS.cell_masks && S.jitter_len == 0;
    // the detailed (counting) pass always uses the converging build; the timed kernels pick by DevFrame::converge.
    // Lean scenes (SmallScene::lean, set only with cell_masks) take the lean build, which does not use the per-thread
    // shadow-origin cache: the part of kSmallSmemBytes before it is all it stages.
    // The *_sweep builds have no lean kernel: a scene that needs them holds a CSG, and a lean one holds none.
#ifndef RTC_CSG_SWEEP_BUILD
    if (!detailed && !F.converge && small && SS.cell_masks && SS.lean) {
        if (drawn)
            render_tiles<false, true, false, true, true><<<grid, kBlockThreads, kSmemOrg * 16, stream>>>(S, SS, F, counters);
        else
            render_tiles<false, true, false, false, true><<<grid, kBlockThreads, kSmemOrg * 16, stream>>>(S, SS, F, counters);
        return;
    }
#endif
    if (drawn) {
        if (detailed)
            render_tiles<true, true, true, true><<<grid, kBlockThreads, kSmallSmemBytes, stream>>>(S, SS, F, counters);
        else if (F.converge)
            render_tiles<false, true, true, true><<<grid, kBlockThreads, kSmallSmemBytes, stream>>>(S, SS, F, counters);
        else
            render_tiles<false, true, false, true><<<grid, kBlockThreads, kSmallSmemBytes, stream>>>(S, SS, F, counters);
    } else if (detailed) {
        if (small)
            render_tiles<true, true, true, false><<<grid, kBlockThreads, kSmallSmemBytes, stream>>>(S, SS, F, counters);
        else
            render_tiles<true, false, true, false><<<grid, kBlockThreads, 0, stream>>>(S, SS, F, counters);
    } else if (small) {
        if (F.converge)
            render_tiles<false, true, true, false><<<grid, kBlockThreads, kSmallSmemBytes, stream>>>(S, SS, F, counters);
        else
            render_tiles<false, true, false, false><<<grid, kBlockThreads, kSmallSmemBytes, stream>>>(S, SS, F, counters);
    } else {
        if (F.converge)
            render_tiles<false, false, true, false><<<grid, kBlockThreads, 0, stream>>>(S, SS, F, counters);
        else
            render_tiles<false, false, false, false><<<grid, kBlockThreads, 0, stream>>>(S, SS, F, counters);
    }
}

// A batch of views (rtc_render_views): the kernel choice of launch_render without its detailed pass
void launch_views(const DevScene& S, const SmallScene& SS, const DevFrame& F, const DevView* views, int n_views, DevCounters* counters,
                  cudaStream_t stream) {
    dim3 grid((S.width + kTileW - 1) / kTileW, F.n_bands, n_views);
    if (grid.x == 0 || grid.y == 0 || grid.z == 0) return;
    const bool small = SS.n > 0;
    if (!small && F.stream_counter) {
        render_stream_views<<<F.stream_blocks, kBlockThreads, 0, stream>>>(S, SS, F, counters, views, n_views);
        return;
    }
    const bool drawn = small && SS.cell_masks && S.jitter_len == 0;
#ifndef RTC_CSG_SWEEP_BUILD
    if (!F.converge && small && SS.cell_masks && SS.lean) {
        if (drawn)
            render_tiles_views<true, false, true, true><<<grid, kBlockThreads, kSmemOrg * 16, stream>>>(S, SS, F, counters, views);
        else
            render_tiles_views<true, false, false, true><<<grid, kBlockThreads, kSmemOrg * 16, stream>>>(S, SS, F, counters, views);
        return;
    }
#endif
    if (small) {
        if (drawn && F.converge)
            render_tiles_views<true, true, true, false><<<grid, kBlockThreads, kSmallSmemBytes, stream>>>(S, SS, F, counters, views);
        else if (drawn)
            render_tiles_views<true, false, true, false><<<grid, kBlockThreads, kSmallSmemBytes, stream>>>(S, SS, F, counters, views);
        else if (F.converge)
            render_tiles_views<true, true, false, false><<<grid, kBlockThreads, kSmallSmemBytes, stream>>>(S, SS, F, counters, views);
        else
            render_tiles_views<true, false, false, false><<<grid, kBlockThreads, kSmallSmemBytes, stream>>>(S, SS, F, counters, views);
    } else if (F.converge) {
        render_tiles_views<false, true, false, false><<<grid, kBlockThreads, 0, stream>>>(S, SS, F, counters, views);
    } else {
        render_tiles_views<false, false, false, false><<<grid, kBlockThreads, 0, stream>>>(S, SS, F, counters, views);
    }
}

void launch_trace(const DevScene& S, const SmallScene& SS, int n, const float* origins, const float* directions, int depth,
                  float* out_rgb, float* out_t, int* out_pos, DevCounters* counters, cudaStream_t stream) {
    if (n <= 0) return;
    const bool small = SS.n > 0;
    const bool drawn = small && SS.cell_masks && S.jitter_len == 0;  // the predicate of launch_render
    if (drawn)
        trace_rays<true, true><<<(n + kBlockThreads - 1) / kBlockThreads, kBlockThreads, kSmallSmemBytes, stream>>>(S, SS, n, origins, directions, depth, out_rgb, out_t, out_pos, counters);
    else if (small)
        trace_rays<true, false><<<(n + kBlockThreads - 1) / kBlockThreads, kBlockThreads, kSmallSmemBytes, stream>>>(S, SS, n, origins, directions, depth, out_rgb, out_t, out_pos, counters);
    else
        trace_rays<false, false><<<(n + kBlockThreads - 1) / kBlockThreads, kBlockThreads, 0, stream>>>(S, SS, n, origins, directions, depth, out_rgb, out_t, out_pos, counters);
}

#if !defined(RTC_STRICT) && !defined(RTC_CSG_SWEEP_BUILD)
// K5: 8 independent FMA chains per thread, 4096 iterations: 2 * 8 * 4096 flops per thread.
__global__ void __launch_bounds__(256) fma_peak(float* out, float a, float b, int iters) {
    float x0 = threadIdx.x, x1 = x0 + 1.f, x2 = x0 + 2.f, x3 = x0 + 3.f, x4 = x0 + 4.f, x5 = x0 + 5.f, x6 = x0 + 6.f, x7 = x0 + 7.f;
    for (int i = 0; i < iters; i++) {
        x0 = fmaf(x0, a, b);
        x1 = fmaf(x1, a, b);
        x2 = fmaf(x2, a, b);
        x3 = fmaf(x3, a, b);
        x4 = fmaf(x4, a, b);
        x5 = fmaf(x5, a, b);
        x6 = fmaf(x6, a, b);
        x7 = fmaf(x7, a, b);
    }
    float s = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
    if (s == 12345.678f) out[0] = s;  // keep the chains alive
}
void launch_fma_peak(float* out, int blocks, int iters, cudaStream_t stream) {
    fma_peak<<<blocks, 256, 0, stream>>>(out, 0.999f, 0.001f, iters);
}
#endif

}  // namespace RTC_NS
}  // namespace rtc
