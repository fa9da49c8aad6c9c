// rtc_kernels.cu — the sm_100a kernels.  Compiled twice into the library: as namespace `fast` (FMA
// contraction on) and, with -DRTC_STRICT -fmad=false, as namespace `strict` (the Rust / IEEE evaluation
// order bit for bit).  rtc_api.cu picks one per scene (RTC_OPT_STRICT_FP).
//
// K1 render_tiles : Camera::render (camera.rs:76-91) — one thread per pixel, 128-thread blocks covering a
//                   16x8 pixel tile as four 8x4 warps so that a warp's rays stay coherent; writes the f32
//                   RGB canvas and the 8-bit canvas (canvas.rs:39-43) in the same pass.
//                   render_tiles_views / render_tiles_samples / render_tiles_views_samples: the same for a batch of
//                   views, for n x n samples per pixel (rtc_render_samples), and for both at once
//                   (rtc_render_views_samples); render_stream* the pixel-stream forms for branching tree scenes.
// K4 trace_rays   : World::color_at for caller-supplied rays (the unit-test probe).
// K5 fma_peak     : dependent-FMA micro-benchmark for the measured FP32 roofline denominator.
// Each is compiled once more with -DRTC_CSG_SWEEP_BUILD, as `fast_sweep` / `strict_sweep`: the builds that evaluate CSGs
// beyond csg_eval's limits with csg_sweep (dev_bvh.cuh), used only for scenes that hold one.
// The kernels' bodies are in dev_kernels.cuh; this file holds the launch functions, which switch on the variant
// rtc_launch.h's frame_variant / trace_variant choose.
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

#include "dev_kernels.cuh"

namespace rtc {
namespace RTC_NS {

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

void launch_render(const DevScene& S, const SmallScene& SS, const DevFrame& F, DevCounters* counters, bool detailed,
                   cudaStream_t stream) {
    dim3 grid((S.width + kTileW - 1) / kTileW, F.n_bands);
    if (grid.x == 0 || grid.y == 0) return;
    const KernelVariant v = frame_variant(S, SS, F, detailed, kHasLean);
    if (v.stream) {
        if (v.stats)
            render_stream<true><<<F.stream_blocks, kBlockThreads, 0, stream>>>(S, SS, F, counters);
        else
            render_stream<false><<<F.stream_blocks, kBlockThreads, 0, stream>>>(S, SS, F, counters);
        return;
    }
    const int smem = dynamic_smem(v);
    switch (variant_code(v)) {
#define RTC_LAUNCH_TILES(ST, SM, CV, DR, LE)                                                                  \
    case variant_code(ST, SM, CV, DR, LE):                                                                   \
        render_tiles<ST, SM, CV, DR, LE><<<grid, kBlockThreads, smem, stream>>>(S, SS, F, counters); \
        break;
        RTC_TILE_VARIANTS(RTC_LAUNCH_TILES)
#undef RTC_LAUNCH_TILES
    }
}

// A batch of views (rtc_render_views): the kernel choice of launch_render without its detailed pass
void launch_views(const DevScene& S, const SmallScene& SS, const DevFrame& F, const DevView* views, int n_views, DevCounters* counters,
                  cudaStream_t stream) {
    dim3 grid((S.width + kTileW - 1) / kTileW, F.n_bands, n_views);
    if (grid.x == 0 || grid.y == 0 || grid.z == 0) return;
    const KernelVariant v = frame_variant(S, SS, F, false, kHasLean);
    if (v.stream) {
        render_stream_views<<<F.stream_blocks, kBlockThreads, 0, stream>>>(S, SS, F, counters, views, n_views);
        return;
    }
    const int smem = dynamic_smem(v);
    switch (variant_code(v)) {
#define RTC_LAUNCH_VIEWS(ST, SM, CV, DR, LE) RTC_LAUNCH_VIEWS_##ST(SM, CV, DR, LE)
#define RTC_LAUNCH_VIEWS_true(SM, CV, DR, LE)  // the counting pass has no views kernel
#define RTC_LAUNCH_VIEWS_false(SM, CV, DR, LE)                                                                    \
    case variant_code(false, SM, CV, DR, LE):                                                                    \
        render_tiles_views<SM, CV, DR, LE><<<grid, kBlockThreads, smem, stream>>>(S, SS, F, counters, views); \
        break;
        RTC_TILE_VARIANTS(RTC_LAUNCH_VIEWS)
#undef RTC_LAUNCH_VIEWS
#undef RTC_LAUNCH_VIEWS_true
#undef RTC_LAUNCH_VIEWS_false
    }
}

// n x n samples per pixel (rtc_render_samples): launch_views' kernel choice for one view, the sample camera C
void launch_samples(const DevScene& S, const SmallScene& SS, const DevFrame& F, const DevView& C, int n, DevCounters* counters,
                    cudaStream_t stream) {
    dim3 grid((S.width + kTileW - 1) / kTileW, F.n_bands);
    if (grid.x == 0 || grid.y == 0) return;
    const KernelVariant v = frame_variant(S, SS, F, false, kHasLean);
    if (v.stream) {
        render_stream_samples<<<F.stream_blocks, kBlockThreads, 0, stream>>>(S, SS, F, counters, C, n);
        return;
    }
    const int smem = dynamic_smem(v);
    switch (variant_code(v)) {
#define RTC_LAUNCH_SAMPLES(ST, SM, CV, DR, LE) RTC_LAUNCH_SAMPLES_##ST(SM, CV, DR, LE)
#define RTC_LAUNCH_SAMPLES_true(SM, CV, DR, LE)  // the counting pass has no samples kernel
#define RTC_LAUNCH_SAMPLES_false(SM, CV, DR, LE)                                                                      \
    case variant_code(false, SM, CV, DR, LE):                                                                        \
        render_tiles_samples<SM, CV, DR, LE><<<grid, kBlockThreads, smem, stream>>>(S, SS, F, counters, C, n); \
        break;
        RTC_TILE_VARIANTS(RTC_LAUNCH_SAMPLES)
#undef RTC_LAUNCH_SAMPLES
#undef RTC_LAUNCH_SAMPLES_true
#undef RTC_LAUNCH_SAMPLES_false
    }
}

// A batch of views with n x n samples per pixel (rtc_render_views_samples): launch_samples' kernel choice, views[v] view v's
// sample camera, view z of the grid view v's frame as in launch_views
void launch_views_samples(const DevScene& S, const SmallScene& SS, const DevFrame& F, const DevView* views, int n_views, int n,
                          DevCounters* counters, cudaStream_t stream) {
    dim3 grid((S.width + kTileW - 1) / kTileW, F.n_bands, n_views);
    if (grid.x == 0 || grid.y == 0 || grid.z == 0) return;
    const KernelVariant v = frame_variant(S, SS, F, false, kHasLean);
    if (v.stream) {
        render_stream_views_samples<<<F.stream_blocks, kBlockThreads, 0, stream>>>(S, SS, F, counters, views, n_views, n);
        return;
    }
    const int smem = dynamic_smem(v);
    switch (variant_code(v)) {
#define RTC_LAUNCH_VIEWS_SAMPLES(ST, SM, CV, DR, LE) RTC_LAUNCH_VIEWS_SAMPLES_##ST(SM, CV, DR, LE)
#define RTC_LAUNCH_VIEWS_SAMPLES_true(SM, CV, DR, LE)  // the counting pass has no samples kernel
#define RTC_LAUNCH_VIEWS_SAMPLES_false(SM, CV, DR, LE)                                                                         \
    case variant_code(false, SM, CV, DR, LE):                                                                                 \
        render_tiles_views_samples<SM, CV, DR, LE><<<grid, kBlockThreads, smem, stream>>>(S, SS, F, counters, views, n); \
        break;
        RTC_TILE_VARIANTS(RTC_LAUNCH_VIEWS_SAMPLES)
#undef RTC_LAUNCH_VIEWS_SAMPLES
#undef RTC_LAUNCH_VIEWS_SAMPLES_true
#undef RTC_LAUNCH_VIEWS_SAMPLES_false
    }
}

void launch_trace(const DevScene& S, const SmallScene& SS, int n, const float* origins, const float* directions, int depth,
                  float* out_rgb, float* out_t, int* out_pos, DevCounters* counters, cudaStream_t stream) {
    if (n <= 0) return;
    const KernelVariant v = trace_variant(S, SS);
    const int blocks = (n + kBlockThreads - 1) / kBlockThreads, smem = dynamic_smem(v);
    switch (variant_code(v)) {
#define RTC_LAUNCH_TRACE(SM, DR)                                                                                                  \
    case variant_code(false, SM, true, DR, false):                                                                               \
        trace_rays<SM, DR><<<blocks, kBlockThreads, smem, stream>>>(S, SS, n, origins, directions, depth, out_rgb, out_t, out_pos, \
                                                                   counters);                                                   \
        break;
        RTC_TRACE_VARIANTS(RTC_LAUNCH_TRACE)
#undef RTC_LAUNCH_TRACE
    }
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
