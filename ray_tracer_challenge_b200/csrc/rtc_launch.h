// rtc_launch.h — host-callable launchers of the kernel builds (see rtc_kernels.cu).
#pragma once
#include <cuda_runtime.h>

#include "rtc_types.h"

namespace rtc {
// The kernel a launch function runs for its inputs.  launch_render, launch_views, launch_samples, launch_views_samples and
// launch_trace (rtc_kernels.cu) switch on it, and so does the host harness of the kernels (tests/emu/emu_kernels.cpp), which
// thus runs the kernel the GPU runs.
struct KernelVariant {
    bool stream;  // render_stream / render_stream_views / render_stream_samples / render_stream_views_samples: a tree scene
                  // whose lanes draw pixels from F.stream_counter
    // otherwise the template flags of render_tiles / render_tiles_views / render_tiles_samples / render_tiles_views_samples /
    // trace_rays
    bool stats, small, converge, drawn, lean;
};
constexpr int variant_code(bool stats, bool small, bool converge, bool drawn, bool lean) {
    return (stats ? 16 : 0) | (small ? 8 : 0) | (converge ? 4 : 0) | (drawn ? 2 : 0) | (lean ? 1 : 0);
}
constexpr int variant_code(const KernelVariant& v) { return variant_code(v.stats, v.small, v.converge, v.drawn, v.lean); }

// A frame or a batch of views.  detailed: the counting pass (launch_render only), which always uses the converging build;
// the timed kernels pick by DevFrame::converge.  Small scenes whose area light draws its samples (jitter None) need the
// build with the drawn-sample cell loop.  Lean scenes (SmallScene::lean, set only with cell_masks) take the lean build,
// which does not use the per-thread shadow-origin cache: the part of kSmallSmemBytes before it is all it stages.
// has_lean: the build has the lean kernel (the *_sweep builds have none: a scene that needs them holds a CSG, and a lean
// one holds none).
inline KernelVariant frame_variant(const DevScene& S, const SmallScene& SS, const DevFrame& F, bool detailed, bool has_lean) {
    const bool small = SS.n > 0;
    if (!small && F.stream_counter) return {true, detailed, false, true, false, false};  // the host zeroed the counter
    const bool drawn = small && SS.cell_masks && S.jitter_len == 0;
    const bool lean = has_lean && !detailed && !F.converge && small && SS.cell_masks && SS.lean;
    return {false, detailed, small, detailed || F.converge != 0, drawn, lean};
}
// Caller-supplied rays: always the converging build, drawn by the predicate of frame_variant
inline KernelVariant trace_variant(const DevScene& S, const SmallScene& SS) {
    const bool small = SS.n > 0;
    return {false, false, small, true, small && SS.cell_masks && S.jitter_len == 0, false};
}
// The dynamic shared memory of a tile or trace kernel: small scenes stage their table (dev_small.cuh); the lean build
// stages only the part of kSmallSmemBytes before the shadow-origin cache
inline int dynamic_smem(const KernelVariant& v) { return v.lean ? kSmemOrg * 16 : v.small ? kSmallSmemBytes : 0; }

namespace fast {
void launch_render(const DevScene& S, const SmallScene& SS, const DevFrame& F, DevCounters* counters, bool detailed,
                   cudaStream_t stream);
// A batch of views of the committed scene (rtc_render_views): F's bands of `n_views` views, view v's camera views[v] and its
// frame at F.rgb / F.u8 + v * width * height * 3; a tree scene with F.stream_counter set renders them as one pixel stream.
void launch_views(const DevScene& S, const SmallScene& SS, const DevFrame& F, const DevView* views, int n_views, DevCounters* counters,
                  cudaStream_t stream);
// n x n samples per pixel of the committed canvas (rtc_render_samples): the bands of F, each output pixel the box filter of
// the pixels (n x + i, n y + j) of `camera`, the reference's Camera::new at n width x n height; a tree scene with
// F.stream_counter set renders them as one pixel stream.
// launch_views_samples: the same for a batch of views (rtc_render_views_samples), cameras[v] view v's sample camera and its
// frame at F.rgb / F.u8 + v * width * height * 3, as launch_views lays them out.
void launch_samples(const DevScene& S, const SmallScene& SS, const DevFrame& F, const DevView& camera, int samples_per_axis,
                    DevCounters* counters, cudaStream_t stream);
void launch_views_samples(const DevScene& S, const SmallScene& SS, const DevFrame& F, const DevView* cameras, int n_views,
                          int samples_per_axis, DevCounters* counters, cudaStream_t stream);
void launch_trace(const DevScene& S, const SmallScene& SS, int n, const float* origins, const float* directions, int depth,
                  float* out_rgb, float* out_t, int* out_pos, DevCounters* counters, cudaStream_t stream);
void launch_fma_peak(float* out, int blocks, int iters, cudaStream_t stream);
// One chunk of a frame (the bands of F) through the wavefront renderer: every kernel of every level, enqueued on `stream`
// with no host synchronisation in between (counts live on the device).  `blocks`: the persistent grid of the tree walks.
void launch_wave(const DevScene& S, const SmallScene& SS, const DevFrame& F, const WavePoolRaw& pool, DevCounters* counters, int blocks,
                 cudaStream_t stream);
}  // namespace fast
namespace strict {
void launch_render(const DevScene& S, const SmallScene& SS, const DevFrame& F, DevCounters* counters, bool detailed,
                   cudaStream_t stream);
void launch_views(const DevScene& S, const SmallScene& SS, const DevFrame& F, const DevView* views, int n_views, DevCounters* counters,
                  cudaStream_t stream);
void launch_samples(const DevScene& S, const SmallScene& SS, const DevFrame& F, const DevView& camera, int samples_per_axis,
                    DevCounters* counters, cudaStream_t stream);
void launch_views_samples(const DevScene& S, const SmallScene& SS, const DevFrame& F, const DevView* cameras, int n_views,
                          int samples_per_axis, DevCounters* counters, cudaStream_t stream);
void launch_trace(const DevScene& S, const SmallScene& SS, int n, const float* origins, const float* directions, int depth,
                  float* out_rgb, float* out_t, int* out_pos, DevCounters* counters, cudaStream_t stream);
void launch_wave(const DevScene& S, const SmallScene& SS, const DevFrame& F, const WavePoolRaw& pool, DevCounters* counters, int blocks,
                 cudaStream_t stream);
}  // namespace strict
// the same two builds with csg_sweep's call sites (scenes holding a CSG beyond csg_eval's limits)
namespace fast_sweep {
void launch_render(const DevScene& S, const SmallScene& SS, const DevFrame& F, DevCounters* counters, bool detailed,
                   cudaStream_t stream);
void launch_views(const DevScene& S, const SmallScene& SS, const DevFrame& F, const DevView* views, int n_views, DevCounters* counters,
                  cudaStream_t stream);
void launch_samples(const DevScene& S, const SmallScene& SS, const DevFrame& F, const DevView& camera, int samples_per_axis,
                    DevCounters* counters, cudaStream_t stream);
void launch_views_samples(const DevScene& S, const SmallScene& SS, const DevFrame& F, const DevView* cameras, int n_views,
                          int samples_per_axis, DevCounters* counters, cudaStream_t stream);
void launch_trace(const DevScene& S, const SmallScene& SS, int n, const float* origins, const float* directions, int depth,
                  float* out_rgb, float* out_t, int* out_pos, DevCounters* counters, cudaStream_t stream);
void launch_wave(const DevScene& S, const SmallScene& SS, const DevFrame& F, const WavePoolRaw& pool, DevCounters* counters, int blocks,
                 cudaStream_t stream);
}  // namespace fast_sweep
namespace strict_sweep {
void launch_render(const DevScene& S, const SmallScene& SS, const DevFrame& F, DevCounters* counters, bool detailed,
                   cudaStream_t stream);
void launch_views(const DevScene& S, const SmallScene& SS, const DevFrame& F, const DevView* views, int n_views, DevCounters* counters,
                  cudaStream_t stream);
void launch_samples(const DevScene& S, const SmallScene& SS, const DevFrame& F, const DevView& camera, int samples_per_axis,
                    DevCounters* counters, cudaStream_t stream);
void launch_views_samples(const DevScene& S, const SmallScene& SS, const DevFrame& F, const DevView* cameras, int n_views,
                          int samples_per_axis, DevCounters* counters, cudaStream_t stream);
void launch_trace(const DevScene& S, const SmallScene& SS, int n, const float* origins, const float* directions, int depth,
                  float* out_rgb, float* out_t, int* out_pos, DevCounters* counters, cudaStream_t stream);
void launch_wave(const DevScene& S, const SmallScene& SS, const DevFrame& F, const WavePoolRaw& pool, DevCounters* counters, int blocks,
                 cudaStream_t stream);
}  // namespace strict_sweep
// rtc_render_ppm (rtc_ppm.cu; one build: no floating point): out[j] = the byte length of the PPM text of R's row j; then
// that text written at out + row_at[j]
void launch_ppm_row_bytes(const PpmRows& R, unsigned long long* out, int sm_count, cudaStream_t stream);
void launch_ppm_write(const PpmRows& R, const unsigned long long* row_at, char* out, int sm_count, cudaStream_t stream);
}  // namespace rtc
