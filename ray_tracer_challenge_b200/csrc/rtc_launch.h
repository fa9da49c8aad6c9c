// rtc_launch.h — host-callable launchers of the kernel builds (see rtc_kernels.cu).
#pragma once
#include <cuda_runtime.h>

#include "rtc_types.h"

namespace rtc {
namespace fast {
void launch_render(const DevScene& S, const SmallScene& SS, const DevFrame& F, DevCounters* counters, bool detailed,
                   cudaStream_t stream);
// A batch of views of the committed scene (rtc_render_views): F's bands of `n_views` views, view v's camera views[v] and its
// frame at F.rgb / F.u8 + v * width * height * 3; a tree scene with F.stream_counter set renders them as one pixel stream.
void launch_views(const DevScene& S, const SmallScene& SS, const DevFrame& F, const DevView* views, int n_views, DevCounters* counters,
                  cudaStream_t stream);
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
void launch_trace(const DevScene& S, const SmallScene& SS, int n, const float* origins, const float* directions, int depth,
                  float* out_rgb, float* out_t, int* out_pos, DevCounters* counters, cudaStream_t stream);
void launch_wave(const DevScene& S, const SmallScene& SS, const DevFrame& F, const WavePoolRaw& pool, DevCounters* counters, int blocks,
                 cudaStream_t stream);
}  // namespace strict_sweep
}  // namespace rtc
