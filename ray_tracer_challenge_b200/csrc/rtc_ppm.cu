// rtc_ppm.cu — the PPM text kernels of rtc_render_ppm and rtc_render_views_ppm (bodies in dev_ppm.cuh).  Compiled once: they do no floating point,
// so the fast / strict builds of rtc_kernels.cu have nothing to differ in.
#define RTC_NS text

#include <algorithm>

#include "rtc_launch.h"

#include "dev_ppm.cuh"

namespace rtc {

namespace {
int ppm_grid(const PpmRows& R, int sm_count) {
    const int warps = text::kPpmThreads / 32;
    return (int)std::min<long long>(((long long)R.n_rows * R.n_views + warps - 1) / warps, (long long)sm_count * 16);
}
}  // namespace

void launch_ppm_row_bytes(const PpmRows& R, unsigned long long* out, int sm_count, cudaStream_t stream) {
    if (R.n_rows <= 0 || R.n_views <= 0) return;
    text::ppm_row_bytes<<<ppm_grid(R, sm_count), text::kPpmThreads, 0, stream>>>(R, out);
}
void launch_ppm_write(const PpmRows& R, const unsigned long long* row_at, char* out, int sm_count, cudaStream_t stream) {
    if (R.n_rows <= 0 || R.n_views <= 0) return;
    text::ppm_write<<<ppm_grid(R, sm_count), text::kPpmThreads, 0, stream>>>(R, row_at, out);
}

}  // namespace rtc
