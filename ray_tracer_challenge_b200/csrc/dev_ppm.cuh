// dev_ppm.cuh — Canvas::to_ppm (canvas.rs:58-96) of the frame's 8-bit plane, written on the device: the kernels of
// rtc_ppm.cu (rtc_render_ppm, rtc_render_views_ppm), apart from their launch functions so that the host harness
// (tests/emu/emu_ppm.cpp) compiles the same bodies.  A launch covers the rows of one device's bands in each of n_views
// frames (PpmRows); a single frame is one view.  Like the other device parts it opens namespace rtc::RTC_NS itself.
//
// A row's text is its 3 * width values in decimal, each followed by exactly one separator byte: after the row's last value
// a newline, after any other a space, or a newline where the line has reached 70 - 3 columns (canvas.rs:47-55).  So a
// value's offset in its row is the sum of (digits + 1) over the values before it, and the row's length that sum over all of
// them, whatever the line breaks: the breaks only decide which separators are newlines.  A line that starts at row offset
// p ends at the first value whose separator lies at or beyond p + 67 (the line is then at least 67 columns long).
#pragma once

namespace rtc {
namespace RTC_NS {

constexpr int kPpmThreads = 128;  // four warps; a warp writes one row at a time
constexpr int kPpmPerLane = 4;    // consecutive values per lane: a warp steps through a row 128 values at a time
constexpr unsigned kPpmNoValue = 256u;

__device__ __forceinline__ unsigned ppm_digits(unsigned v) { return 1u + (v >= 10u) + (v >= 100u); }
__device__ __forceinline__ long long ppm_launch_rows(const PpmRows& R) { return (long long)R.n_rows * R.n_views; }
__device__ __forceinline__ const unsigned char* ppm_row(const PpmRows& R, long long j) {
    const long long v = j / R.n_rows, r = j - v * R.n_rows;  // view v's row r
    const size_t row = (size_t)(R.shard + r / kBandRows * R.n_shards) * kBandRows + (size_t)(r % kBandRows);
    return R.u8 + (size_t)v * R.view_stride + row * (size_t)R.width * 3;
}

// out[j] = the byte length of the text of R's row j
__global__ void __launch_bounds__(kPpmThreads) ppm_row_bytes(PpmRows R, unsigned long long* out) {
    const int lane = threadIdx.x & 31;
    const size_t n = (size_t)R.width * 3;
    const long long warps = (long long)gridDim.x * (kPpmThreads / 32);
    for (long long j = (long long)blockIdx.x * (kPpmThreads / 32) + (threadIdx.x >> 5); j < ppm_launch_rows(R); j += warps) {
        const unsigned char* src = ppm_row(R, j);
        unsigned sum = 0;  // at most 16 bytes per 128 values of the row: below 2^32 for every canvas rtc_set_camera accepts
        for (size_t c = (size_t)lane * kPpmPerLane; c < n; c += 32 * kPpmPerLane)
#pragma unroll
            for (int k = 0; k < kPpmPerLane; k++)
                if (c + k < n) sum += ppm_digits(src[c + k]) + 1u;
        const unsigned hi = __reduce_add_sync(0xffffffffu, sum >> 16), lo = __reduce_add_sync(0xffffffffu, sum & 0xffffu);
        if (lane == 0) out[j] = ((unsigned long long)hi << 16) + lo;
    }
}

// The text of R's row j at text + row_at[j].  A step of a warp: each lane takes 4 consecutive values, a warp scan gives
// their offsets, then the line ends of the step are found one per ballot (a line holds 17 to 34 values, so a step has at
// most 8), and every lane writes its values and separators.
__global__ void __launch_bounds__(kPpmThreads) ppm_write(PpmRows R, const unsigned long long* row_at, char* text) {
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const size_t n = (size_t)R.width * 3;
    const long long warps = (long long)gridDim.x * (kPpmThreads / 32);
    for (long long j = (long long)blockIdx.x * (kPpmThreads / 32) + (threadIdx.x >> 5); j < ppm_launch_rows(R); j += warps) {
        const unsigned char* src = ppm_row(R, j);
        char* dst = text + row_at[j];
        unsigned long long base = 0;  // row offset of the step's first value
        unsigned long long line = 0;  // row offset where the current line starts
        for (size_t c = 0; c < n; c += 32 * kPpmPerLane) {
            const size_t first = c + (size_t)lane * kPpmPerLane;
            unsigned v[kPpmPerLane], end[kPpmPerLane];  // a value (kPpmNoValue past the row's end); lane offset past its separator
            unsigned mine = 0;
#pragma unroll
            for (int k = 0; k < kPpmPerLane; k++) {
                v[k] = first + k < n ? (unsigned)src[first + k] : kPpmNoValue;
                mine += v[k] != kPpmNoValue ? ppm_digits(v[k]) + 1u : 0u;
                end[k] = mine;
            }
            unsigned incl = mine;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const unsigned t = __shfl_sync(full, incl, lane >= d ? lane - d : lane);
                if (lane >= d) incl += t;
            }
            const unsigned before = incl - mine;  // step offset of the lane's first value
            const unsigned step = __shfl_sync(full, incl, 31);
            unsigned breaks = 0;  // bit k: value k's separator ends its line
            for (;;) {
                int k_end = -1;
                unsigned at_end = 0;
#pragma unroll
                for (int k = 0; k < kPpmPerLane; k++)
                    if (k_end < 0 && v[k] != kPpmNoValue && base + before + end[k] >= line + 68) k_end = k, at_end = before + end[k];
                const unsigned who = __ballot_sync(full, k_end >= 0);
                if (!who) break;
                const int owner = __ffs((int)who) - 1;
                if (lane == owner) breaks |= 1u << k_end;
                line = base + __shfl_sync(full, at_end, owner);
            }
            char* p = dst + base + before;
#pragma unroll
            for (int k = 0; k < kPpmPerLane; k++) {
                if (v[k] == kPpmNoValue) continue;
                const unsigned d = ppm_digits(v[k]);
                unsigned x = v[k];
                for (unsigned q = d; q-- > 0; x /= 10u) p[q] = (char)('0' + x % 10u);
                p[d] = (breaks >> k & 1u) || first + k == n - 1 ? '\n' : ' ';
                p += d + 1;
            }
            base += step;
        }
    }
}

}  // namespace RTC_NS
}  // namespace rtc
