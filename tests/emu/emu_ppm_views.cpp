// emu_ppm_views.cpp — TEST INFRASTRUCTURE ONLY (built and loaded by tests/test_views_ppm_on_host.py, never by the product):
// the PPM text kernels of rtc_render_views_ppm (dev_ppm.cuh: ppm_row_bytes, ppm_write) run on the HOST in blocks of 128
// threads and warps of 32 lanes (simt.h) over a batch of 8-bit planes the caller gives, with the libraries' host scan
// (rtc_internal.h: ppm_layout) between them.  As rtc_render_views_ppm writes a chunk, each of n_dev devices encodes its own
// bands of every view in one launch of each kernel, and every (view, band)'s text is then copied to its offset.
#include <vector>

#include "rtc_internal.h"  // PpmRows, ppm_header, ppm_device_rows, ppm_layout
#include "simt.h"

#define RTC_NS emu
#include "dev_ppm.cuh"

namespace {
constexpr int kConcurrent = 8;  // blocks at once: the kernels use no shared memory
// blocks of a launch: rtc_ppm.cu's grid for one SM (16 blocks), so that a warp steps through several rows and views
simt::Dim ppm_grid(const rtc::PpmRows& R) {
    const int warps = rtc::emu::kPpmThreads / 32;
    return simt::Dim{(unsigned)std::min<long long>(16, ((long long)R.n_rows * R.n_views + warps - 1) / warps), 1, 1};
}
}  // namespace

// Canvas::to_ppm of each of n_views width x height 8-bit planes (view v's at u8 + v * width * height * 3) into out (capacity
// bytes, >= n_views * rtc_ppm_bound); view_at[v] receives view v's offset.  Returns the total length, -1 when it does not
// fit, -2 when a device's ppm_write wrote past its text.
extern "C" long long emu_ppm_views(const unsigned char* u8, int width, int height, int n_views, int n_dev, char* out,
                                   long long capacity, unsigned long long* view_at) {
    using namespace rtc;
    const size_t plane = (size_t)width * height * 3;
    std::vector<PpmRows> rows(n_dev);
    std::vector<std::vector<unsigned long long>> lengths(n_dev);
    std::vector<unsigned long long*> lp(n_dev);
    for (int i = 0; i < n_dev; i++) {
        rows[i] = PpmRows{u8, width, i, n_dev, ppm_device_rows((uint32_t)height, i, n_dev), n_views, plane};
        lengths[i].assign((size_t)rows[i].n_rows * n_views + 1, ~0ull);
        lp[i] = lengths[i].data();
        if (rows[i].n_rows > 0)
            simt::launch(ppm_grid(rows[i]), emu::kPpmThreads, 0, kConcurrent, [&] { emu::ppm_row_bytes(rows[i], lp[i]); });
    }
    // the scan writes the headers as it goes: check the total first
    const std::string header = ppm_header((uint32_t)width, (uint32_t)height);
    unsigned long long total = (unsigned long long)n_views * header.size();
    for (int i = 0; i < n_dev; i++)
        for (size_t j = 0; j < (size_t)rows[i].n_rows * n_views; j++) total += lp[i][j];
    if ((long long)total > capacity) return -1;
    PpmLayout L;
    ppm_layout((uint32_t)height, n_dev, header.size(), lp.data(), L, n_views, header.data(), out);
    const int total_bands = (height + kBandRows - 1) / kBandRows;
    for (int i = 0; i < n_dev; i++) {
        std::vector<char> text(L.device_bytes[i] + 1, '\x7f');  // the byte past the device's text must stay untouched
        if (rows[i].n_rows > 0)
            simt::launch(ppm_grid(rows[i]), emu::kPpmThreads, 0, kConcurrent, [&] { emu::ppm_write(rows[i], lp[i], text.data()); });
        if (text.back() != '\x7f') return -2;
        for (int v = 0; v < n_views; v++)
            for (int b = i; b < total_bands; b += n_dev) {
                const size_t vb = (size_t)v * total_bands + b;
                memcpy(out + L.band_at[vb], text.data() + L.band_local[vb], L.band_bytes[vb]);
            }
    }
    for (int v = 0; v < n_views; v++) view_at[v] = L.view_at[v];
    return (long long)L.total;
}
