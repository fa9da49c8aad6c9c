// emu_ppm.cpp — TEST INFRASTRUCTURE ONLY (built and loaded by tests/test_ppm_on_host.py, never by the product): the PPM
// text kernels of rtc_render_ppm (dev_ppm.cuh: ppm_row_bytes, ppm_write) run on the HOST in blocks of 128 threads and warps
// of 32 lanes (simt.h), over an 8-bit plane the caller gives, with rtc_render_ppm's host scan (rtc_internal.h: ppm_layout)
// between them.  A frame split over n_dev devices is encoded device by device, each from its own bands, and every band's
// text is then copied to its offset as rtc_render_ppm copies it.
#include <vector>

#include "rtc_internal.h"  // PpmRows, ppm_header, ppm_device_rows, ppm_layout
#include "simt.h"

#define RTC_NS emu
#include "dev_ppm.cuh"

namespace {
constexpr int kConcurrent = 8;  // blocks at once: the kernels use no shared memory
// blocks of a launch: rtc_ppm.cu's grid for one SM (16 blocks), so that a warp steps through several rows
simt::Dim ppm_grid(const rtc::PpmRows& R) {
    const int warps = rtc::emu::kPpmThreads / 32;
    return simt::Dim{(unsigned)std::min(16, (R.n_rows + warps - 1) / warps), 1, 1};
}
}  // namespace

// Canvas::to_ppm of the width x height 8-bit plane u8 into out (capacity bytes, >= rtc_ppm_bound); returns the text's
// length, or -1 when it does not fit.
extern "C" long long emu_ppm(const unsigned char* u8, int width, int height, int n_dev, char* out, long long capacity) {
    using namespace rtc;
    std::vector<PpmRows> rows(n_dev);
    std::vector<std::vector<unsigned long long>> lengths(n_dev);
    std::vector<unsigned long long*> lp(n_dev);
    for (int i = 0; i < n_dev; i++) {
        rows[i] = PpmRows{u8, width, i, n_dev, ppm_device_rows((uint32_t)height, i, n_dev)};
        lengths[i].assign((size_t)rows[i].n_rows + 1, ~0ull);
        lp[i] = lengths[i].data();
        if (rows[i].n_rows > 0)
            simt::launch(ppm_grid(rows[i]), emu::kPpmThreads, 0, kConcurrent, [&] { emu::ppm_row_bytes(rows[i], lp[i]); });
    }
    const std::string header = ppm_header((uint32_t)width, (uint32_t)height);
    PpmLayout L;
    ppm_layout((uint32_t)height, n_dev, header.size(), lp.data(), L);
    if ((long long)L.total > capacity) return -1;
    memcpy(out, header.data(), header.size());
    const int total_bands = (height + kBandRows - 1) / kBandRows;
    for (int i = 0; i < n_dev; i++) {
        std::vector<char> text(L.device_bytes[i] + 1, '\x7f');  // the byte past the device's text must stay untouched
        if (rows[i].n_rows > 0)
            simt::launch(ppm_grid(rows[i]), emu::kPpmThreads, 0, kConcurrent, [&] { emu::ppm_write(rows[i], lp[i], text.data()); });
        if (text.back() != '\x7f') return -2;
        for (int b = i; b < total_bands; b += n_dev) memcpy(out + L.band_at[b], text.data() + L.band_local[b], L.band_bytes[b]);
    }
    return (long long)L.total;
}

// The byte lengths of the rows of one device's bands (ppm_row_bytes alone), for the row scan's tests
extern "C" int emu_ppm_row_bytes(const unsigned char* u8, int width, int height, int device, int n_dev, unsigned long long* out) {
    const rtc::PpmRows R{u8, width, device, n_dev, rtc::ppm_device_rows((uint32_t)height, device, n_dev)};
    if (R.n_rows > 0) simt::launch(ppm_grid(R), rtc::emu::kPpmThreads, 0, kConcurrent, [&] { rtc::emu::ppm_row_bytes(R, out); });
    return R.n_rows;
}
