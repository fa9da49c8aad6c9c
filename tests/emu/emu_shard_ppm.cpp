// emu_shard_ppm.cpp — TEST INFRASTRUCTURE ONLY (built and loaded by tests/test_shard_ppm_on_host.py, never by the product):
// the PPM text kernels (dev_ppm.cuh: ppm_row_bytes, ppm_write) run on the HOST in blocks of 128 threads and warps of 32 lanes
// (simt.h) over an 8-bit plane the caller gives, as n_shards processes run them through rtc_render_shard_ppm_rows and
// rtc_write_shard_ppm: each shard measures its own rows, and each then lays out the whole text on its own from every row's
// length (rtc_internal.h: ppm_layout_frame_rows) and copies only its bands.
#include <vector>

#include "rtc_internal.h"  // PpmRows, ppm_header, ppm_device_rows, ppm_layout_frame_rows
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

// Canvas::to_ppm of the width x height plane u8 into out (capacity bytes, >= rtc_ppm_bound) as n_shards processes write it:
// every shard runs ppm_row_bytes over its rows and puts their lengths into one height-entry array in frame-row order; then
// every shard lays out the whole text on its own from that array (ppm_layout_frame_rows, with the header text for shard 0
// only), runs ppm_write and copies only its bands into out.  only >= 0: only that shard writes into out (all of them
// compute lengths).  Returns the text's length, -1 when it does not fit, -2 when ppm_write wrote past a shard's text, -3
// when two shards disagree on the length.
extern "C" long long emu_ppm_shards(const unsigned char* u8, int width, int height, int n_shards, int only, char* out,
                                    long long capacity) {
    using namespace rtc;
    std::vector<uint64_t> row_bytes((size_t)height, ~0ull);
    for (int i = 0; i < n_shards; i++) {
        const PpmRows R{u8, width, i, n_shards, ppm_device_rows((uint32_t)height, i, n_shards)};
        std::vector<unsigned long long> own((size_t)R.n_rows + 1, ~0ull);
        if (R.n_rows > 0) simt::launch(ppm_grid(R), emu::kPpmThreads, 0, kConcurrent, [&] { emu::ppm_row_bytes(R, own.data()); });
        for (int y = 0, k = 0; y < height; y++)
            if (y / kBandRows % n_shards == i) row_bytes[y] = own[k++];
    }
    const std::string header = ppm_header((uint32_t)width, (uint32_t)height);
    long long total = -1;
    for (int i = 0; i < n_shards; i++) {
        std::vector<std::vector<unsigned long long>> shard_rows;
        PpmLayout L;
        const bool writes = only < 0 || only == i;
        ppm_layout_frame_rows((uint32_t)height, n_shards, header.size(), row_bytes.data(), shard_rows, L,
                              writes && i == 0 ? header.data() : nullptr, writes && i == 0 ? out : nullptr);
        if ((long long)L.total > capacity) return -1;
        if (total >= 0 && (long long)L.total != total) return -3;
        total = (long long)L.total;
        if (!writes) continue;
        const PpmRows R{u8, width, i, n_shards, (int)shard_rows[i].size()};
        std::vector<char> text(L.device_bytes[i] + 1, '\x7f');  // the byte past the shard's text must stay untouched
        if (R.n_rows > 0)
            simt::launch(ppm_grid(R), emu::kPpmThreads, 0, kConcurrent, [&] { emu::ppm_write(R, shard_rows[i].data(), text.data()); });
        if (text.back() != '\x7f') return -2;
        for (int b = i; b < L.total_bands; b += n_shards) memcpy(out + L.band_at[b], text.data() + L.band_local[b], L.band_bytes[b]);
    }
    return total;
}
