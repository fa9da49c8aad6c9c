// emu_shard_samples.cpp — TEST INFRASTRUCTURE ONLY (built and loaded by tests/test_shard_samples_on_host.py, never by the
// product): one shard of an anti-aliased frame shared by several processes (rtc_render_shard_samples,
// rtc_render_shard_samples_ppm_rows + rtc_write_shard_ppm) on the HOST.  The samples kernels (emu_samples.cpp, included
// whole, and through it emu_kernels.cpp) run with DevFrame.shard / n_shards of the shard over the shard's bands as the host
// plans them (rtc_shard_bands' count, cut into slices); the PPM text kernels (dev_ppm.cuh) then run over the shard's rows of
// that plane, phase by phase: each shard measures its rows, the caller exchanges the lengths, and each shard lays out the
// whole text on its own (rtc_internal.h: ppm_layout_frame_rows) and copies only its bands.
#include "emu_samples.cpp"

#include "dev_ppm.cuh"

namespace {
// blocks of a PPM launch: rtc_ppm.cu's grid for one SM (16 blocks), so that a warp steps through several rows
simt::Dim ppm_grid(const rtc::PpmRows& R) {
    const int warps = rtc::emu::kPpmThreads / 32;
    return simt::Dim{(unsigned)std::min(16, (R.n_rows + warps - 1) / warps), 1, 1};
}
}  // namespace

// rtc_render_shard_samples' render of shard `shard` of n_shards: the shard's bands (as many as rtc_shard_bands counts) in
// n_slices launches of consecutive bands, as render_views_body slices a view.  *variant receives the last launch's kernel.
extern "C" int emu_render_shard_samples(RtcScene* s, int depth, int n, int shard, int n_shards, int n_slices, int converge,
                                        int stream, float* rgb, unsigned char* u8, DevCounters* counters, int* variant) {
    const int nb = rtc_shard_bands(s->height, shard, n_shards, nullptr);
    if (nb < 0) return nb;
    for (int k = 0; k < n_slices; k++) {
        const int b0 = (int)((int64_t)nb * k / n_slices), b1 = (int)((int64_t)nb * (k + 1) / n_slices);
        if (b1 <= b0) continue;
        if (int rc = emu_render_samples(s, depth, shard, n_shards, b0, b1 - b0, n, converge, stream, rgb, u8, counters, variant))
            return rc;
    }
    return 0;
}

// Phase 1's text half: the byte length of the text of every row shard `shard` owns in the width x height plane u8, written
// into row_bytes (height entries, frame-row order) at the shard's rows only.
extern "C" void emu_shard_ppm_rows(const unsigned char* u8, int width, int height, int shard, int n_shards, uint64_t* row_bytes) {
    using namespace rtc;
    const PpmRows R{u8, width, shard, n_shards, ppm_device_rows((uint32_t)height, shard, n_shards)};
    if (R.n_rows == 0) return;
    std::vector<unsigned long long> own((size_t)R.n_rows);
    simt::launch(ppm_grid(R), emu::kPpmThreads, 0, kConcurrent, [&] { emu::ppm_row_bytes(R, own.data()); });
    for (int y = 0, k = 0; y < height; y++)
        if (y / kBandRows % n_shards == shard) row_bytes[y] = own[k++];
}

// Phase 2 (rtc_write_shard_ppm): the layout of the whole text from every row's length, then shard `shard`'s bands of u8
// written at their offsets in out (shard 0 also the header).  Returns the text's length, -1 when it does not fit capacity,
// -2 when ppm_write wrote past the shard's text.
extern "C" long long emu_write_shard_ppm(const unsigned char* u8, int width, int height, int shard, int n_shards,
                                         const uint64_t* row_bytes, char* out, long long capacity) {
    using namespace rtc;
    const std::string header = ppm_header((uint32_t)width, (uint32_t)height);
    std::vector<std::vector<unsigned long long>> shard_rows;
    PpmLayout L;
    ppm_layout_frame_rows((uint32_t)height, n_shards, header.size(), row_bytes, shard_rows, L, shard == 0 ? header.data() : nullptr,
                          shard == 0 ? out : nullptr);
    if ((long long)L.total > capacity) return -1;
    const PpmRows R{u8, width, shard, n_shards, (int)shard_rows[shard].size()};
    std::vector<char> text(L.device_bytes[shard] + 1, '\x7f');  // the byte past the shard's text must stay untouched
    if (R.n_rows > 0)
        simt::launch(ppm_grid(R), emu::kPpmThreads, 0, kConcurrent, [&] { emu::ppm_write(R, shard_rows[shard].data(), text.data()); });
    if (text.back() != '\x7f') return -2;
    for (int b = shard; b < L.total_bands; b += n_shards) memcpy(out + L.band_at[b], text.data() + L.band_local[b], L.band_bytes[b]);
    return (long long)L.total;
}
