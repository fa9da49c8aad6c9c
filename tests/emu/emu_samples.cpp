// emu_samples.cpp — TEST INFRASTRUCTURE ONLY (built and loaded by tests/test_samples_on_host.py, never by the product):
// the harness of the kernels (emu_kernels.cpp, included whole: its launches, scene loading and 32-lane warps) plus the
// kernels of rtc_render_samples (dev_kernels.cuh: render_tiles_samples, render_stream_samples), launched as
// launch_samples (rtc_kernels.cu) launches them, with the sample camera rtc_render_samples derives (rtc_internal.h:
// sample_camera).
#include "emu_kernels.cpp"

namespace {
// the kernel kinds of a samples variant id, after emu_kernels.cpp's Kind: kind * 32 + variant_code
constexpr int kSamples = kWave + 1, kStreamSamples = kWave + 2;
}  // namespace

// Every variant launch_samples can select in this build: out[i] = kind * 32 + variant_code; returns the count
extern "C" int emu_sample_variants(int* out) {
    int n = 0;
#define RTC_EMU_SAMPLES(ST, SM, CV, DR, LE) \
    if (!ST) out[n++] = kSamples * 32 + rtc::variant_code(ST, SM, CV, DR, LE);
    RTC_TILE_VARIANTS(RTC_EMU_SAMPLES)
#undef RTC_EMU_SAMPLES
    out[n++] = kStreamSamples * 32 + rtc::variant_code(false, false, true, false, false);
    return n;
}

// rtc_render_samples' sample camera for n samples per axis (rtc_internal.h: sample_camera): pixel_size, half_width,
// half_height
extern "C" void emu_sample_camera(RtcScene* s, unsigned n, float* out) {
    const RtcView c = rtc::sample_camera(s, n);
    out[0] = c.pixel_size, out[1] = c.half_width, out[2] = c.half_height;
}

// launch_samples with n samples per axis over the bands [band_begin, band_begin + n_bands) of a shard, the sample camera
// rtc_render_samples derives from the scene's
extern "C" int emu_render_samples(RtcScene* s, int depth, int shard, int n_shards, int band_begin, int n_bands, int n, int converge,
                                  int stream, float* rgb, unsigned char* u8, DevCounters* counters, int* variant) {
    using namespace rtc;
    Scene sc;
    if (int rc = load(s, sc)) return rc;
    const RtcView c = sample_camera(s, (uint32_t)n);
    DevView C;
    rows3(c.transform_inverse, C.cam_inv);
    C.half_w = c.half_width, C.half_h = c.half_height, C.pixel_size = c.pixel_size, C.pad = 0.f;
    const DevScene& S = sc.S;
    const SmallScene& SS = sc.SS;
    unsigned stream_counter = 0;
    const bool streams = stream < 0 ? streams_pixels(s, SS) : (SS.n == 0 && stream != 0);
    DevFrame F{rgb, u8, shard, n_shards, depth, n_bands, band_begin, nullptr, nullptr,
               converge < 0 ? frame_converge(s) : converge, streams ? &stream_counter : nullptr, stream_blocks(kEmuSms)};
    memset(counters, 0, sizeof(DevCounters));
    const unsigned tiles_x = (unsigned)(S.width + kTileW - 1) / kTileW;
    if (tiles_x == 0 || n_bands <= 0) return 0;
    const KernelVariant v = frame_variant(S, SS, F, false, emu::kHasLean);
    if (v.stream) {
        *variant = kStreamSamples * 32 + variant_code(v);
        simt::launch(dim(F.stream_blocks), kThreads, 0, kConcurrent, [&] { emu::render_stream_samples(S, SS, F, counters, C, n); });
        return 0;
    }
    *variant = kSamples * 32 + variant_code(v);
    switch (variant_code(v)) {
#define RTC_EMU_SAMPLES(ST, SM, CV, DR, LE) RTC_EMU_SAMPLES_##ST(SM, CV, DR, LE)
#define RTC_EMU_SAMPLES_true(SM, CV, DR, LE)
#define RTC_EMU_SAMPLES_false(SM, CV, DR, LE)                                                                            \
    case variant_code(false, SM, CV, DR, LE):                                                                            \
        simt::launch(dim(tiles_x, (unsigned)n_bands), kThreads, (size_t)dynamic_smem(v), 1,                               \
                     [&] { emu::render_tiles_samples<SM, CV, DR, LE>(S, SS, F, counters, C, n); });                      \
        return 0;
        RTC_TILE_VARIANTS(RTC_EMU_SAMPLES)
#undef RTC_EMU_SAMPLES
#undef RTC_EMU_SAMPLES_true
#undef RTC_EMU_SAMPLES_false
    }
    return fail(RTC_ERR_INVALID, "no kernel for the variant");
}
