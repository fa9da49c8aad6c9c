// emu_views_samples.cpp — TEST INFRASTRUCTURE ONLY (built and loaded by tests/test_views_samples_on_host.py, never by the
// product): the harness of rtc_render_samples' kernels (emu_samples.cpp, included whole, and through it emu_kernels.cpp)
// plus the kernels of rtc_render_views_samples (dev_kernels.cuh: render_tiles_views_samples, render_stream_views_samples),
// launched as launch_views_samples (rtc_kernels.cu) launches them, with the sample cameras rtc_render_views_samples derives
// for its views (rtc_internal.h: sample_camera).
#include "emu_samples.cpp"

namespace {
// the kernel kinds of a batch samples variant id, after emu_samples.cpp's: kind * 32 + variant_code
constexpr int kViewsSamples = kWave + 3, kStreamViewsSamples = kWave + 4;

// The view rtc_render_views takes for the camera of the scene `cam` (its Camera::new fields)
RtcView view_of(const RtcScene* cam) {
    RtcView v;
    v.half_width = cam->half_w, v.half_height = cam->half_h, v.pixel_size = cam->pixel_size;
    memcpy(v.transform_inverse, cam->cam_inv, sizeof(v.transform_inverse));
    return v;
}
}  // namespace

// Every variant launch_views_samples can select in this build: out[i] = kind * 32 + variant_code; returns the count
extern "C" int emu_views_sample_variants(int* out) {
    int n = 0;
#define RTC_EMU_VIEWS_SAMPLES(ST, SM, CV, DR, LE) \
    if (!ST) out[n++] = kViewsSamples * 32 + rtc::variant_code(ST, SM, CV, DR, LE);
    RTC_TILE_VARIANTS(RTC_EMU_VIEWS_SAMPLES)
#undef RTC_EMU_VIEWS_SAMPLES
    out[n++] = kStreamViewsSamples * 32 + rtc::variant_code(false, false, true, false, false);
    return n;
}

// The sample camera rtc_render_views_samples derives for the view of `cam` on a width-pixel canvas with n samples per axis
// (rtc_internal.h: sample_camera's RtcView overload): pixel_size, half_width, half_height
extern "C" void emu_view_sample_camera(RtcScene* cam, unsigned width, unsigned n, float* out) {
    const RtcView c = rtc::sample_camera(view_of(cam), width, n);
    out[0] = c.pixel_size, out[1] = c.half_width, out[2] = c.half_height;
}

// launch_views_samples with n samples per axis for n_views views whose cameras are those of the scenes cams[v], over the
// bands [band_begin, band_begin + n_bands) of a shard: view v's frame at rgb / u8 + v * width * height * 3.  A launch of the
// views [v0, v1) of a batch is this call with cams + v0 and the planes at view v0, as the host's plan cuts it.
extern "C" int emu_render_views_samples(RtcScene* s, int depth, int shard, int n_shards, int band_begin, int n_bands,
                                        RtcScene* const* cams, int n_views, int n, int converge, int stream, float* rgb,
                                        unsigned char* u8, DevCounters* counters, int* variant) {
    using namespace rtc;
    Scene sc;
    if (int rc = load(s, sc)) return rc;
    std::vector<DevView> table((size_t)(n_views > 0 ? n_views : 0));
    for (int i = 0; i < n_views; i++) {  // the view table rtc_render_views_samples uploads: the views' sample cameras
        const RtcView c = sample_camera(view_of(cams[i]), s->width, (uint32_t)n);
        DevView& d = table[(size_t)i];
        rows3(c.transform_inverse, d.cam_inv);
        d.half_w = c.half_width, d.half_h = c.half_height, d.pixel_size = c.pixel_size, d.pad = 0.f;
    }
    const DevView* views = table.data();
    const DevScene& S = sc.S;
    const SmallScene& SS = sc.SS;
    unsigned stream_counter = 0;
    const bool streams = stream < 0 ? streams_pixels(s, SS) : (SS.n == 0 && stream != 0);
    DevFrame F{rgb, u8, shard, n_shards, depth, n_bands, band_begin, nullptr, nullptr,
               converge < 0 ? frame_converge(s) : converge, streams ? &stream_counter : nullptr, stream_blocks(kEmuSms)};
    memset(counters, 0, sizeof(DevCounters));
    const unsigned tiles_x = (unsigned)(S.width + kTileW - 1) / kTileW;
    if (tiles_x == 0 || n_bands <= 0 || n_views <= 0) return 0;
    const KernelVariant v = frame_variant(S, SS, F, false, emu::kHasLean);
    if (v.stream) {
        *variant = kStreamViewsSamples * 32 + variant_code(v);
        simt::launch(dim(F.stream_blocks), kThreads, 0, kConcurrent,
                     [&] { emu::render_stream_views_samples(S, SS, F, counters, views, n_views, n); });
        return 0;
    }
    *variant = kViewsSamples * 32 + variant_code(v);
    const simt::Dim grid = dim(tiles_x, (unsigned)n_bands, (unsigned)n_views);
    switch (variant_code(v)) {
#define RTC_EMU_VIEWS_SAMPLES(ST, SM, CV, DR, LE) RTC_EMU_VIEWS_SAMPLES_##ST(SM, CV, DR, LE)
#define RTC_EMU_VIEWS_SAMPLES_true(SM, CV, DR, LE)
#define RTC_EMU_VIEWS_SAMPLES_false(SM, CV, DR, LE)                                                                     \
    case variant_code(false, SM, CV, DR, LE):                                                                           \
        simt::launch(grid, kThreads, (size_t)dynamic_smem(v), 1,                                                         \
                     [&] { emu::render_tiles_views_samples<SM, CV, DR, LE>(S, SS, F, counters, views, n); });            \
        return 0;
        RTC_TILE_VARIANTS(RTC_EMU_VIEWS_SAMPLES)
#undef RTC_EMU_VIEWS_SAMPLES
#undef RTC_EMU_VIEWS_SAMPLES_true
#undef RTC_EMU_VIEWS_SAMPLES_false
    }
    return fail(RTC_ERR_INVALID, "no kernel for the variant");
}
