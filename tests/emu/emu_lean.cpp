// emu_lean.cpp — TEST INFRASTRUCTURE ONLY (built and loaded by tests/test_lean_build.py, never by the product): the
// host harness of emu_color.cpp with one more entry point, World::color_at through the lean kernel build
// (dev_shade.cuh: color_at<.., LEAN = true>, the build render_tiles runs for scenes the commit marks SmallScene::lean).
#include "emu_color.cpp"

// World::color_at for n rays through the lean build; RTC_ERR_INVALID when the commit does not mark the scene lean.
extern "C" int emu_lean_color_at(RtcScene* s, uint32_t n, const float* origins, const float* directions, int depth, float* out_rgb) {
    using namespace rtc;
    Flattened f;
    if (int rc = flatten(s, f)) return rc;
    if (!f.small.lean) return RTC_ERR_INVALID;
    DevScene S;
    host_scene(s, f, S);
    const SmallScene SS = f.small;
    const bool drawn = S.jitter_len == 0;  // the predicate of launch_render
    const emu::Env E{S, SS};
    memset(g_rays, 0, sizeof(g_rays));
    for (uint32_t i = 0; i < n; i++) {
        emu::stage_small_scene(S, SS);
        emu::V3 o = emu::ld3(origins + 3 * (size_t)i), d = emu::ld3(directions + 3 * (size_t)i);
        emu::Ctr<false> k;
        emu::Rays r;
        const emu::V3 c = drawn ? emu::color_at<false, true, false, true, true>(E, true, o, d, depth, i, r, k, nullptr, nullptr)
                                : emu::color_at<false, true, false, false, true>(E, true, o, d, depth, i, r, k, nullptr, nullptr);
        emu::finish_rays(S, r);
        g_rays[0] += r.primary, g_rays[1] += r.secondary, g_rays[2] += r.shadow, g_rays[3] += r.shades;
        out_rgb[3 * (size_t)i] = c.x, out_rgb[3 * (size_t)i + 1] = c.y, out_rgb[3 * (size_t)i + 2] = c.z;
    }
    return 0;
}
