// dev_shade.cuh — World::color_at with the bounded reflect / refract stack, Camera::ray_for_pixel, Canvas::scale_color.
// Part of rtc_device.cuh (include that, not this): compiled once per kernel build inside namespace rtc::RTC_NS.
#pragma once

#include <type_traits>

namespace rtc {
namespace RTC_NS {

__device__ __forceinline__ float powi5(float x) {  // llvm.powi with a constant 5: x * (x^2)^2
    float x2 = x * x;
    return x * (x2 * x2);
}

// One pending shade_hit whose children are still being traced (world.rs:62-86).  The reference adds its three terms
// left to right, `(surface + reflected * R) + refracted * (1 - R)` (world.rs:80-85), so a frame holds ONE colour: the
// surface colour while the reflection subtree is traced, then the first partial sum while the refraction subtree is.
// Only the fields a frame's children need are written (a mirror's frame: acc, reflective, reflectance, path, flags —
// the refraction ray and the transparency are stored for frames that refract); `remaining` is not stored at all: the
// frame at stack index i was pushed by a ray with remaining = depth - i.
struct Frame {
    V3 acc;             // stage 1: surface; stage 2: surface + reflected * R (or surface + reflected)
    float reflective;
    float reflectance;  // Schlick R, or < 0 when the plain sum applies (world.rs:80-85)
    unsigned path;
    int flags;          // bit 0: waiting for the refraction subtree (stage 2); bit 1: a refraction ray is pending
    float transparency;
    V3 refr_o, refr_d;
};
// The frame of the lean build (SmallScene::lean: no transparent material), whose ray trees are reflection chains: every
// frame waits for its reflection subtree alone and combines with the plain sum.  The path (the jitter key of a child's
// shadow rays) is kept only where the light draws its samples.
template <bool PATH>
struct ReflectFrame {
    V3 acc;
    float reflective;
    unsigned path;
};
template <>
struct ReflectFrame<false> {
    V3 acc;
    float reflective;
};

// world.rs:80-85, first and second addition
__device__ __forceinline__ V3 add_reflected(V3 surface, V3 reflected, float reflectance) {
    return reflectance >= 0.0f ? surface + reflected * reflectance : surface + reflected;
}
__device__ __forceinline__ V3 add_refracted(V3 partial, V3 refracted, float reflectance) {
    return reflectance >= 0.0f ? partial + refracted * (1.0f - reflectance) : partial + refracted;
}
__device__ __forceinline__ V3 combine(V3 surface, V3 reflected, V3 refracted, float reflectance) {
    return add_refracted(add_reflected(surface, reflected, reflectance), refracted, reflectance);
}

// Where a lane's rays come from.  OnePixel: the caller's ray, one per thread (render_tiles, trace_rays).  PixelStream:
// a lane whose ray tree is finished stores its pixel and draws the next pixel of the launch from a global counter at
// the converged top of the loop — in scenes whose ray trees differ wildly from pixel to pixel (mirrors and glass among
// 100 k spheres: one pixel traces 2 rays, its neighbour 60) a warp otherwise runs until its deepest tree is done with
// the other lanes idle (ncu, c5: 8 of 32 lanes active per instruction).
struct OnePixel {
    static constexpr bool kStream = false;
    __device__ __forceinline__ bool exhausted() const { return true; }
    __device__ __forceinline__ bool refill(bool&, V3&, V3&, unsigned&) { return false; }
    __device__ __forceinline__ void finish(unsigned, V3) {}
};

__device__ __forceinline__ unsigned char scale_color(float c);
__device__ __forceinline__ void ray_for_pixel(const DevScene& S, int x, int y, V3& o, V3& d);
__device__ __forceinline__ void ray_for_pixel(const DevView& V, int x, int y, V3& o, V3& d);

// Pixels of a launch in stream order: 32 consecutive indices are one 8x4 block (so a warp that refills all its lanes at
// once gets coherent primary rays), blocks run along a band (kBandRows rows: two block rows), bands in the order of
// the shard's band list.
struct PixelStream {
    static constexpr bool kStream = true;
    const DevScene& S;
    const DevFrame& F;
    unsigned* counter;  // next unclaimed stream index of this launch
    unsigned total;     // stream indices of this launch
    int blocks_x;       // 8-pixel blocks across the frame
    bool done = false;  // warp-uniform: the counter has run past the end
    __device__ __forceinline__ bool exhausted() const { return done; }
    // Warp-collective, called converged.  Idle lanes draw new pixels when at least kRefillLanes of them are idle (one
    // atomic per refill); returns true for a lane that starts a new pixel.
    __device__ __forceinline__ bool refill(bool& running, V3& ro, V3& rd, unsigned& pixel) {
        const unsigned idle = __ballot_sync(0xffffffffu, !running);
        if (done || (__popc(idle) < kRefillLanes && idle != 0xffffffffu)) return false;
        const int lane = threadIdx.x & 31, leader = __ffs(idle) - 1;
        unsigned base = 0;
        if (lane == leader) base = atomicAdd(counter, (unsigned)__popc(idle));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (base + (unsigned)__popc(idle) >= total) done = true;
        if (running) return false;
        const unsigned idx = base + (unsigned)__popc(idle & ((1u << lane) - 1u));
        if (idx >= total) return false;
        const unsigned block = idx >> 5, within = idx & 31u;
        const unsigned per_band = (unsigned)blocks_x * 2u;
        const unsigned band_i = block / per_band, b = block - band_i * per_band;
        const int band = F.shard + (F.band_begin + (int)band_i) * F.n_shards;
        const int x = (int)(b >> 1) * 8 + (int)(within & 7u), y = band * kBandRows + (int)(b & 1u) * 4 + (int)(within >> 3);
        if (x >= S.width || y >= S.height) return false;
        pixel = (unsigned)(y * S.width + x);
        if (x >= S.width - 1 || y >= S.height - 1) {  // camera.rs:80-81: never rendered, stays black (canvas.rs:23)
            finish(pixel, mk(0.f, 0.f, 0.f));
            return false;
        }
        ray_for_pixel(S, x, y, ro, rd);
        running = true;
        return true;
    }
    __device__ __forceinline__ void finish(unsigned pixel, V3 c) {  // Canvas::write_pixel + scale_color (canvas.rs:26-43)
        const size_t i = (size_t)pixel * 3;
        if (F.rgb) F.rgb[i] = c.x, F.rgb[i + 1] = c.y, F.rgb[i + 2] = c.z;
        if (F.u8) F.u8[i] = scale_color(c.x), F.u8[i + 1] = scale_color(c.y), F.u8[i + 2] = scale_color(c.z);
    }
};

// The pixel stream of a batch of views (rtc_render_views): the view is the outermost term of the stream index, so the
// pixels a warp draws in one refill lie in one view but at a view's end; view v's frame follows view v - 1's.  The
// arithmetic of PixelStream with the view split off first (a separate type: PixelStream's code stays as it is).
struct ViewPixelStream {
    static constexpr bool kStream = true;
    const DevScene& S;
    const DevFrame& F;
    unsigned* counter;      // next unclaimed stream index of this launch
    unsigned total;         // stream indices of this launch
    int blocks_x;           // 8-pixel blocks across the frame
    const DevView* views;   // the launch's cameras
    unsigned view_blocks;   // 8x4 blocks of one view in this launch
    bool done = false;      // warp-uniform: the counter has run past the end
    size_t out = 0;         // where this lane's view starts in the frame planes (elements)
    __device__ __forceinline__ bool exhausted() const { return done; }
    __device__ __forceinline__ bool refill(bool& running, V3& ro, V3& rd, unsigned& pixel) {
        const unsigned idle = __ballot_sync(0xffffffffu, !running);
        if (done || (__popc(idle) < kRefillLanes && idle != 0xffffffffu)) return false;
        const int lane = threadIdx.x & 31, leader = __ffs(idle) - 1;
        unsigned base = 0;
        if (lane == leader) base = atomicAdd(counter, (unsigned)__popc(idle));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (base + (unsigned)__popc(idle) >= total) done = true;
        if (running) return false;
        const unsigned idx = base + (unsigned)__popc(idle & ((1u << lane) - 1u));
        if (idx >= total) return false;
        const unsigned within = idx & 31u, view = (idx >> 5) / view_blocks, block = (idx >> 5) - view * view_blocks;
        const unsigned per_band = (unsigned)blocks_x * 2u;
        const unsigned band_i = block / per_band, b = block - band_i * per_band;
        const int band = F.shard + (F.band_begin + (int)band_i) * F.n_shards;
        const int x = (int)(b >> 1) * 8 + (int)(within & 7u), y = band * kBandRows + (int)(b & 1u) * 4 + (int)(within >> 3);
        if (x >= S.width || y >= S.height) return false;
        pixel = (unsigned)(y * S.width + x);  // within its view: the jitter generator's key, as in a single-view render
        out = (size_t)view * ((size_t)S.width * S.height * 3);
        if (x >= S.width - 1 || y >= S.height - 1) {  // camera.rs:80-81: never rendered, stays black (canvas.rs:23)
            finish(pixel, mk(0.f, 0.f, 0.f));
            return false;
        }
        ray_for_pixel(views[view], x, y, ro, rd);
        running = true;
        return true;
    }
    __device__ __forceinline__ void finish(unsigned pixel, V3 c) {  // Canvas::write_pixel + scale_color (canvas.rs:26-43)
        const size_t i = out + (size_t)pixel * 3;
        if (F.rgb) F.rgb[i] = c.x, F.rgb[i + 1] = c.y, F.rgb[i + 2] = c.z;
        if (F.u8) F.u8[i] = scale_color(c.x), F.u8[i + 1] = scale_color(c.y), F.u8[i + 2] = scale_color(c.z);
    }
};

// World::color_at (world.rs:88-101) with the recursion of reflected_color / refracted_color replaced by an
// explicit stack of at most depth+1 frames, evaluated in the reference's order (surface, then the whole
// reflection subtree, then the whole refraction subtree) and combined bottom-up with the same arithmetic.
// out_t / out_pos (optional) receive the primary hit.
//
// The loop runs one ray per iteration.  With CONVERGE (the host picks that build for scenes with reflective AND
// transparent materials, whose ray trees branch) EVERY lane of the warp calls this (active = false: no ray) and all
// lanes meet at a warp vote at the top: lanes whose tree is finished wait there, the others start their next ray —
// whichever branch produced it (first child, refraction sibling after a finished reflection subtree) — TOGETHER.
// Without the vote the compiler's reconvergence points leave lanes that took different exits of the body running
// their iterations one after the other (c5: 5 of 32 lanes active in the traversal code; 126 -> 64 ms with it).  Scenes
// whose trees are chains run ~5 % faster without it.
//
// LEAN (small scenes the commit marked SmallScene::lean: no pattern, no transparency, only spheres, planes and
// axis-aligned cubes, an area light on the cell-mask loops): patterns, the n1 / n2 walk, Schlick and refraction are
// not compiled, and the stack holds ReflectFrames.  Same arithmetic in the same order: a frame without a refraction
// child combines with reflectance -1, the plain sum.
template <bool STATS, bool SMALL, bool CONVERGE, bool DRAWN = false, bool LEAN = false, class Source = OnePixel>
__device__ __forceinline__ V3 color_at(const Env& E, bool active, V3 ro, V3 rd, int depth, unsigned pixel, Rays& r, Ctr<STATS>& k,
                                       float* out_t, int* out_pos, Source src = Source()) {
    static_assert(!Source::kStream || CONVERGE, "a pixel stream refills at the converged top of the loop");
    static_assert(!LEAN || (SMALL && !CONVERGE), "the lean build is the chain-order small-scene build");
    const DevScene& S = E.S;
    std::conditional_t<LEAN, ReflectFrame<DRAWN>, Frame> stack[kMaxFrames];
    int sp = 0;
    int remaining = depth;
    unsigned path = 1u;
    bool primary = true, running = active;
    V3 result = mk(0.f, 0.f, 0.f);
    for (;;) {
        if (CONVERGE) {
            if (Source::kStream && src.refill(running, ro, rd, pixel)) sp = 0, remaining = depth, path = 1u;
            if (!__any_sync(0xffffffffu, running)) {
                if (src.exhausted()) break;
                continue;
            }
            if (!running) continue;
        }
        Hit best{kInfF, -1, 0x7fffffff};
        find_hit<STATS, SMALL, LEAN>(E, ro, rd, best, k);
        if (primary) {
            if (out_t) *out_t = best.pos >= 0 ? best.t : -1.0f;
            if (out_pos) *out_pos = best.pos;
            primary = false;
        }
        V3 c = mk(0.f, 0.f, 0.f);
        if (best.pos >= 0) {
            // ---- precompute_values (world.rs:212-283)
            r.shades++;
            const int4 h = __ldg(&S.head[best.pos]);
            const DevMaterial& mat = S.materials[h.x >> 8];
            V3 n, over_point, material_color;
            {
                // everything that needs the hit primitive's transform happens here, BEFORE the light loop, so the
                // twelve registers of `m` (and the hit point) are dead while intensity_at runs; the pattern colour
                // (pattern.rs:15-19, evaluated at over_point, Q4) does not depend on the light
                const Xf m = load_xf(S.xform + 3 * (size_t)h.y);
                const V3 point = ro + rd * best.t;
                const V3 object_point = xf_point(m, point);
                n = norm(xf_normal(m, local_normal(S, h.x & 15, h.z, object_point)));  // shape.rs:148-154,130-145
                if (dot(n, -rd) < 0.0f) n = -n;
                over_point = point + n * kAcne;
                if constexpr (!LEAN) {
                    material_color = ld3(mat.color);
                    if (mat.pattern >= 0) {
                        k.pattern();
                        material_color = pattern_color(S, mat.pattern, xf_point(m, over_point));
                    }
                }
            }
            // ---- shade_hit (world.rs:62-86): light intensity first, then Phong (phong_lighting.rs:12-63)
            const float li = intensity_at<STATS, SMALL, DRAWN, LEAN>(E, over_point, pixel, path, r, k);
            // without patterns the colour is loaded after the light loop instead of held in registers across it
            if constexpr (LEAN) material_color = ld3(mat.color);
            const V3 eye = -rd;
            V3 light_rgb = ld3(S.light_rgb);
            V3 effective = material_color * light_rgb;
            V3 ambient = effective * mat.ambient;
            V3 surface = ambient;
            if (li != 0.f) {
                V3 to_light = norm(ld3(S.light_pos) - over_point);
                float lnc = dot(to_light, n);
                V3 diffuse = mk(0.f, 0.f, 0.f), specular = mk(0.f, 0.f, 0.f);
                if (!(lnc < 0.0f)) {
                    diffuse = effective * mat.diffuse * lnc;
                    V3 sr = reflect(-to_light, n);
                    float rec = dot(sr, eye);
                    if (!(rec <= 0.0f)) {
                        // `intensity * specular * factor` (phong_lighting.rs:56-57): with specular == 0 the product
                        // is 0 for every finite factor, so powf is only evaluated when it can matter
                        float factor = (mat.specular == 0.0f && mat.shininess <= 1.0e4f) ? 1.0f : powf(rec, mat.shininess);
                        specular = light_rgb * mat.specular * factor;
                    }
                }
                surface = ambient + (diffuse + specular) * li;
            }
            // ---- children (world.rs:121-162) with the reference's asymmetric guards (Q11)
            bool want_refl = mat.reflective != 0.0f && remaining >= 1;
            bool want_refr = false;
            float reflectance = -1.0f;
            V3 refr_d = mk(0.f, 0.f, 0.f);
            if (!LEAN && mat.transparency != 0.0f) {
                float n1, n2;
                find_containers<STATS>(S, ro, rd, best.pos, n1, n2, k);
                float cos_i = dot(eye, n);
                if (remaining != 0) {
                    float n_ratio = n1 / n2;  // world.rs:196-207
                    float sin2 = (n_ratio * n_ratio) * (1.0f - cos_i * cos_i);
                    if (!(sin2 > 1.0f)) {
                        k.refr_dir();
                        float cos_t = sqrtf(1.0f - sin2);
                        refr_d = n * (n_ratio * cos_i - cos_t) - (eye * n_ratio);
                        want_refr = true;
                    }
                }
                if (mat.reflective > 0.0f && mat.transparency > 0.0f) {  // schlick_reflectance, world.rs:285-303
                    k.schlick();
                    float cosine = cos_i;
                    bool tir = false;
                    if (n1 > n2) {
                        float nn = n1 / n2;
                        float sin2_t = (nn * nn) * (1.0f - cosine * cosine);
                        if (sin2_t > 1.0f)
                            tir = true;
                        else
                            cosine = sqrtf(1.0f - sin2_t);
                    }
                    if (tir) {
                        reflectance = 1.0f;
                    } else {
                        float q = (n1 - n2) / (n1 + n2);
                        float r0 = q * q;
                        reflectance = r0 + (1.0f - r0) * powi5(1.0f - cosine);
                    }
                }
            }
            if ((want_refl || want_refr) && sp < kMaxFrames) {
                auto& f = stack[sp++];
                if constexpr (!LEAN) f.reflectance = reflectance;
                if constexpr (!LEAN || DRAWN) f.path = path;
                r.secondary++;
                remaining = remaining - 1;
                V3 under_point = over_point;
                if constexpr (!LEAN) {
                    if (want_refr) {
                        under_point = (ro + rd * best.t) - n * kAcne;  // `point` again: the same expression, the same bits
                        f.transparency = mat.transparency;
                        f.refr_o = under_point;
                        f.refr_d = refr_d;
                    }
                }
                if (LEAN || want_refl) {
                    f.acc = surface;
                    f.reflective = mat.reflective;
                    if constexpr (!LEAN) f.flags = want_refr ? 2 : 0;
                    // reflect(rd, n) (world.rs:225) is bit-for-bit the same for n and -n — every product and every sum
                    // changes sign twice — so it is evaluated here from the flipped normal instead of being kept live
                    // across the light loop
                    ro = over_point;
                    rd = reflect(rd, n);
                    path = path * 3u + 1u;
                } else if constexpr (!LEAN) {  // no reflection: reflected_color is black (world.rs:126-128)
                    f.acc = add_reflected(surface, mk(0.f, 0.f, 0.f), reflectance);
                    f.flags = 1;
                    ro = under_point;
                    rd = refr_d;
                    path = path * 3u + 2u;
                }
                continue;  // to the vote: trace the child
            }
            c = combine(surface, mk(0.f, 0.f, 0.f), mk(0.f, 0.f, 0.f), reflectance);
        }
        // ---- hand the colour to the waiting frames
        for (;;) {
            if (sp == 0) {
                if (!CONVERGE) return c;
                if (Source::kStream) src.finish(pixel, c);
                result = c;
                running = false;
                break;
            }
            auto& f = stack[sp - 1];
            if constexpr (LEAN) {
                // world.rs:131, 80-85.  The general build rounds `reflected` before the sum (a select on the frame's
                // reflectance sits between them), so the FMA build must not fuse the two here either
                const V3 reflected = mk(mul_rn(c.x, f.reflective), mul_rn(c.y, f.reflective), mul_rn(c.z, f.reflective));
                c = combine(f.acc, reflected, mk(0.f, 0.f, 0.f), -1.0f);
                sp--;
                continue;
            } else {
                const int flags = f.flags;
                const float reflectance = f.reflectance;
                if (!(flags & 1)) {                        // the reflection subtree is done
                    const V3 reflected = c * f.reflective;  // world.rs:131
                    if (flags & 2) {                        // its refraction sibling is next
                        f.acc = add_reflected(f.acc, reflected, reflectance);
                        f.flags = 1;
                        ro = f.refr_o;
                        rd = f.refr_d;
                        remaining = depth - sp;  // the frame's ray had depth - (sp - 1)
                        path = f.path * 3u + 2u;
                        r.secondary++;
                        break;
                    }
                    c = combine(f.acc, reflected, mk(0.f, 0.f, 0.f), reflectance);
                } else {
                    c = add_refracted(f.acc, c * f.transparency, reflectance);  // world.rs:159-160
                }
                sp--;
            }
        }
    }
    return result;
}

// is_shadowed calls of a thread's shades (see Rays)
__device__ __forceinline__ void finish_rays(const DevScene& S, Rays& r) { r.shadow = r.shades * (unsigned)(S.light_is_rect ? S.cells : 1); }

// Camera::ray_for_pixel (camera.rs:60-74), for the committed camera (DevScene) or one view of a batch (DevView): the
// same arithmetic in the same order
template <class Camera>
__device__ __forceinline__ void camera_ray(const Camera& S, int x, int y, V3& o, V3& d) {
    float x_offset = ((float)x + 0.5f) * S.pixel_size;
    float y_offset = ((float)y + 0.5f) * S.pixel_size;
    float world_x = S.half_w - x_offset;
    float world_y = S.half_h - y_offset;
    Xf m{S.cam_inv[0], S.cam_inv[1], S.cam_inv[2]};
    V3 pixel = xf_point(m, mk(world_x, world_y, -1.0f));
    o = xf_point(m, mk(0.f, 0.f, 0.f));
    d = norm(pixel - o);
}
__device__ __forceinline__ void ray_for_pixel(const DevScene& S, int x, int y, V3& o, V3& d) { camera_ray(S, x, y, o, d); }
__device__ __forceinline__ void ray_for_pixel(const DevView& V, int x, int y, V3& o, V3& d) { camera_ray(V, x, y, o, d); }

// Canvas::scale_color (canvas.rs:39-43): clamp, then truncate; NaN -> 255 because f32::min returns the
// non-NaN operand (fminf does the same) and `as u8` saturates.
__device__ __forceinline__ unsigned char scale_color(float c) {
    float s = fmaxf(fminf(c * 255.0f, 255.0f), 0.0f);
    return (unsigned char)__float2uint_rz(s);
}

}  // namespace RTC_NS
}  // namespace rtc
