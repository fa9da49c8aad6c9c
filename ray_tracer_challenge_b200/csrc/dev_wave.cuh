// dev_wave.cuh — Camera::render for tree scenes as a WAVEFRONT: rays are work items, not lanes' private property.
// Part of rtc_device.cuh (include that, not this): compiled once per kernel build inside namespace rtc::RTC_NS.
//
// Why.  In a scene of 10^5 primitives with mirrors and glass the cost of a ray is its walk through the tree, and walks
// differ wildly in length (a ray that hits the sphere in front of it visits a dozen nodes, a shadow ray that reaches the
// light crosses the whole field).  With one pixel — or one ray tree — per lane a warp walks until its longest ray is
// done: ncu shows 8.7 of 32 lanes active in the box tests of render_stream although 89 % of the lanes hold a ray.  Here
// the tree walks are a kernel of their own (wave_trace) whose lanes draw the next ray from the level's queue the
// moment theirs ends, and everything between two walks is a kernel of fully converged, one-thread-per-ray shading:
//
//   level L = 0 .. depth (the rays with `remaining = depth - L`, world.rs:121-162), per chunk of the frame:
//     wave_trace<nearest>   World::intersect + Intersection::hit of every ray of the level          (world.rs:52-60)
//     wave_hit              the hit record's geometry; emits the shadow ray                          (world.rs:212-233, 104-111)
//     wave_trace<shadow>    World::is_shadowed of every shadow ray                                   (world.rs:112-119)
//     wave_shade            Phong, n1 / n2, Schlick; appends reflection / refraction rays to level L + 1 (world.rs:62-86, 121-162)
//   then level depth .. 0:
//     wave_combine          surface + reflected * R + refracted * (1 - R) into the parent's node, or the pixel (world.rs:80-85)
//
// The arithmetic of every ray is the arithmetic of color_at (dev_shade.cuh), statement for statement: frames are
// bit-identical to render_tiles / render_stream (tests/test_gpu_parity.py runs the tree scenes through both).  Only point
// lights take this path (one shadow ray per shade); the host falls back to render_stream for anything else, for the
// detailed (counting) pass, and when a chunk's ray pool overflows — never silently.
#pragma once

namespace rtc {
namespace RTC_NS {

// One ray of a ray tree and what tracing it found (96 B).
struct WaveRay {
    float ox, oy, oz, dx, dy, dz;  // the ray
    float t;                       // nearest hit distance, or < 0
    int pos;                       // ... and primitive position, or -1
    unsigned pixel, path;          // frame pixel (y * width + x) and jitter path id
    int parent;                    // pool index of the ray whose shade spawned this one, or -1 (primary)
    int slot;                      // 0: the parent's reflection, 1: its refraction
    float sx, sy, sz, sdx, sdy, sdz;  // the shadow ray of this ray's hit point (over_point -> light, normalised)
    float smax;                    // its length limit (the light's distance), or < 0: no shadow ray
    int shadowed;                  // wave_trace<shadow>'s verdict
    int pad0, pad1, pad2, pad3;
};
static_assert(sizeof(WaveRay) == 96, "WaveRay layout");

// What the combine pass needs of a shaded ray (64 B).
struct WaveNode {
    float sr, sg, sb;       // surface colour (black for a miss)
    float reflective, transparency, reflectance;
    float rr, rg, rb;       // the reflection child's colour, raw (written by that child's combine)
    float fr, fg, fb;       // the refraction child's colour, raw
    int flags;              // bit 0: hit; bit 1: has a reflection child; bit 2: has a refraction child
    int parent, slot;
    unsigned pixel;
};
static_assert(sizeof(WaveNode) == 64, "WaveNode layout");

struct WavePool {
    WaveRay* rays;
    WaveNode* nodes;
    int capacity;       // rays the pool holds
    int* base;          // [kMaxFrames + 1] first pool index of every level
    int* count;         // [kMaxFrames + 1] rays of every level
    int* cursor;        // [2 * (kMaxFrames + 1)] wave_trace's next unclaimed ray: nearest, shadow — per level
    unsigned long long* overflow;   // rays that did not fit: the chunk is rendered again by render_stream
    unsigned long long* secondary;  // this chunk's secondary rays and shades (the host adds the records of the chunks it keeps)
    unsigned long long* shades;
};

// the pool as the host hands it to the launchers (rtc_types.h), typed
__device__ __forceinline__ WavePool wave_pool(const WavePoolRaw& raw) {
    WavePool P;
    P.rays = static_cast<WaveRay*>(raw.rays), P.nodes = static_cast<WaveNode*>(raw.nodes), P.capacity = raw.capacity;
    P.base = raw.ints, P.count = raw.ints + kWaveLevels, P.cursor = raw.ints + 2 * kWaveLevels;
    P.overflow = raw.record, P.secondary = raw.record + 1, P.shades = raw.record + 2;
    return P;
}

// between the appends to a level and its first walk (one thread): the level keeps the rays that were written, and the
// next level starts where it ends.  wave_append counts every ray, also those that did not fit (the overflow record has
// them and the chunk is rendered again); left in the count they would send the level's kernels past the pool's end.
__device__ __forceinline__ void wave_next_level(const WavePool& P, int level) {
    const int n = min(P.count[level], P.capacity - P.base[level]);
    P.count[level] = n;
    P.base[level + 1] = P.base[level] + n;
}

// ---- chunk start: the primary rays of bands [band_begin, band_begin + n_bands) of the shard ------------------------
__device__ __forceinline__ int wave_append(const WavePool& P, int level, bool want) {
    // warp-aggregated: one atomic per warp, lanes in order
    const unsigned mask = __ballot_sync(0xffffffffu, want);
    if (mask == 0u) return -1;
    const int lane = threadIdx.x & 31, leader = __ffs(mask) - 1;
    int first = 0;
    if (lane == leader) first = atomicAdd(&P.count[level], __popc(mask));
    first = __shfl_sync(0xffffffffu, first, leader);
    if (!want) return -1;
    const int idx = P.base[level] + first + __popc(mask & ((1u << lane) - 1u));
    if (idx >= P.capacity) {
        atomicAdd(P.overflow, 1ull);
        return -1;
    }
    return idx;
}

__device__ __forceinline__ void wave_primary(const DevScene& S, const DevFrame& F, const WavePool& P) {
    const int blocks_x = (S.width + 7) / 8;
    const unsigned total = (unsigned)F.n_bands * (unsigned)blocks_x * 2u * 32u;  // stream order of PixelStream
    const unsigned stride = gridDim.x * blockDim.x;
    for (unsigned base = blockIdx.x * blockDim.x; base < total; base += stride) {  // warp-uniform trip count
        const unsigned idx = base + threadIdx.x;
        bool rendered = false;
        int x = 0, y = 0;
        if (idx < total) {
            const unsigned block = idx >> 5, within = idx & 31u;
            const unsigned per_band = (unsigned)blocks_x * 2u;
            const unsigned band_i = block / per_band, b = block - band_i * per_band;
            const int band = F.shard + (F.band_begin + (int)band_i) * F.n_shards;
            x = (int)(b >> 1) * 8 + (int)(within & 7u), y = band * kBandRows + (int)(b & 1u) * 4 + (int)(within >> 3);
            if (x < S.width && y < S.height) {
                rendered = x < S.width - 1 && y < S.height - 1;
                if (!rendered) {  // camera.rs:80-81: never rendered, stays black (canvas.rs:23)
                    const size_t i = ((size_t)y * S.width + x) * 3;
                    if (F.rgb) F.rgb[i] = 0.f, F.rgb[i + 1] = 0.f, F.rgb[i + 2] = 0.f;
                    if (F.u8) F.u8[i] = 0, F.u8[i + 1] = 0, F.u8[i + 2] = 0;
                }
            }
        }
        const int slot = wave_append(P, 0, rendered);
        if (slot >= 0) {
            V3 o, d;
            ray_for_pixel(S, x, y, o, d);
            WaveRay& r = P.rays[slot];
            r.ox = o.x, r.oy = o.y, r.oz = o.z, r.dx = d.x, r.dy = d.y, r.dz = d.z;
            r.t = -1.0f, r.pos = -1, r.pixel = (unsigned)(y * S.width + x), r.path = 1u, r.parent = -1, r.slot = 0;
            r.smax = -1.0f, r.shadowed = 0;
        }
    }
}

// ---- the tree walks ---------------------------------------------------------------------------------------------------
// Every lane owns one ray at a time and draws the next one from the level's queue when its walk ends (the refill
// happens at a converged point, when at least kRefillLanes lanes are idle: one atomic per refill).  The walk itself is
// nearest_hit's (dev_bvh.cuh): linear list first, then while-while through the tree with the per-thread stack.
// SHADOW: the ray is a shadow ray (sx.., limit smax, world.rs:104-119) and the result is `shadowed`.
template <bool SHADOW>
__device__ __forceinline__ void wave_trace(const DevScene& S, const WavePool& P, int level) {
    const int n = P.count[level], base = P.base[level];
    int* cursor = &P.cursor[2 * level + (SHADOW ? 1 : 0)];
    const int lane = threadIdx.x & 31;
    Ctr<false> k;
    bool live = false, exhausted = false;
    int mine = -1, node = 0, sp = 0;
    int stack[kBvhStack];
    V3 o = mk(0.f, 0.f, 0.f), d = mk(0.f, 0.f, 1.f), inv = d, noi = d;
    Hit best{0.f, -1, 0};
    ObjRay cache;
    const bool any_hit = SHADOW && S.all_cast_shadow;
    constexpr int kDone = -0x7fffffff - 1;
    for (;;) {
        // ---- refill (converged)
        const unsigned idle = __ballot_sync(0xffffffffu, !live);
        if (!exhausted && idle != 0u && (__popc(idle) >= kRefillLanes || idle == 0xffffffffu)) {
            const int leader = __ffs(idle) - 1;
            int first = 0;
            if (lane == leader) first = atomicAdd(cursor, __popc(idle));
            first = __shfl_sync(0xffffffffu, first, leader);
            if (first + __popc(idle) >= n) exhausted = true;
            if (!live) {
                const int q = first + __popc(idle & ((1u << lane) - 1u));
                if (q < n) {
                    mine = base + q;
                    const WaveRay& r = P.rays[mine];
                    bool wanted = true;
                    if (SHADOW) {
                        o = mk(r.sx, r.sy, r.sz), d = mk(r.sdx, r.sdy, r.sdz);
                        best = Hit{r.smax, -1, -1};  // order -1: a hit AT the light distance is never accepted (`<`, world.rs:116)
                        wanted = r.smax >= 0.0f;
                    } else {
                        o = mk(r.ox, r.oy, r.oz), d = mk(r.dx, r.dy, r.dz);
                        best = Hit{kInfF, -1, 0x7fffffff};
                    }
                    if (wanted) {
                        cache = ObjRay();
                        bool done = false;
#pragma unroll 1
                        for (int i = 0; i < S.n_linear && !done; i++) {
                            test_prim<false>(S, __ldg(&S.linear[i]), o, d, cache, best, k);
                            done = any_hit && best.pos >= 0;
                        }
                        if (!done && S.bvh_root >= 0) {
                            inv = mk(tree_inverse(d.x), tree_inverse(d.y), tree_inverse(d.z));
                            noi = mk(-(o.x * inv.x), -(o.y * inv.y), -(o.z * inv.z));
                            node = S.bvh_root, sp = 0, live = true;
                        }
                    }
                    if (!live) {  // settled without a walk
                        WaveRay& w = P.rays[mine];
                        if (SHADOW)
                            w.shadowed = wanted && best.pos >= 0 && (any_hit || ((__ldg(&S.head[best.pos]).x >> 4) & kFlagCastsShadow));
                        else
                            w.t = best.pos >= 0 ? best.t : -1.0f, w.pos = best.pos;
                    }
                }
            }
        }
        if (!__any_sync(0xffffffffu, live)) {
            if (exhausted) break;
            continue;
        }
        // ---- a burst of the walk: until this lane's ray is done, or too few lanes are still walking
        if (live) {
            bool done = false;
            for (;;) {
                while (node >= 0) {
                    const float4* np = reinterpret_cast<const float4*>(S.bvh + node);
                    const float4 a = __ldg(np), b = __ldg(np + 1), c = __ldg(np + 2);
                    const int4 link = __ldg(reinterpret_cast<const int4*>(np + 3));
                    float t0, t1;
                    const bool h0 = slab(noi, inv, a.x, a.y, a.z, a.w, b.x, b.y, best.t, t0);
                    const bool h1 = slab(noi, inv, b.z, b.w, c.x, c.y, c.z, c.w, best.t, t1);
                    if (h0 && h1) {
                        int near = link.x, far = link.y;
                        if (t1 < t0) near = link.y, far = link.x;
                        if (sp < kBvhStack) stack[sp++] = far;  // the builder bounds the depth (rtc_commit.cu, rtc_lbvh.cu)
                        node = near;
                    } else if (h0) {
                        node = link.x;
                    } else if (h1) {
                        node = link.y;
                    } else {
                        node = sp == 0 ? kDone : stack[--sp];
                    }
                }
                if (node == kDone) {
                    done = true;
                    break;
                }
                {
                    const int code = ~node;
                    const int first = code >> 4, count = (code & 15) + 1;
                    for (int i = 0; i < count && !done; i++) {
                        test_prim<false>(S, first + i, o, d, cache, best, k);
                        done = any_hit && best.pos >= 0;
                    }
                }
                if (done || sp == 0) {
                    done = true;
                    break;
                }
                node = stack[--sp];
                if (__popc(__activemask()) <= 32 - kRefillLanes && !exhausted) break;  // enough lanes idle: go and refill
            }
            if (done) {
                WaveRay& w = P.rays[mine];
                if (SHADOW)
                    w.shadowed = best.pos >= 0 && (any_hit || ((__ldg(&S.head[best.pos]).x >> 4) & kFlagCastsShadow));
                else
                    w.t = best.pos >= 0 ? best.t : -1.0f, w.pos = best.pos;
                live = false;
            }
        }
    }
}

// ---- between the walks ---------------------------------------------------------------------------------------------------
// precompute_values' geometry (world.rs:212-233), exactly as color_at spells it
struct WaveHit {
    V3 n, over_point;
    int4 head;
};
__device__ __forceinline__ WaveHit wave_hit_record(const DevScene& S, V3 ro, V3 rd, float t, int pos) {
    WaveHit h;
    h.head = __ldg(&S.head[pos]);
    const Xf m = load_xf(S.xform + 3 * (size_t)h.head.y);
    const V3 point = ro + rd * t;
    const V3 object_point = xf_point(m, point);
    V3 n = norm(xf_normal(m, local_normal(S, h.head.x & 15, h.head.z, object_point)));  // shape.rs:148-154,130-145
    if (dot(n, -rd) < 0.0f) n = -n;
    h.n = n;
    h.over_point = point + n * kAcne;
    return h;
}

// after wave_trace<nearest>: the shadow ray of every hit (world.rs:104-111; point lights only: one per shade)
__device__ __forceinline__ void wave_hit(const DevScene& S, const WavePool& P, int level) {
    const int n = P.count[level], base = P.base[level];
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < n; q += gridDim.x * blockDim.x) {
        WaveRay& r = P.rays[base + q];
        if (r.pos < 0) {
            r.smax = -1.0f;
            continue;
        }
        const WaveHit h = wave_hit_record(S, mk(r.ox, r.oy, r.oz), mk(r.dx, r.dy, r.dz), r.t, r.pos);
        const V3 v = ld3(S.light_pos) - h.over_point;
        const float distance = magnitude(v);
        const V3 direction = div3(v, distance);
        r.sx = h.over_point.x, r.sy = h.over_point.y, r.sz = h.over_point.z;
        r.sdx = direction.x, r.sdy = direction.y, r.sdz = direction.z;
        r.smax = distance;
    }
}

// after wave_trace<shadow>: shade_hit (world.rs:62-86) and the children (world.rs:121-162) — color_at's statements
__device__ __forceinline__ void wave_shade(const DevScene& S, const WavePool& P, int level, int depth) {
    const int n = P.count[level], base = P.base[level];
    const int remaining = depth - level;
    unsigned secondary = 0, shades = 0;
    Ctr<false> k;
    const int trips = (n + gridDim.x * blockDim.x - 1) / (gridDim.x * blockDim.x);  // warp-uniform: wave_append is collective
    for (int trip = 0; trip < trips; trip++) {
        const int q = trip * gridDim.x * blockDim.x + blockIdx.x * blockDim.x + threadIdx.x;
        const bool valid = q < n;
        const int idx = base + (valid ? q : 0);
        WaveNode node;
        node.sr = node.sg = node.sb = 0.f, node.reflective = node.transparency = 0.f, node.reflectance = -1.0f;
        node.rr = node.rg = node.rb = node.fr = node.fg = node.fb = 0.f;
        node.flags = 0;
        bool want_refl = false, want_refr = false;
        V3 refl_o = mk(0.f, 0.f, 0.f), refl_d = refl_o, refr_o = refl_o, refr_d = refl_o;
        unsigned pixel = 0, path = 1;
        if (valid) {
            const WaveRay r = P.rays[idx];
            node.parent = r.parent, node.slot = r.slot, node.pixel = r.pixel;
            pixel = r.pixel, path = r.path;
            if (r.pos >= 0) {
                shades++;
                const V3 ro = mk(r.ox, r.oy, r.oz), rd = mk(r.dx, r.dy, r.dz);
                const WaveHit h = wave_hit_record(S, ro, rd, r.t, r.pos);
                const V3 nrm = h.n, over_point = h.over_point;
                const DevMaterial& mat = S.materials[h.head.x >> 8];
                V3 material_color = ld3(mat.color);
                if (mat.pattern >= 0) {
                    const Xf m = load_xf(S.xform + 3 * (size_t)h.head.y);
                    material_color = pattern_color(S, mat.pattern, xf_point(m, over_point));  // pattern.rs:15-19 at over_point (Q4)
                }
                const float li = r.shadowed ? 0.f : 1.f;  // point_light.rs:28-34
                const V3 eye = -rd;
                const V3 light_rgb = ld3(S.light_rgb);
                const V3 effective = material_color * light_rgb;
                const V3 ambient = effective * mat.ambient;
                V3 surface = ambient;
                if (li != 0.f) {
                    const V3 to_light = norm(ld3(S.light_pos) - over_point);
                    const float lnc = dot(to_light, nrm);
                    V3 diffuse = mk(0.f, 0.f, 0.f), specular = mk(0.f, 0.f, 0.f);
                    if (!(lnc < 0.0f)) {
                        diffuse = effective * mat.diffuse * lnc;
                        const V3 sr = reflect(-to_light, nrm);
                        const float rec = dot(sr, eye);
                        if (!(rec <= 0.0f)) {
                            const float factor = (mat.specular == 0.0f && mat.shininess <= 1.0e4f) ? 1.0f : powf(rec, mat.shininess);
                            specular = light_rgb * mat.specular * factor;
                        }
                    }
                    surface = ambient + (diffuse + specular) * li;
                }
                want_refl = mat.reflective != 0.0f && remaining >= 1;
                float reflectance = -1.0f;
                if (mat.transparency != 0.0f) {
                    float n1, n2;
                    find_containers<false>(S, ro, rd, r.pos, n1, n2, k);
                    const float cos_i = dot(eye, nrm);
                    if (remaining != 0) {
                        const float n_ratio = n1 / n2;  // world.rs:196-207
                        const float sin2 = (n_ratio * n_ratio) * (1.0f - cos_i * cos_i);
                        if (!(sin2 > 1.0f)) {
                            const float cos_t = sqrtf(1.0f - sin2);
                            refr_d = nrm * (n_ratio * cos_i - cos_t) - (eye * n_ratio);
                            want_refr = true;
                        }
                    }
                    if (mat.reflective > 0.0f && mat.transparency > 0.0f) {  // schlick_reflectance, world.rs:285-303
                        float cosine = cos_i;
                        bool tir = false;
                        if (n1 > n2) {
                            const float nn = n1 / n2;
                            const float sin2_t = (nn * nn) * (1.0f - cosine * cosine);
                            if (sin2_t > 1.0f)
                                tir = true;
                            else
                                cosine = sqrtf(1.0f - sin2_t);
                        }
                        if (tir) {
                            reflectance = 1.0f;
                        } else {
                            const float q0 = (n1 - n2) / (n1 + n2);
                            const float r0 = q0 * q0;
                            reflectance = r0 + (1.0f - r0) * powi5(1.0f - cosine);
                        }
                    }
                }
                // color_at only opens a frame (and counts its children) below kMaxFrames levels; depth <= kMaxFrames - 1
                if (want_refr) refr_o = (ro + rd * r.t) - nrm * kAcne;  // under_point
                if (want_refl) refl_o = over_point, refl_d = reflect(rd, nrm);
                node.sr = surface.x, node.sg = surface.y, node.sb = surface.z;
                node.reflective = mat.reflective, node.transparency = mat.transparency, node.reflectance = reflectance;
                node.flags = 1 | (want_refl ? 2 : 0) | (want_refr ? 4 : 0);
            }
            P.nodes[idx] = node;
        }
        // children: reflection first, then refraction (their order in the queue is irrelevant: a child knows its parent)
        const int c0 = wave_append(P, level + 1, want_refl);
        if (c0 >= 0) {
            WaveRay& c = P.rays[c0];
            c.ox = refl_o.x, c.oy = refl_o.y, c.oz = refl_o.z, c.dx = refl_d.x, c.dy = refl_d.y, c.dz = refl_d.z;
            c.t = -1.0f, c.pos = -1, c.pixel = pixel, c.path = path * 3u + 1u, c.parent = idx, c.slot = 0, c.smax = -1.0f, c.shadowed = 0;
        }
        const int c1 = wave_append(P, level + 1, want_refr);
        if (c1 >= 0) {
            WaveRay& c = P.rays[c1];
            c.ox = refr_o.x, c.oy = refr_o.y, c.oz = refr_o.z, c.dx = refr_d.x, c.dy = refr_d.y, c.dz = refr_d.z;
            c.t = -1.0f, c.pos = -1, c.pixel = pixel, c.path = path * 3u + 2u, c.parent = idx, c.slot = 1, c.smax = -1.0f, c.shadowed = 0;
        }
        secondary += (want_refl ? 1u : 0u) + (want_refr ? 1u : 0u);
    }
    const unsigned s2 = __reduce_add_sync(0xffffffffu, secondary), s3 = __reduce_add_sync(0xffffffffu, shades);
    if ((threadIdx.x & 31) == 0) {
        if (s2) atomicAdd(P.secondary, (unsigned long long)s2);
        if (s3) atomicAdd(P.shades, (unsigned long long)s3);
    }
}

// a level's colours go up: into the parent's node, or (level 0) into the frame
__device__ __forceinline__ void wave_combine(const DevScene& S, const DevFrame& F, const WavePool& P, int level) {
    const int n = P.count[level], base = P.base[level];
    for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < n; q += gridDim.x * blockDim.x) {
        const WaveNode nd = P.nodes[base + q];
        V3 c = mk(0.f, 0.f, 0.f);
        if (nd.flags & 1) {
            const V3 reflected = (nd.flags & 2) ? mk(nd.rr, nd.rg, nd.rb) * nd.reflective : mk(0.f, 0.f, 0.f);     // world.rs:131
            const V3 refracted = (nd.flags & 4) ? mk(nd.fr, nd.fg, nd.fb) * nd.transparency : mk(0.f, 0.f, 0.f);  // world.rs:159-160
            c = combine(mk(nd.sr, nd.sg, nd.sb), reflected, refracted, nd.reflectance);
        }
        if (nd.parent >= 0) {
            WaveNode& p = P.nodes[nd.parent];
            if (nd.slot == 0)
                p.rr = c.x, p.rg = c.y, p.rb = c.z;
            else
                p.fr = c.x, p.fg = c.y, p.fb = c.z;
        } else {  // Canvas::write_pixel + scale_color (canvas.rs:26-43)
            const size_t i = (size_t)nd.pixel * 3;
            if (F.rgb) F.rgb[i] = c.x, F.rgb[i + 1] = c.y, F.rgb[i + 2] = c.z;
            if (F.u8) F.u8[i] = scale_color(c.x), F.u8[i + 1] = scale_color(c.y), F.u8[i + 2] = scale_color(c.z);
        }
    }
}

}  // namespace RTC_NS
}  // namespace rtc
