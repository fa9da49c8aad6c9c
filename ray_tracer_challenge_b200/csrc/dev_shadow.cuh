// dev_shadow.cuh — World::is_shadowed and Light::intensity_at: the shadow filter, the exact test, the cell-mask loops of area lights.
// Part of rtc_device.cuh (include that, not this): compiled once per kernel build inside namespace rtc::RTC_NS.
#pragma once

namespace rtc {
namespace RTC_NS {

// ---------------------------------------------------------------------------------------------------
// Shadow filter (small scenes made of spheres, planes and axis-aligned cubes only — SmallScene::filter_ok).
//
// World::is_shadowed only needs a BOOLEAN per light sample: "is the nearest hit in [0, distance) a shadow caster".
// The reference gets it the expensive way: normalise the direction (sqrt + 3 divisions), intersect everything,
// divide out every root.  Away from the decision boundaries the boolean does not depend on any of that rounding, so
// the filter evaluates the same predicate on the UN-normalised segment point -> light (parameter s in [0, 1),
// t = s * distance) with fused multiply-adds and approximate reciprocals, carries a forward error bound that covers
// both its own rounding and the reference's (object-space origins are the reference's own values, bit for bit; only
// the direction differs), and answers only when every comparison it needs is decided by a margin larger than that
// bound.  Anything closer than the margin — tangent rays, roots at the light, ties between objects, NaN / inf —
// returns F_UNSURE and the caller runs the exact test.  Frames are therefore bit-identical with the filter on or off
// (tests/test_gpu_parity.py::test_shadow_filter_changes_no_pixel).
enum : int { F_MISS = 0, F_HIT = 1, F_UNSURE = 2 };
struct FRes {
    int code;
    float s, e;  // F_HIT: segment parameter of the nearest hit and its error bound
};

// sphere.rs:47-70 on the segment o + s * d, d = M * (light - point).  `tol` = SmallScene::tol_sphere, which scales
// with the worst condition number of the spheres' transforms (set at commit).
// The part that runs once the discriminant is clearly positive: which root is Intersection::hit's, is it in [0, 1).
__device__ __forceinline__ FRes sphere_roots(float a, float b, float oo, float spread, float disc, float tol) {
    const float rs = rsqrtf(disc), ia = rcp_(a);
    const float sq = disc * rs;
    const float s0 = (-b - sq) * ia, s1 = (-b + sq) * ia;
    const float x = oo * ia;
    // |error of a root| <= tol * (sqrt(oo / a) + spread / sqrt(disc) + |root|); + tol for the comparison with 1
    const float e = tol * (x * rsqrtf(x + 1e-30f) + spread * rs + fmaxf(fabsf(s0), fabsf(s1)) + 1.0f);
    const bool p0 = s0 > e, n0 = s0 < -e, p1 = s1 > e, n1 = s1 < -e;
    if (n0 && n1) return FRes{F_MISS, 0.f, 0.f};
    if (!(p0 || (n0 && p1))) return FRes{F_UNSURE, 0.f, 0.f};
    const float cand = p0 ? s0 : s1;  // Intersection::hit: the smallest non-negative root
    if (cand < 1.0f - e) return FRes{F_HIT, cand, e};
    if (cand > 1.0f + e) return FRes{F_MISS, 0.f, 0.f};
    return FRes{F_UNSURE, 0.f, 0.f};
}
__device__ __forceinline__ FRes filter_sphere(const Xf& m, V3 o, V3 v, float tol) {
    const float dx = fma_(m.r0.x, v.x, fma_(m.r0.y, v.y, m.r0.z * v.z));
    const float dy = fma_(m.r1.x, v.x, fma_(m.r1.y, v.y, m.r1.z * v.z));
    const float dz = fma_(m.r2.x, v.x, fma_(m.r2.y, v.y, m.r2.z * v.z));
    const float a = fma_(dx, dx, fma_(dy, dy, dz * dz));
    const float b = fma_(dx, o.x, fma_(dy, o.y, dz * o.z));  // half the reference's b
    const float oo = fma_(o.x, o.x, fma_(o.y, o.y, o.z * o.z));
    const float c = oo - 1.0f;
    const float disc = fma_(b, b, -(a * c));                 // a quarter of the reference's discriminant (times |v|^2)
    const float spread = oo + fabsf(c);
    const float td = tol * (a * spread);                     // a * spread >= b^2 + |a c|
    if (disc < -td) return FRes{F_MISS, 0.f, 0.f};
    if (!(disc > td)) return FRes{F_UNSURE, 0.f, 0.f};
    return sphere_roots(a, b, oo, spread, disc, tol);
}

// plane.rs:45-56: only the y row of the inverse is needed.  `len` ~ |light - point| (the reference compares the
// NORMALISED direction's y with EPSILON).
// `upper`: len is only an upper bound of the length (the cell-mask path passes the 1-norm): a direction that is not
// clearly steeper than EPSILON against the bound is undecided rather than a miss.
template <bool NEED_S>
__device__ __forceinline__ FRes filter_plane(float4 r1, float oy, V3 v, float len, bool upper = false) {
    const float px = r1.x * v.x, py = r1.y * v.y, pz = r1.z * v.z;
    const float dy = px + py + pz;
    const float edy = kTolP * (fabsf(px) + fabsf(py) + fabsf(pz));
    const float mag = fabsf(dy), thr = kAcne * len;
    if (!upper && mag + edy < thr * (1.0f - kTolP)) return FRes{F_MISS, 0.f, 0.f};  // plane.rs:49
    if (!(mag - edy > thr * (1.0f + kTolP)) || oy == 0.0f) return FRes{F_UNSURE, 0.f, 0.f};
    if ((oy < 0.0f) == (dy < 0.0f)) return FRes{F_MISS, 0.f, 0.f};  // t = -oy / dy < 0
    const float aoy = fabsf(oy);
    if (aoy < (mag - edy) * (1.0f - kTolP)) {
        if (!NEED_S) return FRes{F_HIT, 0.f, 0.f};
        const float im = rcp_(mag), s = aoy * im;
        return FRes{F_HIT, s, s * (edy * im + 4.0f * kTolP)};
    }
    if (aoy > (mag + edy) * (1.0f + kTolP)) return FRes{F_MISS, 0.f, 0.f};
    return FRes{F_UNSURE, 0.f, 0.f};
}

// cube.rs:55-63 + 90-129 for a cube whose inverse has a diagonal 3x3 part (checked at commit): every direction
// component is ONE product, so each slab distance differs from the reference's by a few ulp, never by cancellation.
__device__ __forceinline__ FRes filter_cube(const Xf& m, V3 o, V3 v) {
    const float dx = m.r0.x * v.x, dy = m.r1.y * v.y, dz = m.r2.z * v.z;
    if (dx == 0.0f || dy == 0.0f || dz == 0.0f) return FRes{F_UNSURE, 0.f, 0.f};
    const float ix = rcp_(dx), iy = rcp_(dy), iz = rcp_(dz);
    float p = (-1.0f - o.x) * ix, q = (1.0f - o.x) * ix;
    float lo = fminf(p, q), hi = fmaxf(p, q);
    p = (-1.0f - o.y) * iy, q = (1.0f - o.y) * iy;
    lo = fmaxf(lo, fminf(p, q)), hi = fminf(hi, fmaxf(p, q));
    p = (-1.0f - o.z) * iz, q = (1.0f - o.z) * iz;
    lo = fmaxf(lo, fminf(p, q)), hi = fminf(hi, fmaxf(p, q));
    const float e = kTolP * (fabsf(lo) + fabsf(hi) + 1.0f);
    const float g = hi - fmaxf(lo, 0.0f);
    if (g < -e) return FRes{F_MISS, 0.f, 0.f};
    if (!(g > e) || !(fabsf(lo) > e)) return FRes{F_UNSURE, 0.f, 0.f};
    const float cand = lo > 0.0f ? lo : hi;
    if (cand < 1.0f - e) return FRes{F_HIT, cand, e};
    if (cand > 1.0f + e) return FRes{F_MISS, 0.f, 0.f};
    return FRes{F_UNSURE, 0.f, 0.f};
}

// The items [begin, ends.z) of the small-scene table against the segment.  MODE 0: casters, any hit decides
// (every object casts); MODE 1: casters, keep the nearest hit (s_c, e_c); MODE 2: non-casters against the nearest
// caster hit.  Returns F_UNSURE as soon as some test is undecided; otherwise F_HIT / F_MISS, meaning
//   MODE 0/1: some / no caster is hit in [0, 1);  MODE 2: F_HIT = a non-caster is clearly nearer than every caster.
template <bool STATS, int MODE>
__device__ __forceinline__ int filter_scan(const Env& E, bool cached, int begin, int4 ends, V3 p, V3 v, float len, float& s_c,
                                           float& e_c, Ctr<STATS>& k) {
    const float4* tab = small_tab();
    const float tol = E.SS.tol_sphere;
    int result = F_MISS;
    auto take = [&](const FRes& r) -> bool {  // true: the scan is decided
        if (r.code == F_UNSURE) {
            result = F_UNSURE;
            return true;
        }
        if (r.code == F_MISS) return false;
        if (MODE == 0) {
            result = F_HIT;
            return true;
        }
        if (MODE == 1) {
            result = F_HIT;
            e_c = r.s < s_c ? r.e : e_c;
            s_c = fminf(s_c, r.s);
            return false;
        }
        if (r.s + r.e < s_c - e_c) {  // clearly in front of the nearest caster: the point is lit (world.rs:113-118)
            result = F_HIT;
            return true;
        }
        if (r.s - r.e > s_c + e_c) return false;  // clearly behind it
        result = F_UNSURE;
        return true;
    };
    int i = begin;
#pragma unroll 1
    for (; i < ends.x; i++) {
        Xf m{tab[i * kSmallStride + 1], tab[i * kSmallStride + 2], tab[i * kSmallStride + 3]};
        k.xform();
        k.prim(T_SPHERE);
        if (take(filter_sphere(m, small_origin(cached, i, m, p), v, tol))) return result;
    }
#pragma unroll 1
    for (; i < ends.y; i++) {
        float4 r1 = tab[i * kSmallStride + 2];
        float oy;
        if (cached && i < kOrgCache)
            oy = small_org()[(i * 3 + 1) * kBlockThreads];
        else
            oy = r1.x * p.x + r1.y * p.y + r1.z * p.z + r1.w;
        k.xform();
        k.prim(T_PLANE);
        if (take(filter_plane<MODE != 0>(r1, oy, v, len))) return result;
    }
#pragma unroll 1
    for (; i < ends.z; i++) {
        Xf m{tab[i * kSmallStride + 1], tab[i * kSmallStride + 2], tab[i * kSmallStride + 3]};
        k.xform();
        k.prim(T_CUBE);
        if (take(filter_cube(m, small_origin(cached, i, m, p), v))) return result;
    }
    return result;
}

// 0: lit, 1: shadowed, 2: undecided (run the exact test)
template <bool STATS>
__device__ __forceinline__ int shadow_filter(const Env& E, bool cached, V3 light_position, V3 p, Ctr<STATS>& k) {
    const SmallScene& SS = E.SS;
    const V3 v = light_position - p;
    const float vv = fma_(v.x, v.x, fma_(v.y, v.y, v.z * v.z));
    const float len = vv * rsqrtf(vv);
    float s_c = kInfF, e_c = 0.0f;
    if (E.S.all_cast_shadow) return filter_scan<STATS, 0>(E, cached, 0, SS.caster_end, p, v, len, s_c, e_c, k);
    int r = filter_scan<STATS, 1>(E, cached, 0, SS.caster_end, p, v, len, s_c, e_c, k);
    if (r != F_HIT) return r == F_MISS ? 0 : 2;
    r = filter_scan<STATS, 2>(E, cached, SS.caster_end.w, SS.other_end, p, v, len, s_c, e_c, k);
    return r == F_UNSURE ? 2 : (r == F_HIT ? 0 : 1);
}

// World::is_shadowed (world.rs:104-119): nearest hit on the point->light ray; shadowed iff that object
// casts a shadow and is nearer than the light (Q9).
//
// Small scenes test the shadow casters first: with no caster in [0, distance) the answer is "lit" whatever
// the non-casting objects do, and otherwise only a non-casting object NEARER than the nearest caster (same
// (t, depth-first order) comparison as Intersection::hit) can un-shadow the point.  Same predicate as the
// reference's, evaluated with fewer intersection tests.
template <bool STATS, bool LEAN>
__device__ __forceinline__ bool shadow_exact_small(const Env& E, bool cached, V3 light_position, V3 p, Ctr<STATS>& k) {
    const DevScene& S = E.S;
    const SmallScene& SS = E.SS;
    V3 v = light_position - p;
    float distance = magnitude(v);
    V3 direction = div3(v, distance);
    // order -1: a hit AT the light distance is never accepted (`<`, world.rs:116)
    Hit best{distance, -1, -1};
    if (!LEAN && (!SS.two_pass_shadows || SS.has_cull_chain)) {  // a CSG root or a cull chain: plain nearest-hit search
#pragma unroll 1
        for (int i = 0; i < SS.n; i++) test_small<STATS>(E, i, cached, p, direction, best, k);
        return best.pos >= 0 && ((__ldg(&S.head[best.pos]).x >> 4) & kFlagCastsShadow);
    }
    if (S.all_cast_shadow)  // every object casts: any hit in [0, distance) shadows the point
        return scan_small<STATS, true, LEAN>(E, cached, 0, SS.caster_end, p, direction, best, k);
    int begin = 0, caster = -1;
    int4 ends = SS.caster_end;
#pragma unroll 1
    for (int seg = 0; seg < 2; seg++) {  // casters, then non-casters: one copy of the loops
        scan_small<STATS, false, LEAN>(E, cached, begin, ends, p, direction, best, k);
        if (seg == 0) {
            if (best.pos < 0) return false;
            caster = best.pos;
        }
        begin = ends.w;
        ends = SS.other_end;
    }
    return best.pos == caster;
}
// One shadow ray of a small scene, out of line (ONE copy of the filter and of the exact test in the kernel: the
// kernel's instruction footprint, not its arithmetic, limits the issue rate).  skip_filter: the caller already
// knows the filter cannot decide this ray.  LEAN: a lean scene is filter-eligible, holds no CSG root, cull chain or
// "everything else" item, and its cell-mask loops never fill the origin cache.
template <bool STATS, bool LEAN = false>
__device__ __noinline__ bool shadow_query_small(const Env& E, bool cached, bool skip_filter, V3 light_position, V3 p, Ctr<STATS>& k) {
    if (LEAN) cached = false;
    if (LEAN || E.SS.filter_ok) {
        const int f = skip_filter ? 2 : shadow_filter<STATS>(E, cached, light_position, p, k);
        if (f != 2) return f == 1;
        k.refiltered();
    }
    return shadow_exact_small<STATS, LEAN>(E, cached, light_position, p, k);
}
template <bool STATS, bool SMALL, bool CACHED>
__device__ __forceinline__ bool is_shadowed(const Env& E, V3 light_position, V3 p, Rays& r, Ctr<STATS>& k) {
    if (SMALL) return shadow_query_small<STATS>(E, CACHED, false, light_position, p, k);
    const DevScene& S = E.S;
    V3 v = light_position - p;
    float distance = magnitude(v);
    V3 direction = div3(v, distance);
    Hit best{distance, -1, -1};  // order -1: a hit AT the light distance is never accepted (`<`, world.rs:116)
    if (S.all_cast_shadow) {
        nearest_hit<STATS, true>(S, p, direction, best, k);
        return best.pos >= 0;
    }
    nearest_hit<STATS, false>(S, p, direction, best, k);
    return best.pos >= 0 && ((__ldg(&S.head[best.pos]).x >> 4) & kFlagCastsShadow);
}

// RectangleLight::intensity_at (rectangle_light.rs:76-88) for filter_ok scenes with a table-mode light: the light
// samples are the same for every shade (staged in shared memory), so the loops are turned inside out — primitive
// outside, light cell inside — and the per-shade part of every test (object-space origin, |o|^2, ...) leaves the
// cell loop.  Pass 1 runs the shadow filter of every CASTER against up to 32 cells at a time and keeps two bit
// masks: cells where some caster is clearly hit, cells where some test was undecided.  Cells in neither mask are
// lit.  Pass 2 revisits the others one by one: hit cells need the nearest-caster / non-caster comparison
// (shadow_filter) when the scene has non-casting objects, undecided cells run the exact test.
// Distances from p to a bounding ball {centre, radius}: no point of the ball is farther than ball_reach, none is
// nearer than ball_gap (negative inside).  Approximate square roots: the callers compare with a 0.1 % margin.
__device__ __forceinline__ float ball_reach(float4 ball, V3 p) {
    const float dx = p.x - ball.x, dy = p.y - ball.y, dz = p.z - ball.z;
    const float ww = fma_(dx, dx, fma_(dy, dy, dz * dz));
    return ww * rsqrtf(ww + 1e-30f) + ball.w;
}
__device__ __forceinline__ float ball_gap(float4 ball, V3 p) {
    const float dx = p.x - ball.x, dy = p.y - ball.y, dz = p.z - ball.z;
    const float ww = fma_(dx, dx, fma_(dy, dy, dz * dz));
    return ww * rsqrtf(ww + 1e-30f) - ball.w;
}

// filter_plane with the per-(plane, cell) constants of plane_cell_constants: q = {r1.L, tol*|r1||L|, eps'*|L|_1},
// rp = r1.p, erp = tol * sum|r1_k p_k|, p1 = eps' * |p|_1 (per shade).  |L - p| <= |L|_1 + |p|_1 stands in for the length
// in the reference's `direction.y.abs() < EPSILON` test (plane.rs:49), so a direction that is not clearly steeper than
// that is undecided rather than a miss.
__device__ __forceinline__ int filter_plane_cell(float4 q, float oy, float rp, float erp, float p1) {
    const float dy = q.x - rp;
    const float edy = q.y + erp;
    const float mag = fabsf(dy), lo = mag - edy;
    if (!(lo > q.z + p1) || oy == 0.0f) return F_UNSURE;
    if ((oy < 0.0f) == (dy < 0.0f)) return F_MISS;  // t = -oy / dy < 0
    const float aoy = fabsf(oy);
    if (aoy < lo * (1.0f - kTolP)) return F_HIT;
    if (aoy > (mag + edy) * (1.0f + kTolP)) return F_MISS;
    return F_UNSURE;
}

// Bundle reject: every shadow segment of a shade runs from p to a light sample inside the ball (Lc, Rl), so all of
// them lie in the cone-like solid { x : |x - (p + s (Lc - p))| <= s Rl, 0 <= s <= 1 }.  A primitive whose bounding ball
// (C, R) stays outside it — f(s) = |w + s u|^2 - (R + s Rl)^2 > 0 on [0, 1], w = p - C, u = Lc - p — cannot be hit by
// any of them.  R is padded by 0.1 % plus 2^-17 * |w|^2 / R: beyond that clearance neither this filter nor the
// reference's f32 discriminant (whose rounding error grows with |w|^2 / R^2) can report a hit.
__device__ __forceinline__ bool bundle_misses(float4 ball, float pad_over_r, float4 light_ball, V3 p) {
    const V3 w = mk(p.x - ball.x, p.y - ball.y, p.z - ball.z);
    const V3 u = mk(light_ball.x - p.x, light_ball.y - p.y, light_ball.z - p.z);
    const float ww = fma_(w.x, w.x, fma_(w.y, w.y, w.z * w.z));
    const float R = fma_(pad_over_r, ww, ball.w), Rl = light_ball.w;
    const float A = fma_(u.x, u.x, fma_(u.y, u.y, u.z * u.z)) - Rl * Rl;
    const float B = fma_(w.x, u.x, fma_(w.y, u.y, w.z * u.z)) - R * Rl;
    const float C = ww - R * R;
    if (!(C > 0.0f) || !(A + 2.0f * B + C > 0.0f)) return false;  // an end of the bundle touches the ball
    if (!(A > 0.0f)) return A <= 0.0f;      // concave or linear: the minimum over [0, 1] is at an end (NaN: no reject)
    if (B >= 0.0f || -B >= A) return true;  // convex, vertex outside (0, 1)
    return C * A > B * B * 1.0001f;
}

// point_on_light (rectangle_light.rs:60-66) for the cells [c0, c0 + nc) of a shade with generated jitter: two values per
// cell in the reference's order `for v { for u { j_u, j_v } }`
__device__ __forceinline__ void draw_light_samples(const DevScene& S, unsigned pixel, unsigned path, int c0, int nc, float4* drawn) {
    const V3 corner = ld3(S.corner), u_vec = ld3(S.u_vec), v_vec = ld3(S.v_vec);
    const unsigned key = jitter_key(S.seed, pixel, path);
    for (int j = 0; j < nc; j++) {
        const unsigned cell = (unsigned)(c0 + j);
        const int v = (int)cell / S.u_steps, u = (int)cell - v * S.u_steps;
        const float j1 = jitter_value(key, 2u * cell);
        const float j2 = jitter_value(key, 2u * cell + 1u);
        const V3 lp = corner + u_vec * ((float)u + j1) + v_vec * ((float)v + j2);
        drawn[j] = make_float4(lp.x, lp.y, lp.z, 0.f);
    }
}

// TABLE: the light samples are the staged table.  Otherwise (jitter `None`, rectangle_light.rs:46: the counter-based
// generator) a chunk's sample points are drawn first — two jitter values per cell in the reference's order
// `for v { for u { j_u, j_v } }`, point_on_light's arithmetic (rectangle_light.rs:60-66) — into a per-thread array,
// and the same loops read them from there.
template <bool STATS, bool TABLE, bool LEAN>
__device__ __forceinline__ float intensity_cells(const Env& E, V3 p, unsigned pixel, unsigned path, Rays& r, Ctr<STATS>& k) {
    const DevScene& S = E.S;
    const SmallScene& SS = E.SS;
    const float4* tab = small_tab();
    const float4* table = small_samples();
    const int cells = S.cells;
    const float tol = SS.tol_sphere;
    const int4 ends = SS.caster_end;
    int lit = 0;
    float4 drawn[TABLE ? 1 : 32];
    for (int c0 = 0; c0 < cells; c0 += 32) {
        const int nc = min(32, cells - c0);
        const unsigned full = nc == 32 ? 0xffffffffu : ((1u << nc) - 1u);
        // Generated jitter: the chunk's sample points are drawn only when the first caster that the bundle tests cannot
        // dismiss needs them — most shades of a floor under a light are settled for every cell by those tests alone, and
        // the points of a cell depend on nothing but (seed, pixel, path, cell), so drawing them late draws the same points.
        bool have_samples = TABLE;
#define RTC_DRAW_SAMPLES()                                                   \
    do {                                                                     \
        if (!TABLE && !have_samples) {                                       \
            have_samples = true;                                             \
            draw_light_samples(S, pixel, path, c0, nc, drawn);               \
        }                                                                    \
    } while (0)
        const float4* smp = TABLE ? table + c0 : drawn;
        unsigned hit = 0u, unsure = 0u;
        float far_hit = 0.0f;  // no caster hit of this chunk is farther from p than this (bounding balls)
        int i = 0;
#pragma unroll 1
        for (; i < ends.x && (hit | unsure) != full; i++) {  // caster spheres
            if (bundle_misses(tab[i * kSmallStride + 5], tab[i * kSmallStride + 4].w, SS.light_ball, p)) continue;
            const unsigned hit_before = hit;
            RTC_DRAW_SAMPLES();
            const Xf m{tab[i * kSmallStride + 1], tab[i * kSmallStride + 2], tab[i * kSmallStride + 3]};
            const V3 o = xf_point(m, p);  // the reference's object-space origin (shape.rs:60-70), once per shade
            const float oo = fma_(o.x, o.x, fma_(o.y, o.y, o.z * o.z));
            const float c = oo - 1.0f;
            const float spread = oo + fabsf(c);
            const float ts = tol * spread;
#pragma unroll 4
            for (int j = 0; j < nc; j++) {
                const float4 L = smp[j];
                const float vx = L.x - p.x, vy = L.y - p.y, vz = L.z - p.z;
                const float dx = fma_(m.r0.x, vx, fma_(m.r0.y, vy, m.r0.z * vz));
                const float dy = fma_(m.r1.x, vx, fma_(m.r1.y, vy, m.r1.z * vz));
                const float dz = fma_(m.r2.x, vx, fma_(m.r2.y, vy, m.r2.z * vz));
                const float a = fma_(dx, dx, fma_(dy, dy, dz * dz));
                const float b = fma_(dx, o.x, fma_(dy, o.y, dz * o.z));
                const float disc = fma_(b, b, -(a * c));
                const float td = a * ts;
                if (!(disc < -td)) {  // not a clear miss
                    const int code = disc > td ? sphere_roots(a, b, oo, spread, disc, tol).code : F_UNSURE;
                    hit |= (unsigned)(code == F_HIT) << j;
                    unsure |= (unsigned)(code == F_UNSURE) << j;
                }
            }
            for (int j = 0; j < nc; j++) {
                k.xform();
                k.prim(T_SPHERE);
            }
            if (hit != hit_before) far_hit = fmaxf(far_hit, ball_reach(tab[i * kSmallStride + 5], p));
        }
#pragma unroll 1
        for (i = ends.x; i < ends.y && (hit | unsure) != full; i++) {  // caster planes
            const unsigned hit_before = hit;
            const float4 r1 = tab[i * kSmallStride + 2];
            const float tx = r1.x * p.x, ty = r1.y * p.y, tz = r1.z * p.z;
            const float rp = tx + ty + tz;
            const float oy = rp + r1.w;  // the reference's object-space origin.y (shape.rs:60-70)
            const float erp = kTolP * (fabsf(tx) + fabsf(ty) + fabsf(tz));
            const float p1 = (kAcne * (1.0f + 2.0f * kTolP)) * (fabsf(p.x) + fabsf(p.y) + fabsf(p.z));
            if (i - ends.x < 2) {
                // the whole bundle at once: with the bounds of the cell constants (table mode) or of the light's rectangle
                // (generated jitter), every cell's direction is clearly steep and points away from the plane's side the
                // point is on (a floor under a light above it): the per-cell test would answer F_MISS for each of them
                // (a NaN bound — no bundle data for this plane — fails both comparisons)
                const float4 pb = SS.plane_bundle[i - ends.x];
                const float slack = pb.z + erp + pb.w + p1;
                if ((oy > 0.0f && (pb.x - rp) > slack) || (oy < 0.0f && (rp - pb.y) > slack)) continue;
            }
            if (SS.plane_cells) {
                const float4* pc = small_plane_cells() + (i - ends.x) * cells + c0;
#pragma unroll 4
                for (int j = 0; j < nc; j++) {
                    const int code = filter_plane_cell(pc[j], oy, rp, erp, p1);
                    hit |= (unsigned)(code == F_HIT) << j;
                    unsure |= (unsigned)(code == F_UNSURE) << j;
                }
                for (int j = 0; j < nc; j++) {
                    k.xform();
                    k.prim(T_PLANE);
                }
                if (hit != hit_before) far_hit = kInfF;  // a plane has no bounding ball
                continue;
            }
            RTC_DRAW_SAMPLES();
#pragma unroll 4
            for (int j = 0; j < nc; j++) {
                const float4 L = smp[j];
                const V3 v = mk(L.x - p.x, L.y - p.y, L.z - p.z);
                // |v| <= |v|_1: a conservative stand-in for the length in the `direction.y.abs() < EPSILON` test
                const int code = filter_plane<false>(r1, oy, v, fabsf(v.x) + fabsf(v.y) + fabsf(v.z), true).code;
                hit |= (unsigned)(code == F_HIT) << j;
                unsure |= (unsigned)(code == F_UNSURE) << j;
            }
            for (int j = 0; j < nc; j++) {
                k.xform();
                k.prim(T_PLANE);
            }
            if (hit != hit_before) far_hit = kInfF;
        }
#pragma unroll 1
        for (i = ends.y; i < ends.z && (hit | unsure) != full; i++) {  // caster cubes
            if (bundle_misses(tab[i * kSmallStride + 5], tab[i * kSmallStride + 4].w, SS.light_ball, p)) continue;
            const unsigned hit_before = hit;
            RTC_DRAW_SAMPLES();
            const Xf m{tab[i * kSmallStride + 1], tab[i * kSmallStride + 2], tab[i * kSmallStride + 3]};
            const V3 o = xf_point(m, p);
#pragma unroll 2
            for (int j = 0; j < nc; j++) {
                const float4 L = smp[j];
                const int code = filter_cube(m, o, mk(L.x - p.x, L.y - p.y, L.z - p.z)).code;
                hit |= (unsigned)(code == F_HIT) << j;
                unsure |= (unsigned)(code == F_UNSURE) << j;
            }
            for (int j = 0; j < nc; j++) {
                k.xform();
                k.prim(T_CUBE);
            }
            if (hit != hit_before) far_hit = fmaxf(far_hit, ball_reach(tab[i * kSmallStride + 5], p));
        }
        for (int j = 0; j < nc; j++) k.cell();
        // pass 2.  A non-caster only matters where it is NEARER than the nearest caster hit (world.rs:113-118): when
        // every non-caster's bounding ball begins beyond the reach of every caster that was hit, the hit cells are
        // shadowed as they stand.
        bool hits_final = S.all_cast_shadow != 0;
        if (!hits_final && (hit & ~unsure) != 0u) {
            float near_other = kInfF;
#pragma unroll 1
            for (int q = ends.w; q < SS.other_end.z; q++) {
                const float4 ball = tab[q * kSmallStride + 5];
                const bool has_ball = q < SS.other_end.x || q >= SS.other_end.y;  // spheres and cubes; planes have none
                near_other = fminf(near_other, has_ball ? ball_gap(ball, p) : 0.0f);
            }
            hits_final = far_hit * 1.001f < near_other;  // false for NaN
        }
        unsigned todo = hits_final ? unsure : (hit | unsure);
        lit += __popc(full & ~(hit | unsure));
        if (todo) RTC_DRAW_SAMPLES();
        while (todo) {
            const int j = __ffs(todo) - 1;
            todo &= todo - 1u;
            const float4 L = smp[j];
            lit += !shadow_query_small<STATS, LEAN>(E, false, (unsure >> j) & 1u, mk(L.x, L.y, L.z), p, k);
        }
    }
    return (float)lit / (float)cells;  // `total += 1.0` per lit cell is exact in f32
#undef RTC_DRAW_SAMPLES
}

// Light::intensity_at (point_light.rs:28-34, rectangle_light.rs:76-88).  DRAWN: the kernel build for small scenes whose
// area light draws its jitter from the counter-based generator (only that build carries intensity_cells<.., false>).
// LEAN: the scene's light takes the cell-mask loops (SmallScene::lean implies SmallScene::cell_masks).
template <bool STATS, bool SMALL, bool DRAWN, bool LEAN = false>
__device__ __forceinline__ float intensity_at(const Env& E, V3 p, unsigned pixel, unsigned path, Rays& r, Ctr<STATS>& k) {
    const DevScene& S = E.S;
    if (!LEAN && !S.light_is_rect) return is_shadowed<STATS, SMALL, false>(E, ld3(S.light_pos), p, r, k) ? 0.f : 1.f;
    if (SMALL && (LEAN || E.SS.cell_masks))
        return DRAWN ? intensity_cells<STATS, false, LEAN>(E, p, pixel, path, r, k) : intensity_cells<STATS, true, LEAN>(E, p, pixel, path, r, k);
    if (SMALL) cache_origins(E, p);
    const unsigned key = S.jitter_len > 0 ? 0u : jitter_key(S.seed, pixel, path);
    float total = 0.f;
    int cell = 0;
    for (int v = 0; v < S.v_steps; v++) {
        for (int u = 0; u < S.u_steps; u++, cell++) {
            V3 lp;
            k.cell();
            if (S.jitter_len > 0) {
                float4 s = __ldg(&S.samples[cell]);  // table mode: point_on_light is the same for every shade
                lp = mk(s.x, s.y, s.z);
            } else {
                float j1 = jitter_value(key, 2u * cell);
                float j2 = jitter_value(key, 2u * cell + 1u);
                // rectangle_light.rs:60-66
                lp = ld3(S.corner) + ld3(S.u_vec) * ((float)u + j1) + ld3(S.v_vec) * ((float)v + j2);
            }
            if (!is_shadowed<STATS, SMALL, SMALL>(E, lp, p, r, k)) total += 1.0f;
        }
    }
    return total / (float)S.cells;
}

}  // namespace RTC_NS
}  // namespace rtc
