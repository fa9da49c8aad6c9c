// dev_small.cuh — the small-scene path: shared-memory table, typed nearest-hit loops, ray-vs-ball pre-test.
// Part of rtc_device.cuh (include that, not this): compiled once per kernel build inside namespace rtc::RTC_NS.
#pragma once

// The declaration of the dynamic shared-memory block.  The host harness of the device code (tests/emu/simt.h) turns
// __shared__ into `static` for the static arrays, so it spells this one as a plain `extern` array instead.
#ifndef RTC_EXTERN_SHARED
#define RTC_EXTERN_SHARED extern __shared__
#endif

namespace rtc {
namespace RTC_NS {

// ---------------------------------------------------------------------------------------------------
// What a thread needs to trace: the scene and the small-scene table (both in the kernel parameter block).
struct Env {
    const DevScene& S;
    const SmallScene& SS;
};

// Small scenes keep these in (dynamic) shared memory, kSmallSmemBytes in all:
//   tab     : the primitive table, kSmallStride x float4 per primitive {head, row0, row1, row2, bound, ball} — every
//             thread of a warp reads the same entry, so a row is one broadcast LDS.128 with an immediate offset;
//   samples : table-mode area light: the `cells` sample points (cell-mask loops, intensity_cells);
//   plane cells : per (caster plane, cell) the constants of filter_plane_cell (rtc_types.h: plane_cell_constants);
//   org     : per thread, the object-space origin of the current shade's shadow rays for the first kOrgCache
//             primitives (element (i, c) of thread t at org[(i * 3 + c) * kBlockThreads + t]) — the per-cell shadow loop.
// The first three are the same for every block: stage_small_scene copies them from the scene's image.
__device__ __forceinline__ const float4* small_tab() {
    RTC_EXTERN_SHARED float4 rtc_smem[];
    return rtc_smem;
}
__device__ __forceinline__ float* small_org() {
    RTC_EXTERN_SHARED float4 rtc_smem[];
    return reinterpret_cast<float*>(rtc_smem + kSmemOrg) + threadIdx.x;
}
__device__ __forceinline__ const float4* small_plane_cells() {
    RTC_EXTERN_SHARED float4 rtc_smem[];
    return rtc_smem + kSmemPlaneCells;
}
__device__ __forceinline__ const float4* small_samples() {  // table-mode light samples (SmallScene::cell_masks)
    RTC_EXTERN_SHARED float4 rtc_smem[];
    return rtc_smem + kSmemSamples;
}
// A block's staging: three coalesced copies out of the scene's image (L2 / L1 resident after the first blocks), each
// started by a different warp so that no warp does all of it while the others wait at the barrier.  Every kernel that
// stages runs blocks of kBlockThreads threads: with the block size a constant the start offsets and trip counts are
// shifts and masks, not the integer divisions a runtime blockDim.x costs every block (the host harnesses of
// tests/emu stage with one thread, emu_color.cpp, or with kBlockThreads, emu_kernels.cpp).
__device__ __forceinline__ void stage_small_scene(const DevScene& S, const SmallScene& SS) {
    RTC_EXTERN_SHARED float4 rtc_smem[];
    const float4* img = S.small_image;
#ifdef __CUDA_ARCH__
    constexpr int nt = kBlockThreads;
#else
    const int nt = blockDim.x;
#endif
    const int t = threadIdx.x;
    // at most kPlaneCellCap / kBlockThreads iterations each: not unrolled, the prologue stays short
#pragma unroll 1
    for (int i = t; i < SS.n * kSmallStride; i += nt) rtc_smem[i] = __ldg(img + i);
    if (SS.cell_masks && S.jitter_len > 0) {
#pragma unroll 1
        for (int i = (t + nt - 32) % nt; i < S.cells; i += nt) rtc_smem[kSmemSamples + i] = __ldg(img + kSmemSamples + i);
        if (SS.plane_cells) {
            const int n = (SS.caster_end.y - SS.caster_end.x) * S.cells;
#pragma unroll 1
            for (int i = (t + nt - 64) % nt; i < n; i += nt) rtc_smem[kSmemPlaneCells + i] = __ldg(img + kSmemPlaneCells + i);
        }
    }
    __syncthreads();
}

// Object-space origin of primitive i: from the per-shade cache (all shadow rays of one shade share their
// origin, so `inverse * origin`, shape.rs:60-70, is evaluated once per primitive instead of once per light
// cell — the same arithmetic, hoisted) or computed.
__device__ __forceinline__ V3 small_origin(bool cached, int i, const Xf& m, V3 o) {
    if (cached && i < kOrgCache) {
        const float* org = small_org();
        return mk(org[(i * 3 + 0) * kBlockThreads], org[(i * 3 + 1) * kBlockThreads], org[(i * 3 + 2) * kBlockThreads]);
    }
    return xf_point(m, o);
}

__device__ __forceinline__ void cache_origins(const Env& E, V3 o) {
    const int n = E.SS.n < kOrgCache ? E.SS.n : kOrgCache;
    const float4* tab = small_tab();
    float* org = small_org();
    for (int i = 0; i < n; i++) {
        Xf m{tab[i * kSmallStride + 1], tab[i * kSmallStride + 2], tab[i * kSmallStride + 3]};
        V3 o2 = xf_point(m, o);
        org[(i * 3 + 0) * kBlockThreads] = o2.x;
        org[(i * 3 + 1) * kBlockThreads] = o2.y;
        org[(i * 3 + 2) * kBlockThreads] = o2.z;
    }
}

// Ray-vs-bounding-ball pre-test of the small-scene loops: true when the LINE o + t d stays clear of the primitive's
// world-space ball {centre, radius} grown by `pad_rate * |centre - o|^2` (SmallPrim::ball / bound.w) — then the
// reference's intersection test reports no hit either, with any sign of t (its f32 error, which for a far, small
// object grows with the squared distance over the radius, is inside the padding), and the exact test is skipped.
// ~14 instructions against ~90 for a sphere and ~250 for a cylinder or cone.  NaN ball (planes, CSG): never true.
__device__ __forceinline__ bool ball_missed(float4 ball, float pad_rate, V3 o, V3 d) {
    const float wx = ball.x - o.x, wy = ball.y - o.y, wz = ball.z - o.z;
    const float ww = fma_(wx, wx, fma_(wy, wy, wz * wz));
    const float wd = fma_(wx, d.x, fma_(wy, d.y, wz * d.z));
    const float dd = fma_(d.x, d.x, fma_(d.y, d.y, d.z * d.z));
    const float R = fma_(pad_rate, ww, ball.w);
    // squared distance of the centre from the line, times |d|^2, against the squared radius times |d|^2 (0.1 % margin)
    return fma_(ww, dd, -(wd * wd)) > R * R * dd * 1.001f;
}

// One item of a small scene of any kind (primitive or CSG root), honouring the cull chain: the general form
// (out of line: cylinders, cones, triangles and CSG roots are the rare members of small scenes).
template <bool STATS>
__device__ __noinline__ void test_small(const Env& E, int i, bool cached, V3 o, V3 d, Hit& best, Ctr<STATS>& k) {
    const float4* tab = small_tab();
    const int4 head = *reinterpret_cast<const int4*>(tab + i * kSmallStride);
    const int type = head.x & 15;
    if (type == T_CSG) {
        if (((head.x >> 4) & kFlagHasParent) && !ancestors_pass(E.S, head.y, o, d)) return;  // RTC_OPT_EXACT_GROUPS
        if constexpr (kWithCsgSweep) {
            if (E.S.csg_ops[head.z].pad < 0) {  // marked at commit: beyond csg_eval's limits
                csg_sweep_nearest<STATS>(E.S, head.z, o, d, best, k);
                return;
            }
        }
        float ht[kCsgHitCap];
        int hp[kCsgHitCap];
        int n = csg_eval<STATS>(E.S, head.z, o, d, ht, hp, k);
        for (int j = 0; j < n; j++) {
            if (ht[j] >= 0.0f) {
                consider(best, ht[j], hp[j], __ldg(&E.S.head[hp[j]]).w);
                break;
            }
        }
        return;
    }
    Xf m{tab[i * kSmallStride + 1], tab[i * kSmallStride + 2], tab[i * kSmallStride + 3]};
    V3 o2 = cached ? small_origin(true, i, m, o) : xf_point(m, o);
    V3 d2 = xf_vec(m, d);
    k.xform();
    k.prim(type);
    float tn = nearest_t(E.S, type, head.z, tab[i * kSmallStride + 4], o2, d2);
    if (((head.x >> 4) & kFlagHasParent) && tn >= 0.0f && would_win(best, tn, head.w) && !ancestors_pass(E.S, head.y, o, d)) return;
    consider(best, tn, i, head.w);
}

// Nearest hit among the items [begin, ends.w) of a small scene, which are runs of spheres, planes, cubes and
// "everything else" ending at ends.x / .y / .z / .w: one tight loop per kind, no per-item dispatch.
// ANY: return true as soon as some item is hit in [0, best.t) (shadow rays when every object casts a shadow).
// LEAN: the lean kernel build (render_tiles), for scenes the commit marked SmallScene::lean — no "everything else" run.
template <bool STATS, bool LEAN>
__device__ __forceinline__ bool scan_small_impl(const Env& E, bool cached, const bool any, int begin, int4 ends, V3 o, V3 d, Hit& best,
                                                Ctr<STATS>& k) {
    const float4* tab = small_tab();
    int i = begin;
#pragma unroll 1
    for (; i < ends.x; i++) {  // spheres — sphere.rs:47-70
        if (ball_missed(tab[i * kSmallStride + 5], tab[i * kSmallStride + 4].w, o, d)) continue;
        Xf m{tab[i * kSmallStride + 1], tab[i * kSmallStride + 2], tab[i * kSmallStride + 3]};
        V3 o2 = small_origin(cached, i, m, o);
        V3 d2 = xf_vec(m, d);
        k.xform();
        k.prim(T_SPHERE);
        float t = nearest_t(E.S, T_SPHERE, 0, make_float4(0.f, 0.f, 0.f, 0.f), o2, d2);
        if (any && t >= 0.0f && t < best.t) return true;
        consider(best, t, i, __float_as_int(tab[i * kSmallStride].w));
    }
#pragma unroll 1
    for (; i < ends.y; i++) {  // planes — plane.rs:45-56 only reads the y components of the object-space ray
        float4 r1 = tab[i * kSmallStride + 2];
        float oy;
        if (cached && i < kOrgCache)
            oy = small_org()[(i * 3 + 1) * kBlockThreads];
        else
            oy = r1.x * o.x + r1.y * o.y + r1.z * o.z + r1.w;
        float dy = r1.x * d.x + r1.y * d.y + r1.z * d.z;
        k.xform();
        k.prim(T_PLANE);
        float t = (fabsf(dy) < kAcne) ? -1.0f : -oy / dy;
        if (any && t >= 0.0f && t < best.t) return true;
        consider(best, t, i, __float_as_int(tab[i * kSmallStride].w));
    }
#pragma unroll 1
    for (; i < ends.z; i++) {  // cubes — cube.rs:55-63
        if (ball_missed(tab[i * kSmallStride + 5], tab[i * kSmallStride + 4].w, o, d)) continue;
        Xf m{tab[i * kSmallStride + 1], tab[i * kSmallStride + 2], tab[i * kSmallStride + 3]};
        V3 o2 = small_origin(cached, i, m, o);
        V3 d2 = xf_vec(m, d);
        k.xform();
        k.prim(T_CUBE);
        float t = nearest_t(E.S, T_CUBE, 0, make_float4(0.f, 0.f, 0.f, 0.f), o2, d2);
        if (any && t >= 0.0f && t < best.t) return true;
        consider(best, t, i, __float_as_int(tab[i * kSmallStride].w));
    }
#pragma unroll 1
    for (; !LEAN && i < ends.w; i++) {  // cylinders, cones, triangles, CSG roots
        if (ball_missed(tab[i * kSmallStride + 5], tab[i * kSmallStride + 4].w, o, d)) continue;
        const int before = best.pos;
        test_small<STATS>(E, i, cached, o, d, best, k);
        if (any && best.pos != before) return true;
    }
    return false;
}
#ifdef RTC_SHARED_SCAN
// One out-of-line copy of the four loops for every caller (nearest hit, both shadow passes); `any` at run time.
template <bool STATS, bool LEAN>
__device__ __noinline__ Hit scan_small_shared(const Env& E, bool cached, bool any, int begin, int4 ends, V3 o, V3 d, Hit best, Ctr<STATS>& k) {
    if (scan_small_impl<STATS, LEAN>(E, cached, any, begin, ends, o, d, best, k)) best.pos = -2;  // any: found
    return best;
}
template <bool STATS, bool ANY, bool LEAN = false>
__device__ __forceinline__ bool scan_small(const Env& E, bool cached, int begin, int4 ends, V3 o, V3 d, Hit& best, Ctr<STATS>& k) {
    best = scan_small_shared<STATS, LEAN>(E, cached, ANY, begin, ends, o, d, best, k);
    if (ANY && best.pos == -2) {
        best.pos = -1;
        return true;
    }
    return false;
}
#else
template <bool STATS, bool ANY, bool LEAN = false>
__device__ __forceinline__ bool scan_small(const Env& E, bool cached, int begin, int4 ends, V3 o, V3 d, Hit& best, Ctr<STATS>& k) {
    return scan_small_impl<STATS, LEAN>(E, cached, ANY, begin, ends, o, d, best, k);
}
#endif

// World::intersect + Intersection::hit for the nearest hit, general (BVH) or small-scene form.
template <bool STATS, bool SMALL, bool LEAN = false>
__device__ __forceinline__ void find_hit(const Env& E, V3 o, V3 d, Hit& best, Ctr<STATS>& k) {
    if (SMALL) {
        const SmallScene& SS = E.SS;
        if (!LEAN && SS.has_cull_chain) {
#pragma unroll 1
            for (int i = 0; i < SS.n; i++) test_small<STATS>(E, i, false, o, d, best, k);
        } else {
            int begin = 0;
            int4 ends = SS.caster_end;
#pragma unroll 1
            for (int seg = 0; seg < 2; seg++) {  // casters, then non-casters: one copy of the loops
                scan_small<STATS, false, LEAN>(E, false, begin, ends, o, d, best, k);
                begin = ends.w;
                ends = SS.other_end;
            }
        }
    } else {
        nearest_hit<STATS, false>(E.S, o, d, best, k);
    }
}

}  // namespace RTC_NS
}  // namespace rtc
