// dev_bvh.cuh — nearest hit through the BVH (while-while), CSG programs, cull chains, the n1 / n2 container walk.
// Part of rtc_device.cuh (include that, not this): compiled once per kernel build inside namespace rtc::RTC_NS.
#pragma once

namespace rtc {
namespace RTC_NS {

// ---------------------------------------------------------------------------------------------------
// Nearest hit so far.  `order` is the primitive's depth-first index: the reference's tie-break (Q8).
struct Hit {
    float t;
    int pos;
    int order;
};
__device__ __forceinline__ void consider(Hit& best, float t, int pos, int order) {
    const bool better = t >= 0.0f && (t < best.t || (t == best.t && order < best.order));
    best.t = better ? t : best.t;
    best.pos = better ? pos : best.pos;
    best.order = better ? order : best.order;
}
// A candidate with t >= 0 that consider() would take.  The cull-chain walk runs only for such a candidate: one that loses
// leaves `best` as it was whether its chain passes or not.
__device__ __forceinline__ bool would_win(const Hit& best, float t, int order) {
    return t < best.t || (t == best.t && order < best.order);
}

// The world ray as seen by the primitive being tested; cached by transform id so that a mesh whose
// triangles share one transform pays for one ray transform per traversal, not one per triangle.
struct ObjRay {
    int xf_id = -1;
    V3 o, d;
};

// Every enclosing GroupShape culls with the forward ray (group.rs:119-125); the walk stops at a CSG because
// CSG subtrees are evaluated whole by csg_eval.
__device__ __noinline__ bool ancestors_pass(const DevScene& S, int node, V3 o, V3 d) {
    while (node >= 0) {
        const DevNode& n = S.nodes[node];
        float lo, hi;
        if (!aabb_ref(o, d, ld3(n.bmin), ld3(n.bmax), lo, hi)) return false;
        node = n.parent;
    }
    return true;
}

// The one-box certificate for a hit at distance t >= 0 of a primitive whose innermost group is `node`: true only when
// ancestors_pass would be true.  The hit point o + t d lies inside the node's box by the margin 2^-21 (max(|mn|, |mx|) +
// |o| + |p|) + 2^-100 on every axis, and every ancestor's box contains its child's (DevNode::pad, set at commit), so the
// reference's aabb_intersection of each box of the chain brackets t on every axis (DESIGN.md §4, "Exact group culls: the
// certificate's margin").  A direction component below 2^-60, an infinite bound, a non-finite point or an unmarked node
// never certifies: the chain is then walked.
__device__ __forceinline__ bool axis_certified(float mn, float mx, float o, float d, float t) {
    const float p = o + t * d;
    const float m = 4.76837158203125e-07f * (fmaxf(fabsf(mn), fabsf(mx)) + fabsf(o) + fabsf(p)) + 7.888609052210118e-31f;
    return fabsf(d) >= 8.673617379884035e-19f && m <= 1e30f && mn + m <= p && p + m <= mx;
}
__device__ __forceinline__ bool chain_certified(const DevScene& S, int node, V3 o, V3 d, float t) {
    const DevNode& n = S.nodes[node];
    return n.pad == 1 && axis_certified(n.bmin[0], n.bmax[0], o.x, d.x, t) && axis_certified(n.bmin[1], n.bmax[1], o.y, d.y, t) &&
           axis_certified(n.bmin[2], n.bmax[2], o.z, d.z, t);
}

// CSG::local_intersect (csg.rs:87-104) for a whole CSG subtree, flattened at commit time into a post-order
// instruction list.  ht/hp receive the filtered hits (distance, primitive position) in the reference's
// sorted order; returns their count.
template <bool STATS>
__device__ __noinline__ int csg_eval(const DevScene& S, int pc, V3 wo, V3 wd, float* ht, int* hp, Ctr<STATS>& k) {
    V3 ro[kCsgRayDepth], rd[kCsgRayDepth];
    int s_mark[kCsgRayDepth], m_mark[kCsgRayDepth];
    int rsp = 0, n = 0;
    ro[0] = wo;
    rd[0] = wd;
    k.prim(T_CSG);
    const int end = S.csg_ops[pc].skip;  // the root's ENTER skips to one past its EXIT
    while (pc < end) {
        DevCsgOp op = S.csg_ops[pc];
        switch (op.op) {
            case OP_CSG_ENTER: {
                const DevNode& nd = S.nodes[op.arg];
                Xf m{nd.inv[0], nd.inv[1], nd.inv[2]};
                V3 o2 = xf_point(m, ro[rsp]), d2 = xf_vec(m, rd[rsp]);  // shape.rs:60-70 on the CSG itself
                k.xform();
                float lo, hi;
                k.node();
                if (!aabb_ref(o2, d2, ld3(nd.bmin), ld3(nd.bmax), lo, hi)) {  // csg.rs:90-93
                    pc = op.skip;
                    break;
                }
                rsp++;
                ro[rsp] = o2;
                rd[rsp] = d2;
                s_mark[rsp] = n;
                pc++;
                break;
            }
            case OP_CSG_MID:
                m_mark[rsp] = n;
                pc++;
                break;
            case OP_CSG_EXIT: {
                const int s = s_mark[rsp], m = m_mark[rsp], e = n;
                const int csg_op = S.nodes[op.arg].op;
                for (int i = s; i < m; i++) hp[i] |= 0x40000000;  // came from s1 (csg.rs:46 `s1.includes`)
                for (int i = s + 1; i < e; i++) {                 // stable insertion sort by distance (csg.rs:101)
                    float ti = ht[i];
                    int pi = hp[i];
                    int j = i - 1;
                    while (j >= s && ht[j] > ti) {
                        ht[j + 1] = ht[j];
                        hp[j + 1] = hp[j];
                        j--;
                    }
                    ht[j + 1] = ti;
                    hp[j + 1] = pi;
                }
                bool in1 = false, in2 = false;  // csg.rs:37-58
                int w = s;
                for (int i = s; i < e; i++) {
                    bool hit1 = (hp[i] & 0x40000000) != 0;
                    bool allowed;
                    if (csg_op == 0)
                        allowed = (hit1 && !in2) || (!hit1 && !in1);
                    else if (csg_op == 1)
                        allowed = (hit1 && in2) || (!hit1 && in1);
                    else
                        allowed = (hit1 && !in2) || (!hit1 && in1);
                    if (allowed) {
                        ht[w] = ht[i];
                        hp[w] = hp[i] & 0x3fffffff;
                        w++;
                    }
                    if (hit1)
                        in1 = !in1;
                    else
                        in2 = !in2;
                }
                n = w;
                rsp--;
                pc++;
                break;
            }
            case OP_GROUP: {
                const DevNode& nd = S.nodes[op.arg];
                float lo, hi;
                k.node();
                if (!aabb_ref(ro[rsp], rd[rsp], ld3(nd.bmin), ld3(nd.bmax), lo, hi))  // group.rs:122-125
                    pc = op.skip;
                else
                    pc++;
                break;
            }
            default: {  // OP_PRIM
                int4 h = __ldg(&S.head[op.arg]);
                Xf m = load_xf(S.xform + 3 * (size_t)h.y);
                V3 o2 = xf_point(m, ro[rsp]), d2 = xf_vec(m, rd[rsp]);
                k.xform();
                float t[4];
                int type = h.x & 15;
                k.prim(type);
                int c = local_intersect(S, type, h.z, load_bound(S, type, h.z), o2, d2, t);
                for (int i = 0; i < c; i++) {
                    if (n < kCsgHitCap) {
                        ht[n] = t[i];
                        hp[n] = op.arg;
                        n++;
                    } else {
                        k.overflow();
                    }
                }
                pc++;
                break;
            }
        }
    }
    return n;
}

// ---------------------------------------------------------------------------------------------------
// csg_sweep's call sites are compiled into the kernel builds for scenes that hold a CSG marked for it
// (RTC_CSG_SWEEP_BUILD, rtc_kernels.cu) and into host builds of this code; every other kernel build is exactly the
// csg_eval-only code, so the sweep costs the scenes that do not use it no registers.
#if defined(RTC_CSG_SWEEP_BUILD) || !defined(__CUDA_ARCH__)
constexpr bool kWithCsgSweep = true;
#else
constexpr bool kWithCsgSweep = false;
#endif

// csg_sweep: the same filtered hit list as csg_eval, in the same order, delivered one hit at a time in memory that does
// not depend on the size of the tree (CSGs beyond csg_eval's limits, marked at commit: rtc_types.h, DevCsgOp::pad).
//
// Order.  csg.rs:101 stable-sorts at every CSG and groups concatenate, so a CSG's filtered list is ordered by the key
// (t, position of the leaf's PRIM instruction, index of the hit in the leaf's local_intersect output): key = t and
// (PRIM position << 2 | index).  t compares as a float (-0 == +0: the tie goes to the rest of the key).
// Pass.  Walk the program as csg_eval does (same ENTER transforms and box culls, same GROUP culls, same PRIM arithmetic)
// and keep the kCsgSweepPass (= kCsgHitCap) smallest leaf hits whose key is above a cursor, sorted.
// Filter by climbing.  Each buffered hit, in order, climbs its chain of CSG ancestors: at each it is tested with
// intersection_allowed (csg.rs:63-74) against that CSG's in_s1 / in_s2, then the flag of the side it came from toggles
// (csg.rs:37-58); it stops at the first CSG that does not allow it.  A hit that clears the root is the next output.
// Every CSG thereby sees its operands' outputs merged in key order, which is what the stable sort gives it.
// Repeat from the last key of the pass until the consumer stops or no hit is left.  The cursor moves strictly forward
// (keys are distinct), so every ray ends.  A NaN distance is above no cursor: such a hit is never buffered and never
// delivered (the reference cannot order it either: its sort panics), where csg_eval would keep it in some position.
// Hits per pass: kCsgHitCap (a smaller figure is a test aid: every ray then takes several passes).
#ifndef RTC_CSG_SWEEP_PASS
#define RTC_CSG_SWEEP_PASS kCsgHitCap
#endif
constexpr int kCsgSweepPass = RTC_CSG_SWEEP_PASS;
static_assert(kCsgSweepPass >= 1 && kCsgSweepPass <= kCsgHitCap, "csg_sweep: 1 .. kCsgHitCap hits per pass");
__device__ __forceinline__ bool csg_key_less(float ta, int ka, float tb, int kb) { return ta < tb || (ta == tb && ka < kb); }

// One pass: the up to kCsgSweepPass smallest leaf hits above the cursor {bt, bk}[kCsgSweepPass] into bt / bk, sorted;
// returns the count.  ro[0] / rd[0] hold the world ray.  The world ray and the cursor are read from local memory rather
// than held in registers through the walk: that keeps the sweep's register footprint, which every caller of
// test_prim_other, test_small and container_csg in the sweep builds makes room for, near csg_eval's.
template <bool STATS>
__device__ __forceinline__ int csg_sweep_pass(const DevScene& S, int root, V3* ro, V3* rd, float* bt, int* bk, Ctr<STATS>& k) {
    int rsp = 0, n = 0, pc = root;
    k.prim(T_CSG);
    const int end = S.csg_ops[root].skip;
#pragma unroll 1
    while (pc < end) {
        DevCsgOp op = S.csg_ops[pc];
        switch (op.op) {
            case OP_CSG_ENTER: {
                const DevNode& nd = S.nodes[op.arg];
                Xf m{nd.inv[0], nd.inv[1], nd.inv[2]};
                V3 o2 = xf_point(m, ro[rsp]), d2 = xf_vec(m, rd[rsp]);  // shape.rs:60-70 on the CSG itself
                k.xform();
                float lo, hi;
                k.node();
                if (!aabb_ref(o2, d2, ld3(nd.bmin), ld3(nd.bmax), lo, hi)) {  // csg.rs:90-93
                    pc = op.skip;
                    break;
                }
                rsp++;
                ro[rsp] = o2;
                rd[rsp] = d2;
                pc++;
                break;
            }
            case OP_CSG_MID:
                pc++;
                break;
            case OP_CSG_EXIT:
                rsp--;
                pc++;
                break;
            case OP_GROUP: {
                const DevNode& nd = S.nodes[op.arg];
                float lo, hi;
                k.node();
                if (!aabb_ref(ro[rsp], rd[rsp], ld3(nd.bmin), ld3(nd.bmax), lo, hi))  // group.rs:122-125
                    pc = op.skip;
                else
                    pc++;
                break;
            }
            default: {  // OP_PRIM
                int4 h = __ldg(&S.head[op.arg]);
                Xf m = load_xf(S.xform + 3 * (size_t)h.y);
                V3 o2 = xf_point(m, ro[rsp]), d2 = xf_vec(m, rd[rsp]);
                k.xform();
                float t[4];
                int type = h.x & 15;
                k.prim(type);
                int c = local_intersect(S, type, h.z, load_bound(S, type, h.z), o2, d2, t);
#pragma unroll 1
                for (int i = 0; i < c; i++) {
                    const float ti = t[i];
                    const int ki = (pc << 2) | i;
                    const float ct = *(volatile float*)&bt[kCsgSweepPass];
                    const int ck = *(volatile int*)&bk[kCsgSweepPass];
                    if (!csg_key_less(ct, ck, ti, ki)) continue;  // not above the cursor (or NaN)
                    if (n == kCsgSweepPass && !csg_key_less(ti, ki, bt[n - 1], bk[n - 1])) continue;
                    int j = n < kCsgSweepPass ? n++ : n - 1;  // a full buffer drops its largest key
                    while (j > 0 && csg_key_less(ti, ki, bt[j - 1], bk[j - 1])) {
                        bt[j] = bt[j - 1];
                        bk[j] = bk[j - 1];
                        j--;
                    }
                    bt[j] = ti;
                    bk[j] = ki;
                }
                pc++;
                break;
            }
        }
    }
    return n;
}

// The sweep driver.  Both consumers stop at the first output hit with t >= 0 (nearest hit: it is the answer; container
// walk: the hits before it are the ones behind the origin), so the driver returns that hit in t_out / pos_out (pos_out
// -1: none).  NEG: the output hits with t < 0 are compacted, in order, into bt / bk (distance, primitive position) and
// handed to neg(bt, bk, m) after each pass's climb, so the consumer's state is not live through the climb.
template <bool STATS, bool NEG, class Neg>
__device__ __forceinline__ void csg_sweep(const DevScene& S, int root, V3 wo, V3 wd, Neg& neg, float& t_out, int& pos_out,
                                          Ctr<STATS>& k) {
    float bt[kCsgSweepPass + 1];  // [kCsgSweepPass]: the cursor
    int bk[kCsgSweepPass + 1];
    V3 ro[kCsgSweepDepth], rd[kCsgSweepDepth];
    ro[0] = wo;
    rd[0] = wd;
    unsigned state[2 * kCsgSweepNodes / 32];  // in_s1 / in_s2 of CSG node s: bits 2 s and 2 s + 1
    const int words = (2 * -S.csg_ops[root].pad + 31) / 32;  // the root ENTER's pad: -(CSG nodes of the program)
#pragma unroll 1
    for (int w = 0; w < words; w++) state[w] = 0u;
    bt[kCsgSweepPass] = -kInfF;
    bk[kCsgSweepPass] = -1;  // below every key: the first pass takes every hit that is not NaN
    pos_out = -1;
#pragma unroll 1
    for (;;) {
        const int n = csg_sweep_pass<STATS>(S, root, ro, rd, bt, bk, k);
        if (n == 0) return;
        bt[kCsgSweepPass] = bt[n - 1];  // the next pass starts above this one's last key
        bk[kCsgSweepPass] = bk[n - 1];
        int m = 0;
#pragma unroll 1
        for (int j = 0; j < n && pos_out < 0; j++) {
            const DevCsgOp leaf = S.csg_ops[bk[j] >> 2];
            int e = root + (leaf.pad >> 1);
            bool left = leaf.pad & 1;
#pragma unroll 1
            for (;;) {
                const DevCsgOp enter = S.csg_ops[e];
                const int sidx = S.csg_ops[enter.skip - 1].pad >> 1;
                const unsigned word = state[sidx >> 4];
                const int shift = 2 * (sidx & 15);
                const bool in1 = (word >> shift) & 1u, in2 = (word >> (shift + 1)) & 1u;
                const int csg_op = S.nodes[enter.arg].op;
                bool allowed;  // csg.rs:63-74
                if (csg_op == 0)
                    allowed = (left && !in2) || (!left && !in1);
                else if (csg_op == 1)
                    allowed = (left && in2) || (!left && in1);
                else
                    allowed = (left && !in2) || (!left && in1);
                state[sidx >> 4] = word ^ (1u << (shift + (left ? 0 : 1)));
                if (!allowed) break;
                if (e == root) {  // an output hit
                    if (bt[j] >= 0.0f) {
                        t_out = bt[j];
                        pos_out = leaf.arg;
                    } else if (NEG) {
                        bt[m] = bt[j];  // m <= j: the keys still to climb are untouched
                        bk[m] = leaf.arg;
                        m++;
                    }
                    break;
                }
                left = S.csg_ops[enter.skip - 1].pad & 1;
                e = root + enter.pad;
            }
        }
        if (NEG) neg(bt, bk, m);
        if (pos_out >= 0 || n < kCsgSweepPass) return;
    }
}

// csg_sweep's consumers.  Nearest hit: the first output hit with t >= 0.  Inlined into test_prim_other and test_small,
// which costs their callers fewer registers than one more level of call.
struct CsgSweepNoNeg {
    __device__ __forceinline__ void operator()(const float*, const int*, int) {}
};
template <bool STATS>
__device__ __forceinline__ void csg_sweep_nearest(const DevScene& S, int pc, V3 o, V3 d, Hit& best, Ctr<STATS>& k) {
    CsgSweepNoNeg none;
    float t;
    int pos;
    csg_sweep<STATS, false>(S, pc, o, d, none, t, pos, k);
    if (pos >= 0) consider(best, t, pos, __ldg(&S.head[pos]).w);
}

// Marks a capacity overflow of csg_sweep in the render's DevCounters::overflows, in every kernel build: the render then
// fails with RTC_ERR_CAPACITY rather than being silently wrong.  A plain store, not an atomic: any nonzero value fails
// the render (the counters are zeroed before each one), and an atomic here costs every caller of the container walk
// registers.
__device__ __forceinline__ void flag_csg_overflow(const DevScene& S) {
#ifdef __CUDA_ARCH__
    *S.csg_overflows = 1ull;
#else
    if (S.csg_overflows) *S.csg_overflows = 1ull;
#endif
}

// Test one stored primitive against the world ray for the nearest-hit search: test_prim, below, does a mesh triangle
// itself and sends the rest here.
// Everything but a mesh triangle: CSG trees and the analytic shapes.  Out of line: the traversal loop then holds only
// the slab tests and the triangle test, which is what keeps it inside the instruction cache (profiles/README.md).
template <bool STATS>
__device__ __noinline__ void test_prim_other(const DevScene& S, int pos, int4 h, V3 o, V3 d, Hit& best, Ctr<STATS>& k) {
    const float4* rec = S.rec + 4 * (size_t)pos;
    int type = h.x & 15;
    if (type == T_CSG) {
        // a CSG inside groups (RTC_OPT_EXACT_GROUPS): the enclosing groups cull before it is evaluated (group.rs:122-125)
        if (((h.x >> 4) & kFlagHasParent) && !ancestors_pass(S, __ldg(&S.head[pos + S.n_prims]).x, o, d)) return;
        if constexpr (kWithCsgSweep) {
            if (S.csg_ops[h.z].pad < 0) {  // marked at commit: beyond csg_eval's limits
                csg_sweep_nearest<STATS>(S, h.z, o, d, best, k);
                return;
            }
        }
        float ht[kCsgHitCap];
        int hp[kCsgHitCap];
        int n = csg_eval<STATS>(S, h.z, o, d, ht, hp, k);
        for (int i = 0; i < n; i++) {
            if (ht[i] >= 0.0f) {
                consider(best, ht[i], hp[i], __ldg(&S.head[hp[i]]).w);
                break;  // the list is sorted: the first non-negative entry is this CSG's nearest
            }
        }
        return;
    }
    k.prim(type);
    Xf m = load_xf(rec + 1);  // the primitive's own inverse transform travels in its record
    k.xform();
    float tn = nearest_t(S, type, h.z, load_bound(S, type, h.z), xf_point(m, o), xf_vec(m, d));
    if (!(tn >= 0.0f)) return;
    if (((h.x >> 4) & kFlagHasParent) && would_win(best, tn, h.w)) {
        const int parent = __ldg(&S.head[pos + S.n_prims]).x;
        if (!chain_certified(S, parent, o, d, tn) && !ancestors_pass(S, parent, o, d)) return;
    }
    consider(best, tn, pos, h.w);
}

template <bool STATS>
__device__ __forceinline__ void test_prim(const DevScene& S, int pos, V3 o, V3 d, ObjRay& cache, Hit& best, Ctr<STATS>& k) {
    const float4* rec = S.rec + 4 * (size_t)pos;
    int4 h = __ldg(reinterpret_cast<const int4*>(rec));
    if ((h.x & 15) != T_TRIANGLE) {
        test_prim_other<STATS>(S, pos, h, o, d, best, k);
        return;
    }
    k.prim(T_TRIANGLE);
    // a mesh's triangles share one transform: the object-space ray is kept across primitives (shape.rs:60-70)
    if (h.y != cache.xf_id) {
        Xf m = load_xf(S.xform + 3 * (size_t)h.y);
        cache.o = xf_point(m, o);
        cache.d = xf_vec(m, d);
        cache.xf_id = h.y;
        k.xform();
    }
    float tn = nearest_t(S, T_TRIANGLE, h.z, make_float4(0.f, 0.f, 0.f, 0.f), cache.o, cache.d, rec + 1);
    if (!(tn >= 0.0f)) return;
    if (((h.x >> 4) & kFlagHasParent) && would_win(best, tn, h.w)) {
        const int parent = __ldg(&S.head[pos + S.n_prims]).x;
        if (!chain_certified(S, parent, o, d, tn) && !ancestors_pass(S, parent, o, d)) return;
    }
    consider(best, tn, pos, h.w);
}

// Conservative slab test for the acceleration structure (boxes are padded at build time, so this never rejects a
// primitive the reference would have hit; it is not part of the reference's semantics).  The distances are formed as
// fma(plane, 1 / d, -(o / d)) — one FFMA per plane instead of a subtraction and a product, in both kernel builds; the two
// product roundings are at most 2^-22 of the scene's extent in length, which the builder's padding includes
// (rtc_commit.cu).  A direction component below 2^-60 in magnitude is replaced by +-2^-60 first (tree_inverse): its
// reciprocal stays finite, so no inf - inf = NaN can appear — a ray parallel to a slab gets distances of +-1e18 with the
// right signs: inside the slab no constraint, outside a miss (and it is the padded box the ray has to clear).
__device__ __forceinline__ bool slab(V3 noi, V3 inv, float lx, float ly, float lz, float hx, float hy, float hz, float tmax,
                                     float& tnear) {
    float a = fma_(lx, inv.x, noi.x), b = fma_(hx, inv.x, noi.x);
    float lo = fminf(a, b), hi = fmaxf(a, b);
    a = fma_(ly, inv.y, noi.y), b = fma_(hy, inv.y, noi.y);
    lo = fmaxf(lo, fminf(a, b));
    hi = fminf(hi, fmaxf(a, b));
    a = fma_(lz, inv.z, noi.z), b = fma_(hz, inv.z, noi.z);
    lo = fmaxf(lo, fminf(a, b));
    hi = fminf(hi, fmaxf(a, b));
    tnear = lo;
    return hi >= fmaxf(lo, 0.0f) && lo <= tmax;
}

__device__ __forceinline__ float tree_inverse(float d) {
    const float tiny = 8.673617379884035e-19f;  // 2^-60
    return 1.0f / (fabsf(d) < tiny ? copysignf(tiny, d) : d);
}

// World::intersect + Intersection::hit (world.rs:52-60, intersection.rs:30-35): nearest t >= 0 with the
// depth-first tie-break, searched through the BVH.  `best.t` on entry is the search limit (exclusive).
// ANY: stop at the first hit (shadow rays when every primitive casts a shadow).
template <bool STATS, bool ANY>
__device__ __noinline__ void nearest_hit(const DevScene& S, V3 o, V3 d, Hit& best, Ctr<STATS>& k) {
    ObjRay cache;
#pragma unroll 1
    for (int i = 0; i < S.n_linear; i++) {
        test_prim<STATS>(S, __ldg(&S.linear[i]), o, d, cache, best, k);
        if (ANY && best.pos >= 0) return;
    }
    if (S.bvh_root < 0) return;
    const V3 inv = mk(tree_inverse(d.x), tree_inverse(d.y), tree_inverse(d.z));
    const V3 noi = mk(-(o.x * inv.x), -(o.y * inv.y), -(o.z * inv.z));
    int stack[kBvhStack];
    int sp = 0;
    int node = S.bvh_root;
    // "while-while" traversal: every lane first descends to its next leaf (lanes that are there already wait), then
    // all lanes test their leaf's primitives together — instead of serialising an inner-node step for some lanes with
    // a leaf for the others in every iteration (ncu: 4.5 of 32 lanes active in the primitive tests before).
    constexpr int kDone = -0x7fffffff - 1;  // never a leaf code: ~((first << 4) | (count - 1)) > INT_MIN
    for (;;) {
        while (node >= 0) {
            const float4* np = reinterpret_cast<const float4*>(S.bvh + node);
            float4 a = __ldg(np), b = __ldg(np + 1), c = __ldg(np + 2);
            int4 link = __ldg(reinterpret_cast<const int4*>(np + 3));
            float t0, t1;
            k.node();
            k.node();
            bool h0 = slab(noi, inv, a.x, a.y, a.z, a.w, b.x, b.y, best.t, t0);
            bool h1 = slab(noi, inv, b.z, b.w, c.x, c.y, c.z, c.w, best.t, t1);
            if (h0 && h1) {
                int near = link.x, far = link.y;
                if (t1 < t0) {
                    near = link.y;
                    far = link.x;
                }
                if (sp < kBvhStack) stack[sp++] = far;
                node = near;
            } else if (h0) {
                node = link.x;
            } else if (h1) {
                node = link.y;
            } else {
                node = sp == 0 ? kDone : stack[--sp];
            }
        }
        if (node == kDone) return;
        {
            int code = ~node;
            int first = code >> 4, count = (code & 15) + 1;
            for (int i = 0; i < count; i++) {
                test_prim<STATS>(S, first + i, o, d, cache, best, k);
                if (ANY && best.pos >= 0) return;
            }
        }
        if (sp == 0) return;
        node = stack[--sp];
    }
}

// ---------------------------------------------------------------------------------------------------
// n1 / n2 (world.rs:235-263) without materialising the sorted list (SURVEY Appendix F2).  In the render
// path the hit is the first t >= 0 entry, so the containers are decided by the NEGATIVE-t intersections:
// an object is open when it has an odd number of them, and the open object whose last negative hit is
// latest in the sorted order (t, then depth-first order) is the innermost one.
struct Containers {
    float best_t = -kInfF;  // innermost open object other than the hit object
    int best_order = -1;
    int best_pos = -1;
    bool hit_open = false;  // the hit object itself is open (we are leaving it)
    float hit_t = -kInfF;
    int hit_order = -1;
};
__device__ __forceinline__ void container_add(Containers& c, int hit_pos, float t_last, int pos, int order) {
    if (pos == hit_pos) {
        c.hit_open = true;
        c.hit_t = t_last;
        c.hit_order = order;
    } else if (t_last > c.best_t || (t_last == c.best_t && order > c.best_order)) {
        c.best_t = t_last;
        c.best_order = order;
        c.best_pos = pos;
    }
}
// container_csg's parity and last negative hit per leaf, from csg_sweep's output hits with t < 0: a plane or triangle has
// one hit, so an output hit opens it for good and goes to container_add directly; the other leaves toggle in and out of
// a list of the open ones, which holds their latest hit.  More than kCsgHitCap solids of one CSG open at once along the
// backward ray is an overflow: counted, so the render fails.
struct CsgSweepOpen {
    const DevScene& S;
    Containers& c;
    int hit_pos;
    int n = 0;
    int pos[kCsgHitCap];
    float last[kCsgHitCap];
    __device__ __forceinline__ void operator()(const float* ht, const int* hp, int m) {
#pragma unroll 1
        for (int i = 0; i < m; i++) {
            const int p = hp[i];
            const int4 h = __ldg(&S.head[p]);
            const int type = h.x & 15;
            if (type == T_PLANE || type == T_TRIANGLE) {
                container_add(c, hit_pos, ht[i], p, h.w);
                continue;
            }
            int j = 0;
#pragma unroll 1
            while (j < n && pos[j] != p) j++;
            if (j < n) {  // an even count: closed again
                n--;
                pos[j] = pos[n];
                last[j] = last[n];
            } else if (n < kCsgHitCap) {
                pos[n] = p;
                last[n] = ht[i];
                n++;
            } else {
                flag_csg_overflow(S);
            }
        }
    }
};
template <bool STATS>
__device__ __noinline__ void csg_sweep_containers(const DevScene& S, int pc, V3 o, V3 d, int hit_pos, Containers& c, Ctr<STATS>& k) {
    CsgSweepOpen open{S, c, hit_pos};
    float t;
    int pos;
    csg_sweep<STATS, true>(S, pc, o, d, open, t, pos, k);
#pragma unroll 1
    for (int j = 0; j < open.n; j++) container_add(c, hit_pos, open.last[j], open.pos[j], __ldg(&S.head[open.pos[j]]).w);
}

// The CSG case of container_prim, out of line (one copy for both of its call sites; rarely taken).
template <bool STATS>
__device__ __noinline__ void container_csg(const DevScene& S, int pc, V3 o, V3 d, int hit_pos, Containers& c, Ctr<STATS>& k) {
    if constexpr (kWithCsgSweep) {
        if (S.csg_ops[pc].pad < 0) {  // marked at commit: beyond csg_eval's limits
            csg_sweep_containers<STATS>(S, pc, o, d, hit_pos, c, k);
            return;
        }
    }
    float ht[kCsgHitCap];
    int hp[kCsgHitCap];
    int n = csg_eval<STATS>(S, pc, o, d, ht, hp, k);
    // per leaf: parity and last negative hit among the filtered hits
#pragma unroll 1
    for (int i = 0; i < n; i++) {
        if (!(ht[i] < 0.0f)) break;
        int p = hp[i];
        bool seen = false;
#pragma unroll 1
        for (int j = 0; j < i; j++) seen |= (hp[j] == p);
        if (seen) continue;
        int cnt = 0;
        float last = 0.f;
#pragma unroll 1
        for (int j = i; j < n && ht[j] < 0.0f; j++)
            if (hp[j] == p) {
                cnt++;
                last = ht[j];
            }
        if (cnt & 1) container_add(c, hit_pos, last, p, __ldg(&S.head[p]).w);
    }
}
template <bool STATS>
__device__ __forceinline__ void container_prim(const DevScene& S, int pos, V3 o, V3 d, ObjRay& cache, int hit_pos, Containers& c,
                                               Ctr<STATS>& k) {
    int4 h = __ldg(&S.head[pos]);
    int type = h.x & 15;
    if (type == T_CSG) {
        if (((h.x >> 4) & kFlagHasParent) && !ancestors_pass(S, __ldg(&S.head[pos + S.n_prims]).x, o, d)) return;
        container_csg<STATS>(S, h.z, o, d, hit_pos, c, k);
        return;
    }
    if (h.y != cache.xf_id) {
        Xf m = load_xf(S.xform + 3 * (size_t)h.y);
        cache.o = xf_point(m, o);
        cache.d = xf_vec(m, d);
        cache.xf_id = h.y;
        k.xform();
    }
    float t[4];
    k.prim(type);
    int n = local_intersect(S, type, h.z, load_bound(S, type, h.z), cache.o, cache.d, t);
    int cnt = 0;
    float last = -kInfF;
    for (int i = 0; i < n; i++)
        if (t[i] < 0.0f) {
            cnt++;
            last = fmaxf(last, t[i]);
        }
    if (!(cnt & 1)) return;
    // a grouped primitive only reports hits when every enclosing group's box passes the forward ray (Q6)
    int parent = __ldg(&S.head[pos + S.n_prims]).x;
    if (parent >= 0 && !ancestors_pass(S, parent, o, d)) return;
    container_add(c, hit_pos, last, pos, h.w);
}
template <bool STATS>
__device__ __noinline__ void find_containers(const DevScene& S, V3 o, V3 d, int hit_pos, float& n1, float& n2, Ctr<STATS>& k) {
    Containers c;
    ObjRay cache;
#pragma unroll 1
    for (int i = 0; i < S.n_linear; i++) container_prim<STATS>(S, __ldg(&S.linear[i]), o, d, cache, hit_pos, c, k);
    if (S.bvh_root >= 0) {
        // walk the backward half-line: the forward half-line of the reversed ray
        const V3 inv = mk(tree_inverse(-d.x), tree_inverse(-d.y), tree_inverse(-d.z));
        const V3 noi = mk(-(o.x * inv.x), -(o.y * inv.y), -(o.z * inv.z));
        int stack[kBvhStack];
        int sp = 0;
        int node = S.bvh_root;
        constexpr int kDone = -0x7fffffff - 1;
        for (;;) {  // while-while, as in nearest_hit
            while (node >= 0) {
                const float4* np = reinterpret_cast<const float4*>(S.bvh + node);
                float4 a = __ldg(np), b = __ldg(np + 1), cc = __ldg(np + 2);
                int4 link = __ldg(reinterpret_cast<const int4*>(np + 3));
                float t0, t1;
                k.node();
                k.node();
                // A sphere or a cube has an odd number of hits behind the origin only when the origin is inside it (both
                // roots of an outside origin have one sign, cube.rs:124-128 rejects a box that is not straddled), and
                // the tree's boxes are padded far beyond f32 rounding: subtrees of such primitives are culled with a
                // point-in-box test instead of the unbounded backward ray (a refraction hit deep in a 100 k-sphere
                // field no longer walks every node along the whole half-line).
                bool h0, h1;
                if (link.z & 1)
                    h0 = o.x >= a.x && o.x <= a.w && o.y >= a.y && o.y <= b.x && o.z >= a.z && o.z <= b.y;
                else
                    h0 = slab(noi, inv, a.x, a.y, a.z, a.w, b.x, b.y, kInfF, t0);
                if (link.z & 2)
                    h1 = o.x >= b.z && o.x <= cc.y && o.y >= b.w && o.y <= cc.z && o.z >= cc.x && o.z <= cc.w;
                else
                    h1 = slab(noi, inv, b.z, b.w, cc.x, cc.y, cc.z, cc.w, kInfF, t1);
                if (h0 && h1) {
                    if (sp < kBvhStack) stack[sp++] = link.y;
                    node = link.x;
                } else if (h0) {
                    node = link.x;
                } else if (h1) {
                    node = link.y;
                } else {
                    node = sp == 0 ? kDone : stack[--sp];
                }
            }
            if (node == kDone) break;
            {
                int code = ~node;
                int first = code >> 4, count = (code & 15) + 1;
#pragma unroll 1
                for (int i = 0; i < count; i++) container_prim<STATS>(S, first + i, o, d, cache, hit_pos, c, k);
            }
            if (sp == 0) break;
            node = stack[--sp];
        }
    }
    auto index_of = [&](int pos) { return S.materials[(__ldg(&S.head[pos]).x >> 8)].refractive_index; };
    float other = (c.best_pos >= 0) ? index_of(c.best_pos) : 1.0f;  // REFRACTION_VACCUM, world.rs:242
    if (c.hit_open) {
        // leaving the hit object: n1 is the innermost open object (possibly the hit object itself)
        bool hit_is_inner = c.best_pos < 0 || c.hit_t > c.best_t || (c.hit_t == c.best_t && c.hit_order > c.best_order);
        n1 = hit_is_inner ? index_of(hit_pos) : other;
        n2 = other;
    } else {
        n1 = other;
        n2 = index_of(hit_pos);
    }
}

}  // namespace RTC_NS
}  // namespace rtc
