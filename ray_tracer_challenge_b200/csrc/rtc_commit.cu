// rtc_commit.cu — the host half of rtc_scene_commit: validation of the flattened scene, binned-SAH BVH over the book's
// bounding boxes (top levels built by several threads), device positions and transform table, CSG programs, traversal
// records, shading tables, and the small-scene table with its shadow-filter plan.  No device calls: rtc_scene_inspect
// runs exactly this on machines without a GPU.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <future>
#include <map>
#include <thread>
#include <tuple>
#include <unordered_map>

#include "rtc_internal.h"

namespace rtc {

namespace {

// ---- binned-SAH BVH over the top-level items -----------------------------------------------------------
struct BuildItem {
    Box box;
    float centroid[3];
    int item;     // index into the bounded item list
    bool closed;  // sphere or cube: it has an odd number of hits behind a ray origin only if the origin is inside it
};
struct Builder {
    RawVector<BuildItem>& items;
    RawVector<DevBvhNode>& nodes;
    int leaf_size;
    // returns the link for the range [b, e): >= 0 inner node, < 0 leaf code
    // The traversal stack holds one deferred child per level (kBvhStack entries, dev_bvh.cuh) and a full stack must
    // never drop a subtree, so the tree's depth is bounded HERE: SAH splits are free to be lopsided only while
    // `depth + ceil(log2 n)` leaves room; past that every split is the balanced median (depth grows by exactly
    // ceil(log2 n) from there), so no path is longer than kBvhDepthCap whatever the scene (10^5 coincident centroids
    // included).  max_depth records what was built; flatten() refuses a tree that exceeds the cap.
    static constexpr int kBvhDepthCap = kBvhStack - 2;
    int max_depth = 0;
    static int ceil_log2(int n) {
        int l = 0;
        while ((1 << l) < n) l++;
        return l;
    }
    int build(int b, int e, int depth) {
        int n = e - b;
        max_depth = std::max(max_depth, depth);
        if (n <= leaf_size) return ~((b << 4) | (n - 1));
        if (depth + ceil_log2(n) + 1 >= kBvhDepthCap) {  // balanced from here on
            int mid = (b + e) / 2;
            Box cb;
            for (int i = b; i < e; i++)
                for (int a = 0; a < 3; a++)
                    cb.lo[a] = std::min(cb.lo[a], items[i].centroid[a]), cb.hi[a] = std::max(cb.hi[a], items[i].centroid[a]);
            int axis = 0;
            for (int a = 1; a < 3; a++)
                if (cb.hi[a] - cb.lo[a] > cb.hi[axis] - cb.lo[axis]) axis = a;
            std::nth_element(items.begin() + b, items.begin() + mid, items.begin() + e,
                             [&](const BuildItem& x, const BuildItem& y) { return x.centroid[axis] < y.centroid[axis]; });
            return make_inner(b, mid, e, depth);
        }
        Box cb;
        for (int i = b; i < e; i++)
            for (int a = 0; a < 3; a++)
                cb.lo[a] = std::min(cb.lo[a], items[i].centroid[a]), cb.hi[a] = std::max(cb.hi[a], items[i].centroid[a]);
        int axis = 0;
        float ext = cb.hi[0] - cb.lo[0];
        for (int a = 1; a < 3; a++)
            if (cb.hi[a] - cb.lo[a] > ext) axis = a, ext = cb.hi[a] - cb.lo[a];
        int mid = -1;
        if (ext > 0.f) {
            constexpr int kBins = 16;
            Box bins[kBins];
            int counts[kBins] = {0};
            float scale = kBins / ext;
            auto bin_of = [&](const BuildItem& it) {
                int k = (int)((it.centroid[axis] - cb.lo[axis]) * scale);
                return std::min(std::max(k, 0), kBins - 1);
            };
            for (int i = b; i < e; i++) {
                int k = bin_of(items[i]);
                bins[k].grow(items[i].box);
                counts[k]++;
            }
            float right_area[kBins];
            int right_count[kBins];
            Box acc;
            int cnt = 0;
            for (int k = kBins - 1; k > 0; k--) {
                acc.grow(bins[k]);
                cnt += counts[k];
                right_area[k] = acc.area();
                right_count[k] = cnt;
            }
            Box left;
            int lcnt = 0, best_k = -1;
            float best_cost = INFINITY;
            for (int k = 0; k < kBins - 1; k++) {
                left.grow(bins[k]);
                lcnt += counts[k];
                if (lcnt == 0 || right_count[k + 1] == 0) continue;
                float cost = left.area() * lcnt + right_area[k + 1] * right_count[k + 1];
                if (cost < best_cost) best_cost = cost, best_k = k;
            }
            if (best_k >= 0) {
                auto it = std::partition(items.begin() + b, items.begin() + e,
                                         [&](const BuildItem& x) { return bin_of(x) <= best_k; });
                mid = (int)(it - items.begin());
            }
        }
        if (mid <= b || mid >= e) {  // degenerate: equal centroids — split by count
            mid = (b + e) / 2;
            std::nth_element(items.begin() + b, items.begin() + mid, items.begin() + e,
                             [&](const BuildItem& x, const BuildItem& y) { return x.centroid[axis] < y.centroid[axis]; });
        }
        return make_inner(b, mid, e, depth);
    }
    // Subtrees of the top `par_depth` levels are built by separate threads into their own node arrays (the ranges of
    // `items` they partition are disjoint) and appended afterwards with their inner links shifted.
    int par_depth = 0;
    static void append(RawVector<DevBvhNode>& dst, RawVector<DevBvhNode>& sub, int& link) {
        const int off = (int)dst.size();
        for (DevBvhNode& n : sub) {
            if (n.d.x >= 0) n.d.x += off;
            if (n.d.y >= 0) n.d.y += off;
        }
        if (link >= 0) link += off;
        dst.insert(dst.end(), sub.begin(), sub.end());
    }
    int make_inner(int b, int mid, int e, int depth) {
        int idx = (int)nodes.size();
        nodes.emplace_back();
        Box b0, b1;
        for (int i = b; i < mid; i++) b0.grow(items[i].box);
        for (int i = mid; i < e; i++) b1.grow(items[i].box);
        int c0, c1;
        if (depth < par_depth && e - b > 4096) {
            RawVector<DevBvhNode> left_nodes, right_nodes;
            Builder left{items, left_nodes, leaf_size}, right{items, right_nodes, leaf_size};
            left.par_depth = right.par_depth = par_depth;
            auto task = std::async(std::launch::async, [&] { return left.build(b, mid, depth + 1); });
            c1 = right.build(mid, e, depth + 1);
            c0 = task.get();
            max_depth = std::max(max_depth, std::max(left.max_depth, right.max_depth));
            append(nodes, left_nodes, c0);
            append(nodes, right_nodes, c1);
        } else {
            c0 = build(b, mid, depth + 1);
            c1 = build(mid, e, depth + 1);
        }
        DevBvhNode& n = nodes[idx];
        n.a = make_float4(b0.lo[0], b0.lo[1], b0.lo[2], b0.hi[0]);
        n.b = make_float4(b0.hi[1], b0.hi[2], b1.lo[0], b1.lo[1]);
        n.c = make_float4(b1.lo[2], b1.hi[0], b1.hi[1], b1.hi[2]);
        // d.z bit i: child i holds closed primitives only (find_containers may cull it with a point-in-box test)
        bool closed0 = true, closed1 = true;
        for (int i = b; i < mid; i++) closed0 = closed0 && items[i].closed;
        for (int i = mid; i < e; i++) closed1 = closed1 && items[i].closed;
        n.d = make_int4(c0, c1, (closed0 ? 1 : 0) | (closed1 ? 2 : 0), 0);
        return idx;
    }
};

// worst-case number of intersections a leaf kind can emit (cone: 2 walls + 2 caps)
int max_hits(int type) {
    switch (type) {
        case RTC_SPHERE: return 2;
        case RTC_PLANE: return 1;
        case RTC_CUBE: return 2;
        case RTC_CYLINDER: return 3;
        case RTC_CONE: return 4;
        default: return 1;
    }
}

// The lowest i in [0, n) with pred(i), or n: a scan by all threads.
template <class Pred>
int first_index(int n, Pred pred, size_t grain = 16384) {
    std::atomic<int> first{n};
    parallel_for((size_t)n, grain, [&](size_t b, size_t e, int) {
        for (size_t i = b; i < e && (int)i < first.load(std::memory_order_relaxed); i++)
            if (pred((int)i)) {
                int seen = first.load();
                while ((int)i < seen && !first.compare_exchange_weak(seen, (int)i)) {
                }
                break;
            }
    });
    return first.load();
}

// Every index the flattened scene carries must point inside its table (the reference cannot express a dangling
// reference; a foreign host can).
int validate_scene(const RtcScene* s) {
    const int np = (int)s->prims.size(), nn = (int)s->nodes.size();
    // ---- validate references (the primitive passes run on all threads; the lowest failing index is the one reported)
    auto prim_error = [&](int i) -> const char* {
        const RtcPrim& p = s->prims[i];
        if (p.type < RTC_SPHERE || p.type > RTC_TRIANGLE) return "bad type";
        if (p.material < 0 || p.material >= (int)s->materials.size()) return "bad material index";
        if (p.parent < -1 || p.parent >= nn) return "bad parent";
        return nullptr;
    };
    {
        const int bad = first_index(np, [&](int i) { return prim_error(i) != nullptr; });
        if (bad < np) return fail(RTC_ERR_INVALID, "primitive " + std::to_string(bad) + ": " + prim_error(bad));
    }
    for (int i = 0; i < nn; i++) {
        const RtcNode& n = s->nodes[i];
        if (n.kind != RTC_NODE_GROUP && n.kind != RTC_NODE_CSG) return fail(RTC_ERR_INVALID, "node: bad kind");
        if (n.parent < -1 || n.parent >= nn || n.parent == i) return fail(RTC_ERR_INVALID, "node: bad parent");
        if (n.child_begin < 0 || n.child_count < 0 || n.child_begin + n.child_count > (int)s->refs.size())
            return fail(RTC_ERR_INVALID, "node: bad child range");
        if (n.kind == RTC_NODE_CSG && (n.child_count != 2 || n.op < 0 || n.op > 2)) return fail(RTC_ERR_INVALID, "csg node: needs 2 children and a valid operator");
        for (int c = 0; c < n.child_count; c++) {
            int r = s->refs[n.child_begin + c];
            if (r >= np || (r < 0 && ~r >= nn)) return fail(RTC_ERR_INVALID, "node: bad child reference");
        }
    }
    // ---- the node graph must be a forest whose parent and child links agree (the reference's Box<dyn Shape> tree
    // cannot be anything else; a foreign host's arrays can): every child reference names an item whose `parent` is the
    // referring node, no item is referenced twice, every item with a parent is in that parent's list, and parent chains
    // end.  A parent cycle would spin the device's cull-chain walk forever; a reference cycle would recurse the CSG
    // emitter without bound.
    // (a node marks only children whose parent field names it, so the marks of different nodes never collide and the
    // nodes can be checked on all threads)
    std::vector<unsigned char> prim_seen(np, 0), node_seen(nn, 0);
    auto link_error = [&](int i) -> const char* {
        const RtcNode& n = s->nodes[i];
        for (int c = 0; c < n.child_count; c++) {
            const int r = s->refs[n.child_begin + c];
            if ((r >= 0 ? s->prims[r].parent : s->nodes[~r].parent) != i) return "child's parent field does not point back";
        }
        for (int c = 0; c < n.child_count; c++) {
            const int r = s->refs[n.child_begin + c];
            unsigned char& seen = r >= 0 ? prim_seen[r] : node_seen[~r];
            if (seen) return "a child is referenced twice";
            seen = 1;
        }
        return nullptr;
    };
    {
        std::vector<const char*> why(nn, nullptr);
        const int bad = first_index(nn, [&](int i) { return (why[i] = link_error(i)) != nullptr; }, 512);
        if (bad < nn) return fail(RTC_ERR_INVALID, "node " + std::to_string(bad) + ": " + why[bad]);
    }
    {
        const int bad = first_index(np, [&](int i) { return s->prims[i].parent >= 0 && !prim_seen[i]; });
        if (bad < np) return fail(RTC_ERR_INVALID, "primitive " + std::to_string(bad) + ": not in its parent's child list");
    }
    {
        const int orphan = first_index(nn, [&](int i) { return s->nodes[i].parent >= 0 && !node_seen[i]; }, 4096);
        const int cyclic = first_index(nn, [&](int i) {
            int steps = 0;
            for (int a = s->nodes[i].parent; a >= 0; a = s->nodes[a].parent)
                if (++steps > nn) return true;
            return false;
        }, 512);
        if (orphan < nn && orphan <= cyclic) return fail(RTC_ERR_INVALID, "node " + std::to_string(orphan) + ": not in its parent's child list");
        if (cyclic < nn) return fail(RTC_ERR_INVALID, "node parents form a cycle");
    }
    for (const RtcMaterial& m : s->materials)
        if (m.pattern < -1 || m.pattern >= (int)s->patterns.size()) return fail(RTC_ERR_INVALID, "material: bad pattern index");
    for (const RtcPattern& p : s->patterns) {
        if (p.kind < RTC_PAT_STRIPES || p.kind > RTC_PAT_CUBIC_MAP) return fail(RTC_ERR_INVALID, "pattern: bad kind");
        int need = p.kind == RTC_PAT_TEXTURE_MAP ? 1 : (p.kind == RTC_PAT_CUBIC_MAP ? 6 : 0);
        for (int i = 0; i < need; i++)
            if (p.uv[i] < 0 || p.uv[i] >= (int)s->uvs.size()) return fail(RTC_ERR_INVALID, "pattern: bad uv pattern index");
    }
    return 0;
}

// Materials, patterns, UV patterns and image texels in their device layout, and the table-mode light samples.
int build_shading_tables(RtcScene* s, Flattened& f) {
    // ---- shading tables
    s->has_branching_materials = false;
    for (const RtcMaterial& m : s->materials) {
        if (m.reflective != 0.0f && m.transparency != 0.0f) s->has_branching_materials = true;
        DevMaterial d{};
        memcpy(d.color, m.color, sizeof(d.color));
        d.ambient = m.ambient, d.diffuse = m.diffuse, d.specular = m.specular, d.shininess = m.shininess;
        d.reflective = m.reflective, d.transparency = m.transparency, d.refractive_index = m.refractive_index;
        d.pattern = m.pattern;
        f.materials.push_back(d);
    }
    for (const RtcPattern& p : s->patterns) {
        DevPattern d{};
        rows3(p.inv, d.inv);
        memcpy(d.a, p.a, sizeof(d.a));
        memcpy(d.b, p.b, sizeof(d.b));
        d.kind = p.kind, d.mapping = p.mapping;
        memcpy(d.uv, p.uv, sizeof(d.uv));
        f.patterns.push_back(d);
    }
    std::vector<size_t> texel_base;
    for (const RtcScene::Texture& t : s->textures) {
        texel_base.push_back(f.texels.size());
        for (size_t i = 0; i < (size_t)t.width * t.height; i++)
            f.texels.push_back(make_float4(t.rgb[3 * i], t.rgb[3 * i + 1], t.rgb[3 * i + 2], 0.f));
    }
    if (f.texels.size() >= (1u << 30)) return fail(RTC_ERR_CAPACITY, "image textures exceed 2^30 pixels");
    for (const RtcUvPattern& u : s->uvs) {
        DevUvPattern d{};
        d.kind = u.kind;
        memcpy(d.p, u.params, sizeof(d.p));
        if (u.kind == RTC_UV_IMAGE) {  // {first texel, width, height} as integers
            const int t = (int)u.params[0];
            if (t < 0 || t >= (int)s->textures.size() || (float)t != u.params[0]) return fail(RTC_ERR_INVALID, "uv image: bad texture index");
            const int base = (int)texel_base[t], w = (int)s->textures[t].width, h = (int)s->textures[t].height;
            if (w < 1 || h < 1) return fail(RTC_ERR_INVALID, "uv image: empty canvas");
            memcpy(&d.p[0], &base, 4), memcpy(&d.p[1], &w, 4), memcpy(&d.p[2], &h, 4);
        }
        f.uvs.push_back(d);
    }
    // ---- table-mode light samples: point_on_light (rectangle_light.rs:60-66) is the same for every shade
    if (s->light_is_rect && !s->jitter.empty()) {
        size_t cursor = 0, L = s->jitter.size();
        for (int v = 0; v < s->v_steps; v++)
            for (int u = 0; u < s->u_steps; u++) {
                float j1 = s->jitter[cursor % L], j2 = s->jitter[(cursor + 1) % L];
                cursor += 2;
                float su = (float)u + j1, sv = (float)v + j2;
                float p[3];
                for (int a = 0; a < 3; a++) {
                    volatile float t1 = s->u_cell[a] * su;  // volatile: no host-side contraction / reassociation
                    volatile float t2 = s->corner[a] + t1;
                    volatile float t3 = s->v_cell[a] * sv;
                    p[a] = t2 + t3;
                }
                f.samples.push_back(make_float4(p[0], p[1], p[2], 0.f));
            }
    }
    return 0;
}

// The small-scene table of the kernel parameter block (every demo scene: no tree, at most kSmallCap items in the
// linear list) and the plan of its shadow filter: per-item bounding balls, filter eligibility, the cell-mask loops
// of an area light, the ball around the light's samples and the per-plane bundle constants (dev_shadow.cuh: shadow
// filter, intensity_cells, bundle_misses, ball_missed).
void plan_small_scene(const RtcScene* s, Flattened& f, int n_items) {
    // ---- small-scene table (kernel parameter block): no tree, every item in the linear list, few enough of them
    memset(&f.small, 0, sizeof(f.small));
    if (f.bvh_root < 0 && n_items > 0 && n_items <= kSmallCap) {
        f.small.n = n_items;
        f.small.two_pass_shadows = 1;
        int ends[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (int i = 0; i < n_items; i++) {
            SmallPrim& sp = f.small.p[i];
            int4 h = f.head[i];
            sp.head = make_int4(h.x, f.head[f.n_pos + i].x, h.z, h.w);
            int type = h.x & 15;
            bool caster = type == T_CSG || ((h.x >> 4) & kFlagCastsShadow);
            int bucket = (caster ? 0 : 4) + (type == T_SPHERE ? 0 : type == T_PLANE ? 1 : type == T_CUBE ? 2 : 3);
            for (int b = bucket; b < 8; b++) ends[b] = i + 1;
            if ((h.x >> 4) & kFlagHasParent) f.small.has_cull_chain = 1;
            sp.ball = make_float4(NAN, NAN, NAN, NAN);  // a NaN ball never rejects
            if (type == T_CSG) {
                f.small.two_pass_shadows = 0;
                sp.r0 = sp.r1 = sp.r2 = sp.bound = make_float4(0.f, 0.f, 0.f, 0.f);
                continue;
            }
            sp.r0 = f.xform[3 * (size_t)h.y], sp.r1 = f.xform[3 * (size_t)h.y + 1], sp.r2 = f.xform[3 * (size_t)h.y + 2];
            sp.bound = (type == T_CYLINDER || type == T_CONE) ? f.bound[h.z] : make_float4(0.f, 0.f, 0.f, 0.f);
            // ---- world-space bounding ball (dev_small.cuh: ball_missed, dev_shadow.cuh: bundle_misses).  Sphere / cube: centre =
            // forward transform of the origin, radius = the largest stretch of the forward 3x3 (bounded by
            // sqrt(|T|_1 |T|_inf)), times sqrt(3) for a cube's corners; other bounded shapes: the ball around their
            // world box.  bound.w = 2^-17 cond^2 / radius is the rate at which the tested radius grows with the squared
            // distance of the ray origin: beyond that clearance no f32 intersection test of the reference reports a hit.
            {
                const double m[3][4] = {{sp.r0.x, sp.r0.y, sp.r0.z, sp.r0.w}, {sp.r1.x, sp.r1.y, sp.r1.z, sp.r1.w}, {sp.r2.x, sp.r2.y, sp.r2.z, sp.r2.w}};
                const double det = m[0][0] * (m[1][1] * m[2][2] - m[1][2] * m[2][1]) - m[0][1] * (m[1][0] * m[2][2] - m[1][2] * m[2][0]) +
                                   m[0][2] * (m[1][0] * m[2][1] - m[1][1] * m[2][0]);
                double t[3][3], n1 = 0.0, ninf = 0.0, mi = 0.0;  // t = forward 3x3 = inverse of m's 3x3
                for (int a = 0; a < 3; a++)
                    for (int b = 0; b < 3; b++) {
                        const int a1 = (a + 1) % 3, a2 = (a + 2) % 3, b1 = (b + 1) % 3, b2 = (b + 2) % 3;
                        t[a][b] = (m[b1][a1] * m[b2][a2] - m[b1][a2] * m[b2][a1]) / det;
                    }
                for (int a = 0; a < 3; a++) {
                    n1 = std::max(n1, std::fabs(t[0][a]) + std::fabs(t[1][a]) + std::fabs(t[2][a]));
                    ninf = std::max(ninf, std::fabs(t[a][0]) + std::fabs(t[a][1]) + std::fabs(t[a][2]));
                    mi = std::max(mi, std::fabs(m[a][0]) + std::fabs(m[a][1]) + std::fabs(m[a][2]));
                }
                const double cond = std::max(1.0, mi * ninf);
                double c[3], radius;
                if (type == T_SPHERE || type == T_CUBE) {
                    radius = std::sqrt(n1 * ninf) * (type == T_CUBE ? std::sqrt(3.0) : 1.0);
                    for (int a = 0; a < 3; a++) c[a] = -(t[a][0] * m[0][3] + t[a][1] * m[1][3] + t[a][2] * m[2][3]);
                } else {
                    const RtcPrim& pr = s->prims[h.w];
                    double d2 = 0.0;
                    for (int a = 0; a < 3; a++) {
                        c[a] = 0.5 * ((double)pr.bbox_min[a] + pr.bbox_max[a]);
                        d2 += 0.25 * ((double)pr.bbox_max[a] - pr.bbox_min[a]) * ((double)pr.bbox_max[a] - pr.bbox_min[a]);
                    }
                    radius = std::sqrt(d2);
                }
                if (std::isfinite(radius) && std::isfinite(c[0]) && std::isfinite(c[1]) && std::isfinite(c[2]) && radius > 0.0 &&
                    std::isfinite(cond)) {
                    sp.ball = make_float4((float)c[0], (float)c[1], (float)c[2], (float)(radius * 1.001 + 1e-6));
                    sp.bound.w = (float)(std::ldexp(1.0, -17) * cond * cond / radius);
                }
            }
        }
        f.small.caster_end = make_int4(ends[0], ends[1], ends[2], ends[3]);
        f.small.other_end = make_int4(ends[4], ends[5], ends[6], ends[7]);
        // ---- shadow-filter eligibility (dev_shadow.cuh: shadow_filter): spheres whose transform is well conditioned
        // (the filter's error bound scales with the condition number), planes (term-wise bound: any transform),
        // cubes whose inverse has a diagonal 3x3 part (every direction component is a single product)
        bool ok = f.small.two_pass_shadows && !f.small.has_cull_chain && ends[2] == ends[3] && ends[6] == ends[7];
        double worst_tol = 64.0;  // in units of u = 2^-24
        for (int i = 0; i < n_items && ok; i++) {
            const SmallPrim& sp = f.small.p[i];
            const int type = sp.head.x & 15;
            const double m[3][3] = {{sp.r0.x, sp.r0.y, sp.r0.z}, {sp.r1.x, sp.r1.y, sp.r1.z}, {sp.r2.x, sp.r2.y, sp.r2.z}};
            for (int a = 0; a < 3; a++)
                for (int b = 0; b < 3; b++) ok = ok && std::isfinite(m[a][b]);
            if (type == T_CUBE) {
                for (int a = 0; a < 3; a++)
                    for (int b = 0; b < 3; b++) ok = ok && (a == b ? m[a][b] != 0.0 : m[a][b] == 0.0);
            } else if (type == T_SPHERE) {
                const double det = m[0][0] * (m[1][1] * m[2][2] - m[1][2] * m[2][1]) - m[0][1] * (m[1][0] * m[2][2] - m[1][2] * m[2][0]) +
                                   m[0][2] * (m[1][0] * m[2][1] - m[1][1] * m[2][0]);
                double norm_m = 0.0, norm_i = 0.0;
                for (int a = 0; a < 3; a++) {
                    double row_m = 0.0, row_i = 0.0;
                    for (int b = 0; b < 3; b++) {
                        const int a1 = (a + 1) % 3, a2 = (a + 2) % 3, b1 = (b + 1) % 3, b2 = (b + 2) % 3;
                        row_m += std::fabs(m[a][b]);
                        row_i += std::fabs((m[b1][a1] * m[b2][a2] - m[b1][a2] * m[b2][a1]) / det);  // inverse = adjugate / det
                    }
                    norm_m = std::max(norm_m, row_m), norm_i = std::max(norm_i, row_i);
                }
                const double cond = norm_m * norm_i;
                ok = ok && std::isfinite(cond) && cond <= 64.0;
                // a diagonal 3x3 part (translation x axis-aligned scaling: every sphere of the demo scenes): each direction
                // component is ONE product, nothing cancels, and the bound does not grow with the condition number
                bool diagonal = true;
                for (int a = 0; a < 3; a++)
                    for (int b = 0; b < 3; b++) diagonal = diagonal && (a == b || m[a][b] == 0.0);
                if (ok) worst_tol = std::max(worst_tol, diagonal ? 64.0 : 128.0 * cond + 32.0);
            }
        }
        f.small.filter_ok = ok ? 1 : 0;
        // cell-mask path: a table-mode light whose samples fit the staging area, or the counter-mode generator
        const bool table_light = s->light_is_rect && !f.samples.empty() && f.samples.size() <= (size_t)kSampleCap;
        const bool counter_light = s->light_is_rect && s->jitter.empty() && s->u_steps > 0 && s->v_steps > 0;
        f.small.cell_masks = ok && (table_light || counter_light);
        // the lean kernel build (dev_shade.cuh: color_at<.., LEAN>): cell_masks already rules out CSG roots, cull chains,
        // kinds other than spheres, planes and axis-aligned cubes, and point lights; no material of the table may have a
        // pattern or transparency.  RTC_LEAN=0 (test aid, read on every commit) keeps such scenes on the general build,
        // so that the two builds' frames can be compared.
        const char* lean_env = getenv("RTC_LEAN");
        bool lean = f.small.cell_masks && !(lean_env && atoi(lean_env) == 0);
        for (int i = 0; i < n_items && lean; i++) {
            const DevMaterial& m = f.materials[f.small.p[i].head.x >> 8];
            lean = m.pattern < 0 && m.transparency == 0.0f;
        }
        f.small.lean = lean ? 1 : 0;
        if (f.small.cell_masks) {
            // the bundle reject (dev_shadow.cuh: bundle_misses): a ball around the light samples, and for every sphere /
            // cube its world-space bounding ball — centre = forward transform of the origin, radius = the largest
            // stretch of the forward 3x3 (bounded by sqrt(|T|_1 |T|_inf)), times sqrt(3) for a cube's corners
            // the light's possible sample points: the table's, or (counter mode: jitter in (0, 1]) the whole rectangle
            std::vector<float4> pts = f.samples;
            if (pts.empty())
                for (int cu = 0; cu < 2; cu++)
                    for (int cv = 0; cv < 2; cv++)
                        pts.push_back(make_float4(s->corner[0] + s->u_cell[0] * (cu * s->u_steps) + s->v_cell[0] * (cv * s->v_steps),
                                                  s->corner[1] + s->u_cell[1] * (cu * s->u_steps) + s->v_cell[1] * (cv * s->v_steps),
                                                  s->corner[2] + s->u_cell[2] * (cu * s->u_steps) + s->v_cell[2] * (cv * s->v_steps), 0.f));
            double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
            for (const float4& q : pts) {
                const double v[3] = {q.x, q.y, q.z};
                for (int a = 0; a < 3; a++) lo[a] = std::min(lo[a], v[a]), hi[a] = std::max(hi[a], v[a]);
            }
            const double lc[3] = {0.5 * (lo[0] + hi[0]), 0.5 * (lo[1] + hi[1]), 0.5 * (lo[2] + hi[2])};
            double rl = 0.0;
            for (const float4& q : pts)
                rl = std::max(rl, std::sqrt((q.x - lc[0]) * (q.x - lc[0]) + (q.y - lc[1]) * (q.y - lc[1]) + (q.z - lc[2]) * (q.z - lc[2])));
            f.small.light_ball = make_float4((float)lc[0], (float)lc[1], (float)lc[2], (float)(rl * 1.001 + 1e-6));
            const int n_planes = ends[1] - ends[0];
            f.small.plane_cells = table_light && n_planes > 0 && (size_t)n_planes * f.samples.size() <= (size_t)kPlaneCellCap;
            // bounds of the per-(plane, cell) constants over all cells (dev_small.cuh: plane_cell_constants), padded
            // beyond the f32 rounding of the device's own evaluation: lets a shade settle the plane for every cell at once
            for (int q = 0; q < 2; q++) {
                f.small.plane_bundle[q] = make_float4(NAN, NAN, NAN, NAN);  // NaN: the bundle test never decides
                // table mode: over the table's sample points; counter mode (samples drawn per shade): over the corners of
                // the light's rectangle, which bound every drawn point — r1.L is linear in L, the two error terms convex
                if (!(f.small.plane_cells || counter_light) || q >= n_planes) continue;
                const float4 r1 = f.small.p[ends[0] + q].r1;
                double lo = 1e300, hi = -1e300, e_max = 0.0, l1_max = 0.0;
                for (const float4& L : (f.small.plane_cells ? f.samples : pts)) {
                    const double px = (double)r1.x * L.x, py = (double)r1.y * L.y, pz = (double)r1.z * L.z;
                    const double a = std::fabs(px) + std::fabs(py) + std::fabs(pz);
                    lo = std::min(lo, px + py + pz - 1e-6 * a), hi = std::max(hi, px + py + pz + 1e-6 * a);
                    e_max = std::max(e_max, 3.814697265625e-06 * a * 1.000001);
                    l1_max = std::max(l1_max, 1.1920929e-3 * (1.0 + 7.7e-6) * (std::fabs(L.x) + std::fabs(L.y) + std::fabs(L.z)) * 1.000001);
                }
                f.small.plane_bundle[q] = make_float4((float)lo, (float)hi, (float)e_max, (float)l1_max);
                // round outwards
                f.small.plane_bundle[q].x = std::nextafter(f.small.plane_bundle[q].x, -INFINITY);
                f.small.plane_bundle[q].y = std::nextafter(f.small.plane_bundle[q].y, INFINITY);
                f.small.plane_bundle[q].z = std::nextafter(f.small.plane_bundle[q].z, INFINITY);
                f.small.plane_bundle[q].w = std::nextafter(f.small.plane_bundle[q].w, INFINITY);
            }
        }
        // the sphere filter's relative bound, DESIGN.md "Shadow filter: where the bounds come from": the two discriminants
        // (reference: normalised direction, no fusing; filter: fused, unnormalised) are each within (4 eps + 14 u) a spread
        // of the exact one.  General transform: eps <= 18 k u and <= 9 k u (k = inf-norm condition number, u = 2^-24),
        // together (108 k + 28) u, shipped (128 k + 32) u.  Diagonal 3x3 part: eps <= 4 u and <= u, together 48 u, shipped 64 u.
        f.small.tol_sphere = (float)(std::ldexp(1.0, -24) * worst_tol);
        // ---- the image every block stages into shared memory (dev_small.cuh: stage_small_scene)
        f.small_image.assign(kSmemOrg, make_float4(0.f, 0.f, 0.f, 0.f));
        memcpy(f.small_image.data(), f.small.p, (size_t)n_items * sizeof(SmallPrim));
        static_assert(sizeof(SmallPrim) == kSmallStride * sizeof(float4), "table entry layout");
        if (table_light) {
            std::copy(f.samples.begin(), f.samples.end(), f.small_image.begin() + kSmemSamples);
            if (f.small.plane_cells)
                for (int q = 0; q < ends[1] - ends[0]; q++)
                    for (size_t c = 0; c < f.samples.size(); c++)
                        f.small_image[kSmemPlaneCells + (size_t)q * f.samples.size() + c] =
                            plane_cell_constants(f.small.p[ends[0] + q].r1, f.samples[c]);
        }
    }
}

}  // namespace

int flatten(RtcScene* s, Flattened& f, TreeBuilderFn tree_builder, void* tree_builder_ctx) {
    const int np = (int)s->prims.size(), nn = (int)s->nodes.size();
    const bool timing = getenv("RTC_TIMING") != nullptr;  // tuning aid: phase times of the host half on stderr
    auto t_last = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (!timing) return;
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[rtc commit] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - t_last).count());
        t_last = now;
    };
    if (int rc = validate_scene(s)) return rc;
    lap("  validate");

    // ---- which CSG (if any) is the outermost CSG ancestor of each node / primitive
    std::vector<int> top_csg_of_node(nn, -1);
    auto resolve = [&](int node) {
        int top = -1, guard = 0;
        for (int a = node; a >= 0; a = s->nodes[a].parent) {
            if (s->nodes[a].kind == RTC_NODE_CSG) top = a;
            if (++guard > nn) return -2;
        }
        return top;
    };
    parallel_for((size_t)nn, 512, [&](size_t b, size_t e, int) {
        for (size_t i = b; i < e; i++) top_csg_of_node[i] = resolve((int)i);
    });
    for (int i = 0; i < nn; i++)
        if (top_csg_of_node[i] == -2) return fail(RTC_ERR_INVALID, "node parents form a cycle");
    // (the passes over the primitives below run on all threads — rtc_parallel.h — and keep primitive order)
    constexpr size_t kGrain = 16384;
    std::vector<int> prim_top_csg(np, -1);
    parallel_for((size_t)np, kGrain, [&](size_t b, size_t e, int) {
        for (size_t i = b; i < e; i++) prim_top_csg[i] = s->prims[i].parent >= 0 ? top_csg_of_node[s->prims[i].parent] : -1;
    });

    lap("  csg ancestors");
    // ---- top-level items: free primitives and outermost CSG nodes.  Two passes over the primitives: tally (how many
    // bounded and unbounded items each chunk holds, the scene's extent, the triangles), then write at the offsets.
    struct Item {
        int prim;  // >= 0 primitive, else ~csg node
        float lo[3], hi[3];
        Box box() const {
            Box b;
            for (int a = 0; a < 3; a++) b.lo[a] = lo[a], b.hi[a] = hi[a];
            return b;
        }
    };
    auto make_item = [](int ref, const float* lo, const float* hi) {
        Item it;
        it.prim = ref;
        for (int a = 0; a < 3; a++) it.lo[a] = lo[a], it.hi[a] = hi[a];
        return it;
    };
    auto reach = [](const Item& it) {  // the largest coordinate of a bounded item
        float m = 0.f;
        for (int a = 0; a < 3; a++) m = std::max(m, std::max(std::fabs(it.lo[a]), std::fabs(it.hi[a])));
        return m;
    };
    RawVector<Item> bounded;
    std::vector<Item> unbounded;
    float extent = 0.f;  // the largest coordinate a ray of this scene starts from or aims at (bounded items; camera and light below)
    size_t n_triangles = 0;
    {
        struct Tally {
            int bounded = 0;
            size_t triangles = 0;
            float extent = 0.f;
            std::vector<Item> unbounded;
        };
        const int n_parts = parallel_chunks((size_t)np, kGrain);
        std::vector<Tally> tally(n_parts);
        parallel_for((size_t)np, kGrain, [&](size_t b, size_t e, int part) {
            Tally t;
            for (size_t i = b; i < e; i++) {
                if (prim_top_csg[i] >= 0) continue;
                const Item it = make_item((int)i, s->prims[i].bbox_min, s->prims[i].bbox_max);
                if (it.box().finite())
                    t.bounded++, t.triangles += s->prims[i].type == RTC_TRIANGLE, t.extent = std::max(t.extent, reach(it));
                else
                    t.unbounded.push_back(it);
            }
            tally[part] = std::move(t);
        });
        std::vector<Item> csg_bounded;
        for (int i = 0; i < nn; i++)
            if (s->nodes[i].kind == RTC_NODE_CSG && top_csg_of_node[i] == i) {
                const Item it = make_item(~i, s->nodes[i].world_bbox_min, s->nodes[i].world_bbox_max);
                if (it.box().finite())
                    csg_bounded.push_back(it), extent = std::max(extent, reach(it));
                else
                    tally.back().unbounded.push_back(it);  // after every primitive, as a sequential walk lists them
            }
        std::vector<int> base(n_parts + 1, 0);
        for (int part = 0; part < n_parts; part++) {
            base[part + 1] = base[part] + tally[part].bounded;
            n_triangles += tally[part].triangles, extent = std::max(extent, tally[part].extent);
            unbounded.insert(unbounded.end(), tally[part].unbounded.begin(), tally[part].unbounded.end());
        }
        bounded.resize((size_t)base[n_parts] + csg_bounded.size());
        parallel_for((size_t)np, kGrain, [&](size_t b, size_t e, int part) {
            Item* out = bounded.data() + base[part];
            for (size_t i = b; i < e; i++) {
                if (prim_top_csg[i] >= 0) continue;
                const Item it = make_item((int)i, s->prims[i].bbox_min, s->prims[i].bbox_max);
                if (it.box().finite()) *out++ = it;
            }
        });
        std::copy(csg_bounded.begin(), csg_bounded.end(), bounded.begin() + base[n_parts]);
    }
    if ((int)bounded.size() < s->bvh_min_prims) {  // tiny scene: test everything for every ray, no tree
        unbounded.insert(unbounded.end(), bounded.begin(), bounded.end());
        bounded.clear();
        // group the linear list by (shadow casters first, kind) — the small-scene kernels loop over runs of one
        // kind; depth-first order inside a run (ties are broken by the stored order field, not by position)
        std::stable_sort(unbounded.begin(), unbounded.end(), [&](const Item& a, const Item& b) {
            auto key = [&](const Item& it) {
                int dfs = it.prim >= 0 ? it.prim : np + ~it.prim;
                int caster = it.prim >= 0 ? (s->prims[it.prim].casts_shadow ? 0 : 1) : 0;
                int type = it.prim >= 0 ? s->prims[it.prim].type : 99;
                int bucket = type == RTC_SPHERE ? 0 : type == RTC_PLANE ? 1 : type == RTC_CUBE ? 2 : 3;
                return std::make_tuple(caster, bucket, dfs);
            };
            return key(a) < key(b);
        });
    }

    lap("  item lists");
    // ---- BVH
    // the scene's extent also covers the camera and the light
    {
        float m[16], cam[3] = {0.f, 0.f, 0.f};
        memcpy(m, s->cam_inv, sizeof(m));  // the camera's origin = inverse * (0, 0, 0): the translation column
        for (int a = 0; a < 3; a++) cam[a] = m[a * 4 + 3];
        for (int a = 0; a < 3; a++) {
            extent = std::max(extent, std::fabs(cam[a]));
            float l = std::fabs(s->light_pos[a]);
            if (s->light_is_rect)
                l = std::max(l, std::fabs(s->corner[a]) + std::fabs(s->u_cell[a]) * s->u_steps + std::fabs(s->v_cell[a]) * s->v_steps);
            if (std::isfinite(l)) extent = std::max(extent, l);
        }
        f.reach = extent;
    }
    RawVector<BuildItem> build_items(bounded.size());
    parallel_for(bounded.size(), kGrain, [&](size_t begin, size_t end, int) {
        for (size_t i = begin; i < end; i++) {
            BuildItem& b = build_items[i];
            b.box = bounded[i].box();
            b.item = (int)i;
            b.closed = bounded[i].prim >= 0 && (s->prims[bounded[i].prim].type == RTC_SPHERE || s->prims[bounded[i].prim].type == RTC_CUBE);
            for (int a = 0; a < 3; a++) {
                // pad: the tree must never reject a hit the reference would report (it is only an accelerator).  The last
                // term covers the traversal's own arithmetic: slab distances are formed as fma(plane, 1/d, -(o * 1/d)), two
                // roundings of products as large as the ray origin's coordinate, and 1/d is rounded once — together below 2^-21 of
                // the scene's extent in length; 2^-20 is added
                float ext = b.box.hi[a] - b.box.lo[a];
                float pad = 1e-4f * ext + 1e-5f * std::max(std::fabs(b.box.lo[a]), std::fabs(b.box.hi[a])) + 1e-6f + 9.54e-7f * extent;
                b.box.lo[a] -= pad;
                b.box.hi[a] += pad;
                b.centroid[a] = 0.5f * (b.box.lo[a] + b.box.hi[a]);
            }
        }
    });
    lap("  padded boxes");
    if (!build_items.empty()) {
        // Leaf size: a mesh's triangles share one transform (the object-space ray is cached), so a few per leaf cost
        // less than the extra boxes; every other primitive pays its own ray transform, and one per leaf wins
        // (measured on B200: 102 k triangles 0.50 ms at 4 vs 0.58 at 1; 100 k spheres 38.7 ms at 1 vs 51.7 at 4).
        int leaf = s->leaf_size > 0 ? s->leaf_size : (2 * n_triangles > bounded.size() ? 4 : 1);
        if (const char* env = getenv("RTC_BVH_LEAF")) leaf = atoi(env);  // tuning aid
        f.leaf_size = std::min(std::max(leaf, 1), 16);
        int root = 0;
        s->built_on_device = 0;
        if (tree_builder && build_items.size() >= 1024) {  // the device builder: the same padded boxes, Morton order
            RawVector<float> boxes(6 * build_items.size());
            RawVector<unsigned char> closed(build_items.size());
            parallel_for(build_items.size(), kGrain, [&](size_t b, size_t e, int) {
                for (size_t i = b; i < e; i++) {
                    for (int a = 0; a < 3; a++) boxes[6 * i + a] = build_items[i].box.lo[a], boxes[6 * i + 3 + a] = build_items[i].box.hi[a];
                    closed[i] = build_items[i].closed;
                }
            });
            TreeBuildOutput out;
            lap("  builder input");
            if (tree_builder(tree_builder_ctx, TreeBuildInput{boxes.data(), closed.data(), (int)build_items.size(), f.leaf_size}, out) == 0) {
                RawVector<BuildItem> sorted(build_items.size());
                parallel_for(sorted.size(), kGrain, [&](size_t b, size_t e, int) {
                    for (size_t i = b; i < e; i++) sorted[i] = build_items[out.order[i]];
                });
                build_items.swap(sorted);
                lap("  device builder + reorder");
                f.bvh.swap(out.nodes);
                root = out.root;
                f.bvh_depth = out.depth;
                s->built_on_device = 1;
            }
        }
        if (!s->built_on_device) {
            Builder builder{build_items, f.bvh, f.leaf_size};
            const unsigned hw = std::max(1u, std::thread::hardware_concurrency());
            while ((1u << builder.par_depth) < hw && builder.par_depth < 5) builder.par_depth++;  // up to 32 subtree tasks
            f.bvh.reserve(build_items.size());
            root = builder.build(0, (int)build_items.size(), 0);
            // max_depth is the most inner nodes above a leaf; a tree that is one leaf gets the wrapping node below
            f.bvh_depth = std::max(builder.max_depth, 1);
        }
        if (f.bvh_depth > kBvhStack - 1)  // cannot happen (Builder::build balances before the cap); never silent if it does
            return fail(RTC_ERR_CAPACITY, "BVH depth " + std::to_string(f.bvh_depth) + " exceeds the traversal stack (" +
                                              std::to_string(kBvhStack) + ")");
        if (root < 0) {  // a single leaf: wrap it so the traversal always starts at an inner node
            DevBvhNode n;
            Box b;
            bool closed = true;
            for (auto& it : build_items) b.grow(it.box), closed = closed && it.closed;
            n.a = make_float4(b.lo[0], b.lo[1], b.lo[2], b.hi[0]);
            n.b = make_float4(b.hi[1], b.hi[2], NAN, NAN);  // second child: a NaN box never passes the slab test
            n.c = make_float4(NAN, NAN, NAN, NAN);
            n.d = make_int4(root, root, closed ? 1 : 0, 0);
            f.bvh.push_back(n);
            root = (int)f.bvh.size() - 1;
        }
        f.bvh_root = root;
    }

    lap("bvh build");
    // ---- device positions: BVH order, then the linear list, then CSG-internal primitives
    const int n_tree = (int)build_items.size();
    const int n_items = n_tree + (int)unbounded.size();
    std::vector<int> item_refs(n_items);
    parallel_for((size_t)n_tree, kGrain, [&](size_t b, size_t e, int) {
        for (size_t i = b; i < e; i++) item_refs[i] = bounded[build_items[i].item].prim;
    });
    for (size_t i = 0; i < unbounded.size(); i++) item_refs[n_tree + i] = unbounded[i].prim;
    std::vector<int> prim_pos(np, -1), csg_pos(nn, -1);
    parallel_for((size_t)n_items, kGrain, [&](size_t b, size_t e, int) {
        for (size_t i = b; i < e; i++) {
            if (item_refs[i] >= 0)
                prim_pos[item_refs[i]] = (int)i;
            else
                csg_pos[~item_refs[i]] = (int)i;
        }
    });
    int next = n_items;
    for (int i = 0; i < np; i++)
        if (prim_top_csg[i] >= 0) prim_pos[i] = next++;
    f.n_pos = next;
    for (int i = n_tree; i < n_items; i++) f.linear.push_back(i);

    // ---- transforms, triangle and bound tables, heads.  Transform table: one slot per non-triangle primitive in
    // primitive order, then the triangles' transforms de-duplicated bitwise in first-use order (only a mesh's triangles
    // share transforms in practice, and only they profit: the object-space ray is cached by transform id).  Two passes
    // over the primitives on all threads — count, then write at the offsets the counts fix — with the same result
    // for any number of threads.
    struct XfKey {
        uint32_t w[12];
        bool operator==(const XfKey& o) const { return memcmp(w, o.w, sizeof(w)) == 0; }
    };
    struct XfHash {
        size_t operator()(const XfKey& k) const {  // FNV-1a over the 12 words
            uint64_t h = 1469598103934665603ull;
            for (uint32_t v : k.w) h = (h ^ v) * 1099511628211ull;
            return (size_t)h;
        }
    };
    struct Part {
        int plain = 0, tris = 0, bounds = 0;  // non-triangle primitives, triangles, cylinders + cones of the chunk
        bool all_cast = true;
        std::vector<XfKey> keys;     // the chunk's distinct triangle transforms, first use first
        std::vector<int> tri_key;    // per triangle of the chunk: index into `keys`, later the global transform id
    };
    const int n_parts = parallel_chunks((size_t)np, kGrain);
    std::vector<Part> parts(n_parts);
    parallel_for((size_t)np, kGrain, [&](size_t b, size_t e, int c) {
        Part& part = parts[c];
        std::unordered_map<XfKey, int, XfHash> ids;
        XfKey last_key{};
        int last_id = -1;
        for (size_t i = b; i < e; i++) {
            const RtcPrim& p = s->prims[i];
            part.all_cast = part.all_cast && p.casts_shadow;
            if (p.type != RTC_TRIANGLE) {
                part.plain++;
                part.bounds += p.type == RTC_CYLINDER || p.type == RTC_CONE;
                continue;
            }
            part.tris++;
            XfKey key;
            memcpy(key.w, p.inv, sizeof(key.w));
            if (last_id < 0 || !(key == last_key)) {  // a mesh's triangles share one transform
                last_key = key;
                auto it = ids.find(key);
                if (it == ids.end()) {
                    it = ids.emplace(key, (int)part.keys.size()).first;
                    part.keys.push_back(key);
                }
                last_id = it->second;
            }
            part.tri_key.push_back(last_id);
        }
    });
    std::vector<int> plain_base(n_parts + 1, 0), tri_base(n_parts + 1, 0), bound_base(n_parts + 1, 0);
    for (int c = 0; c < n_parts; c++) {
        plain_base[c + 1] = plain_base[c] + parts[c].plain, tri_base[c + 1] = tri_base[c] + parts[c].tris;
        bound_base[c + 1] = bound_base[c] + parts[c].bounds;
        if (!parts[c].all_cast) f.all_cast_shadow = 0;
    }
    const int n_plain = plain_base[n_parts];
    {
        std::unordered_map<XfKey, int, XfHash> ids;
        std::vector<XfKey> distinct;
        std::vector<std::vector<int>> global(n_parts);
        for (int c = 0; c < n_parts; c++)
            for (const XfKey& key : parts[c].keys) {
                auto it = ids.find(key);
                if (it == ids.end()) {
                    it = ids.emplace(key, (int)distinct.size()).first;
                    distinct.push_back(key);
                }
                global[c].push_back(n_plain + it->second);
            }
        f.xform.resize(3 * ((size_t)n_plain + distinct.size()));
        for (size_t k = 0; k < distinct.size(); k++) {
            float m[16] = {0};
            memcpy(m, distinct[k].w, sizeof(distinct[k].w));
            rows3(m, &f.xform[3 * ((size_t)n_plain + k)]);
        }
        parallel_for((size_t)n_parts, 1, [&](size_t b, size_t e, int) {
            for (size_t c = b; c < e; c++)
                for (int& k : parts[c].tri_key) k = global[c][k];
        });
    }
    f.head.resize(2 * (size_t)f.n_pos);
    s->pos_to_prim.resize(f.n_pos);
    for (int i = 0; i < nn; i++)
        if (csg_pos[i] >= 0) s->pos_to_prim[csg_pos[i]] = -1;  // a CSG's own position is no primitive
    f.tri.resize(3 * (size_t)tri_base[n_parts]);
    f.bound.resize(bound_base[n_parts]);
    parallel_for((size_t)np, kGrain, [&](size_t b, size_t e, int c) {
        int plain = plain_base[c], tri = tri_base[c], bound = bound_base[c], k = 0;
        for (size_t i = b; i < e; i++) {
            const RtcPrim& p = s->prims[i];
            const int pos = prim_pos[i];
            int aux = 0, xf;
            if (p.type == RTC_TRIANGLE) {
                aux = tri;
                const float* q = p.params;  // p1, e1, e2, normal
                f.tri[3 * (size_t)tri] = make_float4(q[0], q[1], q[2], q[3]);
                f.tri[3 * (size_t)tri + 1] = make_float4(q[4], q[5], q[6], q[7]);
                f.tri[3 * (size_t)tri + 2] = make_float4(q[8], q[9], q[10], q[11]);
                tri++;
                xf = parts[c].tri_key[k++];
            } else {
                if (p.type == RTC_CYLINDER || p.type == RTC_CONE) {
                    aux = bound;
                    f.bound[bound++] = make_float4(p.params[0], p.params[1], p.params[2] != 0.f ? 1.f : 0.f, 0.f);
                }
                xf = plain;
                rows3(p.inv, &f.xform[3 * (size_t)plain]);
                plain++;
            }
            int flags = p.casts_shadow ? kFlagCastsShadow : 0;
            // the group cull chain (Q6): always for the items tested for every ray; for the tree's primitives too under
            // RTC_OPT_EXACT_GROUPS (a CSG's own primitives never: csg_eval culls their groups exactly)
            const bool in_linear = pos >= n_tree && pos < n_items;
            if ((in_linear || (s->exact_groups && prim_top_csg[i] < 0)) && p.parent >= 0) flags |= kFlagHasParent;
            f.head[pos] = make_int4(p.type | (flags << 4) | (p.material << 8), xf, aux, (int)i);
            f.head[f.n_pos + pos] = make_int4(prim_top_csg[i] < 0 ? p.parent : -1, (int)i, 0, 0);
            s->pos_to_prim[pos] = (int)i;
        }
    });
    lap("positions, transforms, heads");
    // ---- reference shape-tree nodes
    f.nodes.resize(nn);
    for (int i = 0; i < nn; i++) {
        const RtcNode& n = s->nodes[i];
        DevNode& d = f.nodes[i];
        rows3(n.inv, d.inv);
        for (int a = 0; a < 3; a++) d.bmin[a] = n.bbox_min[a], d.bmax[a] = n.bbox_max[a];
        d.kind = n.kind;
        d.parent = n.parent;
        d.op = n.op;
        d.pad = 0;
    }
    // ---- loose group boxes: a group whose cached box does not contain a child's parent-space box (exact f32 compare; a
    // NaN bound counts as loose).  The reference caches a group's box on first use and never invalidates it
    // (group.rs:19), so a later add_child or set_transformation leaves it culling with the old box.
    {
        std::atomic<int> loose{0};
        parallel_for((size_t)nn, 4096, [&](size_t b, size_t e, int) {
            int count = 0;
            for (size_t i = b; i < e; i++) {
                const RtcNode& n = s->nodes[i];
                if (n.kind != RTC_NODE_GROUP) continue;
                bool contains = true;
                for (int c = 0; c < n.child_count && contains; c++) {
                    const int r = s->refs[n.child_begin + c];
                    const float* lo = r >= 0 ? s->prims[r].bbox_min : s->nodes[~r].world_bbox_min;
                    const float* hi = r >= 0 ? s->prims[r].bbox_max : s->nodes[~r].world_bbox_max;
                    for (int a = 0; a < 3; a++) contains = contains && n.bbox_min[a] <= lo[a] && hi[a] <= n.bbox_max[a];
                }
                count += !contains;
            }
            loose += count;
        });
        f.loose_group_boxes = loose.load();
        // RTC_OPT_EXACT_GROUPS: DevNode::pad = 1 marks a group whose chain is nested: every box on the way up contains the
        // box below it (the boxes the culls use, exact f32 compare), so a hit point inside this group's box by the rounding
        // margin passes every box of the chain (dev_bvh.cuh: chain_certified).  A stale box breaks the chains through it.
        // RTC_EXACT_GROUPS_CERT=0 (test and timing aid, read on every commit) leaves every node unmarked: every chain walks.
        const char* cert_env = getenv("RTC_EXACT_GROUPS_CERT");
        if (s->exact_groups && !(cert_env && atoi(cert_env) == 0))
            parallel_for((size_t)nn, 4096, [&](size_t b, size_t e, int) {
                for (size_t i = b; i < e; i++) {
                    if (s->nodes[i].kind != RTC_NODE_GROUP) continue;
                    bool ok = true;
                    for (int c = (int)i, a = s->nodes[i].parent; a >= 0 && ok; c = a, a = s->nodes[a].parent) {
                        const RtcNode &in = s->nodes[c], &out = s->nodes[a];
                        ok = out.kind == RTC_NODE_GROUP;
                        for (int k = 0; k < 3; k++) ok = ok && out.bbox_min[k] <= in.bbox_min[k] && in.bbox_max[k] <= out.bbox_max[k];
                    }
                    f.nodes[i].pad = ok ? 1 : 0;
                }
            });
    }

    // ---- CSG programs
    struct Emit {
        RtcScene* s;
        Flattened& f;
        std::vector<int>& prim_pos;
        int max_depth = 0;  // CSG nesting of the program being emitted
        int emit(int ref, int csg_depth) {  // returns worst-case hit count of the subtree
            if (ref >= 0) {
                f.ops.push_back(DevCsgOp{OP_PRIM, prim_pos[ref], 0, 0});
                return max_hits(s->prims[ref].type);
            }
            int node = ~ref;
            const RtcNode& n = s->nodes[node];
            int total = 0;
            if (n.kind == RTC_NODE_GROUP) {
                size_t idx = f.ops.size();
                f.ops.push_back(DevCsgOp{OP_GROUP, node, 0, 0});
                for (int c = 0; c < n.child_count; c++) total += emit(s->refs[n.child_begin + c], csg_depth);
                f.ops[idx].skip = (int)f.ops.size();
            } else {
                max_depth = std::max(max_depth, csg_depth + 1);
                size_t idx = f.ops.size();
                f.ops.push_back(DevCsgOp{OP_CSG_ENTER, node, 0, 0});
                total += emit(s->refs[n.child_begin], csg_depth + 1);
                f.ops.push_back(DevCsgOp{OP_CSG_MID, node, 0, 0});
                total += emit(s->refs[n.child_begin + 1], csg_depth + 1);
                f.ops.push_back(DevCsgOp{OP_CSG_EXIT, node, 0, 0});
                f.ops[idx].skip = (int)f.ops.size();
            }
            return total;
        }
    } emitter{s, f, prim_pos};
    // The links csg_sweep climbs (rtc_types.h: DevCsgOp::pad) for the program [start, f.ops.size()); returns its CSG nodes.
    auto link_for_sweep = [&f](int start) {
        struct Open {
            int enter;
            bool left;
        };
        std::vector<Open> open;
        int n_csg = 0;
        for (int pc = start; pc < (int)f.ops.size(); pc++) {
            DevCsgOp& op = f.ops[pc];
            if (op.op == OP_CSG_ENTER) {
                if (!open.empty()) op.pad = open.back().enter - start;
                f.ops[op.skip - 1].pad = (n_csg++ << 1) | (!open.empty() && open.back().left ? 1 : 0);
                open.push_back(Open{pc, true});
            } else if (op.op == OP_CSG_MID) {
                open.back().left = false;
            } else if (op.op == OP_CSG_EXIT) {
                open.pop_back();
            } else if (op.op == OP_PRIM) {
                op.pad = ((open.back().enter - start) << 1) | (open.back().left ? 1 : 0);
            }
        }
        f.ops[start].pad = -n_csg;
        return n_csg;
    };
    // RTC_CSG_SWEEP=1 (test aid, read on every commit): every CSG goes to csg_sweep, so that scenes csg_eval accepts can
    // be rendered both ways and compared.
    const char* sweep_env = getenv("RTC_CSG_SWEEP");
    const bool sweep_all = sweep_env && atoi(sweep_env) != 0;
    for (int i = 0; i < nn; i++) {
        if (csg_pos[i] < 0) continue;
        int start = (int)f.ops.size();
        emitter.max_depth = 0;
        const int worst = emitter.emit(~i, 0);
        if (sweep_all || worst > kCsgHitCap || emitter.max_depth > kCsgRayDepth - 1) {
            // beyond csg_eval's hit buffer or ray stack: the same program, evaluated by csg_sweep
            if (emitter.max_depth > kCsgSweepDepth - 1)
                return fail(RTC_ERR_CAPACITY, "CSG nesting depth " + std::to_string(emitter.max_depth) + " exceeds " +
                                                  std::to_string(kCsgSweepDepth - 1));
            const int n_csg = link_for_sweep(start);
            f.csg_sweep = true;
            if (n_csg > kCsgSweepNodes)
                return fail(RTC_ERR_CAPACITY, "a CSG holds " + std::to_string(n_csg) + " CSG nodes; at most " +
                                                  std::to_string(kCsgSweepNodes) + " are supported");
        }
        int pos = csg_pos[i];
        // order: depth-first index of the CSG's first leaf (ties are resolved with the leaves' own orders)
        // RTC_OPT_EXACT_GROUPS: a CSG inside a group is evaluated only when its chain of group boxes passes
        const int csg_flags = kFlagCastsShadow | (s->exact_groups && s->nodes[i].parent >= 0 ? kFlagHasParent : 0);
        f.head[pos] = make_int4(T_CSG | (csg_flags << 4), 0, start, 0);
        f.head[f.n_pos + pos] = make_int4(s->nodes[i].parent, -1, 0, 0);
    }

    if (f.ops.size() >= (1u << 29))  // csg_sweep's keys hold a PRIM instruction's position << 2
        return fail(RTC_ERR_CAPACITY, "CSG programs exceed 2^29 instructions");
    lap("nodes + csg programs");
    // ---- traversal records: head + the rows the intersection test needs, one 64 B fetch per primitive
    f.rec.resize(4 * (size_t)f.n_pos);
    parallel_for((size_t)f.n_pos, kGrain, [&](size_t b, size_t e, int) {
        for (size_t pos = b; pos < e; pos++) {
            int4 h = f.head[pos];
            memcpy(&f.rec[4 * pos], &h, sizeof(h));
            int type = h.x & 15;
            if (type == T_CSG) {
                for (int r = 0; r < 3; r++) f.rec[4 * pos + 1 + r] = make_float4(0.f, 0.f, 0.f, 0.f);
                continue;
            }
            const float4* src = (type == T_TRIANGLE) ? &f.tri[3 * (size_t)h.z] : &f.xform[3 * (size_t)h.y];
            for (int r = 0; r < 3; r++) f.rec[4 * pos + 1 + r] = src[r];
        }
    });

    if (int rc = build_shading_tables(s, f)) return rc;
    plan_small_scene(s, f, n_items);
    lap("records, tables, small scene");
    s->n_bvh_nodes = (int)f.bvh.size();
    s->n_linear = (int)f.linear.size();
    s->n_xforms = (int)f.xform.size() / 3;
    return 0;
}

}  // namespace rtc
