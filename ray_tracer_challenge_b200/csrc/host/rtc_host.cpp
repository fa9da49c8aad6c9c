// rtc_host.cpp — the flat C binding (include/rtc_scene.h) of the C++ host mirror in rtc_host.hpp, the OBJ
// loader, and Camera::render_b200: flatten -> rtc_scene_commit -> rtc_render through the C ABI of
// include/rtc_b200.h.  This library links against librtc_b200.so and nothing else; in particular it never
// touches the CPU oracle.
#include "rtc_host.hpp"

#include <chrono>
#include <memory>
#include <sstream>

#include "../../../include/rtc_scene.h"

using namespace rtch;

namespace rtch {

namespace {
void normalize_vertices(std::vector<Vec3>& v) {  // obj_parser.rs:250-264
    Bounds b;
    for (size_t i = 1; i < v.size(); i++) b.add(v[i]);
    float span[3] = {b.hi[0] - b.lo[0], b.hi[1] - b.lo[1], b.hi[2] - b.lo[2]};
    float scale = fmaxf(span[0], fmaxf(span[1], span[2])) / 2.f;
    for (size_t i = 1; i < v.size(); i++) {
        v[i].x = (v[i].x - (b.lo[0] + span[0] / 2.f)) / scale;
        v[i].y = (v[i].y - (b.lo[1] + span[1] / 2.f)) / scale;
        v[i].z = (v[i].z - (b.lo[2] + span[2] / 2.f)) / scale;
    }
}
}  // namespace

int SceneGraph::parse_obj(const std::string& text) {
    std::vector<Vec3> vertices{Vec3{}}, normals{Vec3{}};  // 1-based, obj_parser.rs:104-105
    std::vector<std::string> names;
    std::vector<int> group_ids;
    int current = -1;
    bool normalized = false;
    auto open_group = [&](const std::string& name) {
        int g = add(GROUP);
        for (size_t i = 0; i < names.size(); i++)
            if (names[i] == name) {  // HashMap::insert replaces an existing entry
                group_ids[i] = g;
                return g;
            }
        names.push_back(name);
        group_ids.push_back(g);
        return g;
    };
    std::istringstream in(text);
    std::string line;
    int line_no = 0;
    auto where = [&]() { return " at line " + std::to_string(line_no); };
    for (; std::getline(in, line); line_no++) {
        std::istringstream ls(line);
        std::string head, tok;
        if (!(ls >> head)) continue;
        if (head == "v" || head == "vn") {
            if (head == "v" && normalized) throw Error("vertices must all be specified before any faces" + where());
            float c[3];
            int n = 0;
            while (ls >> tok) {
                char* end = nullptr;
                float f = strtof(tok.c_str(), &end);
                if (end == tok.c_str() || *end) throw Error("malformed number" + where());
                if (n < 3) c[n] = f;
                n++;
            }
            if (n != 3) throw Error("wrong number of coordinates" + where());
            (head == "v" ? vertices : normals).push_back(Vec3{c[0], c[1], c[2]});
        } else if (head == "f") {
            if (!normalized) {
                normalize_vertices(vertices);
                normalized = true;
            }
            std::vector<size_t> vi;
            bool first_has_normal = false;
            while (ls >> tok) {  // parse_face, obj_parser.rs:224-247: v, v/t, v//n, v/t/n
                size_t s1 = tok.find('/');
                std::string vs = tok.substr(0, s1);
                if (vs.empty()) throw Error("Missing vertex index");
                for (char ch : tok)
                    if (ch != '/' && (ch < '0' || ch > '9')) throw Error("malformed face index" + where());
                bool has_normal = false;
                if (s1 != std::string::npos) {
                    size_t s2 = tok.find('/', s1 + 1);
                    has_normal = s2 != std::string::npos && s2 + 1 < tok.size();
                }
                if (vi.empty()) first_has_normal = has_normal;
                vi.push_back((size_t)strtoull(vs.c_str(), nullptr, 10));
            }
            if (vi.size() < 3) throw Error("not enough vertices to form a face" + where());
            if (current < 0) current = open_group("");
            for (size_t i = 1; i + 1 < vi.size(); i++) {  // fan_triangulation, obj_parser.rs:267-293
                size_t idx[3] = {vi[0], vi[i], vi[i + 1]};
                for (size_t k : idx) {
                    if (k >= vertices.size()) throw Error("vertex index out of range" + where());
                    // smooth triangles index the normals with the vertex index (obj_parser.rs:283-285)
                    if (first_has_normal && k >= normals.size()) throw Error("normal index out of range" + where());
                }
                const Vec3 &a = vertices[idx[0]], &b = vertices[idx[1]], &c = vertices[idx[2]];
                float p1[3] = {a.x, a.y, a.z}, p2[3] = {b.x, b.y, b.z}, p3[3] = {c.x, c.y, c.z};
                int t = add_triangle(p1, p2, p3, first_has_normal);
                add_child(current, t);
            }
        } else if (head == "g") {
            std::string name;
            if (!(ls >> name)) throw Error("Missing group name" + where());
            current = open_group(name);
        }
    }
    if (group_ids.empty()) throw Error("OBJ data defines no faces");
    if (group_ids.size() == 1) return group_ids[0];
    int all = add(GROUP);
    for (int g : group_ids) add_child(all, g);
    return all;
}

}  // namespace rtch

// ---------------------------------------------------------------------------------------------- C binding
namespace {
thread_local std::string g_err;
int fail(const std::string& m) {
    g_err = m;
    return -1;
}
struct Prepared {
    RtcScene* scene = nullptr;
    FlatScene flat;
    uint32_t width = 0, height = 0;  // the committed canvas
};
}  // namespace

struct sg_ctx {
    SceneGraph graph;
    std::vector<Material> materials;
    std::vector<World> worlds;
    std::vector<Camera> cameras;
    RenderOptions options;
    RtcStats last_stats{};
    std::vector<std::unique_ptr<Prepared>> prepared;
    ~sg_ctx() {
        for (auto& p : prepared)
            if (p && p->scene) rtc_scene_destroy(p->scene);
    }
};

#define SG_GUARD(...)                      \
    try {                                  \
        __VA_ARGS__                        \
    } catch (const std::exception& e) {    \
        return fail(e.what());             \
    }

static Mat4 mat(const float* p) {
    Mat4 m;
    memcpy(m.m, p, sizeof(m.m));
    return m;
}
static void out16(const Mat4& m, float* o) { memcpy(o, m.m, sizeof(m.m)); }

static void to_sg_stats(const RtcStats& r, sg_stats* s) {
    if (!s) return;
    s->primary_rays = r.primary_rays, s->secondary_rays = r.secondary_rays, s->shadow_rays = r.shadow_rays;
    s->shades = r.shades, s->flops = r.flops, s->ms = r.kernel_ms, s->ms_total = r.total_ms;
}

// one_shot: the scene is rendered once and dropped (Camera::render_b200: the reference's render consumes its World,
// camera.rs:76) — for a big scene the tree is then built on the device (RTC_OPT_BVH_BUILDER), where a millisecond buys a
// tree a little worse than the host's 25-30 ms binned SAH; a scene kept resident (sg_prepare) gets the better tree.
static int commit(sg_ctx* c, RtcScene* scene, bool one_shot, size_t n_prims) {
    const RenderOptions& o = c->options;
    if (rtc_set_option(scene, RTC_OPT_FMA_CONTRACTION, o.fma ? 1 : 0)) return fail(rtc_last_error());
    const bool device_tree = o.bvh_builder < 0 ? (one_shot && n_prims >= 10000) : o.bvh_builder != 0;
    if (rtc_set_option(scene, RTC_OPT_BVH_BUILDER, device_tree ? 1 : 0)) return fail(rtc_last_error());
    if (rtc_set_option(scene, RTC_OPT_EXACT_GROUPS, o.exact_groups ? 1 : 0)) return fail(rtc_last_error());
    const int32_t* ids = o.device_ids.empty() ? nullptr : o.device_ids.data();
    int n = o.device_ids.empty() ? o.n_devices : (int)o.device_ids.size();
    if (rtc_scene_commit(scene, n, ids)) return fail(rtc_last_error());
    return 0;
}

extern "C" {

const char* sg_last_error(void) { return g_err.c_str(); }

void sg_translation(float x, float y, float z, float out[16]) { out16(translation(x, y, z), out); }
void sg_scaling(float x, float y, float z, float out[16]) { out16(scaling(x, y, z), out); }
void sg_rotation_x(float r, float out[16]) { out16(rotation_x(r), out); }
void sg_rotation_y(float r, float out[16]) { out16(rotation_y(r), out); }
void sg_rotation_z(float r, float out[16]) { out16(rotation_z(r), out); }
void sg_shearing(float xy, float xz, float yx, float yz, float zx, float zy, float out[16]) {
    out16(shearing(xy, xz, yx, yz, zx, zy), out);
}
void sg_view_transform(const float from[3], const float to[3], const float up[3], float out[16]) {
    out16(view_transform(Vec3{from[0], from[1], from[2]}, Vec3{to[0], to[1], to[2]}, Vec3{up[0], up[1], up[2]}), out);
}
void sg_matmul(const float a[16], const float b[16], float out[16]) { out16(mat(a) * mat(b), out); }
void sg_inverse(const float m[16], float out[16]) { out16(inverse(mat(m)), out); }
void sg_transpose(const float m[16], float out[16]) { out16(transpose(mat(m)), out); }
float sg_determinant(const float m[16]) { return determinant(mat(m)); }

sg_ctx* sg_create(void) { return new sg_ctx(); }
void sg_destroy(sg_ctx* c) { delete c; }

int sg_pattern_new(sg_ctx* c, int kind, const float a[3], const float b[3]) {
    if (kind < SG_PAT_STRIPES || kind > SG_PAT_TEST) return fail("sg_pattern_new: bad kind");
    Pattern p;
    p.kind = kind;
    if (a) memcpy(p.a, a, 12);
    if (b) memcpy(p.b, b, 12);
    c->graph.patterns.push_back(p);
    return (int)c->graph.patterns.size() - 1;
}
int sg_pattern_set_transform(sg_ctx* c, int pattern, const float m[16]) {
    if (pattern < 0 || pattern >= (int)c->graph.patterns.size()) return fail("bad pattern handle");
    c->graph.patterns[pattern].inv = inverse(mat(m));  // pattern.rs:53-55
    return 0;
}
int sg_uv_pattern_new(sg_ctx* c, int kind, const float* params, int n) {
    if (!((kind == SG_UV_CHECKERS && n == 8) || (kind == SG_UV_ALIGN_CHECK && n == 15))) return fail("bad uv pattern parameters");
    UvPattern u;
    u.kind = kind;
    memcpy(u.params, params, n * sizeof(float));
    c->graph.uvs.push_back(u);
    return (int)c->graph.uvs.size() - 1;
}
int sg_canvas_new(sg_ctx* c, int w, int h, const float* rgb) {
    if (w < 0 || h < 0) return fail("bad canvas size");
    CanvasRec cv;
    cv.width = w, cv.height = h;
    cv.rgb.assign((size_t)w * h * 3, 0.0f);  // Canvas::new: black (canvas.rs:19-25)
    if (rgb) memcpy(cv.rgb.data(), rgb, cv.rgb.size() * sizeof(float));
    c->graph.canvases.push_back(std::move(cv));
    return (int)c->graph.canvases.size() - 1;
}
int sg_canvas_from_ppm(sg_ctx* c, const char* text, int64_t n) {
    SG_GUARD(c->graph.canvases.push_back(canvas_from_ppm(text, (size_t)n)); return (int)c->graph.canvases.size() - 1;)
}
int sg_canvas_size(sg_ctx* c, int cv, int* w, int* h) {
    if (cv < 0 || cv >= (int)c->graph.canvases.size()) return fail("bad canvas handle");
    *w = c->graph.canvases[cv].width, *h = c->graph.canvases[cv].height;
    return 0;
}
int sg_canvas_pixels(sg_ctx* c, int cv, float* out) {
    if (cv < 0 || cv >= (int)c->graph.canvases.size()) return fail("bad canvas handle");
    const CanvasRec& k = c->graph.canvases[cv];
    memcpy(out, k.rgb.data(), k.rgb.size() * sizeof(float));
    return 0;
}
int64_t sg_canvas_to_ppm(sg_ctx* c, int cv, char* out, int64_t capacity) {
    if (cv < 0 || cv >= (int)c->graph.canvases.size()) return fail("bad canvas handle");
    SG_GUARD(std::string ppm = canvas_to_ppm(c->graph.canvases[cv]);
             if (out && capacity > 0) memcpy(out, ppm.data(), (size_t)std::min<int64_t>(capacity, (int64_t)ppm.size()));
             return (int64_t)ppm.size();)
}
// Canvas::to_ppm (canvas.rs:58-96) from an 8-bit plane (width * height * 3, the device's scale_color values)
int64_t sg_ppm_from_u8(sg_ctx*, int width, int height, const uint8_t* u8, char* out, int64_t capacity) {
    if (width < 0 || height < 0 || (!u8 && width * height)) return fail("bad 8-bit canvas");
    SG_GUARD(std::string ppm = ppm_from_u8(width, height, u8);
             if (out && capacity > 0) memcpy(out, ppm.data(), (size_t)std::min<int64_t>(capacity, (int64_t)ppm.size()));
             return (int64_t)ppm.size();)
}
int sg_uv_image_new(sg_ctx* c, int cv) {
    if (cv < 0 || cv >= (int)c->graph.canvases.size()) return fail("bad canvas handle");
    if (c->graph.canvases[cv].width < 1 || c->graph.canvases[cv].height < 1) return fail("UVImage needs a non-empty canvas");
    UvPattern u;
    u.kind = SG_UV_IMAGE;
    u.canvas = cv;
    c->graph.uvs.push_back(u);
    return (int)c->graph.uvs.size() - 1;
}
int sg_texture_map_new(sg_ctx* c, int uv, int mapping) {
    if (uv < 0 || uv >= (int)c->graph.uvs.size()) return fail("bad uv handle");
    if (mapping < 0 || mapping > 2) return fail("bad mapping");
    Pattern p;
    p.kind = SG_PAT_TEXTURE_MAP;
    p.uv[0] = uv;
    p.mapping = mapping;
    c->graph.patterns.push_back(p);
    return (int)c->graph.patterns.size() - 1;
}
int sg_cubic_map_new(sg_ctx* c, const int uv[6]) {
    Pattern p;
    p.kind = SG_PAT_CUBIC_MAP;
    for (int i = 0; i < 6; i++) {
        if (uv[i] < 0 || uv[i] >= (int)c->graph.uvs.size()) return fail("bad uv handle");
        p.uv[i] = uv[i];
    }
    c->graph.patterns.push_back(p);
    return (int)c->graph.patterns.size() - 1;
}
int sg_material_new(sg_ctx* c, const float p[10], int pattern) {
    if (pattern >= (int)c->graph.patterns.size()) return fail("bad pattern handle");
    Material m;
    memcpy(m.color, p, 12);
    m.ambient = p[3], m.diffuse = p[4], m.specular = p[5], m.shininess = p[6];
    m.reflective = p[7], m.transparency = p[8], m.refractive_index = p[9];
    m.pattern = pattern < 0 ? -1 : pattern;
    c->materials.push_back(m);
    return (int)c->materials.size() - 1;
}

int sg_shape_new(sg_ctx* c, int kind) {
    switch (kind) {
        case SG_SPHERE: return c->graph.add(SPHERE);
        case SG_PLANE: return c->graph.add(PLANE);
        case SG_CUBE: return c->graph.add(CUBE);
        case SG_CYLINDER: return c->graph.add(CYLINDER);
        case SG_CONE: return c->graph.add(CONE);
        case SG_GROUP: return c->graph.add(GROUP);
    }
    return fail("sg_shape_new: unsupported kind (the reference's TestShape double exists only in the oracle)");
}
int sg_triangle_new(sg_ctx* c, const float p1[3], const float p2[3], const float p3[3]) {
    return c->graph.add_triangle(p1, p2, p3, false);
}
int sg_smooth_triangle_new(sg_ctx* c, const float p[9], const float n[9]) {
    (void)n;  // the render path never reads the vertex normals (smooth_triangle.rs:39-41, SURVEY Q5)
    return c->graph.add_triangle(p, p + 3, p + 6, true);
}
int sg_csg_new(sg_ctx* c, int op, int s1, int s2) {
    if (op < 0 || op > 2) return fail("bad csg op");
    SG_GUARD(return c->graph.add_csg(op, s1, s2);)
}
int sg_shape_clone(sg_ctx* c, int h) { SG_GUARD(return c->graph.clone(h);) }
int sg_shape_set_transform(sg_ctx* c, int h, const float m[16]) { SG_GUARD(c->graph.set_transform(h, mat(m)); return 0;) }
int sg_shape_set_material(sg_ctx* c, int h, int m) {
    if (m < 0 || m >= (int)c->materials.size()) return fail("bad material handle");
    SG_GUARD(c->graph.set_material(h, c->materials[m]); return 0;)
}
int sg_shape_set_casts_shadow(sg_ctx* c, int h, int v) {
    SG_GUARD(c->graph.check(h); c->graph.shapes[h].casts_shadow = v != 0; return 0;)
}
int sg_shape_set_bounds(sg_ctx* c, int h, float lo, float hi, int closed) {
    SG_GUARD(c->graph.check(h); ShapeRec& s = c->graph.shapes[h];
             if (s.kind != CYLINDER && s.kind != CONE) return fail("sg_shape_set_bounds: not a cylinder or cone");
             s.y_min = lo, s.y_max = hi, s.closed = closed != 0; return 0;)
}
int sg_group_add_child(sg_ctx* c, int g, int child) { SG_GUARD(c->graph.add_child(g, child); return 0;) }
int sg_shape_divide(sg_ctx* c, int h, int threshold) { SG_GUARD(c->graph.divide(h, (size_t)threshold); return 0;) }
int sg_parse_obj(sg_ctx* c, const char* text, int64_t n) { SG_GUARD(return c->graph.parse_obj(std::string(text, (size_t)n));) }

int sg_shape_kind(sg_ctx* c, int h) { SG_GUARD(c->graph.check(h); return c->graph.shapes[h].kind;) }
int sg_shape_get_transform(sg_ctx* c, int h, float out[16]) { SG_GUARD(c->graph.check(h); out16(c->graph.shapes[h].t, out); return 0;) }
int sg_shape_get_inverse(sg_ctx* c, int h, float out[16]) { SG_GUARD(c->graph.check(h); out16(c->graph.shapes[h].t_inv, out); return 0;) }
int sg_shape_get_inverse_transpose(sg_ctx* c, int h, float out[16]) {
    SG_GUARD(c->graph.check(h); out16(transpose(c->graph.shapes[h].t_inv), out); return 0;)
}
int sg_shape_bounding_box(sg_ctx* c, int h, float mn[3], float mx[3]) {
    SG_GUARD(Bounds b = c->graph.bounding_box(h); memcpy(mn, b.lo, 12); memcpy(mx, b.hi, 12); return 0;)
}
int sg_shape_parent_space_bounding_box(sg_ctx* c, int h, float mn[3], float mx[3]) {
    SG_GUARD(c->graph.check(h); Bounds b = c->graph.parent_space_box(h); memcpy(mn, b.lo, 12); memcpy(mx, b.hi, 12); return 0;)
}
int sg_group_child_count(sg_ctx* c, int g) {
    SG_GUARD(c->graph.check(g); int k = c->graph.shapes[g].kind; if (k != GROUP && k != CSG) return fail("not a group");
             return (int)c->graph.shapes[g].children.size();)
}
int sg_group_child(sg_ctx* c, int g, int i) {
    SG_GUARD(c->graph.check(g); const auto& kids = c->graph.shapes[g].children;
             if (i < 0 || i >= (int)kids.size()) return fail("child index out of range"); return kids[i];)
}
int sg_triangle_get(sg_ctx* c, int h, float out[12]) {
    SG_GUARD(c->graph.check(h); const ShapeRec& s = c->graph.shapes[h];
             if (s.kind != TRIANGLE && s.kind != SMOOTH_TRIANGLE) return fail("not a triangle");
             memcpy(out, s.tri, sizeof(s.tri)); return 0;)
}

int sg_world_new(sg_ctx* c) {
    c->worlds.emplace_back();
    return (int)c->worlds.size() - 1;
}
int sg_world_add_object(sg_ctx* c, int w, int h) {
    if (w < 0 || w >= (int)c->worlds.size()) return fail("bad world handle");
    SG_GUARD(c->graph.check(h); c->worlds[w].objects.push_back(h); return 0;)
}
int sg_world_set_point_light(sg_ctx* c, int w, const float pos[3], const float intensity[3]) {
    if (w < 0 || w >= (int)c->worlds.size()) return fail("bad world handle");
    Light l;
    l.set = true;
    memcpy(l.position, pos, 12);
    memcpy(l.intensity, intensity, 12);
    c->worlds[w].light = l;
    return 0;
}
int sg_world_set_rect_light(sg_ctx* c, int w, const float intensity[3], const float corner[3], const float u_vec[3], int u_steps,
                            const float v_vec[3], int v_steps, const float* jitter, int n_jitter, uint64_t seed) {
    if (w < 0 || w >= (int)c->worlds.size()) return fail("bad world handle");
    if (u_steps < 1 || v_steps < 1) return fail("light steps must be >= 1");
    c->worlds[w].light = rectangle_light(intensity, corner, u_vec, u_steps, v_vec, v_steps, jitter, n_jitter, seed);
    return 0;
}
int sg_camera_new(sg_ctx* c, uint32_t w, uint32_t h, float fov, const float m[16]) {
    c->cameras.emplace_back(w, h, fov, mat(m));
    return (int)c->cameras.size() - 1;
}

// ---- host-library extensions (not exported by the oracle) ------------------------------------------------
// devices the next render / prepare commits to (device_ids may be NULL: 0..n_devices-1); fma selects the
// FMA-contracted kernel build (RTC_OPT_FMA_CONTRACTION); detailed adds the Appendix-E work counters to the stats.
int sg_set_render_options(sg_ctx* c, int n_devices, const int* device_ids, int fma, int detailed) {
    c->options.n_devices = n_devices;
    c->options.device_ids.clear();
    if (device_ids) c->options.device_ids.assign(device_ids, device_ids + n_devices);
    c->options.fma = fma != 0;
    c->options.detailed = detailed != 0;
    return 0;
}
// -1 (default): automatic — the device builder for one-shot renders of >= 10 000 primitives; 0 / 1: always host / device
int sg_set_bvh_builder(sg_ctx* c, int mode) {
    c->options.bvh_builder = mode < 0 ? -1 : (mode != 0);
    return 0;
}
// RTC_OPT_EXACT_GROUPS (0 / 1) for every later commit of this context: one-shot renders, sg_prepare and sg_inspect
int sg_set_exact_groups(sg_ctx* c, int on) {
    if (on != 0 && on != 1) return fail("exact groups: 0 or 1");
    c->options.exact_groups = on != 0;
    return 0;
}
int sg_last_rtc_stats(sg_ctx* c, RtcStats* out) {
    *out = c->last_stats;
    return 0;
}

// Camera::render_b200 — one call: flatten, commit, render, copy back, release.  With n_shards > 1 the call renders
// and copies only the bands of `shard` (one process per GPU, every process making the same one-shot call on its own
// device for one shared frame); either plane may be null (not copied: the reference's demos only ever serialise the
// 8-bit values, canvas.rs:58-96).
static int camera_render(sg_ctx* c, int cam, int w, int depth, int shard, int n_shards, float* out_rgb, uint8_t* out_u8,
                         sg_stats* stats) {
    if (cam < 0 || cam >= (int)c->cameras.size()) return fail("bad camera handle");
    if (w < 0 || w >= (int)c->worlds.size()) return fail("bad world handle");
    RtcScene* scene = nullptr;
    if (rtc_scene_create(&scene)) return fail(rtc_last_error());
    int rc = 0;
    try {
        auto t0 = std::chrono::steady_clock::now();
        const bool timing = getenv("RTC_TIMING") != nullptr;  // tuning aid: where a one-shot render spends its time
        auto mark = [&, last = t0](const char* what) mutable {
            if (!timing) return;
            const auto now = std::chrono::steady_clock::now();
            fprintf(stderr, "[rtc one-shot] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - last).count());
            last = now;
        };
        FlatScene flat;
        fill_scene(scene, c->graph, c->worlds[w], c->cameras[cam], flat);
        mark("fill_scene");
        rc = commit(c, scene, true, flat.n_prims);
        mark("commit (host half + upload)");
        if (!rc) {
            if (n_shards > 1)
                rc = rtc_render_shard(scene, depth, shard, n_shards, out_rgb, out_u8, &c->last_stats);
            else
                rc = c->options.detailed ? rtc_render_detailed(scene, depth, out_rgb, out_u8, &c->last_stats)
                                         : rtc_render(scene, depth, out_rgb, out_u8, &c->last_stats);
            if (rc) fail(rtc_last_error());
            mark("render + copies");
        }
        c->last_stats.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        to_sg_stats(c->last_stats, stats);
    } catch (const std::exception& e) {
        rc = fail(e.what());
    }
    const auto t1 = std::chrono::steady_clock::now();
    rtc_scene_destroy(scene);
    if (getenv("RTC_TIMING"))
        fprintf(stderr, "[rtc one-shot] %-28s %8.3f ms\n", "scene destroy",
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t1).count());
    return rc ? -1 : 0;
}
int sg_camera_render(sg_ctx* c, int cam, int w, int depth, float* out_rgb, uint8_t* out_u8, sg_stats* stats) {
    return camera_render(c, cam, w, depth, 0, 1, out_rgb, out_u8, stats);
}
int sg_camera_render_shard(sg_ctx* c, int cam, int w, int depth, int shard, int n_shards, float* out_rgb, uint8_t* out_u8,
                           sg_stats* stats) {
    if (n_shards < 1 || shard < 0 || shard >= n_shards) return fail("bad shard index");
    return camera_render(c, cam, w, depth, shard, n_shards, out_rgb, out_u8, stats);
}

// A batch of views: the cameras' RtcViews, every camera of the committed canvas size (or the call fails)
static int camera_views(sg_ctx* c, const int* cams, int n, uint32_t width, uint32_t height, std::vector<RtcView>& out) {
    if (n < 1 || !cams) return fail("a batch needs at least one camera");
    out.clear();
    for (int i = 0; i < n; i++) {
        if (cams[i] < 0 || cams[i] >= (int)c->cameras.size()) return fail("bad camera handle");
        const Camera& k = c->cameras[cams[i]];
        if (k.width != width || k.height != height)
            return fail("camera " + std::to_string(i) + " of the batch is " + std::to_string(k.width) + "x" + std::to_string(k.height) +
                        ", the scene's canvas is " + std::to_string(width) + "x" + std::to_string(height) +
                        ": every view of a batch has the committed canvas size");
        out.push_back(camera_view(k));
    }
    return 0;
}
// The camera of a batch whose origin lies farthest out (largest coordinate magnitude; the first of equals): committing with
// it gives the tree the reach every view of the batch needs (rtc_render_views)
static int farthest_camera(const sg_ctx* c, const int* cams, int n) {
    int best = 0;
    float far = -1.f;
    for (int i = 0; i < n; i++) {
        const Mat4& m = c->cameras[cams[i]].transform_inverse;
        const float r = std::max(std::fabs(m.m[3]), std::max(std::fabs(m.m[7]), std::fabs(m.m[11])));
        if (r > far) far = r, best = i;
    }
    return best;
}

// rtc_scene_inspect for (camera, world): flatten + the host half of the commit, no device needed.  `info` is an
// RtcCommitInfo (include/rtc_b200.h); flatten_ms receives the time of the scene-graph flattening itself.
int sg_inspect(sg_ctx* c, int cam, int w, void* info, double* flatten_ms) {
    if (cam < 0 || cam >= (int)c->cameras.size()) return fail("bad camera handle");
    if (w < 0 || w >= (int)c->worlds.size()) return fail("bad world handle");
    RtcScene* scene = nullptr;
    if (rtc_scene_create(&scene)) return fail(rtc_last_error());
    int rc = 0;
    try {
        FlatScene flat;
        const auto t0 = std::chrono::steady_clock::now();
        fill_scene(scene, c->graph, c->worlds[w], c->cameras[cam], flat);
        if (flatten_ms) *flatten_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        if (rtc_set_option(scene, RTC_OPT_EXACT_GROUPS, c->options.exact_groups ? 1 : 0) ||
            rtc_scene_inspect(scene, static_cast<RtcCommitInfo*>(info)))
            rc = fail(rtc_last_error());
    } catch (const std::exception& e) {
        rc = fail(e.what());
    }
    rtc_scene_destroy(scene);
    return rc;
}

// The flattened (camera, world) as an RtcScene of include/rtc_b200.h that the CALLER owns (rtc_scene_destroy): for a
// host that drives the C ABI itself from here on — rtc_scene_inspect, rtc_scene_commit on devices of its choice,
// rtc_trace_rays — and for the test harness that runs the device code on the host (tests/emu).
int sg_export_scene(sg_ctx* c, int cam, int w, void** out_scene) {
    if (!out_scene) return fail("null out pointer");
    if (cam < 0 || cam >= (int)c->cameras.size()) return fail("bad camera handle");
    if (w < 0 || w >= (int)c->worlds.size()) return fail("bad world handle");
    RtcScene* scene = nullptr;
    if (rtc_scene_create(&scene)) return fail(rtc_last_error());
    try {
        FlatScene flat;
        fill_scene(scene, c->graph, c->worlds[w], c->cameras[cam], flat);
    } catch (const std::exception& e) {
        rtc_scene_destroy(scene);
        return fail(e.what());
    }
    *out_scene = scene;
    return 0;
}

// Keep a committed scene resident on the device(s) for repeated renders (animation / benchmarking).
int sg_prepare(sg_ctx* c, int cam, int w) {
    if (cam < 0 || cam >= (int)c->cameras.size()) return fail("bad camera handle");
    if (w < 0 || w >= (int)c->worlds.size()) return fail("bad world handle");
    auto p = std::make_unique<Prepared>();
    if (rtc_scene_create(&p->scene)) return fail(rtc_last_error());
    try {
        fill_scene(p->scene, c->graph, c->worlds[w], c->cameras[cam], p->flat);
    } catch (const std::exception& e) {
        rtc_scene_destroy(p->scene);
        return fail(e.what());
    }
    if (commit(c, p->scene, false, p->flat.n_prims)) {
        rtc_scene_destroy(p->scene);
        return -1;
    }
    p->width = c->cameras[cam].width, p->height = c->cameras[cam].height;
    c->prepared.push_back(std::move(p));
    return (int)c->prepared.size() - 1;
}
int sg_release_prepared(sg_ctx* c, int h) {
    if (h < 0 || h >= (int)c->prepared.size() || !c->prepared[h]) return fail("bad prepared handle");
    rtc_scene_destroy(c->prepared[h]->scene);
    c->prepared[h].reset();
    return 0;
}
// n_shards == 0: the committed devices split the frame; n_shards >= 1: this process renders only `shard`.
int sg_render_prepared(sg_ctx* c, int h, int depth, int shard, int n_shards, int detailed, int fma, float* out_rgb,
                       uint8_t* out_u8, sg_stats* stats) {
    if (h < 0 || h >= (int)c->prepared.size() || !c->prepared[h]) return fail("bad prepared handle");
    RtcScene* scene = c->prepared[h]->scene;
    if (rtc_set_option(scene, RTC_OPT_FMA_CONTRACTION, fma ? 1 : 0)) return fail(rtc_last_error());
    int rc;
    if (n_shards >= 1)
        rc = rtc_render_shard(scene, depth, shard, n_shards, out_rgb, out_u8, &c->last_stats);
    else if (detailed)
        rc = rtc_render_detailed(scene, depth, out_rgb, out_u8, &c->last_stats);
    else
        rc = rtc_render(scene, depth, out_rgb, out_u8, &c->last_stats);
    to_sg_stats(c->last_stats, stats);
    return rc ? fail(rtc_last_error()) : 0;
}
// rtc_render_views on a prepared scene: n cameras (handles) of its canvas size, frames view-major in out_rgb / out_u8
int sg_render_prepared_views(sg_ctx* c, int h, int depth, int n, const int* cams, int fma, float* out_rgb, uint8_t* out_u8,
                             sg_stats* stats) {
    if (h < 0 || h >= (int)c->prepared.size() || !c->prepared[h]) return fail("bad prepared handle");
    RtcScene* scene = c->prepared[h]->scene;
    std::vector<RtcView> views;
    if (camera_views(c, cams, n, c->prepared[h]->width, c->prepared[h]->height, views)) return -1;
    if (rtc_set_option(scene, RTC_OPT_FMA_CONTRACTION, fma ? 1 : 0)) return fail(rtc_last_error());
    const int rc = rtc_render_views(scene, depth, (uint32_t)n, views.data(), out_rgb, out_u8, &c->last_stats);
    to_sg_stats(c->last_stats, stats);
    return rc ? fail(rtc_last_error()) : 0;
}
// The one-shot form (Camera::render_b200 for a batch of cameras): flatten, commit with the camera whose origin is farthest
// out, render every view, release.  The world is consumed once and n canvases come out.
int sg_camera_render_views(sg_ctx* c, const int* cams, int n, int w, int depth, float* out_rgb, uint8_t* out_u8, sg_stats* stats) {
    if (n < 1 || !cams) return fail("a batch needs at least one camera");
    for (int i = 0; i < n; i++)
        if (cams[i] < 0 || cams[i] >= (int)c->cameras.size()) return fail("bad camera handle");
    if (w < 0 || w >= (int)c->worlds.size()) return fail("bad world handle");
    const Camera& first = c->cameras[cams[farthest_camera(c, cams, n)]];
    std::vector<RtcView> views;
    if (camera_views(c, cams, n, first.width, first.height, views)) return -1;
    RtcScene* scene = nullptr;
    if (rtc_scene_create(&scene)) return fail(rtc_last_error());
    int rc = 0;
    try {
        const auto t0 = std::chrono::steady_clock::now();
        FlatScene flat;
        fill_scene(scene, c->graph, c->worlds[w], first, flat);
        rc = commit(c, scene, true, flat.n_prims);
        if (!rc && rtc_render_views(scene, depth, (uint32_t)n, views.data(), out_rgb, out_u8, &c->last_stats)) rc = fail(rtc_last_error());
        c->last_stats.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        to_sg_stats(c->last_stats, stats);
    } catch (const std::exception& e) {
        rc = fail(e.what());
    }
    rtc_scene_destroy(scene);
    return rc ? -1 : 0;
}
// What a batch hands the device library for a camera (the fields fill_scene passes to rtc_set_camera), and which camera of a
// batch the one-shot form commits with — host arithmetic, no device
int sg_camera_view(sg_ctx* c, int cam, RtcView* out) {
    if (cam < 0 || cam >= (int)c->cameras.size() || !out) return fail("bad camera handle");
    *out = camera_view(c->cameras[cam]);
    return 0;
}
int sg_farthest_camera(sg_ctx* c, const int* cams, int n) {
    if (n < 1 || !cams) return fail("a batch needs at least one camera");
    for (int i = 0; i < n; i++)
        if (cams[i] < 0 || cams[i] >= (int)c->cameras.size()) return fail("bad camera handle");
    return farthest_camera(c, cams, n);
}
// rtc_set_option on a prepared scene (RTC_OPT_* of include/rtc_b200.h)
int sg_set_prepared_option(sg_ctx* c, int h, int option, int64_t value) {
    if (h < 0 || h >= (int)c->prepared.size() || !c->prepared[h]) return fail("bad prepared handle");
    return rtc_set_option(c->prepared[h]->scene, option, value) ? fail(rtc_last_error()) : 0;
}
int sg_flush_l2(sg_ctx* c, int h) {
    if (h < 0 || h >= (int)c->prepared.size() || !c->prepared[h]) return fail("bad prepared handle");
    return rtc_flush_l2(c->prepared[h]->scene) ? fail(rtc_last_error()) : 0;
}
// World::color_at for caller-supplied rays on a prepared scene; out_shape receives the hit SHAPE handle.
int sg_trace_rays(sg_ctx* c, int h, uint32_t n, const float* origins, const float* directions, int depth, int fma,
                  float* out_rgb, float* out_t, int* out_shape) {
    if (h < 0 || h >= (int)c->prepared.size() || !c->prepared[h]) return fail("bad prepared handle");
    Prepared& p = *c->prepared[h];
    if (rtc_set_option(p.scene, RTC_OPT_FMA_CONTRACTION, fma ? 1 : 0)) return fail(rtc_last_error());
    std::vector<int32_t> prim(n);
    if (rtc_trace_rays(p.scene, n, origins, directions, depth, out_rgb, out_t, prim.data())) return fail(rtc_last_error());
    if (out_shape)
        for (uint32_t i = 0; i < n; i++) out_shape[i] = prim[i] >= 0 ? p.flat.prim_shape[prim[i]] : -1;
    return 0;
}
// The flattener's output without touching a device (for CPU-only tests): counts = {prims, nodes, refs,
// materials, patterns, uv patterns}; the arrays are copied out when the pointers are non-null.
int sg_flatten(sg_ctx* c, int w, int counts[6], RtcPrim* prims, RtcNode* nodes, int32_t* refs, int* prim_shapes) {
    if (w < 0 || w >= (int)c->worlds.size()) return fail("bad world handle");
    SG_GUARD(FlatScene flat; Flattener(c->graph, flat).run(c->worlds[w]);
             counts[0] = (int)flat.prims.size(), counts[1] = (int)flat.nodes.size(), counts[2] = (int)flat.refs.size();
             counts[3] = (int)flat.materials.size(), counts[4] = (int)flat.patterns.size(), counts[5] = (int)flat.uvs.size();
             if (prims) memcpy(prims, flat.prims.data(), flat.prims.size() * sizeof(RtcPrim));
             if (nodes) memcpy(nodes, flat.nodes.data(), flat.nodes.size() * sizeof(RtcNode));
             if (refs) memcpy(refs, flat.refs.data(), flat.refs.size() * sizeof(int32_t));
             if (prim_shapes) memcpy(prim_shapes, flat.prim_shape.data(), flat.prim_shape.size() * sizeof(int));
             return 0;)
}

}  // extern "C"
