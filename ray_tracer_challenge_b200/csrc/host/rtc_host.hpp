// rtc_host.hpp — C++ host mirror of the reference's `lib` crate for the Camera::render path.
//
// The reference's host is Rust (no toolchain in this image), so the host side above the C ABI is C++.
// It keeps the reference's scene-construction semantics — transforms baked into group children
// (group.rs:39-44,101-114), material push-down (group.rs:96-100), cached group/CSG boxes
// (group.rs:138-150, csg.rs:119-130), the book's `divide` (group.rs:48-77,158-172), the cofactor inverse
// (matrix.rs:145-212) — and adds the one new thing the B200 path needs: the FLATTENER that lowers a World
// into the POD arrays of include/rtc_b200.h, plus Camera::render_b200 which hands them to the device
// library.  Nothing here intersects a ray or shades a pixel.
//
// Layout: shapes live in an arena (SceneGraph) and are addressed by index; this is deliberately not the
// reference's Box<dyn Shape> tree — the flattener wants arrays, not pointers.
#pragma once
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <limits>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../../include/rtc_b200.h"
#include "../rtc_parallel.h"

namespace rtch {

constexpr float kInf = std::numeric_limits<float>::infinity();

struct Error : std::runtime_error {
    using std::runtime_error::runtime_error;
};

// ------------------------------------------------------------------------------------------- math
struct Vec3 {
    float x = 0, y = 0, z = 0;
};

// 4x4 f32, row-major (matrix.rs:9-12).  Every routine keeps the reference's order of operations so that the
// matrices handed to the device are bit-equal to the ones the Rust code would compute.
struct Mat4 {
    float m[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1};
    float& at(int r, int c) { return m[r * 4 + c]; }
    float at(int r, int c) const { return m[r * 4 + c]; }
};

inline Mat4 operator*(const Mat4& a, const Mat4& b) {  // matrix.rs:86-103
    Mat4 o;
    for (int r = 0; r < 4; r++)
        for (int c = 0; c < 4; c++)
            o.at(r, c) = a.at(r, 0) * b.at(0, c) + a.at(r, 1) * b.at(1, c) + a.at(r, 2) * b.at(2, c) + a.at(r, 3) * b.at(3, c);
    return o;
}
inline Mat4 transpose(const Mat4& a) {  // matrix.rs:134-143
    Mat4 o;
    for (int r = 0; r < 4; r++)
        for (int c = 0; c < 4; c++) o.at(c, r) = a.at(r, c);
    return o;
}
namespace detail {
inline float det2(float a, float b, float c, float d) { return a * d - b * c; }  // matrix.rs:147-148
// determinant of the 3x3 matrix q (row-major) by cofactor expansion along row 0, accumulated from 0.0
// exactly like matrix.rs:149-158
inline float det3(const float q[9]) {
    float c0 = det2(q[4], q[5], q[7], q[8]);
    float c1 = -det2(q[3], q[5], q[6], q[8]);
    float c2 = det2(q[3], q[4], q[6], q[7]);
    float det = 0.0f;
    det += c0 * q[0];
    det += c1 * q[1];
    det += c2 * q[2];
    return det;
}
inline float cofactor4(const Mat4& a, int row, int col) {  // matrix.rs:162-195
    float q[9];
    int k = 0;
    for (int r = 0; r < 4; r++) {
        if (r == row) continue;
        for (int c = 0; c < 4; c++) {
            if (c == col) continue;
            q[k++] = a.at(r, c);
        }
    }
    float minor = det3(q);
    return ((row + col) % 2 == 0) ? minor : -minor;
}
}  // namespace detail
inline float determinant(const Mat4& a) {  // matrix.rs:145-159
    float det = 0.0f;
    for (int c = 0; c < 4; c++) det += detail::cofactor4(a, 0, c) * a.at(0, c);
    return det;
}
inline Mat4 inverse(const Mat4& a) {  // matrix.rs:201-212
    float det = determinant(a);
    Mat4 o;
    for (int r = 0; r < 4; r++)
        for (int c = 0; c < 4; c++) o.at(c, r) = detail::cofactor4(a, r, c) / det;
    return o;
}
// matrix.rs:73-84 for a point (w = 1); returns xyz
inline Vec3 mul_point(const Mat4& a, Vec3 p) {
    return {a.at(0, 0) * p.x + a.at(0, 1) * p.y + a.at(0, 2) * p.z + a.at(0, 3) * 1.0f,
            a.at(1, 0) * p.x + a.at(1, 1) * p.y + a.at(1, 2) * p.z + a.at(1, 3) * 1.0f,
            a.at(2, 0) * p.x + a.at(2, 1) * p.y + a.at(2, 2) * p.z + a.at(2, 3) * 1.0f};
}

// transformations.rs:4-68
inline Mat4 translation(float x, float y, float z) {
    Mat4 o;
    o.at(0, 3) = x, o.at(1, 3) = y, o.at(2, 3) = z;
    return o;
}
inline Mat4 scaling(float x, float y, float z) {
    Mat4 o;
    o.at(0, 0) = x, o.at(1, 1) = y, o.at(2, 2) = z;
    return o;
}
inline Mat4 rotation_x(float r) {
    Mat4 o;
    float c = std::cos(r), s = std::sin(r);
    o.at(1, 1) = c, o.at(1, 2) = -s, o.at(2, 1) = s, o.at(2, 2) = c;
    return o;
}
inline Mat4 rotation_y(float r) {
    Mat4 o;
    float c = std::cos(r), s = std::sin(r);
    o.at(0, 0) = c, o.at(0, 2) = s, o.at(2, 0) = -s, o.at(2, 2) = c;
    return o;
}
inline Mat4 rotation_z(float r) {
    Mat4 o;
    float c = std::cos(r), s = std::sin(r);
    o.at(0, 0) = c, o.at(0, 1) = -s, o.at(1, 0) = s, o.at(1, 1) = c;
    return o;
}
inline Mat4 shearing(float xy, float xz, float yx, float yz, float zx, float zy) {
    Mat4 o;
    o.at(0, 1) = xy, o.at(0, 2) = xz, o.at(1, 0) = yx, o.at(1, 2) = yz, o.at(2, 0) = zx, o.at(2, 1) = zy;
    return o;
}
inline Mat4 view_transform(Vec3 from, Vec3 to, Vec3 up) {  // transformations.rs:57-68
    auto normalise = [](Vec3 v) {  // tuple.rs:29-43 with w = 0
        float mag = std::sqrt(v.x * v.x + v.y * v.y + v.z * v.z + 0.0f * 0.0f);
        return Vec3{v.x / mag, v.y / mag, v.z / mag};
    };
    auto cross = [](Vec3 a, Vec3 b) { return Vec3{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; };
    Vec3 forward = normalise({to.x - from.x, to.y - from.y, to.z - from.z});
    Vec3 left = cross(forward, normalise(up));
    Vec3 true_up = cross(left, forward);
    Mat4 o;
    o.at(0, 0) = left.x, o.at(0, 1) = left.y, o.at(0, 2) = left.z;
    o.at(1, 0) = true_up.x, o.at(1, 1) = true_up.y, o.at(1, 2) = true_up.z;
    o.at(2, 0) = -forward.x, o.at(2, 1) = -forward.y, o.at(2, 2) = -forward.z;
    return o * translation(-from.x, -from.y, -from.z);
}

// bounding_box.rs — only what scene construction needs (no ray test on the host)
struct Bounds {
    float lo[3] = {kInf, kInf, kInf}, hi[3] = {-kInf, -kInf, -kInf};
    void add(Vec3 p) {  // :42-50 — Rust f32::min/max ignore NaN, like fminf/fmaxf
        lo[0] = fminf(lo[0], p.x), lo[1] = fminf(lo[1], p.y), lo[2] = fminf(lo[2], p.z);
        hi[0] = fmaxf(hi[0], p.x), hi[1] = fmaxf(hi[1], p.y), hi[2] = fmaxf(hi[2], p.z);
    }
    void add(const Bounds& b) {  // :52-55
        add(Vec3{b.lo[0], b.lo[1], b.lo[2]});
        add(Vec3{b.hi[0], b.hi[1], b.hi[2]});
    }
    bool contains(Vec3 p) const {  // :57-61
        return p.x >= lo[0] && p.x <= hi[0] && p.y >= lo[1] && p.y <= hi[1] && p.z >= lo[2] && p.z <= hi[2];
    }
    bool contains(const Bounds& b) const {  // :63-65
        return contains(Vec3{b.lo[0], b.lo[1], b.lo[2]}) && contains(Vec3{b.hi[0], b.hi[1], b.hi[2]});
    }
    Bounds transformed(const Mat4& t) const {  // :67-84, corners in the reference's order
        Bounds o;
        for (int i = 0; i < 8; i++) {
            Vec3 c{(i & 4) ? hi[0] : lo[0], (i & 2) ? hi[1] : lo[1], (i & 1) ? hi[2] : lo[2]};
            o.add(mul_point(t, c));
        }
        return o;
    }
    void split(Bounds& left, Bounds& right) const {  // :90-125
        float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
        float greatest = fmaxf(fmaxf(dx, dy), dz);
        float a0[3] = {lo[0], lo[1], lo[2]}, a1[3] = {hi[0], hi[1], hi[2]};
        int axis = (greatest == dx) ? 0 : (greatest == dy) ? 1 : 2;
        float d = (axis == 0) ? dx : (axis == 1) ? dy : dz;
        a0[axis] = a0[axis] + d / 2.f;
        a1[axis] = a0[axis];
        left = *this;
        right = *this;
        for (int a = 0; a < 3; a++) left.hi[a] = a1[a], right.lo[a] = a0[a];
    }
};

// ------------------------------------------------------------------------------------------- scene model
enum Kind : int { SPHERE = 0, PLANE, CUBE, CYLINDER, CONE, TRIANGLE, SMOOTH_TRIANGLE, GROUP, CSG };

struct Pattern {  // pattern/*.rs
    int kind = 0;
    Mat4 inv;  // BasePattern::t_inverse
    float a[3] = {1, 1, 1}, b[3] = {0, 0, 0};
    int mapping = 0;
    int uv[6] = {-1, -1, -1, -1, -1, -1};
};
struct UvPattern {
    int kind = 0;
    float params[15] = {0};
    int canvas = -1;  // UVImage (uv.rs:346-377): the canvas handle
};
struct CanvasRec {  // canvas.rs:6-10 as data: width * height * 3 f32, row-major, row 0 at the top
    int width = 0, height = 0;
    std::vector<float> rgb;
};
struct Material {  // material.rs:19-51
    float color[3] = {1, 1, 1};
    float ambient = 0.1f, diffuse = 0.9f, specular = 0.9f, shininess = 200.0f, reflective = 0.0f, transparency = 0.0f,
          refractive_index = 1.0f;
    int pattern = -1;
};
struct Light {
    bool set = false, rect = false;
    float intensity[3] = {1, 1, 1};
    float position[3] = {0, 0, 0};
    float corner[3] = {0, 0, 0}, u_cell[3] = {0, 0, 0}, v_cell[3] = {0, 0, 0};
    int u_steps = 1, v_steps = 1;
    std::vector<float> jitter;
    uint64_t seed = 0;
};

struct ShapeRec {
    int kind = SPHERE;
    Mat4 t, t_inv;  // BaseShape, base_shape.rs:13-20 (the inverse-transpose is transpose(t_inv))
    Material material;
    bool casts_shadow = true;
    float y_min = -kInf, y_max = kInf;  // cylinder / cone
    bool closed = false;
    float tri[12] = {0};  // p1, e1, e2, normal (triangle.rs:20-33)
    float p2[3] = {0}, p3[3] = {0};
    std::vector<int> children;  // group: children; csg: {s1, s2}
    int csg_op = 0;
    bool box_cached = false;  // group.rs:19, csg.rs:23
    Bounds box;
    bool owned = false;  // already adopted by a group / CSG / world
};

class SceneGraph {
   public:
    std::vector<ShapeRec> shapes;
    std::vector<Pattern> patterns;
    std::vector<UvPattern> uvs;
    std::vector<CanvasRec> canvases;

    int add(int kind) {
        ShapeRec s;
        s.kind = kind;
        shapes.push_back(s);
        return (int)shapes.size() - 1;
    }
    int add_triangle(const float p1[3], const float p2[3], const float p3[3], bool smooth) {  // triangle.rs:20-33
        int id = add(smooth ? SMOOTH_TRIANGLE : TRIANGLE);
        ShapeRec& s = shapes[id];
        float e1[3], e2[3];
        for (int a = 0; a < 3; a++) e1[a] = p2[a] - p1[a], e2[a] = p3[a] - p1[a], s.p2[a] = p2[a], s.p3[a] = p3[a];
        // normal = e2.cross(e1).norm()
        float n[3] = {e2[1] * e1[2] - e2[2] * e1[1], e2[2] * e1[0] - e2[0] * e1[2], e2[0] * e1[1] - e2[1] * e1[0]};
        float mag = std::sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2] + 0.0f * 0.0f);
        for (int a = 0; a < 3; a++) s.tri[a] = p1[a], s.tri[3 + a] = e1[a], s.tri[6 + a] = e2[a], s.tri[9 + a] = n[a] / mag;
        return id;
    }
    int add_csg(int op, int s1, int s2) {
        adopt(s1), adopt(s2);
        int id = add(CSG);
        shapes[id].csg_op = op;
        shapes[id].children = {s1, s2};
        return id;
    }
    void adopt(int id) {
        check(id);
        if (shapes[id].owned) throw Error("shape is already owned by a group, CSG or world");
        shapes[id].owned = true;
    }
    void check(int id) const {
        if (id < 0 || id >= (int)shapes.size()) throw Error("bad shape handle");
    }

    // Shape::set_transformation — base_shape.rs:56-60; GroupShape override group.rs:101-114
    void set_transform(int id, const Mat4& t) {
        check(id);
        if (shapes[id].kind == GROUP && !shapes[id].children.empty()) {
            Mat4 child_transformer = t * shapes[id].t_inv;
            std::vector<int> kids = shapes[id].children;
            for (int c : kids) set_transform(c, child_transformer * shapes[c].t);
        }
        shapes[id].t = t;
        shapes[id].t_inv = inverse(t);
    }
    // Shape::set_material — base_shape.rs:65-67; GroupShape pushes to children instead (group.rs:96-100)
    void set_material(int id, const Material& m) {
        check(id);
        if (shapes[id].kind == GROUP) {
            std::vector<int> kids = shapes[id].children;
            for (int c : kids) set_material(c, m);
        } else {
            shapes[id].material = m;
        }
    }
    void add_child(int group, int child) {  // group.rs:39-44
        check(group);
        if (shapes[group].kind != GROUP) throw Error("not a group");
        adopt(child);
        set_transform(child, shapes[group].t * shapes[child].t);
        shapes[group].children.push_back(child);
    }
    // Shape::bounding_box of each kind
    Bounds bounding_box(int id) {
        check(id);
        ShapeRec& s = shapes[id];
        Bounds b;
        switch (s.kind) {
            case SPHERE:
            case CUBE:
                b.add(Vec3{-1, -1, -1}), b.add(Vec3{1, 1, 1});  // sphere.rs:75-80, cube.rs:82-87
                return b;
            case PLANE:  // plane.rs:61-66
                b.lo[0] = -kInf, b.lo[1] = 0, b.lo[2] = -kInf, b.hi[0] = kInf, b.hi[1] = 0, b.hi[2] = kInf;
                return b;
            case CYLINDER:  // cylinder.rs:74-79
                b.lo[0] = -1, b.lo[1] = s.y_min, b.lo[2] = -1, b.hi[0] = 1, b.hi[1] = s.y_max, b.hi[2] = 1;
                return b;
            case CONE: {  // cone.rs:75-84
                float limit = fmaxf(std::fabs(s.y_min), std::fabs(s.y_max));
                b.lo[0] = -limit, b.lo[1] = s.y_min, b.lo[2] = -limit, b.hi[0] = limit, b.hi[1] = s.y_max, b.hi[2] = limit;
                return b;
            }
            case TRIANGLE:
            case SMOOTH_TRIANGLE:  // triangle.rs:83-89, smooth_triangle.rs:48-51
                b.add(Vec3{s.tri[0], s.tri[1], s.tri[2]});
                b.add(Vec3{s.p2[0], s.p2[1], s.p2[2]});
                b.add(Vec3{s.p3[0], s.p3[1], s.p3[2]});
                return b;
            default:  // group.rs:138-150, csg.rs:119-130 — cached on first use, never invalidated
                if (!s.box_cached) {
                    Bounds acc;
                    std::vector<int> kids = s.children;
                    for (int c : kids) acc.add(parent_space_box(c));
                    shapes[id].box = acc;
                    shapes[id].box_cached = true;
                }
                return shapes[id].box;
        }
    }
    // Shape::parent_space_bounding_box — shape.rs:162-164; group override group.rs:152-156
    Bounds parent_space_box(int id) {
        if (shapes[id].kind == GROUP) return bounding_box(id);
        return bounding_box(id).transformed(shapes[id].t);
    }
    // GroupShape::divide — group.rs:48-77,158-172; CSG::divide csg.rs:132-135
    void divide(int id, size_t threshold) {
        check(id);
        if (shapes[id].kind == CSG) {
            std::vector<int> kids = shapes[id].children;
            for (int c : kids) divide(c, threshold);
            return;
        }
        if (shapes[id].kind != GROUP) return;
        if (threshold <= shapes[id].children.size()) {
            Bounds lb, rb;
            bounding_box(id).split(lb, rb);
            std::vector<int> left, right, keep;
            for (int c : shapes[id].children) {
                Bounds cb = parent_space_box(c);
                if (lb.contains(cb))
                    left.push_back(c);
                else if (rb.contains(cb))
                    right.push_back(c);
                else
                    keep.push_back(c);
            }
            shapes[id].children = keep;
            for (std::vector<int>* part : {&left, &right}) {
                if (part->empty()) continue;
                if (part->size() == 1) {
                    shapes[id].children.push_back((*part)[0]);  // a single shape is not wrapped (group.rs:71-73)
                } else {
                    int g = add(GROUP);
                    shapes[g].owned = true;
                    shapes[g].children = *part;
                    shapes[id].children.push_back(g);
                }
            }
        }
        std::vector<int> kids = shapes[id].children;
        for (int c : kids) divide(c, threshold);
    }
    // dyn_clone of a subtree; caches are reset like the reference's Clone impls (group.rs:175-183)
    int clone(int id) {
        check(id);
        ShapeRec copy = shapes[id];
        copy.owned = false;
        copy.box_cached = false;
        std::vector<int> kids = copy.children;
        for (int& c : kids) {
            c = clone(c);
            shapes[c].owned = true;
        }
        copy.children = kids;
        shapes.push_back(copy);
        return (int)shapes.size() - 1;
    }
    // obj_parser.rs:100-293 + take_all_as_group :33-55 (groups in declaration order)
    int parse_obj(const std::string& text);
};

struct World {  // world.rs:18-21
    std::vector<int> objects;
    Light light;
};

// Camera — camera.rs:8-56
struct Camera {
    uint32_t width = 0, height = 0;
    float field_of_view = 0, half_width = 0, half_height = 0, pixel_size = 0;
    Mat4 transform_inverse;
    Camera() = default;
    Camera(uint32_t w, uint32_t h, float fov, const Mat4& transform) : width(w), height(h), field_of_view(fov) {
        float half_view = std::tan(fov / 2.0f);
        float aspect = (float)w / (float)h;
        if (aspect >= 1.0f) {
            half_width = half_view;
            half_height = half_view / aspect;
        } else {
            half_width = half_view * aspect;
            half_height = half_view;
        }
        pixel_size = (half_width * 2.0f) / (float)w;
        transform_inverse = inverse(transform);
    }
};

// RectangleLight::new — rectangle_light.rs:34-59
inline Light rectangle_light(const float intensity[3], const float corner[3], const float u_vec[3], int u_steps,
                             const float v_vec[3], int v_steps, const float* jitter, int n_jitter, uint64_t seed) {
    Light l;
    l.set = true, l.rect = true;
    for (int a = 0; a < 3; a++) {
        l.intensity[a] = intensity[a];
        l.corner[a] = corner[a];
        l.u_cell[a] = u_vec[a] / (float)u_steps;
        l.v_cell[a] = v_vec[a] / (float)v_steps;
        l.position[a] = corner[a] + (u_vec[a] / 2.f) + (v_vec[a] / 2.f);
    }
    l.u_steps = u_steps, l.v_steps = v_steps;
    if (n_jitter > 0) l.jitter.assign(jitter, jitter + n_jitter);
    l.seed = seed;
    return l;
}

// ------------------------------------------------------------------------------------------- flattener
// World -> the POD arrays of include/rtc_b200.h.  Leaves are emitted in depth-first order of
// World::objects / children / (s1, s2): the reference's emission order, hence its tie-break order.
// ------------------------------------------------------------------------------------------- PPM (canvas.rs)
// Canvas::to_ppm (canvas.rs:58-96), byte for byte, written for speed: one pass over the pixels, a 256-entry table of
// decimal strings, the output reserved up front.  The reference's rule after every value but a row's last: append a
// space if the line is shorter than 70 - 3 columns, else end the line (canvas.rs:47-55); rows end their line.
inline unsigned char scale_color(float rgb) {  // canvas.rs:39-43: f32::min / max keep the non-NaN operand, `as u8` truncates
    float v = rgb * 255.0f;
    v = (v != v) ? 255.0f : (v < 255.0f ? v : 255.0f);
    v = v > 0.0f ? v : 0.0f;
    return (unsigned char)v;
}
// One writer for both sources of 8-bit values: Get(row, i) is channel i of the row through scale_color — computed here
// from the f32 canvas, or taken from the 8-bit plane the device produced with the same conversion (canvas.rs:39-43).
template <class Get>
inline std::string ppm_from(int width, int height, Get get) {
    static const struct Table {
        char text[256][4];
        unsigned char len[256];
        Table() {
            for (int v = 0; v < 256; v++) len[v] = (unsigned char)snprintf(text[v], 4, "%d", v);
        }
    } table;
    std::string out = "P3\n" + std::to_string(width) + " " + std::to_string(height) + "\n255\n";
    out.reserve(out.size() + (size_t)width * height * 12 + 16);
    const size_t n = (size_t)width * 3;
    for (int row = 0; row < height; row++) {
        size_t line = 0;
        for (size_t i = 0; i < n; i++) {
            const unsigned v = get(row, i);
            out.append(table.text[v], table.len[v]);
            line += table.len[v];
            if (i + 1 == n) break;
            if (line < 70 - 3) {
                out.push_back(' ');
                line++;
            } else {
                out.push_back('\n');
                line = 0;
            }
        }
        if (line) out.push_back('\n');
    }
    return out;
}
inline std::string canvas_to_ppm(const CanvasRec& c) {
    const size_t n = (size_t)c.width * 3;
    return ppm_from(c.width, c.height, [&](int row, size_t i) -> unsigned { return scale_color(c.rgb[(size_t)row * n + i]); });
}
// Canvas::to_ppm of a frame of which only the 8-bit plane left the device (Camera::render_b200_u8)
inline std::string ppm_from_u8(int width, int height, const uint8_t* u8) {
    const size_t n = (size_t)width * 3;
    return ppm_from(width, height, [&](int row, size_t i) -> unsigned { return u8[(size_t)row * n + i]; });
}

// canvas_from_ppm (canvas.rs:119-182) + clean_line (184-200).  Error texts start with the reference's ParseError kind.
inline CanvasRec canvas_from_ppm(const char* text, size_t n) {
    auto is_space = [](char ch) { return ch == ' ' || (ch >= '\t' && ch <= '\r'); };
    size_t pos = 0;
    // next line that is neither empty nor a comment, trimmed: [a, b)
    auto next_line = [&](size_t& a, size_t& b) {
        while (pos <= n) {
            size_t end = pos;
            while (end < n && text[end] != '\n') end++;
            a = pos, b = end;
            pos = end + 1;
            while (a < b && is_space(text[a])) a++;
            while (b > a && is_space(text[b - 1])) b--;
            if (a < b && text[a] != '#') return true;
            if (end >= n) break;
        }
        return false;
    };
    auto parse = [&](size_t a, size_t b, uint64_t limit) -> uint64_t {  // str::parse::<u32 / usize>
        const std::string tok(text + a, b - a);
        size_t i = a;
        if (i < b && text[i] == '+') i++;
        if (i >= b) throw Error("ParseIntError: cannot parse integer from '" + tok + "'");
        uint64_t v = 0;
        for (; i < b; i++) {
            if (text[i] < '0' || text[i] > '9') throw Error("ParseIntError: invalid digit found in '" + tok + "'");
            v = v * 10 + (uint64_t)(text[i] - '0');
            if (v > limit) throw Error("ParseIntError: number too large in '" + tok + "'");
        }
        return v;
    };
    size_t a, b;
    if (!next_line(a, b)) throw Error("unexpected end of file in the PPM header");
    if (!(b - a == 2 && text[a] == 'P' && text[a + 1] == '3'))
        throw Error("IncorrectFormat: Incorrect magic number at line 1: expected P3, found " + std::string(text + a, b - a));
    if (!next_line(a, b)) throw Error("unexpected end of file in the PPM header");
    size_t tok[3][2];
    int n_tok = 0;
    for (size_t i = a; i < b;) {
        while (i < b && is_space(text[i])) i++;
        size_t j = i;
        while (j < b && !is_space(text[j])) j++;
        if (j > i) {
            if (n_tok < 3) tok[n_tok][0] = i, tok[n_tok][1] = j;
            n_tok++;
        }
        i = j;
    }
    if (n_tok != 2)
        throw Error("MalformedDimensionHeader: Expected width and height at line 2; found " + std::string(text + a, b - a));
    CanvasRec c;
    c.width = (int)parse(tok[0][0], tok[0][1], 1u << 30);
    c.height = (int)parse(tok[1][0], tok[1][1], 1u << 30);
    if (!next_line(a, b)) throw Error("unexpected end of file in the PPM header");
    const float scale = (float)(uint32_t)parse(a, b, 0xffffffffull);
    const size_t total = (size_t)c.width * c.height * 3;
    c.rgb.assign(total, 0.0f);
    size_t count = 0;  // values consumed; a pixel is written when its third value arrives (canvas.rs:163-176)
    float pending[3];
    while (next_line(a, b)) {
        for (size_t i = a; i < b;) {
            while (i < b && is_space(text[i])) i++;
            size_t j = i;
            while (j < b && !is_space(text[j])) j++;
            if (j > i) {
                pending[count % 3] = (float)(uint32_t)parse(i, j, 0xffffffffull) / scale;
                count++;
                if (count % 3 == 0) {
                    if (count > total) throw Error("more pixel data than width x height");  // data[y][x] panics there
                    memcpy(&c.rgb[count - 3], pending, sizeof(pending));
                }
            }
            i = j;
        }
    }
    return c;
}

struct FlatScene {
    // With `target` set the geometry arrays are written straight into that scene's storage (rtc_map_primitives /
    // rtc_map_nodes: no second copy of a 14 MB array) and the three vectors stay empty.
    RtcScene* target = nullptr;
    size_t n_prims = 0, n_nodes = 0, n_refs = 0;
    rtc::RawVector<RtcPrim> prims;  // resized once, every record written by the walk that owns it
    rtc::RawVector<RtcNode> nodes;
    rtc::RawVector<int32_t> refs;
    std::vector<RtcMaterial> materials;
    std::vector<RtcPattern> patterns;
    std::vector<RtcUvPattern> uvs;
    std::vector<RtcTexture> textures;  // point into the scene graph's canvases
    std::vector<int> prim_shape;  // primitive index -> shape handle
};

// World -> the arrays of include/rtc_b200.h, in the reference's depth-first order (world.rs:18-21, group.rs:16-20,
// csg.rs:18-24): primitive i is the i-th leaf a depth-first walk meets, node j the j-th group / CSG it enters, and a
// node's child references follow those of all its descendants.
//
// A walk over 100 k shapes is bound by cache misses (the arena's records are visited in tree order, not in memory
// order), so a large world is flattened by several threads: the top of the tree is opened level by level until a few
// hundred subtrees are in hand, their sizes are counted in parallel, which fixes where every subtree's records go,
// and each thread then walks its subtrees writing at those offsets — the same arrays, index for index, as one
// sequential walk.  Materials are de-duplicated per thread and merged in subtree order (first-use numbering, as a
// sequential walk would assign).
class Flattener {
   public:
    Flattener(SceneGraph& g, FlatScene& out) : g_(g), out_(out) {}
    void run(const World& w) {
        const bool timing = getenv("RTC_TIMING") != nullptr;
        auto t_last = std::chrono::steady_clock::now();
        auto lap = [&](const char* what) {
            if (!timing) return;
            const auto now = std::chrono::steady_clock::now();
            fprintf(stderr, "[rtc flatten] %-27s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - t_last).count());
            t_last = now;
        };
        const size_t n_shapes = g_.shapes.size();
        const bool threaded = n_shapes >= 8192 && world_has_at_least(w, 4096) && rtc::WorkerPool::instance().threads() > 1;
        // ---- 1. the subtrees to hand out: the world's objects, with the top levels of a large world's groups opened
        std::vector<int> frontier(w.objects.begin(), w.objects.end());
        std::vector<char> opened;
        const int n_threads = threaded ? rtc::WorkerPool::instance().threads() : 1;
        if (threaded) {
            opened.assign(n_shapes, 0);
            std::vector<char> is_leaf(frontier.size(), 0);  // examined before and found to be a leaf: not looked at again
            bool any = true;
            for (int level = 0; level < 10 && any; level++) {
                any = false;
                std::vector<int> next;
                std::vector<char> next_leaf;
                next.reserve(2 * frontier.size()), next_leaf.reserve(2 * frontier.size());
                for (size_t k = 0; k < frontier.size(); k++) {
                    const int id = frontier[k];
                    if (!is_leaf[k]) {
                        g_.check(id);
                        const ShapeRec& s = g_.shapes[id];
                        if ((s.kind == GROUP || s.kind == CSG) && !s.children.empty() && !opened[id]) {
                            opened[id] = 1, any = true;
                            for (int c : s.children) prefetch_kind(c);
                            next.insert(next.end(), s.children.begin(), s.children.end());
                            next_leaf.insert(next_leaf.end(), s.children.size(), 0);
                            continue;
                        }
                    }
                    next.push_back(id), next_leaf.push_back(1);  // a leaf, an empty group, or a group met twice
                }
                frontier.swap(next), is_leaf.swap(next_leaf);
            }
        }
        // ---- 2. their sizes
        std::vector<Counts> counts(frontier.size());
        {
            const size_t n_jobs = threaded ? std::min<size_t>(frontier.size(), 16 * (size_t)n_threads) : 1;
            auto count_range = [&](size_t b, size_t e) {
                for (size_t k = b; k < e; k++) counts[k] = count(frontier[k]);
            };
            if (n_jobs <= 1)
                count_range(0, frontier.size());
            else
                rtc::WorkerPool::instance().run((int)n_jobs, [&](int j) {
                    count_range(frontier.size() * (size_t)j / n_jobs, frontier.size() * (size_t)(j + 1) / n_jobs);
                });
        }
        lap("frontier + subtree sizes");
        // ---- 3. where everything goes: a walk of the opened top of the tree
        struct Entry {
            int id, parent_node;
            Cursor at;
        };
        struct TopNode {
            int id, node, parent_node, child_begin;
            std::vector<int32_t> child_refs;
        };
        std::vector<Entry> entries;
        std::vector<TopNode> tops;
        entries.reserve(frontier.size());
        Cursor cur;
        struct Placer {
            Flattener& f;
            const std::vector<char>& opened;
            const std::vector<Counts>& counts;
            std::vector<Entry>& entries;
            std::vector<TopNode>& tops;
            Cursor& cur;
            int place(int id, int parent_node) {
                if (!opened.empty() && opened[id]) {
                    const ShapeRec& s = f.g_.shapes[id];
                    const size_t me = tops.size();
                    const int node = cur.node++;
                    tops.push_back(TopNode{id, node, parent_node, 0, {}});
                    std::vector<int32_t> refs;
                    refs.reserve(s.children.size());
                    for (int c : s.children) refs.push_back(place(c, node));
                    tops[me].child_begin = cur.ref;
                    cur.ref += (int)refs.size();
                    tops[me].child_refs = std::move(refs);
                    return ~node;
                }
                const Counts& n = counts[entries.size()];
                entries.push_back(Entry{id, parent_node, cur});
                const int ref = n.nodes > 0 ? ~cur.node : cur.prim;  // a group or CSG counts itself as a node
                cur.prim += n.prims, cur.node += n.nodes, cur.ref += n.refs;
                return ref;
            }
        } placer{*this, opened, counts, entries, tops, cur};
        for (int id : w.objects) {
            g_.check(id);
            placer.place(id, -1);
        }
        lap("placement");
        // ---- 4. the records
        out_.n_prims = cur.prim, out_.n_nodes = cur.node, out_.n_refs = cur.ref;
        out_.prim_shape.resize(cur.prim);
        if (out_.target) {
            if (rtc_map_primitives(out_.target, (uint32_t)cur.prim, &prims_) ||
                rtc_map_nodes(out_.target, (uint32_t)cur.node, (uint32_t)cur.ref, &nodes_, &refs_))
                throw Error(rtc_last_error());
        } else {
            out_.prims.resize(cur.prim), out_.nodes.resize(cur.node), out_.refs.resize(cur.ref);
            prims_ = out_.prims.data(), nodes_ = out_.nodes.data(), refs_ = out_.refs.data();
        }
        // contiguous runs of subtrees of about equal weight, a few per thread
        std::vector<size_t> chunk_begin{0};
        if (threaded) {
            const long long total = (long long)cur.prim + cur.node;
            const long long target = std::max<long long>(1024, total / (4 * n_threads));
            long long acc = 0;
            for (size_t k = 0; k < entries.size(); k++) {
                if (acc >= target) chunk_begin.push_back(k), acc = 0;
                acc += counts[k].prims + counts[k].nodes;
            }
        }
        chunk_begin.push_back(entries.size());
        const int n_chunks = (int)chunk_begin.size() - 1;
        std::vector<LocalMaterials> locals(n_chunks);
        std::vector<std::pair<int, int>> prim_range(n_chunks, {0, 0});
        auto emit_chunk = [&](int chunk) {
            const size_t b = chunk_begin[chunk], e = chunk_begin[chunk + 1];
            if (b == e) return;
            LocalMaterials& local = locals[chunk];
            prim_range[chunk].first = entries[b].at.prim;
            Cursor c = entries[b].at;
            for (size_t k = b; k < e; k++) {
                c = entries[k].at;
                emit(entries[k].id, entries[k].parent_node, c, local);
            }
            prim_range[chunk].second = c.prim;
        };
        if (n_chunks == 1)
            emit_chunk(0);
        else
            rtc::WorkerPool::instance().run(n_chunks, emit_chunk);
        lap("records");
        if (timing) {
            fprintf(stderr, "[rtc flatten] %zu shapes, %zu subtrees, %zu opened, %d chunks:", n_shapes, entries.size(), tops.size(), n_chunks);
            for (auto& r : prim_range) fprintf(stderr, " %d", r.second - r.first);
            fprintf(stderr, "\n");
        }
        // ---- 5. one material table (first-use order), the opened nodes' own records
        bool identity = true;
        std::vector<std::vector<int>> remap(n_chunks);
        for (int chunk = 0; chunk < n_chunks; chunk++) {
            for (RtcMaterial r : locals[chunk].list) {
                r.pattern = pattern_index(r.pattern);  // until here: the scene graph's pattern handle
                const int id = material_index(r);
                identity = identity && id == (int)remap[chunk].size();
                remap[chunk].push_back(id);
            }
        }
        if (!identity)
            rtc::WorkerPool::instance().run(n_chunks, [&](int chunk) {
                for (int i = prim_range[chunk].first; i < prim_range[chunk].second; i++)
                    prims_[i].material = remap[chunk][prims_[i].material];
            });
        for (const TopNode& t : tops) {
            std::copy(t.child_refs.begin(), t.child_refs.end(), refs_ + t.child_begin);
            write_node(t.id, t.node, t.parent_node, t.child_begin, (int)t.child_refs.size());
        }
        lap("materials + opened nodes");
    }

   private:
    struct Counts {
        int prims = 0, nodes = 0, refs = 0;
    };
    struct Cursor {  // the next free primitive, node and child-reference slot of a walk
        int prim = 0, node = 0, ref = 0;
    };
    // a walk's own material numbering; `pattern` holds the scene graph's pattern handle until the tables are merged
    struct LocalMaterials {
        std::vector<RtcMaterial> list;
        std::map<std::vector<uint32_t>, int> ids;
        int last = -1;
        int index(const Material& m) {
            RtcMaterial r;
            memcpy(r.color, m.color, sizeof(r.color));
            r.ambient = m.ambient, r.diffuse = m.diffuse, r.specular = m.specular, r.shininess = m.shininess;
            r.reflective = m.reflective, r.transparency = m.transparency, r.refractive_index = m.refractive_index;
            r.pattern = m.pattern < 0 ? -1 : m.pattern;
            // a mesh's triangles share one material: compare with the previous one, then with the first few, before the map
            if (last >= 0 && memcmp(&list[last], &r, 11 * sizeof(uint32_t)) == 0) return last;
            for (size_t i = 0; i < list.size() && i < 16; i++)
                if (memcmp(&list[i], &r, 11 * sizeof(uint32_t)) == 0) return last = (int)i;
            std::vector<uint32_t> key(11);
            memcpy(key.data(), &r, 11 * sizeof(uint32_t));
            auto it = ids.find(key);
            if (it != ids.end()) return last = it->second;
            list.push_back(r);
            return last = ids[key] = (int)list.size() - 1;
        }
    };

    SceneGraph& g_;
    FlatScene& out_;
    RtcPrim* prims_ = nullptr;  // where the walks write: out_'s vectors, or the target scene's mapped arrays
    RtcNode* nodes_ = nullptr;
    int32_t* refs_ = nullptr;
    std::map<std::vector<uint32_t>, int> material_ids_;
    std::map<int, int> pattern_ids_, uv_ids_, texture_ids_;
    int last_material_ = -1;

    int uv_index(int h) {
        if (h < 0 || h >= (int)g_.uvs.size()) throw Error("bad uv pattern handle");
        auto it = uv_ids_.find(h);
        if (it != uv_ids_.end()) return it->second;
        RtcUvPattern u;
        u.kind = g_.uvs[h].kind;
        memcpy(u.params, g_.uvs[h].params, sizeof(u.params));
        if (u.kind == RTC_UV_IMAGE) {  // the canvas travels once, however many patterns share it
            const int cv = g_.uvs[h].canvas;
            auto t = texture_ids_.find(cv);
            if (t == texture_ids_.end()) {
                const CanvasRec& c = g_.canvases.at(cv);
                out_.textures.push_back(RtcTexture{(uint32_t)c.width, (uint32_t)c.height, c.rgb.data()});
                t = texture_ids_.emplace(cv, (int)out_.textures.size() - 1).first;
            }
            u.params[0] = (float)t->second;
        }
        out_.uvs.push_back(u);
        return uv_ids_[h] = (int)out_.uvs.size() - 1;
    }
    int pattern_index(int h) {
        if (h < 0) return -1;
        if (h >= (int)g_.patterns.size()) throw Error("bad pattern handle");
        auto it = pattern_ids_.find(h);
        if (it != pattern_ids_.end()) return it->second;
        const Pattern& p = g_.patterns[h];
        RtcPattern r;
        memset(&r, 0, sizeof(r));
        r.kind = p.kind;
        r.mapping = p.mapping;
        for (int i = 0; i < 6; i++) r.uv[i] = -1;
        if (p.kind == RTC_PAT_TEXTURE_MAP) r.uv[0] = uv_index(p.uv[0]);
        if (p.kind == RTC_PAT_CUBIC_MAP)
            for (int i = 0; i < 6; i++) r.uv[i] = uv_index(p.uv[i]);
        memcpy(r.inv, p.inv.m, sizeof(r.inv));
        memcpy(r.a, p.a, sizeof(r.a));
        if (p.kind == RTC_PAT_GRADIENT || p.kind == RTC_PAT_SINE2D) {
            for (int a = 0; a < 3; a++) r.b[a] = p.b[a] - p.a[a];  // `distance`, gradient.rs:23 / sine_2d.rs:22
        } else {
            memcpy(r.b, p.b, sizeof(r.b));
        }
        out_.patterns.push_back(r);
        return pattern_ids_[h] = (int)out_.patterns.size() - 1;
    }
    int material_index(const RtcMaterial& r) {  // the scene's table: one entry per distinct material
        if (last_material_ >= 0 && memcmp(&out_.materials[last_material_], &r, 11 * sizeof(uint32_t)) == 0) return last_material_;
        for (size_t i = 0; i < out_.materials.size() && i < 16; i++)
            if (memcmp(&out_.materials[i], &r, 11 * sizeof(uint32_t)) == 0) return last_material_ = (int)i;
        std::vector<uint32_t> key(11);
        memcpy(key.data(), &r, 11 * sizeof(uint32_t));
        auto it = material_ids_.find(key);
        if (it != material_ids_.end()) return last_material_ = it->second;
        out_.materials.push_back(r);
        return last_material_ = material_ids_[key] = (int)out_.materials.size() - 1;
    }
    static void put_box(const Bounds& b, float lo[3], float hi[3]) {
        for (int a = 0; a < 3; a++) lo[a] = b.lo[a], hi[a] = b.hi[a];
    }
    // is the world worth several threads?  (a walk that stops at `limit` shapes)
    bool world_has_at_least(const World& w, size_t limit) const {
        std::vector<int> stack(w.objects.begin(), w.objects.end());
        size_t seen = 0;
        while (!stack.empty()) {
            const int id = stack.back();
            stack.pop_back();
            g_.check(id);
            if (++seen >= limit) return true;
            const ShapeRec& s = g_.shapes[id];
            if (s.kind == GROUP || s.kind == CSG) {
                if (seen + s.children.size() >= limit) return true;
                stack.insert(stack.end(), s.children.begin(), s.children.end());
            }
        }
        return false;
    }
    // The walks visit the arena in tree order, not in memory order: every shape record is a cache miss (five lines).
    // A group's children are known before they are visited, so their records are requested a few children ahead.
    static constexpr size_t kAhead = 4;
    void prefetch_kind(int id) const {
        if (id >= 0 && id < (int)g_.shapes.size()) __builtin_prefetch(&g_.shapes[id].kind);
    }
    void prefetch_record(int id) const {
        if (id < 0 || id >= (int)g_.shapes.size()) return;
        const char* p = reinterpret_cast<const char*>(&g_.shapes[id]);
        for (size_t off = 0; off < sizeof(ShapeRec); off += 64) __builtin_prefetch(p + off);
    }
    // records a depth-first walk of `id` emits
    Counts count(int id) const {
        g_.check(id);
        const ShapeRec& s = g_.shapes[id];
        Counts n;
        if (s.kind != GROUP && s.kind != CSG) {
            n.prims = 1;
            return n;
        }
        n.nodes = 1, n.refs = (int)s.children.size();
        const size_t kids = s.children.size();
        for (size_t i = 0; i < kids && i < kAhead; i++) prefetch_kind(s.children[i]);
        for (size_t i = 0; i < kids; i++) {
            if (i + kAhead < kids) prefetch_kind(s.children[i + kAhead]);
            const Counts k = count(s.children[i]);
            n.prims += k.prims, n.nodes += k.nodes, n.refs += k.refs;
        }
        return n;
    }
    void write_node(int id, int node, int parent_node, int child_begin, int child_count) {
        const ShapeRec& s = g_.shapes[id];
        RtcNode n;
        memset(&n, 0, sizeof(n));
        n.kind = (s.kind == GROUP) ? RTC_NODE_GROUP : RTC_NODE_CSG;
        n.parent = parent_node;
        n.op = s.csg_op;
        n.child_begin = child_begin;
        n.child_count = child_count;
        const Mat4 inv = (s.kind == CSG) ? s.t_inv : Mat4();
        memcpy(n.inv, inv.m, sizeof(n.inv));
        put_box(g_.bounding_box(id), n.bbox_min, n.bbox_max);  // cached in the shape on first use (group.rs:138-150)
        put_box(g_.parent_space_box(id), n.world_bbox_min, n.world_bbox_max);
        nodes_[node] = n;
    }
    // the walk: writes the subtree of `id` at the cursor and returns the child reference of what it wrote.  Touches
    // only this subtree's shapes (their cached boxes included), so disjoint subtrees go to different threads.
    int emit(int id, int parent_node, Cursor& c, LocalMaterials& materials) {
        g_.check(id);
        const ShapeRec& s = g_.shapes[id];
        if (s.kind == GROUP || s.kind == CSG) {
            const int node = c.node++;
            std::vector<int32_t> child_refs;
            child_refs.reserve(s.children.size());
            const size_t kids = s.children.size();
            for (size_t i = 0; i < kids && i < kAhead; i++) prefetch_record(s.children[i]);
            for (size_t i = 0; i < kids; i++) {
                if (i + kAhead < kids) prefetch_record(s.children[i + kAhead]);
                child_refs.push_back(emit(s.children[i], node, c, materials));
            }
            std::copy(child_refs.begin(), child_refs.end(), refs_ + c.ref);
            write_node(id, node, parent_node, c.ref, (int)child_refs.size());
            c.ref += (int)child_refs.size();
            return ~node;
        }
        const int i = c.prim++;
        RtcPrim& p = prims_[i];
        memset(&p, 0, sizeof(p));
        switch (s.kind) {
            case SPHERE: p.type = RTC_SPHERE; break;
            case PLANE: p.type = RTC_PLANE; break;
            case CUBE: p.type = RTC_CUBE; break;
            case CYLINDER: p.type = RTC_CYLINDER; break;
            case CONE: p.type = RTC_CONE; break;
            default: p.type = RTC_TRIANGLE; break;  // SmoothTriangle renders as its flat inner triangle (Q5)
        }
        p.material = materials.index(s.material);
        p.casts_shadow = s.casts_shadow ? 1 : 0;
        p.parent = parent_node;
        memcpy(p.inv, s.t_inv.m, sizeof(p.inv));
        if (p.type == RTC_TRIANGLE) {
            memcpy(p.params, s.tri, sizeof(p.params));
        } else if (p.type == RTC_CYLINDER || p.type == RTC_CONE) {
            p.params[0] = s.y_min, p.params[1] = s.y_max, p.params[2] = s.closed ? 1.f : 0.f;
        }
        put_box(g_.parent_space_box(id), p.bbox_min, p.bbox_max);
        out_.prim_shape[i] = id;
        return i;
    }
};

// Camera::render_b200 — the sibling of Camera::render (camera.rs:76-91) that a demo switches to.  Flattens
// the world, commits it to `n_devices` GPUs and renders.  Throws rtch::Error on any failure (no fallback).
struct RenderOptions {
    int n_devices = 1;
    std::vector<int> device_ids;
    bool fma = false;  // RTC_OPT_FMA_CONTRACTION
    bool detailed = false;
    int bvh_builder = -1;  // -1 automatic, 0 host binned SAH, 1 device LBVH (see rtc_host.cpp: commit)
    bool exact_groups = false;  // RTC_OPT_EXACT_GROUPS
};

inline void fill_scene(RtcScene* scene, SceneGraph& g, const World& w, const Camera& cam, FlatScene& flat) {
    auto ck = [](int rc) {
        if (rc) throw Error(rtc_last_error());
    };
    if (!w.light.set) throw Error("World light should be set");  // world.rs:66
    const bool timing = getenv("RTC_TIMING") != nullptr;
    const auto t0 = std::chrono::steady_clock::now();
    flat.target = scene;  // primitives, nodes and child references are written in place
    Flattener(g, flat).run(w);
    if (timing)
        fprintf(stderr, "[rtc host]   %-28s %8.3f ms\n", "scene graph -> flat arrays",
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
    ck(rtc_set_camera(scene, cam.width, cam.height, cam.half_width, cam.half_height, cam.pixel_size, cam.transform_inverse.m));
    ck(rtc_set_materials(scene, (uint32_t)flat.materials.size(), flat.materials.data()));
    ck(rtc_set_patterns(scene, (uint32_t)flat.patterns.size(), flat.patterns.data(), (uint32_t)flat.uvs.size(), flat.uvs.data()));
    ck(rtc_set_textures(scene, (uint32_t)flat.textures.size(), flat.textures.data()));
    const Light& l = w.light;
    if (l.rect)
        ck(rtc_set_rect_light(scene, l.intensity, l.corner, l.u_cell, l.u_steps, l.v_cell, l.v_steps, l.position,
                              l.jitter.data(), (uint32_t)l.jitter.size(), l.seed));
    else
        ck(rtc_set_point_light(scene, l.position, l.intensity));
}

}  // namespace rtch
