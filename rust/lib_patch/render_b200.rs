//! `Camera::render_b200` for the reference's `lib` crate — the drop-in sibling of `Camera::render` (camera.rs:76-91) —
//! and everything it needs: the scene flattener over `Box<dyn Shape>` / `Box<dyn Pattern>` / `Box<dyn Light>`.
//!
//! NOT COMPILED IN THIS REPO (the build image has no Rust toolchain, SURVEY.md §0.2).  The same flattening is
//! implemented and TESTED in C++ (ray_tracer_challenge_b200/csrc/host/rtc_host.hpp: class Flattener, bit-compared with
//! the oracle's construction in tests/test_host_scene.py); this file is its Rust counterpart, complete: every shape
//! kind, every pattern, both lights.  The `#[repr(C)]` structs it fills are checked against include/rtc_b200.h by
//! tests/test_c_abi.py::test_rust_sys_crate_mirrors_the_header.
//!
//! HOW TO APPLY.  The reference keeps its fields private, so the code below is laid out as the blocks a maintainer
//! pastes into the files named in the section headers (each block only touches fields of the type defined in that
//! file), plus three one-line additions to existing traits:
//!
//!   shape/shape.rs    trait Shape    { fn flatten(&self, out: &mut FlatScene, parent: i32) -> i32; }
//!   pattern/pattern.rs trait Pattern { fn lower(&self, out: &mut FlatScene) -> i32; }
//!   pattern/uv.rs     trait UVPattern { fn lower_uv(&self, out: &mut FlatScene) -> i32; }
//!                     trait UVMapping { fn mapping_id(&self) -> i32; }
//!   light/light.rs    trait Light    { fn lower(&self, scene: *mut sys::RtcScene); }
//!
//! and in lib/Cargo.toml:  rtc-b200-sys = { path = "../../rust/rtc-b200-sys" }   (see INTEGRATION.md).
//! A demo then switches paths by one line:  `camera.render(world, 5)`  ->  `camera.render_b200(world, 5)`.
#![allow(dead_code)]
use rtc_b200_sys as sys;

// =====================================================================================================
// lib/src/flat_scene.rs (new file; `pub mod flat_scene;` in lib.rs)
// =====================================================================================================

/// The POD arrays of include/rtc_b200.h, filled in depth-first order of World::objects / GroupShape::children /
/// CSG (s1, s2).  That order is the reference's tie-break between equal distances (world.rs:58: stable sort,
/// intersection.rs:30-35: first minimum), which the device reproduces from the primitive index.
pub struct FlatScene {
    pub prims: Vec<sys::RtcPrim>,
    pub nodes: Vec<sys::RtcNode>,
    pub refs: Vec<i32>,
    pub materials: Vec<sys::RtcMaterial>,
    pub patterns: Vec<sys::RtcPattern>,
    pub uvs: Vec<sys::RtcUvPattern>,
    /// One entry per UVImage canvas (uv.rs:346-377): its f32 pixels row-major, kept alive until the commit.
    pub texture_pixels: Vec<Vec<f32>>,
    pub texture_sizes: Vec<(u32, u32)>,
}

impl FlatScene {
    pub fn new() -> Self {
        FlatScene {
            prims: Vec::new(),
            nodes: Vec::new(),
            refs: Vec::new(),
            materials: Vec::new(),
            patterns: Vec::new(),
            uvs: Vec::new(),
            texture_pixels: Vec::new(),
            texture_sizes: Vec::new(),
        }
    }

    /// Index of `m` in the material table (material.rs:19-51).  A mesh's triangles share one material: equal
    /// pattern-free materials are stored once (bitwise comparison of the ten numbers).
    pub fn material_index(&mut self, m: &Material) -> i32 {
        let pattern = match &m.pattern {
            Some(p) => p.lower(self),
            None => -1,
        };
        let r = sys::RtcMaterial {
            color: [m.color.r, m.color.g, m.color.b],
            ambient: m.ambient,
            diffuse: m.diffuse,
            specular: m.specular,
            shininess: m.shininess,
            reflective: m.reflective,
            transparency: m.transparency,
            refractive_index: m.refractive_index,
            pattern,
        };
        if pattern < 0 {
            let same = |a: &sys::RtcMaterial| {
                a.pattern < 0
                    && a.color.iter().zip(r.color.iter()).all(|(x, y)| x.to_bits() == y.to_bits())
                    && [a.ambient, a.diffuse, a.specular, a.shininess, a.reflective, a.transparency, a.refractive_index]
                        .iter()
                        .zip([r.ambient, r.diffuse, r.specular, r.shininess, r.reflective, r.transparency, r.refractive_index].iter())
                        .all(|(x, y)| x.to_bits() == y.to_bits())
            };
            // newest first: consecutive leaves of one mesh hit the last entry
            if let Some(i) = self.materials.iter().rposition(same) {
                return i as i32;
            }
        }
        self.materials.push(r);
        (self.materials.len() - 1) as i32
    }

    /// A leaf of the shape tree: `params` is {minimum_y, maximum_y, closed} for cylinders / cones and
    /// {p1, e1, e2, normal} for triangles.  Returns the child reference (the primitive index).
    pub fn push_leaf(&mut self, shape: &dyn Shape, kind: i32, params: [f32; 12], parent: i32) -> i32 {
        let b = shape.parent_space_bounding_box(); // shape.rs:162-164
        let material = self.material_index(shape.material());
        self.prims.push(sys::RtcPrim {
            type_: kind,
            material,
            casts_shadow: shape.casts_shadow() as i32, // base_shape.rs:14
            parent,
            inv: mat16(shape.transformation_inverse()), // base_shape.rs:56-60; the device transposes it for normals
            params,
            bbox_min: [b.min.x, b.min.y, b.min.z],
            bbox_max: [b.max.x, b.max.y, b.max.z],
        });
        (self.prims.len() - 1) as i32
    }

    /// An interior node (GroupShape or CSG) and its subtree.  The node's slot is taken BEFORE its children are
    /// visited (pre-order indices), its child references are appended after them; returns `!node` (the child
    /// reference of a node).
    pub fn push_node(&mut self, shape: &dyn Shape, kind: i32, op: i32, children: &[&dyn Shape], parent: i32) -> i32 {
        let node = self.nodes.len();
        self.nodes.push(unsafe { std::mem::zeroed() });
        let child_refs: Vec<i32> = children.iter().map(|c| c.flatten(self, node as i32)).collect();
        let own = shape.bounding_box(); // the cached box the reference culls with (group.rs:119-125, csg.rs:90-93)
        let world = shape.parent_space_bounding_box();
        let identity = {
            let mut m = [0f32; 16];
            m[0] = 1.0;
            m[5] = 1.0;
            m[10] = 1.0;
            m[15] = 1.0;
            m
        };
        self.nodes[node] = sys::RtcNode {
            kind,
            parent,
            op,
            child_begin: self.refs.len() as i32,
            child_count: child_refs.len() as i32,
            // a group has pushed its transform into its children (group.rs:39-44): identity; a CSG keeps its own (csg.rs:78)
            inv: if kind == sys::RTC_NODE_CSG { mat16(shape.transformation_inverse()) } else { identity },
            bbox_min: [own.min.x, own.min.y, own.min.z],
            bbox_max: [own.max.x, own.max.y, own.max.z],
            world_bbox_min: [world.min.x, world.min.y, world.min.z],
            world_bbox_max: [world.max.x, world.max.y, world.max.z],
        };
        self.refs.extend_from_slice(&child_refs);
        !(node as i32)
    }
}

pub fn mat16(m: &Matrix) -> [f32; 16] {
    let mut o = [0f32; 16];
    for r in 0..4 {
        for c in 0..4 {
            o[r * 4 + c] = m.data[r][c];
        }
    }
    o
}

fn rgb(c: Color) -> [f32; 3] {
    [c.r, c.g, c.b]
}

pub fn check(rc: i32) {
    if rc != 0 {
        let msg = unsafe { std::ffi::CStr::from_ptr(sys::rtc_last_error()) };
        panic!("rtc-b200: {}", msg.to_string_lossy()); // the reference's error style is panic (world.rs:66)
    }
}

// =====================================================================================================
// shape/*.rs — `fn flatten` of every Shape implementer (inside each `impl Shape for X { ... }`)
// =====================================================================================================

// shape/sphere.rs
impl Sphere {
    fn flatten(&self, out: &mut FlatScene, parent: i32) -> i32 {
        out.push_leaf(self, sys::RTC_SPHERE, [0.0; 12], parent)
    }
}
// shape/plane.rs
impl Plane {
    fn flatten(&self, out: &mut FlatScene, parent: i32) -> i32 {
        out.push_leaf(self, sys::RTC_PLANE, [0.0; 12], parent)
    }
}
// shape/cube.rs
impl Cube {
    fn flatten(&self, out: &mut FlatScene, parent: i32) -> i32 {
        out.push_leaf(self, sys::RTC_CUBE, [0.0; 12], parent)
    }
}
// shape/cylinder.rs (cylinder.rs:14-19: minimum_y, maximum_y, closed)
impl Cylinder {
    fn flatten(&self, out: &mut FlatScene, parent: i32) -> i32 {
        let mut p = [0f32; 12];
        p[0] = self.minimum_y;
        p[1] = self.maximum_y;
        p[2] = if self.closed { 1.0 } else { 0.0 };
        out.push_leaf(self, sys::RTC_CYLINDER, p, parent)
    }
}
// shape/cone.rs (cone.rs:14-19)
impl Cone {
    fn flatten(&self, out: &mut FlatScene, parent: i32) -> i32 {
        let mut p = [0f32; 12];
        p[0] = self.minimum_y;
        p[1] = self.maximum_y;
        p[2] = if self.closed { 1.0 } else { 0.0 };
        out.push_leaf(self, sys::RTC_CONE, p, parent)
    }
}
// shape/triangle.rs (triangle.rs:9-33: p1 and the e1, e2, normal precomputed by Triangle::new)
impl Triangle {
    pub(crate) fn params(&self) -> [f32; 12] {
        [
            self.p1.x, self.p1.y, self.p1.z, self.e1.x, self.e1.y, self.e1.z, self.e2.x, self.e2.y, self.e2.z, self.normal.x,
            self.normal.y, self.normal.z,
        ]
    }
    fn flatten(&self, out: &mut FlatScene, parent: i32) -> i32 {
        out.push_leaf(self, sys::RTC_TRIANGLE, self.params(), parent)
    }
}
// shape/smooth_triangle.rs — local_intersect delegates to the inner flat Triangle (smooth_triangle.rs:39-41), so the
// intersections name the inner triangle and `local_norm_at` is the flat normal: it renders as RTC_TRIANGLE.  Transform,
// material and casts_shadow are the inner triangle's BaseShape (get_base delegates, smooth_triangle.rs:31-37).
impl SmoothTriangle {
    fn flatten(&self, out: &mut FlatScene, parent: i32) -> i32 {
        out.push_leaf(self, sys::RTC_TRIANGLE, self.base.params(), parent)
    }
}
// shape/group.rs — children in order; the group itself is only a bounding-box cull (group.rs:115-133)
impl GroupShape {
    fn flatten(&self, out: &mut FlatScene, parent: i32) -> i32 {
        let children: Vec<&dyn Shape> = self.children.iter().map(|c| c.as_ref()).collect();
        out.push_node(self, sys::RTC_NODE_GROUP, 0, &children, parent)
    }
}
// shape/csg.rs — (s1, s2) in that order (csg.rs:95-100 intersects s1 first); the operator as RTC_CSG_*
impl CSG {
    fn flatten(&self, out: &mut FlatScene, parent: i32) -> i32 {
        let op = match self.op {
            CSGOperator::Union() => sys::RTC_CSG_UNION,
            CSGOperator::Intersection() => sys::RTC_CSG_INTERSECTION,
            CSGOperator::Difference() => sys::RTC_CSG_DIFFERENCE,
        };
        out.push_node(self, sys::RTC_NODE_CSG, op, &[self.s1.as_ref(), self.s2.as_ref()], parent)
    }
}
// shape/base_shape.rs — BaseShape implements Shape only so that wrappers can delegate to it; like its get_base
// (base_shape.rs:43-49) this is never called
impl BaseShape {
    fn flatten(&self, _out: &mut FlatScene, _parent: i32) -> i32 {
        unimplemented!()
    }
}
// test/utils.rs — TestShape exists for unit tests of Shape's provided methods; it has no surface to render
impl TestShape {
    fn flatten(&self, _out: &mut FlatScene, _parent: i32) -> i32 {
        panic!("TestShape cannot be rendered")
    }
}

// =====================================================================================================
// pattern/*.rs — `fn lower` of every Pattern implementer
// =====================================================================================================

fn push_pattern(out: &mut FlatScene, kind: i32, mapping: i32, uv: [i32; 6], t_inverse: &Matrix, a: Color, b: Color) -> i32 {
    out.patterns.push(sys::RtcPattern { kind, mapping, uv, inv: mat16(t_inverse), a: rgb(a), b: rgb(b) });
    (out.patterns.len() - 1) as i32
}
const NO_UV: [i32; 6] = [-1; 6];
fn black() -> Color {
    Color::new(0.0, 0.0, 0.0)
}

// pattern/stripes.rs:39-45
impl Stripes {
    fn lower(&self, out: &mut FlatScene) -> i32 {
        push_pattern(out, sys::RTC_PAT_STRIPES, 0, NO_UV, self.transformation_inverse(), self.a, self.b)
    }
}
// pattern/gradient.rs:9-36 — `b` carries the precomputed `distance = b - a` (gradient.rs:23)
impl Gradient {
    fn lower(&self, out: &mut FlatScene) -> i32 {
        push_pattern(out, sys::RTC_PAT_GRADIENT, 0, NO_UV, self.transformation_inverse(), self.a, self.distance)
    }
}
// pattern/rings.rs:38-50
impl Rings {
    fn lower(&self, out: &mut FlatScene) -> i32 {
        push_pattern(out, sys::RTC_PAT_RINGS, 0, NO_UV, self.transformation_inverse(), self.a, self.b)
    }
}
// pattern/checkers.rs:38-46
impl Checkers {
    fn lower(&self, out: &mut FlatScene) -> i32 {
        push_pattern(out, sys::RTC_PAT_CHECKERS, 0, NO_UV, self.transformation_inverse(), self.a, self.b)
    }
}
// pattern/sine_2d.rs:39-44 — `b` carries `distance` (sine_2d.rs:22)
impl Sine2D {
    fn lower(&self, out: &mut FlatScene) -> i32 {
        push_pattern(out, sys::RTC_PAT_SINE2D, 0, NO_UV, self.transformation_inverse(), self.a, self.distance)
    }
}
// pattern/pattern.rs:32-63 — BasePattern is "not meant to be instantiated by itself"
impl BasePattern {
    fn lower(&self, _out: &mut FlatScene) -> i32 {
        unimplemented!()
    }
}
// pattern/pattern.rs:66-88
impl TestPattern {
    fn lower(&self, out: &mut FlatScene) -> i32 {
        push_pattern(out, sys::RTC_PAT_TEST, 0, NO_UV, self.transformation_inverse(), black(), black())
    }
}
// pattern/uv.rs:64-93
impl TextureMap {
    fn lower(&self, out: &mut FlatScene) -> i32 {
        let mut uv = NO_UV;
        uv[0] = self.uv_pattern.lower_uv(out);
        push_pattern(out, sys::RTC_PAT_TEXTURE_MAP, self.uv_mapping.mapping_id(), uv, self.transformation_inverse(), black(), black())
    }
}
// pattern/uv.rs:215-283 — uv_patterns is in Face order: Front, Back, Left, Right, Up, Down (uv.rs:229-249)
impl CubicMap {
    fn lower(&self, out: &mut FlatScene) -> i32 {
        let mut uv = NO_UV;
        for (i, p) in self.uv_patterns.iter().enumerate() {
            uv[i] = p.lower_uv(out);
        }
        push_pattern(out, sys::RTC_PAT_CUBIC_MAP, 0, uv, self.transformation_inverse(), black(), black())
    }
}
// pattern/uv.rs:96, 195, 203
impl SphericalMap {
    fn mapping_id(&self) -> i32 {
        sys::RTC_MAP_SPHERICAL
    }
}
impl PlanarMap {
    fn mapping_id(&self) -> i32 {
        sys::RTC_MAP_PLANAR
    }
}
impl CylindricalMap {
    fn mapping_id(&self) -> i32 {
        sys::RTC_MAP_CYLINDRICAL
    }
}
// pattern/uv.rs:21-56 — params: width, height, a.rgb, b.rgb
impl UVCheckers {
    fn lower_uv(&self, out: &mut FlatScene) -> i32 {
        let mut params = [0f32; 15];
        params[0] = self.width;
        params[1] = self.height;
        params[2..5].copy_from_slice(&rgb(self.a));
        params[5..8].copy_from_slice(&rgb(self.b));
        out.uvs.push(sys::RtcUvPattern { kind: sys::RTC_UV_CHECKERS, params });
        (out.uvs.len() - 1) as i32
    }
}
// pattern/uv.rs:135-176 — params: main, ul, ur, bl, br
impl AlignCheck {
    fn lower_uv(&self, out: &mut FlatScene) -> i32 {
        let mut params = [0f32; 15];
        for (i, c) in [self.main, self.ul, self.ur, self.bl, self.br].iter().enumerate() {
            params[3 * i..3 * i + 3].copy_from_slice(&rgb(*c));
        }
        out.uvs.push(sys::RtcUvPattern { kind: sys::RTC_UV_ALIGN_CHECK, params });
        (out.uvs.len() - 1) as i32
    }
}
// pattern/uv.rs:346-377 — the canvas travels once as an RtcTexture; the uv pattern names it by index (params[0])
impl UVImage {
    fn lower_uv(&self, out: &mut FlatScene) -> i32 {
        let (w, h) = (self.canvas.width, self.canvas.height);
        let mut px = Vec::with_capacity(w * h * 3);
        for y in 0..h {
            for x in 0..w {
                let c = self.canvas.pixel_at(x, y);
                px.extend_from_slice(&[c.r, c.g, c.b]);
            }
        }
        out.texture_pixels.push(px);
        out.texture_sizes.push((w as u32, h as u32));
        let mut params = [0f32; 15];
        params[0] = (out.texture_pixels.len() - 1) as f32;
        out.uvs.push(sys::RtcUvPattern { kind: sys::RTC_UV_IMAGE, params });
        (out.uvs.len() - 1) as i32
    }
}

// =====================================================================================================
// light/*.rs — `fn lower` of both Light implementers
// =====================================================================================================

// light/point_light.rs:7-18
impl PointLight {
    fn lower(&self, scene: *mut sys::RtcScene) {
        let p = [self.position.x, self.position.y, self.position.z];
        let i = rgb(self.intensity);
        unsafe { check(sys::rtc_set_point_light(scene, p.as_ptr(), i.as_ptr())) }
    }
}

// light/rectangle_light.rs — after construction u_vec / v_vec are per-CELL edges (:52-53) and `position` is the
// rectangle's centre (:57).  ONE ADDED FIELD: `jitter_is_rng: bool`, set by `new` when jitter_fn_opt is None (:44-47),
// because a boxed closure cannot be asked what it is.
//   * thread_rng (the shipped demos, soft_shadows.rs:72-82): unreproducible by construction — the device draws
//     from its counter-based generator, seeded here from thread_rng (table_len = 0);
//   * a caller's closure (test/utils.rs: constant_jitter, hardcoded_jitter): it is sampled 2 * cells times, in the
//     order intensity_at consumes it (`for v { for u { j_u, j_v } }`, :76-88), and sent as the jitter table.  That is
//     exactly the reference's sequence when the closure's period divides 2 * cells (constant_jitter; tables built for
//     the light), which is also the only case in which every intensity_at call of the reference sees the same values.
impl RectangleLight<'_> {
    fn lower(&self, scene: *mut sys::RtcScene) {
        let intensity = rgb(self.intensity);
        let corner = [self.corner.x, self.corner.y, self.corner.z];
        let u = [self.u_vec.x, self.u_vec.y, self.u_vec.z];
        let v = [self.v_vec.x, self.v_vec.y, self.v_vec.z];
        let position = [self.position.x, self.position.y, self.position.z];
        let (table, seed): (Vec<f32>, u64) = if self.jitter_is_rng {
            (Vec::new(), rand::thread_rng().gen::<u64>())
        } else {
            ((0..2 * self.cells).map(|_| (self.jitter_fn)()).collect(), 0)
        };
        unsafe {
            check(sys::rtc_set_rect_light(
                scene,
                intensity.as_ptr(),
                corner.as_ptr(),
                u.as_ptr(),
                self.u_steps,
                v.as_ptr(),
                self.v_steps,
                position.as_ptr(),
                if table.is_empty() { std::ptr::null() } else { table.as_ptr() },
                table.len() as u32,
                seed,
            ))
        }
    }
}

// =====================================================================================================
// camera.rs — the entry points (inside `impl Camera`, which can read its private fields)
// =====================================================================================================

/// What `Canvas::to_ppm` (canvas.rs:58-96) needs and nothing more: the 8-bit plane, i.e. every channel through
/// `scale_color` (canvas.rs:39-43) on the device.  A 4K frame is 24.9 MB instead of the 99.5 MB of f32 colours.
pub struct CanvasU8 {
    pub width: usize,
    pub height: usize,
    pub rgb: Vec<u8>, // width * height * 3, row-major
}

impl CanvasU8 {
    /// Byte-identical to `Canvas::to_ppm` of the same frame: P3 header, rows of at most 70 columns (canvas.rs:66-93).
    pub fn to_ppm(&self) -> String {
        let mut out = format!("P3\n{} {}\n255\n", self.width, self.height);
        for row in self.rgb.chunks(self.width * 3) {
            let mut line = String::new();
            let n = row.len();
            for (i, v) in row.iter().enumerate() {
                line.push_str(&v.to_string());
                if i != n - 1 {
                    if line.len() < 70 - 3 {
                        line.push(' ');
                    } else {
                        out.push_str(&line);
                        out.push('\n');
                        line.clear();
                    }
                }
            }
            if !line.is_empty() {
                out.push_str(&line);
                out.push('\n');
            }
        }
        out
    }
}

impl Camera {
    /// Flatten `world`, hand it to the device library and commit it on every visible GPU.
    unsafe fn commit_b200(&self, world: &World) -> *mut sys::RtcScene {
        let mut flat = FlatScene::new();
        for o in &world.objects {
            o.flatten(&mut flat, -1); // depth-first: the tie-break order of world.rs:58
        }
        let mut scene = std::ptr::null_mut();
        check(sys::rtc_scene_create(&mut scene));
        check(sys::rtc_set_camera(
            scene,
            self.width_pixels,
            self.height_pixels,
            self.half_width_world,
            self.half_height_world,
            self.pixel_size,
            mat16(&self.transform_inverse).as_ptr(),
        ));
        check(sys::rtc_set_primitives(scene, flat.prims.len() as u32, flat.prims.as_ptr()));
        check(sys::rtc_set_nodes(scene, flat.nodes.len() as u32, flat.nodes.as_ptr(), flat.refs.len() as u32, flat.refs.as_ptr()));
        check(sys::rtc_set_materials(scene, flat.materials.len() as u32, flat.materials.as_ptr()));
        check(sys::rtc_set_patterns(scene, flat.patterns.len() as u32, flat.patterns.as_ptr(), flat.uvs.len() as u32, flat.uvs.as_ptr()));
        let textures: Vec<sys::RtcTexture> = flat
            .texture_pixels
            .iter()
            .zip(&flat.texture_sizes)
            .map(|(px, &(w, h))| sys::RtcTexture { width: w, height: h, rgb: px.as_ptr() })
            .collect();
        check(sys::rtc_set_textures(scene, textures.len() as u32, textures.as_ptr()));
        world.light.as_ref().expect("World light should be set").lower(scene); // world.rs:66
        if flat.prims.len() >= 10_000 {
            // one-shot render of a big scene: build the tree on the device (a millisecond instead of 25-30 ms)
            check(sys::rtc_set_option(scene, sys::RTC_OPT_BVH_BUILDER, 1));
        }
        check(sys::rtc_scene_commit(scene, 0, std::ptr::null())); // 0: every visible GPU, bands interleaved
        scene
    }

    /// Same signature and result as `render` (camera.rs:76): World by value, depth, owned Canvas of f32 colours
    /// (last row and column black, camera.rs:80-81).
    pub fn render_b200(&self, world: World, reflection_recursion_depth: i16) -> Canvas {
        let (w, h) = (self.width_pixels as usize, self.height_pixels as usize);
        let mut rgb = vec![0f32; w * h * 3];
        unsafe {
            let scene = self.commit_b200(&world);
            let mut stats: sys::RtcStats = std::mem::zeroed();
            check(sys::rtc_render(scene, reflection_recursion_depth as i32, rgb.as_mut_ptr(), std::ptr::null_mut(), &mut stats));
            sys::rtc_scene_destroy(scene);
        }
        let mut canvas = Canvas::new(w, h);
        for y in 0..h {
            for x in 0..w {
                let i = (y * w + x) * 3;
                canvas.write_pixel(x, y, Color::new(rgb[i], rgb[i + 1], rgb[i + 2]));
            }
        }
        canvas
    }

    /// `render_b200` anti-aliased: each pixel is the mean of `samples_per_axis`² samples, the pixels of the reference's
    /// `Camera::new(n * hsize, n * vsize, fov, transform).render(world, depth)` (n = samples_per_axis) that fall in it,
    /// summed row by row in f32.  The samples are reduced on the device (`rtc_render_samples`); 1 is `render_b200`.
    pub fn render_b200_samples(&self, world: World, reflection_recursion_depth: i16, samples_per_axis: u32) -> Canvas {
        let (w, h) = (self.width_pixels as usize, self.height_pixels as usize);
        let mut rgb = vec![0f32; w * h * 3];
        unsafe {
            let scene = self.commit_b200(&world);
            let mut stats: sys::RtcStats = std::mem::zeroed();
            check(sys::rtc_render_samples(scene, reflection_recursion_depth as i32, samples_per_axis, rgb.as_mut_ptr(),
                                          std::ptr::null_mut(), &mut stats));
            sys::rtc_scene_destroy(scene);
        }
        let mut canvas = Canvas::new(w, h);
        for y in 0..h {
            for x in 0..w {
                let i = (y * w + x) * 3;
                canvas.write_pixel(x, y, Color::new(rgb[i], rgb[i + 1], rgb[i + 2]));
            }
        }
        canvas
    }

    /// The demos' flow — `camera.render(world, depth).to_ppm()` (e.g. demos/src/bin/soft_shadows.rs:84-87) — without
    /// the f32 plane ever leaving the device: `camera.render_b200_u8(world, depth).to_ppm()`.
    pub fn render_b200_u8(&self, world: World, reflection_recursion_depth: i16) -> CanvasU8 {
        let (w, h) = (self.width_pixels as usize, self.height_pixels as usize);
        let mut out = CanvasU8 { width: w, height: h, rgb: vec![0u8; w * h * 3] };
        unsafe {
            let scene = self.commit_b200(&world);
            let mut stats: sys::RtcStats = std::mem::zeroed();
            check(sys::rtc_render(scene, reflection_recursion_depth as i32, std::ptr::null_mut(), out.rgb.as_mut_ptr(), &mut stats));
            sys::rtc_scene_destroy(scene);
        }
        out
    }

    /// The demos' whole flow in one call: `println!("{}", camera.render_b200_ppm(world, 5))` prints exactly what
    /// `camera.render(world, 5).to_ppm()` prints (canvas.rs:58-96), with the text written on the device (`rtc_render_ppm`)
    /// and copied straight into the String's bytes.
    pub fn render_b200_ppm(&self, world: World, reflection_recursion_depth: i16) -> String {
        let bound = unsafe { sys::rtc_ppm_bound(self.width_pixels, self.height_pixels) };
        let mut text = vec![0u8; bound];
        let mut n = 0usize;
        unsafe {
            let scene = self.commit_b200(&world);
            let mut stats: sys::RtcStats = std::mem::zeroed();
            check(sys::rtc_render_ppm(scene, reflection_recursion_depth as i32, text.as_mut_ptr() as *mut std::os::raw::c_char, bound,
                                      &mut n, &mut stats));
            sys::rtc_scene_destroy(scene);
        }
        text.truncate(n);
        String::from_utf8(text).expect("PPM text is ASCII")
    }

    /// `Camera::render` for several cameras of one canvas size (a turntable, a stereo pair): the world is flattened and
    /// committed once — with the camera whose origin is farthest out, so that the tree's reach covers every view — and all
    /// views come from one `rtc_render_views` batch.  Canvas i is what `cameras[i].render(world, depth)` returns.
    pub fn render_b200_views(cameras: &[Camera], world: World, reflection_recursion_depth: i16) -> Vec<Canvas> {
        let (far, w, h, views) = Camera::batch_views(cameras);
        let mut rgb = vec![0f32; views.len() * w * h * 3];
        unsafe {
            let scene = cameras[far].commit_b200(&world);
            let mut stats: sys::RtcStats = std::mem::zeroed();
            check(sys::rtc_render_views(scene, reflection_recursion_depth as i32, views.len() as u32, views.as_ptr(), rgb.as_mut_ptr(),
                                        std::ptr::null_mut(), &mut stats));
            sys::rtc_scene_destroy(scene);
        }
        rgb.chunks(w * h * 3)
            .map(|frame| {
                let mut canvas = Canvas::new(w, h);
                for y in 0..h {
                    for x in 0..w {
                        let i = (y * w + x) * 3;
                        canvas.write_pixel(x, y, Color::new(frame[i], frame[i + 1], frame[i + 2]));
                    }
                }
                canvas
            })
            .collect()
    }

    /// `Camera::render` then `Canvas::to_ppm` for several cameras of one canvas size, committed once as `render_b200_views`
    /// commits them, with every view's text written on the device (`rtc_render_views_ppm`).  String i is what
    /// `cameras[i].render(world, depth).to_ppm()` returns.
    pub fn render_b200_views_ppm(cameras: &[Camera], world: World, reflection_recursion_depth: i16) -> Vec<String> {
        let (far, w, h, views) = Camera::batch_views(cameras);
        let capacity = views.len() * unsafe { sys::rtc_ppm_bound(w as u32, h as u32) };
        let mut text = vec![0u8; capacity];
        let mut offsets = vec![0usize; views.len() + 1];
        unsafe {
            let scene = cameras[far].commit_b200(&world);
            let mut stats: sys::RtcStats = std::mem::zeroed();
            check(sys::rtc_render_views_ppm(scene, reflection_recursion_depth as i32, views.len() as u32, views.as_ptr(),
                                            text.as_mut_ptr() as *mut std::os::raw::c_char, capacity, offsets.as_mut_ptr(), &mut stats));
            sys::rtc_scene_destroy(scene);
        }
        offsets
            .windows(2)
            .map(|o| String::from_utf8(text[o[0]..o[1]].to_vec()).expect("PPM text is ASCII"))
            .collect()
    }

    /// `render_b200_views` anti-aliased: canvas i is `cameras[i].render_b200_samples(world, depth, samples_per_axis)`, every
    /// view of the batch from one commit and one `rtc_render_views_samples` call.
    pub fn render_b200_views_samples(cameras: &[Camera], world: World, reflection_recursion_depth: i16, samples_per_axis: u32)
                                     -> Vec<Canvas> {
        let (far, w, h, views) = Camera::batch_views(cameras);
        let mut rgb = vec![0f32; views.len() * w * h * 3];
        unsafe {
            let scene = cameras[far].commit_b200(&world);
            let mut stats: sys::RtcStats = std::mem::zeroed();
            check(sys::rtc_render_views_samples(scene, reflection_recursion_depth as i32, views.len() as u32, views.as_ptr(),
                                                samples_per_axis, rgb.as_mut_ptr(), std::ptr::null_mut(), &mut stats));
            sys::rtc_scene_destroy(scene);
        }
        rgb.chunks(w * h * 3)
            .map(|frame| {
                let mut canvas = Canvas::new(w, h);
                for y in 0..h {
                    for x in 0..w {
                        let i = (y * w + x) * 3;
                        canvas.write_pixel(x, y, Color::new(frame[i], frame[i + 1], frame[i + 2]));
                    }
                }
                canvas
            })
            .collect()
    }

    /// `render_b200_views_samples` then `Canvas::to_ppm` of every view, the texts written on the device
    /// (`rtc_render_views_samples_ppm`).  String i is `cameras[i].render_b200_samples(world, depth, samples_per_axis).to_ppm()`.
    pub fn render_b200_views_samples_ppm(cameras: &[Camera], world: World, reflection_recursion_depth: i16, samples_per_axis: u32)
                                         -> Vec<String> {
        let (far, w, h, views) = Camera::batch_views(cameras);
        let capacity = views.len() * unsafe { sys::rtc_ppm_bound(w as u32, h as u32) };
        let mut text = vec![0u8; capacity];
        let mut offsets = vec![0usize; views.len() + 1];
        unsafe {
            let scene = cameras[far].commit_b200(&world);
            let mut stats: sys::RtcStats = std::mem::zeroed();
            check(sys::rtc_render_views_samples_ppm(scene, reflection_recursion_depth as i32, views.len() as u32, views.as_ptr(),
                                                    samples_per_axis, text.as_mut_ptr() as *mut std::os::raw::c_char, capacity,
                                                    offsets.as_mut_ptr(), &mut stats));
            sys::rtc_scene_destroy(scene);
        }
        offsets
            .windows(2)
            .map(|o| String::from_utf8(text[o[0]..o[1]].to_vec()).expect("PPM text is ASCII"))
            .collect()
    }

    /// The anti-aliased demo flow in one call: `camera.render_b200_samples_ppm(world, depth, n)` is
    /// `camera.render_b200_samples(world, depth, n).to_ppm()`, with the text written on the device.
    pub fn render_b200_samples_ppm(&self, world: World, reflection_recursion_depth: i16, samples_per_axis: u32) -> String {
        Camera::render_b200_views_samples_ppm(std::slice::from_ref(self), world, reflection_recursion_depth, samples_per_axis)
            .pop()
            .expect("one view")
    }

    /// A batch's views and the camera it commits with: the one whose origin is farthest out, so that the tree's reach
    /// covers every view.  Every camera must have one canvas size.
    fn batch_views(cameras: &[Camera]) -> (usize, usize, usize, Vec<sys::RtcView>) {
        assert!(!cameras.is_empty(), "a batch needs at least one camera");
        let reach = |c: &Camera| {
            let m = mat16(&c.transform_inverse);
            m[3].abs().max(m[7].abs()).max(m[11].abs())
        };
        let mut far = 0;
        for (i, c) in cameras.iter().enumerate() {
            if reach(c) > reach(&cameras[far]) {
                far = i;
            }
        }
        let (w, h) = (cameras[far].width_pixels as usize, cameras[far].height_pixels as usize);
        let views: Vec<sys::RtcView> = cameras
            .iter()
            .map(|c| {
                assert!(c.width_pixels as usize == w && c.height_pixels as usize == h, "every view of a batch has one canvas size");
                sys::RtcView {
                    half_width: c.half_width_world,
                    half_height: c.half_height_world,
                    pixel_size: c.pixel_size,
                    transform_inverse: mat16(&c.transform_inverse),
                }
            })
            .collect();
        (far, w, h, views)
    }
}
