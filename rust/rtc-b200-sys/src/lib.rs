//! Raw bindings of include/rtc_b200.h.  NOT COMPILED IN THIS REPO'S CI: the build image has no Rust toolchain
//! (SURVEY.md §0.2); the layouts below are kept in sync with the header by hand and mirror the ctypes structures
//! in ray_tracer_challenge_b200/__init__.py, which ARE exercised by the test-suite.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
pub struct RtcScene {
    _private: [u8; 0],
}

pub const RTC_OK: c_int = 0;
pub const RTC_ERR_INVALID: c_int = -1;
pub const RTC_ERR_NO_DEVICE: c_int = -2;
pub const RTC_ERR_CAPACITY: c_int = -3;
pub const RTC_ERR_STATE: c_int = -4;
pub const RTC_ERR_CUDA: c_int = -5;

pub const RTC_SPHERE: i32 = 0;
pub const RTC_PLANE: i32 = 1;
pub const RTC_CUBE: i32 = 2;
pub const RTC_CYLINDER: i32 = 3;
pub const RTC_CONE: i32 = 4;
pub const RTC_TRIANGLE: i32 = 5;
pub const RTC_NODE_GROUP: i32 = 0;
pub const RTC_NODE_CSG: i32 = 1;
pub const RTC_CSG_UNION: i32 = 0;
pub const RTC_CSG_INTERSECTION: i32 = 1;
pub const RTC_CSG_DIFFERENCE: i32 = 2;
pub const RTC_PAT_STRIPES: i32 = 0;
pub const RTC_PAT_GRADIENT: i32 = 1;
pub const RTC_PAT_RINGS: i32 = 2;
pub const RTC_PAT_CHECKERS: i32 = 3;
pub const RTC_PAT_SINE2D: i32 = 4;
pub const RTC_PAT_TEST: i32 = 5;
pub const RTC_PAT_TEXTURE_MAP: i32 = 6;
pub const RTC_PAT_CUBIC_MAP: i32 = 7;
pub const RTC_UV_CHECKERS: i32 = 0;
pub const RTC_UV_ALIGN_CHECK: i32 = 1;
pub const RTC_UV_IMAGE: i32 = 2;
pub const RTC_MAP_SPHERICAL: i32 = 0;
pub const RTC_MAP_PLANAR: i32 = 1;
pub const RTC_MAP_CYLINDRICAL: i32 = 2;
pub const RTC_BAND_ROWS: u32 = 8;
pub const RTC_OPT_FMA_CONTRACTION: i32 = 1;
pub const RTC_OPT_BVH_LEAF_SIZE: i32 = 2;
pub const RTC_OPT_BVH_MIN_PRIMS: i32 = 3;
pub const RTC_OPT_RENDER_SLICES: i32 = 4;
pub const RTC_OPT_ADAPTIVE_ORDER: i32 = 5;
pub const RTC_OPT_SHADOW_FILTER: i32 = 6;
pub const RTC_OPT_BVH_BUILDER: i32 = 7;
pub const RTC_OPT_WAVEFRONT: i32 = 8;
pub const RTC_OPT_EXACT_GROUPS: i32 = 9;

#[repr(C)]
#[derive(Clone, Copy)]
pub struct RtcPrim {
    pub type_: i32,
    pub material: i32,
    pub casts_shadow: i32,
    pub parent: i32,
    pub inv: [f32; 16],
    pub params: [f32; 12],
    pub bbox_min: [f32; 3],
    pub bbox_max: [f32; 3],
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct RtcNode {
    pub kind: i32,
    pub parent: i32,
    pub op: i32,
    pub child_begin: i32,
    pub child_count: i32,
    pub inv: [f32; 16],
    pub bbox_min: [f32; 3],
    pub bbox_max: [f32; 3],
    pub world_bbox_min: [f32; 3],
    pub world_bbox_max: [f32; 3],
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct RtcMaterial {
    pub color: [f32; 3],
    pub ambient: f32,
    pub diffuse: f32,
    pub specular: f32,
    pub shininess: f32,
    pub reflective: f32,
    pub transparency: f32,
    pub refractive_index: f32,
    pub pattern: i32,
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct RtcPattern {
    pub kind: i32,
    pub mapping: i32,
    pub uv: [i32; 6],
    pub inv: [f32; 16],
    pub a: [f32; 3],
    pub b: [f32; 3],
}

pub const RTC_UV_CHECKERS: i32 = 0;
pub const RTC_UV_ALIGN_CHECK: i32 = 1;
pub const RTC_UV_IMAGE: i32 = 2;

#[repr(C)]
#[derive(Clone, Copy)]
pub struct RtcUvPattern {
    pub kind: i32,
    pub params: [f32; 15],
}

/// The Canvas behind a UVImage (canvas.rs:6-10): width * height * 3 f32, row-major, row 0 at the top.
#[repr(C)]
#[derive(Clone, Copy)]
pub struct RtcTexture {
    pub width: u32,
    pub height: u32,
    pub rgb: *const f32,
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct RtcStats {
    pub primary_rays: u64,
    pub secondary_rays: u64,
    pub shadow_rays: u64,
    pub shades: u64,
    pub node_visits: u64,
    pub prim_tests: [u64; 8],
    pub xforms: u64,
    pub patterns: u64,
    pub cells: u64,
    pub schlicks: u64,
    pub refr_dirs: u64,
    pub capacity_overflows: u64,
    pub flops: f64,
    pub kernel_ms: f64,
    pub total_ms: f64,
    pub n_devices: i32,
    pub detailed: i32,
    pub launches: i32,
    pub wave_overflows: i32,
}

/// One camera view of `rtc_render_views`: `Camera::new`'s derived fields (camera.rs:23-56), as `rtc_set_camera` takes them.
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct RtcView {
    pub half_width: f32,
    pub half_height: f32,
    pub pixel_size: f32,
    pub transform_inverse: [f32; 16],
}

/// What `rtc_scene_commit` would build, computed without a device (`rtc_scene_inspect`).
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct RtcCommitInfo {
    pub n_positions: i32,
    pub n_bvh_nodes: i32,
    pub n_linear: i32,
    pub n_xforms: i32,
    pub bvh_leaf_size: i32,
    pub small_n: i32,
    pub filter_ok: i32,
    pub cell_masks: i32,
    pub plane_cells: i32,
    pub converge: i32,
    pub tol_sphere: f32,
    pub light_ball: [f32; 4],
    pub bvh_depth: i32,
    pub host_ms: f64,
    pub digest: u64,
    pub lean: i32,
    pub exact_groups: i32,
    pub loose_group_boxes: i32,
}

extern "C" {
    pub fn rtc_last_error() -> *const c_char;
    pub fn rtc_device_count() -> c_int;
    pub fn rtc_scene_create(out: *mut *mut RtcScene) -> c_int;
    pub fn rtc_scene_destroy(scene: *mut RtcScene);
    pub fn rtc_set_camera(scene: *mut RtcScene, width: u32, height: u32, half_width: f32, half_height: f32,
                          pixel_size: f32, transform_inverse: *const f32) -> c_int;
    pub fn rtc_set_primitives(scene: *mut RtcScene, n: u32, prims: *const RtcPrim) -> c_int;
    pub fn rtc_set_nodes(scene: *mut RtcScene, n_nodes: u32, nodes: *const RtcNode, n_refs: u32, refs: *const i32) -> c_int;
    /// Zero-copy variants: the scene allocates (uninitialised) and the host writes the records in place.
    pub fn rtc_map_primitives(scene: *mut RtcScene, n: u32, prims: *mut *mut RtcPrim) -> c_int;
    pub fn rtc_map_nodes(scene: *mut RtcScene, n_nodes: u32, n_refs: u32, nodes: *mut *mut RtcNode, refs: *mut *mut i32) -> c_int;
    pub fn rtc_set_materials(scene: *mut RtcScene, n: u32, materials: *const RtcMaterial) -> c_int;
    pub fn rtc_set_patterns(scene: *mut RtcScene, n: u32, patterns: *const RtcPattern, n_uv: u32, uv: *const RtcUvPattern) -> c_int;
    pub fn rtc_set_textures(scene: *mut RtcScene, n: u32, textures: *const RtcTexture) -> c_int;
    pub fn rtc_set_point_light(scene: *mut RtcScene, position: *const f32, intensity: *const f32) -> c_int;
    pub fn rtc_set_rect_light(scene: *mut RtcScene, intensity: *const f32, corner: *const f32, u_cell: *const f32,
                              u_steps: i32, v_cell: *const f32, v_steps: i32, position: *const f32,
                              jitter_table: *const f32, table_len: u32, seed: u64) -> c_int;
    pub fn rtc_set_option(scene: *mut RtcScene, option: i32, value: i64) -> c_int;
    pub fn rtc_scene_inspect(scene: *mut RtcScene, out: *mut RtcCommitInfo) -> c_int;
    pub fn rtc_scene_commit(scene: *mut RtcScene, n_devices: i32, device_ids: *const i32) -> c_int;
    pub fn rtc_render(scene: *mut RtcScene, depth: i32, rgb_f32: *mut f32, rgb_u8: *mut u8, stats: *mut RtcStats) -> c_int;
    pub fn rtc_render_shard(scene: *mut RtcScene, depth: i32, shard: i32, n_shards: i32, rgb_f32: *mut f32,
                            rgb_u8: *mut u8, stats: *mut RtcStats) -> c_int;
    pub fn rtc_render_detailed(scene: *mut RtcScene, depth: i32, rgb_f32: *mut f32, rgb_u8: *mut u8, stats: *mut RtcStats) -> c_int;
    pub fn rtc_render_views(scene: *mut RtcScene, depth: i32, n_views: u32, views: *const RtcView, rgb_f32: *mut f32, rgb_u8: *mut u8,
                            stats: *mut RtcStats) -> c_int;
    pub fn rtc_trace_rays(scene: *mut RtcScene, n: u32, origins: *const f32, directions: *const f32, depth: i32,
                          out_rgb: *mut f32, out_t: *mut f32, out_prim: *mut i32) -> c_int;
    pub fn rtc_shard_bands(height: u32, shard: i32, n_shards: i32, first_rows: *mut u32) -> c_int;
    pub fn rtc_host_alloc(bytes: usize) -> *mut c_void;
    pub fn rtc_host_free(ptr: *mut c_void);
    pub fn rtc_host_register(ptr: *mut c_void, bytes: usize) -> c_int;
    pub fn rtc_host_unregister(ptr: *mut c_void) -> c_int;
    pub fn rtc_flush_l2(scene: *mut RtcScene) -> c_int;
    pub fn rtc_measure_fp32_peak(device: i32, tflops: *mut f64, sm_clock_mhz: *mut f64) -> c_int;
}
