/* rtc_b200.h — the drop-in boundary: a C ABI over the B200 (sm_100a) implementation of the reference's
 * `Camera::render` hot path.
 *
 * The reference (garfieldnate/ray_tracer_challenge, Rust) has no FFI of its own; its boundary for this path
 * is the method `Camera::render(&self, world: World, depth: i16) -> Canvas` (lib/src/camera.rs:76-91).
 * A Rust host would add the sibling `Camera::render_b200` which flattens `World` (lib/src/world.rs:18-21)
 * into the POD arrays below and calls this library through a `-sys` crate (see INTEGRATION.md for the
 * binding).  In this repo the same calls are made by the C++ host mirror
 * (ray_tracer_challenge_b200/csrc/host/, Camera::render_b200) and, for tests, by Python/ctypes.
 *
 * Conventions: every function returns 0 on success or a negative RtcStatus; nothing panics or throws
 * across the ABI; rtc_last_error() returns the thread-local message of the last failure.  All pointers
 * are caller-owned and copied before the call returns.  Matrices are 16 f32, row-major.  A scene handle
 * may be used by one host thread at a time.  There is NO CPU fallback: without a CUDA device
 * rtc_scene_commit / rtc_render fail with RTC_ERR_NO_DEVICE.
 */
#ifndef RTC_B200_H
#define RTC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct RtcScene RtcScene;

typedef enum RtcStatus {
    RTC_OK = 0,
    RTC_ERR_INVALID = -1,   /* bad argument / inconsistent scene */
    RTC_ERR_NO_DEVICE = -2, /* no CUDA device is visible (there is no CPU fallback) */
    RTC_ERR_CAPACITY = -3,  /* a documented device-side capacity was exceeded (depth, CSG size) */
    RTC_ERR_STATE = -4,     /* call sequence error (render before commit, ...) */
    RTC_ERR_CUDA = -5       /* a CUDA runtime call failed on a visible device (out of memory, launch failure, ...);
                               rtc_last_error() names the call */
} RtcStatus;

/* Leaf primitive kinds — lib/src/shape/{sphere,plane,cube,cylinder,cone,triangle}.rs.  SmoothTriangle
 * (smooth_triangle.rs:39-41) delegates its intersection to the inner flat Triangle, so it is lowered to
 * RTC_TRIANGLE. */
enum { RTC_SPHERE = 0, RTC_PLANE = 1, RTC_CUBE = 2, RTC_CYLINDER = 3, RTC_CONE = 4, RTC_TRIANGLE = 5 };

/* One leaf of the shape tree, in depth-first order of World::objects / GroupShape::children / CSG s1,s2.
 * That order is the reference's tie-break between equal distances (world.rs:58 stable sort +
 * intersection.rs:30-35 first minimum). */
typedef struct RtcPrim {
    int32_t type;
    int32_t material;     /* index into the material table */
    int32_t casts_shadow; /* BaseShape::casts_shadow, base_shape.rs:14 */
    int32_t parent;       /* index into the node table (enclosing GroupShape / CSG) or -1 */
    float inv[16];        /* Shape::transformation_inverse(), base_shape.rs:56-60; the inverse-transpose used
                             by normal_to_world (shape.rs:130) is its transpose */
    float params[12];     /* cylinder / cone: {minimum_y, maximum_y, closed}; triangle: p1, e1, e2, normal
                             (triangle.rs:20-33) */
    float bbox_min[3];    /* Shape::parent_space_bounding_box(), shape.rs:162-164 */
    float bbox_max[3];
} RtcPrim;

/* Interior node of the shape tree.  Groups have already pushed their transform into their leaves
 * (group.rs:39-44,101-114) and act only as bounding-box culls (group.rs:119-133); CSG nodes keep their own
 * transform (csg.rs:78) and filter their children's sorted hits (csg.rs:37-58,87-104). */
enum { RTC_NODE_GROUP = 0, RTC_NODE_CSG = 1 };
enum { RTC_CSG_UNION = 0, RTC_CSG_INTERSECTION = 1, RTC_CSG_DIFFERENCE = 2 };
typedef struct RtcNode {
    int32_t kind;
    int32_t parent;      /* node index or -1 */
    int32_t op;          /* CSG operator */
    int32_t child_begin; /* into the child reference array */
    int32_t child_count; /* CSG: exactly 2 (s1, s2) */
    float inv[16];       /* CSG: its own transformation_inverse(); groups: identity */
    float bbox_min[3];   /* the node's own bounding_box() as the reference caches it (group.rs:138-150,
                            csg.rs:119-130), in the space its cull test runs in */
    float bbox_max[3];
    float world_bbox_min[3]; /* parent_space_bounding_box() (csg: bounding_box().transform(t)) */
    float world_bbox_max[3];
} RtcNode;
/* child reference: >= 0 is a primitive index, < 0 is ~node_index */

typedef struct RtcMaterial { /* material.rs:19-51 */
    float color[3];
    float ambient, diffuse, specular, shininess, reflective, transparency, refractive_index;
    int32_t pattern; /* index into the pattern table or -1 */
} RtcMaterial;

/* pattern/{stripes,gradient,rings,checkers,sine_2d,pattern,uv}.rs */
enum {
    RTC_PAT_STRIPES = 0,
    RTC_PAT_GRADIENT = 1,
    RTC_PAT_RINGS = 2,
    RTC_PAT_CHECKERS = 3,
    RTC_PAT_SINE2D = 4,
    RTC_PAT_TEST = 5,
    RTC_PAT_TEXTURE_MAP = 6,
    RTC_PAT_CUBIC_MAP = 7
};
enum { RTC_UV_CHECKERS = 0, RTC_UV_ALIGN_CHECK = 1, RTC_UV_IMAGE = 2 };
enum { RTC_MAP_SPHERICAL = 0, RTC_MAP_PLANAR = 1, RTC_MAP_CYLINDRICAL = 2 };
typedef struct RtcPattern {
    int32_t kind;
    int32_t mapping; /* TextureMap */
    int32_t uv[6];   /* TextureMap: uv[0]; CubicMap: Front, Back, Left, Right, Up, Down (uv.rs:229-249) */
    float inv[16];   /* BasePattern::t_inverse, pattern.rs:53-55 */
    float a[3];      /* first colour */
    float b[3];      /* second colour; for Gradient / Sine2D the precomputed `distance = b - a`
                        (gradient.rs:23, sine_2d.rs:22) */
} RtcPattern;
typedef struct RtcUvPattern {
    int32_t kind;
    float params[15]; /* UVCheckers: width, height, a.rgb, b.rgb; AlignCheck: main, ul, ur, bl, br;
                         UVImage (uv.rs:346-377): params[0] = texture index (rtc_set_textures) */
} RtcUvPattern;
/* The Canvas behind a UVImage (canvas.rs:6-10): width * height * 3 f32, row-major, row 0 at the top. */
typedef struct RtcTexture {
    uint32_t width, height;
    const float* rgb; /* caller keeps ownership; copied by rtc_set_textures */
} RtcTexture;

typedef struct RtcStats {
    uint64_t primary_rays;   /* color_at calls from render (camera.rs:83) */
    uint64_t secondary_rays; /* color_at calls from reflected_color / refracted_color (world.rs:129,159) */
    uint64_t shadow_rays;    /* is_shadowed calls (world.rs:104) */
    uint64_t shades;         /* shade_hit calls */
    uint64_t node_visits;    /* BVH boxes tested (detailed pass only) */
    uint64_t prim_tests[8];  /* local_intersect calls by RTC_* type; [6] = CSG evaluations; [7] = shadow rays the
                                shadow filter handed to the exact test (detailed pass only) */
    uint64_t xforms;         /* ray -> object transforms actually performed (detailed pass only) */
    uint64_t patterns, cells, schlicks, refr_dirs;
    uint64_t capacity_overflows; /* CSG hit-buffer overflows: must be 0 for a valid frame */
    double flops;            /* algorithmic FP32 flops (SURVEY.md Appendix E); detailed pass only */
    double kernel_ms;        /* CUDA-event time of the render kernel(s), max over devices */
    double total_ms;         /* host wall time of the call including D2H copies */
    int32_t n_devices;
    int32_t detailed;
    int32_t launches; /* render kernel launches of this call, over all devices */
    int32_t wave_overflows; /* chunks of the frame whose ray pool overflowed in the wavefront renderer and were rendered
                               again by the streaming kernel (0 in the normal case; the frame is complete either way) */
} RtcStats;

const char* rtc_last_error(void);
int rtc_device_count(void); /* >= 0, or a negative RtcStatus */

int rtc_scene_create(RtcScene** out);
void rtc_scene_destroy(RtcScene*);

/* Camera::new's derived fields exactly as the reference computes them (camera.rs:23-56). */
int rtc_set_camera(RtcScene*, uint32_t width, uint32_t height, float half_width, float half_height, float pixel_size,
                   const float transform_inverse[16]);
int rtc_set_primitives(RtcScene*, uint32_t n, const RtcPrim* prims);
int rtc_set_nodes(RtcScene*, uint32_t n_nodes, const RtcNode* nodes, uint32_t n_refs, const int32_t* child_refs);
/* The same without the copy: the scene allocates the arrays and the host writes its records in place (a
 * 100 000-primitive array is 14 MB; a one-shot Camera::render_b200 would otherwise write it twice).  The storage is
 * uninitialised: every record must be written before rtc_scene_commit.  The pointers stay valid until the next
 * rtc_set_* / rtc_map_* call for the same array, or rtc_scene_destroy. */
int rtc_map_primitives(RtcScene*, uint32_t n, RtcPrim** prims);
int rtc_map_nodes(RtcScene*, uint32_t n_nodes, uint32_t n_refs, RtcNode** nodes, int32_t** child_refs);
int rtc_set_materials(RtcScene*, uint32_t n, const RtcMaterial* materials);
int rtc_set_patterns(RtcScene*, uint32_t n, const RtcPattern* patterns, uint32_t n_uv, const RtcUvPattern* uv);
/* Image textures referenced by RTC_UV_IMAGE patterns.  UVImage::color_at (uv.rs:366-377): x = round(u * (width - 1)),
 * y = round((1 - v) * (height - 1)), nearest pixel; where the reference would index outside the canvas and panic
 * (u or v outside [0, 1]) the device clamps to the edge. */
int rtc_set_textures(RtcScene*, uint32_t n, const RtcTexture* textures);
/* PointLight (point_light.rs:7-18) */
int rtc_set_point_light(RtcScene*, const float position[3], const float intensity[3]);
/* RectangleLight after construction (rectangle_light.rs:48-58): u_cell / v_cell are the per-cell edges,
 * `position` the rectangle centre used by phong_lighting (phong_lighting.rs:36).  Jitter: a cyclic table
 * consumed `for v { for u { j_u, j_v } }` (rectangle_light.rs:60-88), or, with table_len == 0, the counter-based
 * generator seeded by `seed` (stand-in for thread_rng, rectangle_light.rs:46).
 * DEVIATION: the reference's table closure (test/utils.rs `hardcoded_jitter`) is ONE stateful cyclic iterator whose
 * cursor carries over from one intensity_at call to the next, in the serial order of the render loop.  Here every
 * intensity_at starts at index 0 (pixels are shaded in parallel; there is no call order).  The two coincide exactly
 * when table_len divides 2 * u_steps * v_steps (every call consumes whole cycles), so any other table_len is
 * REJECTED with RTC_ERR_INVALID rather than rendered with different shadows. */
int rtc_set_rect_light(RtcScene*, const float intensity[3], const float corner[3], const float u_cell[3],
                       int32_t u_steps, const float v_cell[3], int32_t v_steps, const float position[3],
                       const float* jitter_table, uint32_t table_len, uint64_t seed);

/* Options.  RTC_OPT_FMA_CONTRACTION (default 0): the kernels exist in two builds of the same source.  The
 * default one is compiled with -fmad=false and evaluates every expression in the Rust / IEEE order, so frames
 * are bit-for-bit the reference's apart from libm (powf, cosf, atan2f, acosf).  1 selects the FMA-contracted
 * build: a few percent faster, but its last-place differences flip ill-conditioned threshold tests (the
 * discriminant of a distant sphere cancels catastrophically in f32), so it meets the <= 1 LSB bar only on
 * well-conditioned scenes.  It may be changed between renders; the BVH options only before commit. */
enum {
    RTC_OPT_FMA_CONTRACTION = 1,
    RTC_OPT_BVH_LEAF_SIZE = 2, /* primitives per BVH leaf, 1..16; 0 (default) = 4 for triangle meshes, 1 otherwise */
    RTC_OPT_BVH_MIN_PRIMS = 3,
    RTC_OPT_RENDER_SLICES = 4, /* at most this many kernel launches a frame is cut into when it is copied to host memory, so
                                  the copy of one slice overlaps the kernels of the next (default 24, 1..64; never more than
                                  one slice per MiB copied).  The slices rotate over three streams: the blocks of a slice
                                  fill the SMs as the previous one drains */
    RTC_OPT_ADAPTIVE_ORDER = 5, /* default 1: a repeated render of the same shard launches its 16x8-pixel tiles
                                  most-expensive-first (clock cycles per tile recorded by an earlier render) when a
                                  timed trial render shows that order to be faster; changes no pixel */
    RTC_OPT_BVH_BUILDER = 7,   /* 0 (default): the host's binned-SAH builder — the better tree, 25-30 ms for 10^5 primitives;
                                  1: the device builder (Morton codes, sort, Karras topology, refit: K3 lbvh_build) for
                                  scenes of >= 1024 bounded items — a millisecond, a tree that costs more visits per ray:
                                  the choice for a one-shot render, where the build is most of the frame.  Same pixels
                                  either way (the tree only selects which primitives get the exact test).  Before commit */
    RTC_OPT_WAVEFRONT = 8,     /* default 0.  1: tree scenes whose ray trees branch, under a point light, are rendered as a
                                  wavefront — per bounce level a queue of rays, tree walks in a kernel whose lanes draw the
                                  next ray when theirs ends, shading and the post-order combine in kernels of their own —
                                  instead of the streaming kernel.  Same pixels; on B200 it measures ~15 % slower (the walks
                                  are bound by dependent node loads, not by idle lanes), so it is opt-in.  Any time.
                                  rtc_render_views does not use it: a batch takes the streaming kernel */
    RTC_OPT_EXACT_GROUPS = 9,  /* default 0.  1: every bounded primitive, and every outermost CSG, inside a GroupShape reports
                                  a hit only when each enclosing group's cached box passes the forward ray first
                                  (group.rs:115-133), in tree scenes too; with 0 that chain is checked only for the items
                                  tested for every ray (small scenes, unbounded shapes).  The two differ where the reference's
                                  f32 sphere test reports phantom hits at the silhouettes of far, small spheres, and wherever
                                  a group's box is stale (cached before a later add_child or set_transformation, group.rs:19):
                                  then the reference clips what lies outside the old box, and only 1 reproduces that.  Other
                                  values are RTC_ERR_INVALID.  Before commit (it changes the uploaded heads and the digest) */
    RTC_OPT_SHADOW_FILTER = 6   /* default 1: in small scenes of spheres, planes and axis-aligned cubes a shadow ray is
                                  first decided on the un-normalised point->light segment with error bounds; only
                                  undecided rays run the reference's arithmetic.  Changes no pixel (0 = always run
                                  the exact test: the A/B switch the parity tests use) */
};
int rtc_set_option(RtcScene*, int32_t option, int64_t value);

/* What rtc_scene_commit will build for the scene as it stands: runs the host half of the commit (validation, BVH,
 * CSG programs, small-scene table and its shadow-filter eligibility) without touching a device — for tests and
 * tooling on machines without a GPU.  Nothing is uploaded or kept. */
typedef struct RtcCommitInfo {
    int32_t n_positions;     /* device primitive slots (leaves + CSG pseudo-primitives) */
    int32_t n_bvh_nodes;     /* 0: no tree */
    int32_t n_linear;        /* primitives tested for every ray (unbounded shapes, or every item of a small scene) */
    int32_t n_xforms;        /* distinct inverse transforms */
    int32_t bvh_leaf_size;   /* the leaf size used (RTC_OPT_BVH_LEAF_SIZE, or the automatic choice) */
    int32_t small_n;         /* > 0: the small-scene path, with this many table entries */
    int32_t filter_ok;       /* shadow filter eligible (spheres / planes / axis-aligned cubes only) */
    int32_t cell_masks;      /* area light handled by the cell-mask loops */
    int32_t plane_cells;     /* per-(plane, cell) constants staged */
    int32_t converge;        /* some material is reflective and transparent: the converging kernel build */
    float tol_sphere;        /* the filter's relative error bound for spheres */
    float light_ball[4];     /* ball around the light's sample points (cell_masks) */
    int32_t bvh_depth;       /* levels of inner nodes on the longest root-to-leaf path (0: no tree); the builder keeps
                                it below the traversal stack's capacity for every scene */
    double host_ms;          /* time the host half took */
    uint64_t digest;         /* FNV-1a over the arrays a commit would upload for intersection (primitive heads and
                              * records, transforms, triangles, bounds, tree nodes, linear list): equal digests mean
                              * the device would trace the same geometry through the same tree */
    int32_t lean;            /* cell_masks and no pattern or transparency on the small-scene table: the lean kernel build */
    int32_t exact_groups;    /* RTC_OPT_EXACT_GROUPS as applied */
    int32_t loose_group_boxes; /* group nodes whose cached box does not contain the box of one of their children (a stale
                                  box): there the default culls differently from the reference on whole objects */
} RtcCommitInfo;
int rtc_scene_inspect(RtcScene*, RtcCommitInfo* out);

/* Validate, build the BVH over the primitives' bounding boxes and upload one scene replica per device.
 * device_ids == NULL selects devices 0..n_devices-1; n_devices == 0 selects every visible device. */
int rtc_scene_commit(RtcScene*, int32_t n_devices, const int32_t* device_ids);

/* Camera::render.  rgb_f32: width*height*3 (row-major, the Canvas layout, canvas.rs:6-25), rgb_u8: the same
 * pixels through Canvas::scale_color (canvas.rs:39-43); either may be NULL (NULL, NULL = render and leave the
 * frame on the device: kernel timing).  Rows are split in interleaved bands over the committed devices. */
int rtc_render(RtcScene*, int32_t depth, float* rgb_f32, uint8_t* rgb_u8, RtcStats* stats);
/* Same, for one shard of a frame shared by several processes (one process per GPU): only the bands
 * b with b % n_shards == shard are rendered and written; the other rows of the buffers are not touched. */
int rtc_render_shard(RtcScene*, int32_t depth, int32_t shard, int32_t n_shards, float* rgb_f32, uint8_t* rgb_u8,
                     RtcStats* stats);
/* The sharding rule of rtc_render / rtc_render_shard, exposed for hosts that place the shards themselves
 * (pure host arithmetic, no device needed): the frame is cut into bands of RTC_BAND_ROWS rows; band b belongs
 * to shard b % n_shards.  Returns how many bands `shard` owns and writes the first owned row of each to
 * first_rows (may be NULL; capacity >= the return value); a band's rows are [row, min(row + RTC_BAND_ROWS, height)). */
#define RTC_BAND_ROWS 8
int rtc_shard_bands(uint32_t height, int32_t shard, int32_t n_shards, uint32_t* first_rows);
/* As rtc_render but with the detailed work counters (node visits, primitive tests, flops). */
int rtc_render_detailed(RtcScene*, int32_t depth, float* rgb_f32, uint8_t* rgb_u8, RtcStats* stats);

/* One camera view of a batch: Camera::new's derived fields (camera.rs:23-56), as rtc_set_camera takes them. */
typedef struct RtcView {
    float half_width, half_height, pixel_size;
    float transform_inverse[16];
} RtcView;
/* Render n_views camera views of the committed scene, at the committed canvas size, in one batch: the scene stays committed,
 * and the pixels of every view come from one launch per device (per chunk, below), not one launch per view.
 * rgb_f32 / rgb_u8: n_views * height * width * 3 each, view-major (view v at offset v * height * width * 3); either may be
 * NULL (NULL, NULL = leave the frames on the device: kernel timing).  Pinned and pageable destinations both work.
 *   - View v's planes are bit-identical, in f32 and in 8 bits, to rtc_render of the scene committed with that camera, for
 *     every kernel build and option.  With generated jitter a pixel's generator key is its index within its own view
 *     (y * width + x), as in a single-view render.
 *   - The arguments are checked before the scene's state, all with RTC_ERR_INVALID: n_views == 0 or views == NULL; a
 *     non-finite field or pixel_size <= 0; a depth outside [0, 23] (rtc_render's rule).  Then an uncommitted scene is
 *     RTC_ERR_STATE.
 *   - Reach: a scene with a tree pads its boxes for coordinates up to the commit's reach — the largest of the bounded items'
 *     coordinates, the light's reach and the committed camera's origin.  A view whose camera origin (the translation column
 *     of transform_inverse) has a coordinate beyond it is refused with RTC_ERR_INVALID: commit with the farthest camera of
 *     the batch.  Small and tree-less scenes take any finite view.
 *   - With several committed devices each renders its interleaved bands of every view (rtc_shard_bands' rule); copies are
 *     queued after every device has its kernels.  Copied to host memory, the batch is cut into runs of whole views by
 *     rtc_render's slice rule applied to the whole batch (one slice per MiB copied, at most RTC_OPT_RENDER_SLICES); a view
 *     bigger than a slice is cut by bands as rtc_render cuts a frame.  The frames live in a device arena of 2 GiB per
 *     device (environment RTC_VIEW_ARENA_BYTES overrides it); a bigger batch is rendered chunk by chunk through it.  A
 *     pageable destination is staged through pinned host frames of at most 256 MiB per device (one view's planes when
 *     a view alone is bigger), kept with the device for later calls; a chunk then holds no more views than they fit.
 *   - A tree scene whose ray trees branch renders each chunk with one persistent streaming launch, whatever
 *     RTC_OPT_WAVEFRONT says.
 *   - stats: primary_rays = n_views * (width - 1) * (height - 1) over the devices' shares, launches = the launches made,
 *     kernel_ms from the first launch to the last.  With several chunks and a host destination a chunk's launches wait
 *     for the previous chunk's copies, so kernel_ms then includes that copy time; a batch that fits one chunk, or stays
 *     on the device, measures its kernels alone.  There is no detailed variant.
 *   - Nothing of rtc_render's state changes: the committed camera, its frame on the device and its learnt tile order.
 *     rtc_set_camera keeps its meaning (it invalidates the commit). */
int rtc_render_views(RtcScene*, int32_t depth, uint32_t n_views, const RtcView* views, float* rgb_f32, uint8_t* rgb_u8,
                     RtcStats* stats);
/* Anti-aliased Camera::render: n x n samples per pixel (n = samples_per_axis), box-filtered.  The samples of the committed
 * W x H canvas are pixels the reference itself renders: those of Camera::render at n W x n H with the same field of view
 * and transform (the sample camera C_n: Camera::new(n W, n H, fov, transform), camera.rs:23-56 — the committed half_width,
 * half_height and transform_inverse, pixel_size = (half_width * 2) / (float)(n W); C_1 is the committed camera).
 * rgb_f32 / rgb_u8: width * height * 3 each, as rtc_render's; either may be NULL (NULL, NULL = leave the frame on the device).
 *   - Pixel (x, y), x < width - 1 and y < height - 1: sample (i, j), i, j in [0, n), is color_at of C_n's ray for pixel
 *     (n x + i, n y + j); with generated jitter its generator key is that pixel's in the n W x n H frame,
 *     (n y + j) * (n W) + (n x + i).  Per channel in f32: s = sample (0, 0), then s = s + sample (i, j) with j the outer
 *     and i the inner loop, then s / (float)(n * n).  The 8-bit value is Canvas::scale_color of that mean.  The last row and
 *     column are zero in both planes (camera.rs:80-81).
 *   - So n = 1 gives rtc_render's planes bit for bit, and n >= 2 the box filter of rtc_render's frame of the scene
 *     committed with C_n (whose own last row and column are never used), for every kernel build and option.  The samples
 *     are reduced on the device: the n W x n H frame is never stored.
 *   - The arguments are checked before the scene's state, all with RTC_ERR_INVALID: a NULL scene; n outside [1, 16]; a
 *     sample canvas rtc_set_camera would refuse ((n W) * (n H) > 2^31 / 3); a depth outside [0, 23].  Then an uncommitted
 *     scene is RTC_ERR_STATE.
 *   - Destinations and devices as rtc_render_views' for one view: pinned or pageable host memory, each committed device
 *     rendering its interleaved bands of output rows (rtc_shard_bands' rule).  A tree scene whose ray trees branch renders
 *     with one persistent streaming launch, whatever RTC_OPT_WAVEFRONT says.
 *   - stats: primary_rays = n * n * (width - 1) * (height - 1) over the devices' shares, launches = the launches made,
 *     kernel_ms covers the render kernels.  There is no detailed variant.
 *   - Nothing of rtc_render's state changes: the committed camera, its frame on the device and its learnt tile order. */
int rtc_render_samples(RtcScene*, int32_t depth, uint32_t samples_per_axis, float* rgb_f32, uint8_t* rgb_u8, RtcStats* stats);
/* Camera::render followed by Canvas::to_ppm (canvas.rs:58-96), the last step of every demo, with the text written on the
 * device.  rtc_ppm_bound is host arithmetic: the header's length plus width * height * 3 * 4 bytes (three digits and a
 * separator per value), an upper bound on the text of any frame of that size.
 *   - ppm receives exactly the bytes Canvas::to_ppm returns for the rendered canvas: "P3\n{w} {h}\n255\n", then every row's
 *     values in decimal without padding, each followed by a space while the line is shorter than 70 - 3 columns and by a
 *     newline otherwise, and by a newline after the row's last value.  The rows and columns the reference does not render
 *     (camera.rs:80-81) are zeros.  *ppm_bytes receives the length; no terminating NUL is written.
 *   - The arguments are checked before the scene's state, all with RTC_ERR_INVALID: ppm or ppm_bytes NULL; a capacity below
 *     rtc_ppm_bound of the committed canvas; a depth outside [0, 23] (rtc_render's rule).  Then an uncommitted scene is
 *     RTC_ERR_STATE.
 *   - The render is rtc_render's with the frame left on the device; stats are rtc_render's (kernel_ms: the render kernels),
 *     except total_ms, which covers the whole call.  The text is written from the device's 8-bit plane: the value bytes of a
 *     row do not depend on the line breaks, so each device first computes the byte length of each of its rows, the host
 *     scans the lengths of all rows (one small device-to-host copy and a synchronize per call), and each device then writes
 *     its bands' text and copies each band to its offset in ppm.
 *   - Pinned and pageable destinations both work.  A pageable one receives texts of 4 MiB or more through the pinned staging
 *     frame that rtc_render uses for its 8-bit plane, grown to the device's share of the text and kept with the device.
 *   - Device memory kept with each device for later calls: the text of its rows (up to 12 bytes per pixel, 89 MB for a
 *     3840x2160 frame) and 16 bytes per row.
 *   - Not provided: encoding a plane that is not the committed scene's frame. */
size_t rtc_ppm_bound(uint32_t width, uint32_t height);
int rtc_render_ppm(RtcScene*, int32_t depth, char* ppm, size_t capacity, size_t* ppm_bytes, RtcStats* stats);
/* rtc_render_ppm for one shard of a frame shared by several processes (rtc_render_shard's split), in two phases with the
 * callers' exchange of row lengths in between: a row's text length depends only on its values, so once every row's length is
 * known each process can place its own bands.  The library has no communicator: the exchange is the callers' (shared memory
 * and a barrier on one node; an all-reduce of zeroed arrays across nodes).
 *   - Phase 1, rtc_render_shard_ppm_rows: rtc_render_shard with the frame left on the device, then the byte length of the text
 *     of every row the shard owns.  row_bytes has height entries in frame-row order; only the entries of the shard's rows
 *     (rtc_shard_bands) are written, the others are not touched — so the ranks can write into one shared array, or into zeroed
 *     private ones summed by an all-reduce.  stats are rtc_render_shard's, with total_ms covering the whole phase.
 *   - Phase 2, rtc_write_shard_ppm: given every row's length (all shards' entries), writes the text of the shard's bands at
 *     their offsets in ppm; shard 0 also writes the header.  It encodes the 8-bit plane its phase 1 left on the device
 *     (rtc_render_shard_samples_ppm_rows' anti-aliased one, below, as well).  *ppm_bytes receives the whole text's length, the same on every
 *     shard.  A shard writes only [band_at, band_at + band_bytes) of each of its bands (and shard 0 the header): no other byte
 *     of ppm, so the ranks can write into one shared buffer without locking.  No stats.
 *   - The bytes: the union of every shard's writes is byte for byte rtc_render_ppm's text of the same scene — Canvas::to_ppm of
 *     rtc_render's 8-bit plane — for every kernel build and option.
 *   - The arguments are checked before the scene's state, all with RTC_ERR_INVALID: a NULL pointer (stats may be NULL);
 *     n_shards < 1 or shard outside [0, n_shards); in phase 1 a depth outside [0, 23]; in phase 2 a capacity below
 *     rtc_ppm_bound of the committed canvas, and any row_bytes[r] outside [6 * width, 12 * width] (every value takes 2 to 4
 *     bytes with its separator, so an array in range never lays out a text longer than the bound).  Then an uncommitted scene
 *     is RTC_ERR_STATE, and so is a scene committed on more than one device (rtc_render_shard's rule).
 *   - Phase state: phase 2 needs a phase 1 on the same scene with the same shard and n_shards, and no render (of any kind),
 *     rtc_set_* / rtc_map_* or commit in between; otherwise it is RTC_ERR_STATE.  Phase 2 may be repeated (into a second
 *     destination, say).  A failed phase 2 changes nothing.
 *   - The own-row check: phase 2 compares the shard's own entries of row_bytes with the lengths its phase 1 computed (kept
 *     with the scene); a mismatch is a broken exchange and RTC_ERR_INVALID, naming the first such row.  A wrong entry for
 *     another shard's row cannot be detected here: that is the callers' exchange.
 *   - Pinned and pageable destinations both work, as in rtc_render_ppm: a pageable one of 4 MiB or more (the whole text's
 *     length) receives the shard's bands through the device's pinned staging frame, piece by piece.
 *   - Device memory kept with the device for later calls: rtc_render_ppm's buffers (the text of its rows, 16 bytes per row). */
int rtc_render_shard_ppm_rows(RtcScene*, int32_t depth, int32_t shard, int32_t n_shards, uint64_t* row_bytes, RtcStats* stats);
int rtc_write_shard_ppm(RtcScene*, int32_t shard, int32_t n_shards, const uint64_t* row_bytes, char* ppm, size_t capacity,
                        size_t* ppm_bytes);
/* rtc_render_samples for one shard of a frame shared by several processes (one process per GPU): rtc_render_shard's split of
 * an anti-aliased frame, as frames or as PPM text.
 *   - Pixels, rtc_render_shard_samples: only the bands b with b % n_shards == shard (rtc_shard_bands) are rendered and written
 *     into the full-size buffers (width * height * 3 each, as rtc_render_samples'); no other row is touched.  The union over
 *     all shards is rtc_render_samples(n)'s planes bit for bit, in f32 and in 8 bits, for every kernel build and option: pixels
 *     are independent and a sample's generated-jitter key is its index in the n W x n H frame, which a shard does not change.
 *     NULL, NULL leaves the shard's bands on the device.
 *   - Text, rtc_render_shard_samples_ppm_rows: phase 1 of rtc_render_shard_ppm_rows' two phases for that anti-aliased shard —
 *     the shard render above with the frame left on the device, then the byte length of every row the shard owns, written
 *     into row_bytes exactly as rtc_render_shard_ppm_rows writes it.  Phase 2 is rtc_write_shard_ppm, unchanged: it encodes
 *     the plane the last phase 1 of either kind left.  The union of the shards' writes is byte for byte
 *     rtc_render_views_samples_ppm's text of the committed camera (Canvas::to_ppm of rtc_render_samples' 8-bit plane).  Phase
 *     state and the own-row check are rtc_write_shard_ppm's: any render (rtc_render_shard and rtc_render_samples included),
 *     rtc_set_* / rtc_map_* or commit in between voids phase 1.
 *   - The arguments are checked before the scene's state, in this order, all with RTC_ERR_INVALID: a NULL scene; (text call)
 *     row_bytes NULL; n_shards < 1 or shard outside [0, n_shards); samples_per_axis outside [1, 16] or a sample canvas
 *     rtc_set_camera would refuse (rtc_render_samples' rule); a depth outside [0, 23].  Then an uncommitted scene is
 *     RTC_ERR_STATE, and so is a scene committed on more than one device (rtc_render_shard's rule).
 *   - The render is rtc_render_samples' one-view path — slices, pinned and pageable destinations (staged through the
 *     device's pinned frames), one persistent streaming launch for a tree scene whose ray trees branch — over the shard's
 *     bands only.  Nothing of rtc_render's state changes.
 *   - stats: primary_rays = n * n * (width - 1) * (the shard's rows below height - 1); launches and kernel_ms as
 *     rtc_render_samples'; for the text call total_ms covers the whole phase.
 *   - Device memory kept with the device for later calls: rtc_render_samples' frame in the view arena, and rtc_render_ppm's
 *     text buffers. */
int rtc_render_shard_samples(RtcScene*, int32_t depth, uint32_t samples_per_axis, int32_t shard, int32_t n_shards,
                             float* rgb_f32, uint8_t* rgb_u8, RtcStats* stats);
int rtc_render_shard_samples_ppm_rows(RtcScene*, int32_t depth, uint32_t samples_per_axis, int32_t shard, int32_t n_shards,
                                      uint64_t* row_bytes, RtcStats* stats);
/* rtc_render_views followed by Canvas::to_ppm of every view, with the text written on the device.
 *   - ppm receives the views' texts one after the other, no terminating NUL: view v's text is ppm[view_offsets[v] ..
 *     view_offsets[v + 1]).  view_offsets has n_views + 1 entries: view_offsets[0] = 0, view_offsets[n_views] the total.
 *   - View v's text is byte for byte what rtc_render_ppm returns for the scene committed with that camera — Canvas::to_ppm
 *     of rtc_render_views' 8-bit plane of that view — for every kernel build and option.
 *   - The arguments are checked before the scene's state, all with RTC_ERR_INVALID: ppm or view_offsets NULL; every check
 *     rtc_render_views makes on n_views and views; a capacity below n_views * rtc_ppm_bound of the committed canvas (a
 *     product that overflows size_t too); a depth outside [0, 23].  Then an uncommitted scene is RTC_ERR_STATE, and a view
 *     beyond the committed reach of a tree scene is refused as rtc_render_views refuses it.
 *   - The render is rtc_render_views' with the frames left on the device: the same chunks through the same arena
 *     (RTC_VIEW_ARENA_BYTES), one render launch per chunk per device (a branching tree scene: one pixel stream per chunk).
 *     A pageable destination of 4 MiB or more also caps a chunk at as many views as fit 256 MiB of text bound.  Then, per
 *     chunk and device: one launch computes the byte length of every row the device owns in every view of the chunk, one
 *     copy of those lengths to the host and a synchronize, the host's scan, one launch writes the text, and the copies into
 *     ppm, queued once every device has its kernels.  Several devices each write only their own bands of every view.
 *   - Pinned and pageable destinations both work.  A pageable one receives a chunk's text of 4 MiB or more through the
 *     pinned staging frame kept with each device, in pieces of about 4 MiB that the host's threads move on as they arrive.
 *   - stats are rtc_render_views' (primary_rays = n_views * (width - 1) * (height - 1), launches = the render launches,
 *     kernel_ms = the render kernels), except total_ms, which covers the whole call.
 *   - Nothing of rtc_render's state changes: the committed camera, its frame on the device and its learnt tile order.
 *   - Device memory kept with each device for later calls, grow-only: rtc_render_ppm's buffers, grown to the text of the
 *     largest chunk and 16 bytes per row of a chunk (its row lengths, on the device and pinned on the host). */
int rtc_render_views_ppm(RtcScene*, int32_t depth, uint32_t n_views, const RtcView* views, char* ppm, size_t capacity,
                         size_t* view_offsets, RtcStats* stats);
/* Anti-aliased batches: rtc_render_samples for every view of an rtc_render_views batch, as frames or as PPM text.
 *   - Pixels: view v's planes (f32 and 8-bit) are bit for bit what rtc_render_samples(n) returns for the scene committed with
 *     view v's camera, for every kernel build and option.  View v's sample camera has the view's half_width, half_height and
 *     transform_inverse, and pixel_size = the view's own when n = 1, else (half_width * 2) / (float)(n W).  A sample's
 *     generated-jitter key is its index in that view's own n W x n H frame; the f32 sum order and the zero last row and column
 *     are rtc_render_samples'.  So n = 1 gives rtc_render_views' planes bit for bit.  rgb_f32 / rgb_u8 are view-major as in
 *     rtc_render_views; NULL, NULL leaves the frames on the device.
 *   - Text: rtc_render_views_samples_ppm lays out its texts and view_offsets as rtc_render_views_ppm does; view v's text is
 *     byte for byte Canvas::to_ppm of view v's 8-bit plane above.
 *   - The arguments are checked before the scene's state, in this order, all with RTC_ERR_INVALID: a NULL scene; every check
 *     rtc_render_views makes on n_views and views; samples_per_axis outside [1, 16]; a sample canvas rtc_set_camera would
 *     refuse (rtc_render_samples' rule); a depth outside [0, 23]; for the text call, ppm or view_offsets NULL, or a capacity
 *     below n_views * rtc_ppm_bound of the committed canvas (a product that overflows size_t too).  Then an uncommitted scene
 *     is RTC_ERR_STATE, and a view beyond the committed reach of a tree scene is refused as rtc_render_views refuses it.
 *   - Chunks, slices, staging, devices and destinations are rtc_render_views' and rtc_render_views_ppm's (RTC_VIEW_ARENA_BYTES,
 *     the 256 MiB cap on a pageable destination's staged text).  A tree scene whose ray trees branch renders each chunk with
 *     one persistent streaming launch, whatever RTC_OPT_WAVEFRONT says.  The samples are reduced on the device: no view's
 *     n W x n H frame is stored.
 *   - stats: primary_rays = n * n * n_views * (width - 1) * (height - 1) over the devices' shares; the other fields are the
 *     views calls' (the text call's total_ms covers the whole call).
 *   - Nothing of rtc_render's state changes: the committed camera, its frame on the device and its learnt tile order. */
int rtc_render_views_samples(RtcScene*, int32_t depth, uint32_t n_views, const RtcView* views, uint32_t samples_per_axis,
                             float* rgb_f32, uint8_t* rgb_u8, RtcStats* stats);
int rtc_render_views_samples_ppm(RtcScene*, int32_t depth, uint32_t n_views, const RtcView* views, uint32_t samples_per_axis,
                                 char* ppm, size_t capacity, size_t* view_offsets, RtcStats* stats);
/* World::color_at (world.rs:88-101) for caller-supplied rays: origins / directions are n*3 f32; out_rgb n*3;
 * out_t (optional) the hit distance or -1; out_prim (optional) the hit primitive index or -1. */
int rtc_trace_rays(RtcScene*, uint32_t n, const float* origins, const float* directions, int32_t depth,
                   float* out_rgb, float* out_t, int32_t* out_prim);

/* Pinned host memory for canvases (page-locked so the device-to-host copy runs at PCIe speed). */
void* rtc_host_alloc(size_t bytes);
void rtc_host_free(void*);
int rtc_host_register(void* ptr, size_t bytes);
int rtc_host_unregister(void* ptr);
/* Evict the L2 between timed iterations (writes a buffer larger than the 126 MB L2). */
int rtc_flush_l2(RtcScene*);
/* Sustained FP32 FMA throughput of device `device` in TFLOP/s (micro-benchmark; the roofline's measured
 * denominator). */
int rtc_measure_fp32_peak(int32_t device, double* tflops, double* sm_clock_mhz);

#ifdef __cplusplus
}
#endif
#endif
