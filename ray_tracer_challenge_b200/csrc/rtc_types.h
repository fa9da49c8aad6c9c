// rtc_types.h — device-resident scene layout shared by the host (rtc_api.cu) and the kernels.
//
// Everything a ray touches lives in a handful of flat arrays in HBM (L2-resident for every BASELINE config:
// 100 k primitives ~ 8 MB):
//   head[i]   int4   {type | flags<<4 | material<<8, xform id, aux, dfs order}         16 B / primitive
//   xform[k]  3xfloat4 rows of the primitive's inverse transform (deduplicated)        48 B / transform
//   tri[a]    3xfloat4 {p1.xyz e1.x | e1.yz e2.xy | e2.z n.xyz}                        48 B / triangle
//   bound[a]  float4 {minimum_y, maximum_y, closed, 0}                                 16 B / cylinder, cone
//   bvh[n]    4xfloat4 two child boxes + two child links                               64 B / node
// Primitives are stored in BVH leaf order; `dfs order` keeps the reference's depth-first emission order,
// which is the tie-break between equal hit distances (world.rs:58, intersection.rs:30-35).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#include <cuda_runtime.h>
#else
#include <vector_types.h>
#endif

#if defined(__CUDACC__)
#define RTC_HD __host__ __device__
#else
#define RTC_HD
#endif

namespace rtc {

enum : int { T_SPHERE = 0, T_PLANE = 1, T_CUBE = 2, T_CYLINDER = 3, T_CONE = 4, T_TRIANGLE = 5, T_CSG = 6 };

constexpr int kFlagCastsShadow = 1;   // BaseShape::casts_shadow
constexpr int kFlagHasParent = 2;     // has an enclosing group / CSG whose cull must be honoured exactly
constexpr int kMaxFrames = 24;        // explicit reflect/refract stack: depth + 1 frames (depth <= 23)
// A CSG whose worst case stays within kCsgHitCap leaf hits and kCsgRayDepth - 1 nesting levels is evaluated whole by
// csg_eval (dev_bvh.cuh); any other is marked at commit and evaluated by csg_sweep, whose memory does not depend on the
// hit count: it holds kCsgHitCap hits at a time and needs nesting <= kCsgSweepDepth - 1 and <= kCsgSweepNodes CSG nodes.
constexpr int kCsgHitCap = 32;        // csg_eval: leaf hits held at once; csg_sweep: hits per pass, open solids per CSG
constexpr int kCsgRayDepth = 6;       // csg_eval: nested CSG transforms
constexpr int kCsgSweepDepth = 64;    // csg_sweep: nested CSG transforms
constexpr int kCsgSweepNodes = 1024;  // csg_sweep: CSG nodes of one outermost CSG (2 state bits each)
constexpr int kBvhStack = 48;  // traversal stack entries per thread: one deferred child per level (the builder bounds the depth)

struct DevMaterial {  // 48 B
    float color[3];
    float ambient, diffuse, specular, shininess, reflective, transparency, refractive_index;
    int pattern;
    int pad;
};

struct DevPattern {  // 112 B
    float4 inv[3];
    float a[3];
    float b[3];
    int kind, mapping;
    int uv[6];
};

struct DevUvPattern {  // 64 B
    int kind;
    float p[15];
};

struct DevNode {  // group / CSG node of the reference shape tree (cull chain + CSG evaluation)
    float4 inv[3];
    float bmin[3];
    float bmax[3];
    int kind, parent, op, pad;
};

// One instruction of a flattened CSG tree (post-order), see csg_eval and csg_sweep in dev_bvh.cuh.
enum : int { OP_CSG_ENTER = 0, OP_CSG_MID = 1, OP_CSG_EXIT = 2, OP_GROUP = 3, OP_PRIM = 4 };
struct DevCsgOp {
    int op;    // OP_*
    int arg;   // node index (ENTER/MID/EXIT/GROUP) or primitive position (PRIM)
    int skip;  // ENTER/GROUP: instruction to jump to when the bounding-box cull rejects the ray
    int pad;   // 0, except in a program evaluated by csg_sweep (offsets are from the root ENTER):
               //   root ENTER  -(number of CSG nodes in the program): < 0 marks the program for csg_sweep
               //   ENTER       offset of the parent CSG's ENTER
               //   EXIT        state index << 1 | 1 when the CSG is in its parent's left operand (s1)
               //   PRIM        offset of the innermost enclosing CSG's ENTER << 1 | 1 when in its left operand
};

struct DevBvhNode {  // 64 B
    float4 a;  // lo0.xyz, hi0.x
    float4 b;  // hi0.yz, lo1.xy
    float4 c;  // lo1.z, hi1.xyz
    int4 d;    // child0, child1 (>= 0 inner node; < 0 leaf: ~((first << 4) | (count - 1))); z: bit i = child i holds closed
               // primitives only (find_containers culls it with a point-in-box test); w unused
};

struct DevScene {
    // camera (camera.rs:8-20)
    float4 cam_inv[3];
    float half_w, half_h, pixel_size;
    int width, height;
    // light
    int light_is_rect;
    float light_pos[3];  // PointLight::position or the rectangle centre
    float light_rgb[3];
    float corner[3], u_vec[3], v_vec[3];  // per-cell edges
    int u_steps, v_steps, cells;
    int jitter_len;            // > 0: table mode
    const float* jitter;       // table
    const float4* samples;     // table mode: the `cells` precomputed point_on_light positions
    const float4* small_image; // small scenes: the first kSmemOrg float4 of a block's shared memory, ready to copy
    unsigned long long seed;   // counter mode
    // geometry
    const int4* head;
    const float4* rec;    // traversal records, 64 B / primitive: {head, 3 x float4}: the inverse-transform rows, or for a
                          // triangle its p1 / e1 / e2 / normal (its transform is shared: head.y indexes `xform`)
    const float4* xform;
    const float4* tri;
    const float4* bound;
    const DevBvhNode* bvh;
    const int* linear;  // primitive positions tested for every ray (unbounded shapes, or every shape of a tiny scene)
    int n_linear;
    int bvh_root;       // -1: no BVH
    int n_prims;
    const DevNode* nodes;
    const DevCsgOp* csg_ops;
    // shading
    const DevMaterial* materials;
    const DevPattern* patterns;
    const DevUvPattern* uvs;
    const float4* texels;  // image textures, one float4 {r, g, b, 0} per pixel, all canvases back to back
    int all_cast_shadow;  // every primitive casts a shadow: shadow rays may stop at the first hit
    unsigned long long* csg_overflows;  // DevCounters::overflows of the render: csg_sweep flags an overflow here in every build
};

// Small scenes (every BASELINE demo scene: 4..13 primitives) skip the tree: their primitives travel in the
// kernel's parameter block (constant bank), so the per-ray loop over them is warp-uniform — matrix rows come
// through the uniform datapath, no global loads, no address arithmetic, no divergence on the type switch.
constexpr int kSmallCap = 16;   // primitives (or CSG roots) held in the parameter block
constexpr int kOrgCache = 8;    // object-space shadow-ray origins cached per thread in shared memory
constexpr int kSmallStride = 6;  // float4 per table entry
struct SmallPrim {              // 96 B
    int4 head;                  // type | flags << 4 | material << 8, cull-chain parent node, aux, dfs order
    float4 r0, r1, r2;          // rows of the inverse transform
    float4 bound;               // cylinder / cone: minimum_y, maximum_y, closed; .w = the ball's padding rate (below)
    float4 ball;                // world-space bounding ball {centre, radius * 1.001} (NaN: unbounded, never rejects);
                                // tested with radius + bound.w * |centre - origin|^2 (bound.w = 2^-17 cond^2 / radius)
};
// The table is sorted by (casts shadow first, then kind) so every loop over it is a run of ONE kind:
//   casters:     spheres [0, c.x) planes [c.x, c.y) cubes [c.y, c.z) everything else [c.z, c.w)
//   non-casters: spheres [c.w, o.x) planes [o.x, o.y) cubes [o.y, o.z) everything else [o.z, o.w = n)
// (hit ties are broken by the stored depth-first order, so the storage order is free).
struct SmallScene {
    int n;                      // 0: the scene does not qualify, use the general path
    int two_pass_shadows;       // no CSG roots among them: shadow rays may test casters first (see is_shadowed)
    int has_cull_chain;         // some unbounded primitive sits inside a group whose cull must be honoured (Q6)
    int filter_ok;              // spheres / planes / axis-aligned cubes only: shadow rays go through the filter first
    float tol_sphere;           // the filter's relative error bound for spheres (grows with the transforms' condition)
    int cell_masks;             // filter_ok, table-mode area light with <= kSampleCap cells: intensity_cells path
    int plane_cells;            // cell_masks and (caster planes x cells) <= kPlaneCellCap: per-(plane, cell) constants staged
    int lean;                   // cell_masks, and no material of the table has a pattern or transparency: the lean kernel build
    float4 light_ball;          // cell_masks: ball around the light samples (centre, radius) for the bundle reject
    float4 plane_bundle[2];     // cell_masks, first two caster planes: over all light cells (table) or the whole light
                                // rectangle (generated jitter) {min r1.L, max r1.L,
                                // max tol*|r1||L|, max eps'*|L|_1} (bounds of plane_cell_constants, padded)
    int4 caster_end, other_end;
    SmallPrim p[kSmallCap];
};
constexpr int kSampleCap = 128;     // table-mode light samples staged in shared memory
constexpr int kPlaneCellCap = 256;  // (caster plane, light cell) constants staged in shared memory
// A block renders one tile of kTileW x kTileH pixels, one thread per pixel, as 8x4-pixel warps (kTileW / 8 across).
#ifndef RTC_TILE_W
#define RTC_TILE_W 16
#endif
// Shadow filter, plane test with the light sample folded in (SmallScene::plane_cells, dev_shadow.cuh:
// filter_plane_cell): for light point L and shading point p the object-space direction's y is r1.L - r1.p, so everything
// that depends on L alone is computed once per scene, in f32, by the commit: {r1.L, tol * sum|r1_k L_k|, EPSILON' * |L|_1}.
constexpr float kTolP = 3.814697265625e-06f;  // 2^-18 = 64 ulp: planes and cubes (bounds are term-wise, no conditioning)
RTC_HD inline float4 plane_cell_constants(float4 r1, float4 L) {
    const float px = r1.x * L.x, py = r1.y * L.y, pz = r1.z * L.z;
    const float ax = px < 0.f ? -px : px, ay = py < 0.f ? -py : py, az = pz < 0.f ? -pz : pz;
    const float lx = L.x < 0.f ? -L.x : L.x, ly = L.y < 0.f ? -L.y : L.y, lz = L.z < 0.f ? -L.z : L.z;
    float4 q;
    q.x = px + py + pz;
    q.y = kTolP * (ax + ay + az);
    q.z = (1.1920929e-3f * (1.0f + 2.0f * kTolP)) * (lx + ly + lz);
    q.w = 0.0f;
    return q;
}

constexpr int kTileW = RTC_TILE_W, kTileH = 8;
constexpr int kBlockThreads = kTileW * kTileH;
constexpr int kWarpsX = kTileW / 8;
static_assert(kTileW % 8 == 0 && kBlockThreads <= 1024, "tile width: whole 8x4-pixel warps");
// Dynamic shared memory of the small-scene kernels, in float4 units: [table | light samples | (plane, cell) constants |
// per-thread shadow-origin cache].  Everything before the cache is the same for every block of a scene: the commit lays
// it out once (Flattened::small_image -> DevScene::small_image) and a block's staging is a plain coalesced copy.
constexpr int kSmemSamples = kSmallCap * kSmallStride;
constexpr int kSmemPlaneCells = kSmemSamples + kSampleCap;
constexpr int kSmemOrg = kSmemPlaneCells + kPlaneCellCap;
constexpr int kSmallSmemBytes = kSmemOrg * 16 + kOrgCache * 3 * kBlockThreads * 4;

struct DevFrame {  // where a render writes
    float* rgb;            // width*height*3 f32 or null
    unsigned char* u8;     // width*height*3 or null
    int shard, n_shards;   // interleaved bands of kBandRows rows
    int depth;
    int n_bands;           // bands this launch renders ...
    int band_begin;        // ... starting at this index of the shard's band list
    const int* tile_order; // this shard's tiles (band * tiles_x + tile column) in launch order, or null: natural order
    unsigned* tile_cost;   // per frame tile: clock cycles its block ran (learns the launch order), or null
    int converge;          // color_at: all lanes of a warp meet at a vote before every ray (see color_at)
    unsigned* stream_counter;  // render_stream: next unclaimed pixel of the launch (zeroed by the host), or null
    int stream_blocks;         // render_stream: resident blocks to launch (a persistent grid)
};
// One camera of a batch of views (rtc_render_views): Camera::new's derived fields (camera.rs:23-56), read by
// ray_for_pixel in place of DevScene's.  The batch's table lives in device memory, one entry per view of the call.
struct DevView {  // 64 B
    float4 cam_inv[3];
    float half_w, half_h, pixel_size, pad;
};
static_assert(sizeof(DevView) == 64, "DevView: 64 B per view");

#ifndef RTC_REFILL_LANES
#define RTC_REFILL_LANES 8
#endif
constexpr int kRefillLanes = RTC_REFILL_LANES;  // render_stream: idle lanes of a warp that trigger a refill

constexpr int kBandRows = kTileH;

// The wavefront renderer's per-chunk ray pool as the host hands it to the launchers (dev_wave.cuh: WavePool holds the
// same pointers, typed).
struct WavePoolRaw {
    void* rays;    // capacity x 96 B
    void* nodes;   // capacity x 64 B
    int capacity;
    int* ints;     // base[L], count[L], cursor[2 L] for L <= kMaxFrames: see rtc_kernels.cu: wave_pool
    unsigned long long* record;  // this chunk's {rays that did not fit the pool, secondary rays, shades}
};
constexpr int kWaveLevels = kMaxFrames + 1;
constexpr int kWaveInts = 4 * kWaveLevels;
constexpr int kWaveMaxChunks = 64;         // chunk records per render
constexpr int kWaveRaysPerPixel = 6;       // pool capacity per pixel of a chunk (a chunk that needs more is re-rendered by render_stream)

struct DevCounters {  // accumulated with one atomic per warp
    unsigned long long primary, secondary, shadow, shades;
    unsigned long long node_visits, prim_tests[8], xforms, patterns, cells, schlicks, refr_dirs, overflows;
};

}  // namespace rtc
