// rtc_internal.h — structures shared by the two host translation units of librtc_b200.so: rtc_api.cu (C ABI, device
// resources, upload, render) and rtc_commit.cu (the host half of a commit: validation, BVH, CSG programs, tables).
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/rtc_b200.h"
#include "rtc_parallel.h"
#include "rtc_types.h"

namespace rtc {

// records the message for rtc_last_error() (thread-local) and returns `code`
int fail(int code, const std::string& msg);

// the first three rows of a row-major 4x4 (an affine inverse transform) as the device keeps them
inline void rows3(const float m[16], float4 out[3]) {
    for (int r = 0; r < 3; r++) out[r] = make_float4(m[r * 4], m[r * 4 + 1], m[r * 4 + 2], m[r * 4 + 3]);
}

struct Box {
    float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    void grow(const Box& o) {
        for (int a = 0; a < 3; a++) lo[a] = std::min(lo[a], o.lo[a]), hi[a] = std::max(hi[a], o.hi[a]);
    }
    float area() const {
        float dx = hi[0] - lo[0], dy = hi[1] - lo[1], dz = hi[2] - lo[2];
        if (dx < 0 || dy < 0 || dz < 0) return 0.f;
        return 2.f * (dx * dy + dy * dz + dz * dx);
    }
    bool finite() const {
        for (int a = 0; a < 3; a++)
            if (!std::isfinite(lo[a]) || !std::isfinite(hi[a]) || lo[a] > hi[a]) return false;
        return true;
    }
};

// Device-side resources that outlive a scene: creating streams / events and allocating the frame and scene
// buffers costs more than rendering a small frame, so they are pooled per device and leased to a scene at
// commit (Camera::render_b200 commits a fresh scene on every call, like the reference's render takes its
// World by value).
struct DeviceSlot {
    int device = -1;
    cudaStream_t stream = nullptr;       // kernels
    cudaStream_t copy_stream = nullptr;  // device-to-host copies, overlapped with the kernels of later slices
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::vector<cudaEvent_t> slice_done;
    // a caller's pageable canvas: the frame lands here (pinned, full frame, grown on demand) slice by slice and the
    // host's threads move each slice on while the device renders the next ones (rtc_api.cu: render_impl)
    char* h_stage_rgb = nullptr;
    char* h_stage_u8 = nullptr;
    size_t h_stage_rgb_bytes = 0, h_stage_u8_bytes = 0;
    std::vector<cudaEvent_t> copy_done;
    DevCounters* h_counters = nullptr;  // pinned: the frame's counters arrive behind its last kernel, no extra round trip
    cudaStream_t slice_stream[2] = {nullptr, nullptr};  // with `stream`: the slices of a frame rotate over three streams
    float* d_rgb = nullptr;
    unsigned char* d_u8 = nullptr;
    size_t frame_px = 0;
    DevCounters* d_counters = nullptr;
    unsigned* d_tile_cost = nullptr;  // clock cycles per frame tile, recorded by the render that learns the order
    int* d_tile_order = nullptr;      // launch order of this shard's tiles
    int tile_capacity = 0;
    int sm_count = 148;
    char* arena = nullptr;  // scene arrays, one allocation
    size_t arena_bytes = 0;
    char* staging = nullptr;  // pinned host mirror of the arena for one asynchronous upload
    size_t staging_bytes = 0;
    char* lbvh_scratch = nullptr;  // the device tree builder's buffers (grow-only, kept with the slot)
    size_t lbvh_scratch_bytes = 0;
    char* lbvh_pinned = nullptr;   // ... and its pinned staging (boxes up, order and nodes down)
    size_t lbvh_pinned_bytes = 0;
    // the wavefront renderer's ray pool (one chunk of a frame at a time) and its per-chunk records
    void* d_wave_rays = nullptr;
    void* d_wave_nodes = nullptr;
    int* d_wave_ints = nullptr;
    int wave_capacity = 0;
    int wave_rays_per_pixel = kWaveRaysPerPixel;  // doubled after a chunk overflowed
    unsigned* d_stream_counter = nullptr;  // render_stream's pixel counters, one per slice of a render
    void* d_flush = nullptr;
    size_t flush_bytes = 0;
    // rtc_render_views: the batch's view table (device, and its pinned staging) and the frames of one chunk of views, apart
    // from d_rgb / d_u8 so that a batch leaves rtc_render's frame alone (all grow-only)
    DevView* d_views = nullptr;
    DevView* h_views = nullptr;
    uint32_t views_capacity = 0;
    char* d_view_frames = nullptr;
    size_t view_frames_bytes = 0;
    // rtc_render_ppm and rtc_render_views_ppm (grow-only): the text of this device's rows (of a frame, or of every view of a
    // chunk), and their byte lengths, then offsets, on the device and pinned on the host.  A pageable destination is staged
    // through h_stage_u8.
    char* d_ppm = nullptr;
    size_t ppm_bytes = 0;
    unsigned long long* d_ppm_rows = nullptr;
    unsigned long long* h_ppm_rows = nullptr;
    size_t ppm_rows = 0;
};

// One committed replica of the scene on one device.
struct Replica {
    DeviceSlot* slot = nullptr;
    DevScene scene{};
    SmallScene small{};
    int cell_masks_eligible = 0, plane_cells_eligible = 0;
    int filter_eligible = 0;  // SmallScene::filter_ok as computed at commit (RTC_OPT_SHADOW_FILTER masks it per render)
    bool csg_sweep = false;   // Flattened::csg_sweep
    // Longest-first launch order learnt from the previous render of the same shard (see render_impl)
    int order_shard = -1, order_n_shards = -1, order_depth = -1, order_filter = -1;  // what d_tile_order was learnt for
    // The learnt order is kept only if it wins a timed trial: after the render that records the costs, one more in
    // natural order and two in the learnt order are timed (stages 1..3) and the minima compared.
    // order_verdict: 0 undecided, 1 the learnt order won and is used, -1 it lost (natural order is kept)
    // A lost trial is repeated (two natural-order and two learnt-order renders again) after 32 more renders of the same
    // shard, at most three times: one noisy sample must not pin a shard to the slower order for the life of the scene
    // (with eight ranks the frame is as slow as the unluckiest one).
    int order_verdict = 0, order_stage = 0;
    int order_retrials = 0, renders_since_loss = 0;
    bool order_lost_here = false;  // this render uses natural order because the trial was lost
    bool order_timed = false;  // this render is one of the timed trial renders
    float natural_ms = 0.f, ordered_ms = 0.f;
    int renders_done = 0;  // the first render of a replica is cold (module load, caches): its time is not compared
    bool learning = false;  // this render records the tile costs
    int wave_chunks = 0;    // chunks the wavefront renderer launched in this render
};

// Everything rtc_scene_commit derives from the scene on the host, ready for upload (rtc_commit.cu: flatten).
struct Flattened {
    RawVector<int4> head;  // 2 * n_pos entries: [pos] main, [n_pos + pos] {cull-chain parent node, api prim, 0, 0}
    RawVector<float4> xform, tri, bound, rec;  // (raw: sized once, every element written by the pass that owns it)
    RawVector<DevBvhNode> bvh;
    std::vector<int> linear;
    std::vector<DevNode> nodes;
    std::vector<DevCsgOp> ops;
    std::vector<DevMaterial> materials;
    std::vector<DevPattern> patterns;
    std::vector<DevUvPattern> uvs;
    std::vector<float4> texels;
    int leaf_size = 0;  // the BVH leaf size used
    int bvh_depth = 0;  // inner-node levels of the tree (<= kBvhStack - 1, enforced by the builder)
    std::vector<float4> samples;
    std::vector<float4> small_image;  // small scenes: what every block stages (rtc_types.h: kSmemOrg float4)
    SmallScene small{};
    int bvh_root = -1;
    int n_pos = 0;
    int all_cast_shadow = 1;
    bool csg_sweep = false;  // some CSG is evaluated by csg_sweep: the scene renders with the *_sweep kernel builds
    int loose_group_boxes = 0;  // group nodes whose cached box does not contain some child's box (RtcCommitInfo)
    float reach = 0.f;  // the largest coordinate the tree's box padding allows for (bounded items, light, camera origin)
};

}  // namespace rtc

struct RtcScene {
    bool have_camera = false, have_light = false, committed = false;
    uint32_t width = 0, height = 0;
    float half_w = 0, half_h = 0, pixel_size = 0;
    float cam_inv[16];
    rtc::RawVector<RtcPrim> prims;  // copied in by all threads (rtc_set_primitives)
    rtc::RawVector<RtcNode> nodes;
    std::vector<int32_t> refs;
    std::vector<RtcMaterial> materials;
    std::vector<RtcPattern> patterns;
    std::vector<RtcUvPattern> uvs;
    struct Texture {
        uint32_t width, height;
        std::vector<float> rgb;
    };
    std::vector<Texture> textures;
    bool light_is_rect = false;
    float light_pos[3], light_rgb[3], corner[3], u_cell[3], v_cell[3];
    int u_steps = 1, v_steps = 1;
    std::vector<float> jitter;
    uint64_t seed = 0;
    int strict_fp = 1, leaf_size = 0 /* automatic */, bvh_min_prims = rtc::kSmallCap + 1;
    int bvh_builder = 0;       // RTC_OPT_BVH_BUILDER: 0 host binned SAH, 1 device LBVH (scenes of >= kLbvhMinItems bounded items)
    int built_on_device = 0;   // the last commit's tree came from the device builder
    int exact_groups = 0;      // RTC_OPT_EXACT_GROUPS: grouped tree primitives and CSG roots carry the cull chain too
    int render_slices = 24;  // kernel / copy pipeline depth when rendering into host memory
    int adaptive_order = 1;  // launch a shard's bands longest-first, learnt from the previous render
    int shadow_filter = 1;   // RTC_OPT_SHADOW_FILTER
    int wavefront = 0;         // RTC_OPT_WAVEFRONT: tree scenes with branching ray trees and a point light go through the
                               // wavefront renderer (dev_wave.cuh) instead of render_stream — measured slower on B200, so opt-in
    int stream = -1;           // tree scenes: lanes draw pixels from a counter (render_stream): -1 automatic (branching ray
                               // trees), 0 / 1 forced (RTC_STREAM)
    int converge = -1;         // color_at warp vote: -1 automatic (branching ray trees), 0 / 1 forced (RTC_CONVERGE)
    bool has_branching_materials = false;  // some material is reflective AND transparent (set at commit)
    int order_max_waves = 128;  // the longest-first order is not even tried for launches longer than this many waves
    std::vector<rtc::Replica> replicas;
    std::vector<int> replica_devices;
    rtc::RawVector<int> pos_to_prim;  // device position -> API primitive index (-1 for CSG pseudo-primitives)
    // commit statistics
    int n_bvh_nodes = 0, n_linear = 0, n_xforms = 0;
    float reach = 0.f;  // Flattened::reach of the commit: rtc_render_views refuses camera origins beyond it in tree scenes
    // rtc_render_shard_ppm_rows / rtc_render_shard_samples_ppm_rows -> rtc_write_shard_ppm: the shard the last phase 1 encoded
    // (n_shards 0: none), the device's 8-bit plane it encoded (the slot's d_u8, or the samples render's in the view arena) and
    // the byte lengths it computed for the shard's rows in frame-row order.  Any render, rtc_set_* / rtc_map_* or commit clears
    // it.  (The slot's h_ppm_rows cannot serve: ppm_layout turns it into offsets in place.)
    struct ShardPpm {
        int shard = -1, n_shards = 0;
        const unsigned char* plane = nullptr;
        std::vector<unsigned long long> rows;
    } shard_ppm;
};

namespace rtc {
// What a render of the scene decides before it picks a kernel (rtc_launch.h: frame_variant), shared with the host harness
// of the kernels (tests/emu/emu_kernels.cpp).  Tree scenes stream pixels (render_stream) when their ray trees branch,
// unless RTC_STREAM forces it; `small` is the replica's small-scene table.
inline bool streams_pixels(const RtcScene* s, const SmallScene& small) {
    return small.n == 0 && (s->stream < 0 ? s->has_branching_materials : s->stream != 0);
}
// DevFrame::converge: the warp vote before every ray when the ray trees branch, unless RTC_CONVERGE forces it
inline int frame_converge(const RtcScene* s) { return s->converge < 0 ? (int)s->has_branching_materials : s->converge; }
// The sample camera C_n of rtc_render_samples, shared with the host harness of the kernels: Camera::new(n W, n H, fov,
// transform) (camera.rs:23-56).  n W / n H is the same real number as W / H, so the aspect and the half-sizes are the
// committed ones; only pixel_size is derived again.  C_1 is the committed camera.  The RtcView overload is the same for one
// view of a batch (rtc_render_views_samples) of a width-pixel canvas.
inline RtcView sample_camera(const RtcView& view, uint32_t width, uint32_t n) {
    RtcView c = view;
    if (n != 1) c.pixel_size = (view.half_width * 2.0f) / (float)(n * width);
    return c;
}
inline RtcView sample_camera(const RtcScene* s, uint32_t n) {
    RtcView v;
    v.half_width = s->half_w, v.half_height = s->half_h, v.pixel_size = s->pixel_size;
    memcpy(v.transform_inverse, s->cam_inv, sizeof(v.transform_inverse));
    return sample_camera(v, s->width, n);
}
// DevFrame::stream_blocks: render_stream's persistent grid, the resident blocks of its launch bounds (RTC_STREAM_MINBLOCKS)
inline int stream_blocks(int sm_count) { return sm_count * 6; }

// The host scan of rtc_render_ppm (one view) and rtc_render_views_ppm (n_views).  In: for each of n_dev devices, the byte
// lengths of the text of its rows, view after view and in its band order within a view (PpmRows); header: the length of a
// view's header.  Out: the same arrays holding each row's offset in that device's text (view-major as well), and where
// every view and every (view, band) goes; the texts of the views follow each other.  With `text`, each view's header
// (header_text, `header` bytes: ppm_header) is written at its offset there; text must hold the whole (a view's text is at
// most rtc_ppm_bound).  Shared with the host harnesses of the PPM kernels (tests/emu/emu_ppm.cpp: one frame, the header
// left to the caller; tests/emu/emu_ppm_views.cpp).
struct PpmLayout {
    int total_bands = 0;               // bands of one frame
    std::vector<size_t> view_at;       // view v: the offset of its text (its header) in the whole text
    std::vector<size_t> band_at;       // band b of view v (index v * total_bands + b): its offset in the whole text
    std::vector<size_t> band_local;    // ... and in its device's text
    std::vector<size_t> band_bytes;
    std::vector<size_t> device_bytes;  // each device's text
    size_t total = 0;                  // the whole text, headers included
};
inline std::string ppm_header(uint32_t width, uint32_t height) {  // canvas.rs:60-64
    return "P3\n" + std::to_string(width) + " " + std::to_string(height) + "\n255\n";
}
inline int ppm_device_rows(uint32_t height, int device, int n_dev) {
    const int total_bands = ((int)height + kBandRows - 1) / kBandRows;
    int rows = 0;
    for (int b = device; b < total_bands; b += n_dev) rows += std::min<int>(kBandRows, (int)height - b * kBandRows);
    return rows;
}
inline void ppm_layout(uint32_t height, int n_dev, size_t header, unsigned long long* const* rows, PpmLayout& L, int n_views = 1,
                       const char* header_text = nullptr, char* text = nullptr) {
    const int total_bands = ((int)height + kBandRows - 1) / kBandRows;
    std::vector<size_t> dev_rows(n_dev);
    for (int i = 0; i < n_dev; i++) dev_rows[i] = (size_t)ppm_device_rows(height, i, n_dev);
    L.total_bands = total_bands;
    L.view_at.assign(n_views, 0);
    L.band_at.assign((size_t)n_views * total_bands, 0), L.band_local.assign((size_t)n_views * total_bands, 0);
    L.band_bytes.assign((size_t)n_views * total_bands, 0);
    L.device_bytes.assign(n_dev, 0);
    size_t at = 0;
    for (int v = 0; v < n_views; v++) {
        L.view_at[v] = at;
        if (text) memcpy(text + at, header_text, header);
        at += header;
        for (int b = 0; b < total_bands; b++) {
            const int dev = b % n_dev;
            const size_t j0 = (size_t)v * dev_rows[dev] + (size_t)(b / n_dev * kBandRows), vb = (size_t)v * total_bands + b;
            const int n_rows = std::min<int>(kBandRows, (int)height - b * kBandRows);
            size_t& local = L.device_bytes[dev];
            L.band_at[vb] = at, L.band_local[vb] = local;
            for (int k = 0; k < n_rows; k++) {
                const size_t len = rows[dev][j0 + k];
                rows[dev][j0 + k] = local;
                local += len, at += len;
            }
            L.band_bytes[vb] = at - L.band_at[vb];
        }
    }
    L.total = at;
}
// rtc_write_shard_ppm's scan: ppm_layout of one frame cut into n_shards shards, from the byte lengths of all its rows in
// frame-row order (row_bytes, every shard's rtc_render_shard_ppm_rows put together by the callers).  shard_rows[i] receives
// shard i's rows in its band order — its frame rows in increasing order — and, after the scan, their offsets in shard i's
// text.  Every process lays out the whole frame on its own; only shard 0 passes header_text and text, so the header is
// written once.  Shared with the host harness (tests/emu/emu_ppm.cpp: emu_ppm_shards).
inline void ppm_layout_frame_rows(uint32_t height, int n_shards, size_t header, const uint64_t* row_bytes,
                                  std::vector<std::vector<unsigned long long>>& shard_rows, PpmLayout& L,
                                  const char* header_text = nullptr, char* text = nullptr) {
    shard_rows.assign(n_shards, {});
    for (int i = 0; i < n_shards; i++) shard_rows[i].reserve(ppm_device_rows(height, i, n_shards));
    for (uint32_t y = 0; y < height; y++) shard_rows[y / kBandRows % n_shards].push_back(row_bytes[y]);
    std::vector<unsigned long long*> rows(n_shards);
    for (int i = 0; i < n_shards; i++) rows[i] = shard_rows[i].data();
    ppm_layout(height, n_shards, header, rows.data(), L, 1, header_text, text);
}

// A tree builder other than the host's binned SAH (rtc_lbvh.cu: the device LBVH).  In: the padded boxes of the bounded
// items (6 floats each: lo.xyz, hi.xyz), their "closed primitive" flags, the leaf size.  Out: the items' leaf order, the
// binary nodes, the root link (>= 0 node, < 0 a leaf code: the whole tree is one leaf) and the tree's depth.  A non-zero
// return means "not built": flatten() then uses the host builder.
struct TreeBuildInput {
    const float* boxes;
    const unsigned char* closed;
    int n, leaf_size;
};
struct TreeBuildOutput {
    RawVector<int> order;
    RawVector<DevBvhNode> nodes;
    int root = -1, depth = 0;
};
using TreeBuilderFn = int (*)(void* ctx, const TreeBuildInput&, TreeBuildOutput&);
struct LbvhContext {  // lbvh_build's ctx: the stream to build on and the slot's grow-only scratch buffers
    cudaStream_t stream;
    char** scratch;
    size_t* scratch_bytes;
    char** pinned;
    size_t* pinned_bytes;
};
int lbvh_build(void* ctx, const TreeBuildInput& in, TreeBuildOutput& out);

// The host half of a commit: fills `f` from the scene (and the scene's commit statistics).  No device calls of its own:
// rtc_scene_inspect runs it without a GPU; rtc_scene_commit may pass the device tree builder.
int flatten(RtcScene* s, Flattened& f, TreeBuilderFn tree_builder = nullptr, void* tree_builder_ctx = nullptr);
}  // namespace rtc
