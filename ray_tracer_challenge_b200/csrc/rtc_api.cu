// rtc_api.cu — the C ABI of include/rtc_b200.h: scene intake, commit (validation, transform
// de-duplication, binned-SAH BVH over the book's bounding boxes, CSG flattening, upload of one replica per
// device) and the render entry points that drive the kernels of rtc_kernels.cu.
//
// There is no CPU rendering path in this library: every pixel comes from the sm_100a kernels, and every
// entry point that needs a device fails with RTC_ERR_NO_DEVICE when there is none.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <future>
#include <map>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <string>
#include <tuple>
#include <vector>

#include <cuda_runtime.h>

#include "rtc_internal.h"
#include "rtc_launch.h"

using namespace rtc;

namespace {

thread_local std::string g_error;
}  // namespace
namespace rtc {
int fail(int code, const std::string& msg) {
    g_error = msg;
    return code;
}
}  // namespace rtc
namespace {
// no usable device -> RTC_ERR_NO_DEVICE (the "no CPU fallback" contract); anything else a visible device reports
// (out of memory, launch failure, bad argument) -> RTC_ERR_CUDA
int cuda_status(cudaError_t e) {
    switch (e) {
        case cudaErrorNoDevice:
        case cudaErrorInsufficientDriver:
        case cudaErrorInvalidDevice:
        case cudaErrorDevicesUnavailable:
        case cudaErrorInitializationError:
        case cudaErrorSystemNotReady:
        case cudaErrorSystemDriverMismatch:
        case cudaErrorCompatNotSupportedOnDevice:
        case cudaErrorStubLibrary:
        case cudaErrorNoKernelImageForDevice:  // not an sm_100a part: this library has kernels for nothing else
            return RTC_ERR_NO_DEVICE;
        default: return RTC_ERR_CUDA;
    }
}
#define CUDA_TRY(expr)                                                                                          \
    do {                                                                                                        \
        cudaError_t _e = (expr);                                                                                \
        if (_e != cudaSuccess)                                                                                  \
            return fail(cuda_status(_e), std::string(#expr) + ": " + cudaGetErrorString(_e));                    \
    } while (0)



std::mutex g_pool_mutex;
std::vector<DeviceSlot*> g_pool;  // idle slots

int lease_slot(int device, DeviceSlot** out) {
    {
        std::lock_guard<std::mutex> lock(g_pool_mutex);
        for (size_t i = 0; i < g_pool.size(); i++)
            if (g_pool[i]->device == device) {
                *out = g_pool[i];
                g_pool.erase(g_pool.begin() + i);
                return 0;
            }
    }
    CUDA_TRY(cudaSetDevice(device));
    DeviceSlot* d = new DeviceSlot();
    d->device = device;
    CUDA_TRY(cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&d->copy_stream, cudaStreamNonBlocking));
    for (cudaStream_t& st : d->slice_stream) CUDA_TRY(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreate(&d->ev0));
    CUDA_TRY(cudaEventCreate(&d->ev1));
    CUDA_TRY(cudaMalloc(&d->d_counters, sizeof(DevCounters)));
    CUDA_TRY(cudaHostAlloc(&d->h_counters, sizeof(DevCounters), cudaHostAllocDefault));
    CUDA_TRY(cudaMalloc(&d->d_stream_counter, 64 * sizeof(unsigned)));  // RTC_OPT_RENDER_SLICES <= 64
    CUDA_TRY(cudaDeviceGetAttribute(&d->sm_count, cudaDevAttrMultiProcessorCount, device));
    // the kernels keep their bounce and traversal stacks in local memory
    size_t have = 0;
    cudaDeviceGetLimit(&have, cudaLimitStackSize);
    if (have < 8192) CUDA_TRY(cudaDeviceSetLimit(cudaLimitStackSize, 8192));
    *out = d;
    return 0;
}
void return_slot(DeviceSlot* d) {
    if (!d) return;
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    g_pool.push_back(d);
}
int ensure_frame(DeviceSlot* d, size_t px) {
    if (px <= d->frame_px) return 0;
    CUDA_TRY(cudaSetDevice(d->device));
    if (d->d_rgb) cudaFree(d->d_rgb);
    if (d->d_u8) cudaFree(d->d_u8);
    d->d_rgb = nullptr, d->d_u8 = nullptr, d->frame_px = 0;
    CUDA_TRY(cudaMalloc(&d->d_rgb, std::max<size_t>(px * 3 * sizeof(float), 16)));
    CUDA_TRY(cudaMalloc(&d->d_u8, std::max<size_t>(px * 3, 16)));
    d->frame_px = px;
    return 0;
}
int ensure_tiles(DeviceSlot* d, int total_tiles) {
    if (total_tiles <= d->tile_capacity) return 0;
    CUDA_TRY(cudaSetDevice(d->device));
    if (d->d_tile_cost) cudaFree(d->d_tile_cost);
    if (d->d_tile_order) cudaFree(d->d_tile_order);
    d->tile_capacity = 0;
    CUDA_TRY(cudaMalloc(&d->d_tile_cost, (size_t)total_tiles * sizeof(unsigned)));
    CUDA_TRY(cudaMalloc(&d->d_tile_order, (size_t)total_tiles * sizeof(int)));
    d->tile_capacity = total_tiles;
    return 0;
}
int ensure_arena(DeviceSlot* d, size_t bytes) {
    CUDA_TRY(cudaSetDevice(d->device));
    if (bytes > d->arena_bytes) {
        if (d->arena) cudaFree(d->arena);
        d->arena = nullptr, d->arena_bytes = 0;
        size_t cap = std::max<size_t>(bytes + bytes / 4, 1 << 16);
        CUDA_TRY(cudaMalloc(&d->arena, cap));
        d->arena_bytes = cap;
    }
    if (bytes > d->staging_bytes) {
        if (d->staging) cudaFreeHost(d->staging);
        d->staging = nullptr, d->staging_bytes = 0;
        size_t cap = std::max<size_t>(bytes + bytes / 4, 1 << 16);
        CUDA_TRY(cudaHostAlloc(&d->staging, cap, cudaHostAllocDefault));
        d->staging_bytes = cap;
    }
    return 0;
}


}  // namespace


namespace {

void release(RtcScene* s) {
    for (Replica& r : s->replicas) {
        if (!r.slot) continue;
        cudaSetDevice(r.slot->device);
        cudaStreamSynchronize(r.slot->stream);
        cudaStreamSynchronize(r.slot->copy_stream);
        return_slot(r.slot);
        r.slot = nullptr;
    }
    s->replicas.clear();
    s->committed = false;
}

// Packs the scene arrays into one staging buffer (256-byte aligned sections) for a single upload.
struct ArenaWriter {
    size_t bytes = 0;
    struct Part {
        const void* src;
        size_t n, off;
    };
    std::vector<Part> parts;
    template <class T, class A>
    size_t add(const std::vector<T, A>& v) {
        size_t off = bytes;
        if (!v.empty()) {
            parts.push_back({v.data(), v.size() * sizeof(T), off});
            bytes = (bytes + v.size() * sizeof(T) + 255) & ~size_t(255);
        }
        return off;
    }
};

// The kernel build a scene renders with: IEEE (strict) or FMA-contracted (fast), with csg_sweep's call sites when the scene
// holds a CSG beyond csg_eval's limits (rtc_kernels.cu).
struct KernelBuild {
    decltype(&fast::launch_render) render;
    decltype(&fast::launch_trace) trace;
    decltype(&fast::launch_wave) wave;
    decltype(&fast::launch_views) views;
};
const KernelBuild& kernel_build(bool strict_fp, bool csg_sweep) {
    static const KernelBuild builds[4] = {{fast::launch_render, fast::launch_trace, fast::launch_wave, fast::launch_views},
                                          {strict::launch_render, strict::launch_trace, strict::launch_wave, strict::launch_views},
                                          {fast_sweep::launch_render, fast_sweep::launch_trace, fast_sweep::launch_wave, fast_sweep::launch_views},
                                          {strict_sweep::launch_render, strict_sweep::launch_trace, strict_sweep::launch_wave,
                                           strict_sweep::launch_views}};
    return builds[(strict_fp ? 1 : 0) + (csg_sweep ? 2 : 0)];
}

int upload_replica(RtcScene* s, const Flattened& f, Replica& r, int device) {
    int rc;
    if ((rc = lease_slot(device, &r.slot))) return rc;
    DeviceSlot* slot = r.slot;
    CUDA_TRY(cudaSetDevice(device));
    DevScene& d = r.scene;
    memset(&d, 0, sizeof(d));
    rows3(s->cam_inv, d.cam_inv);
    d.half_w = s->half_w, d.half_h = s->half_h, d.pixel_size = s->pixel_size;
    d.width = (int)s->width, d.height = (int)s->height;
    d.light_is_rect = s->light_is_rect;
    memcpy(d.light_pos, s->light_pos, 12);
    memcpy(d.light_rgb, s->light_rgb, 12);
    memcpy(d.corner, s->corner, 12);
    memcpy(d.u_vec, s->u_cell, 12);
    memcpy(d.v_vec, s->v_cell, 12);
    d.u_steps = s->u_steps, d.v_steps = s->v_steps, d.cells = s->u_steps * s->v_steps;
    d.jitter_len = (int)s->jitter.size();
    d.seed = s->seed;
    ArenaWriter w;
    size_t o_jitter = w.add(s->jitter), o_samples = w.add(f.samples), o_head = w.add(f.head), o_rec = w.add(f.rec);
    size_t o_xform = w.add(f.xform), o_tri = w.add(f.tri), o_bound = w.add(f.bound), o_bvh = w.add(f.bvh);
    size_t o_linear = w.add(f.linear), o_nodes = w.add(f.nodes), o_ops = w.add(f.ops), o_mat = w.add(f.materials);
    size_t o_pat = w.add(f.patterns), o_uv = w.add(f.uvs), o_tex = w.add(f.texels), o_img = w.add(f.small_image);
    if ((rc = ensure_arena(slot, std::max<size_t>(w.bytes, 256)))) return rc;
    const bool timing = getenv("RTC_TIMING") != nullptr;  // tuning aid (adds a synchronize)
    auto t0 = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (!timing) return;
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[rtc upload] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - t0).count());
        t0 = now;
    };
    for (const auto& p : w.parts) parallel_stream_copy(slot->staging + p.off, p.src, p.n);
    lap("arrays -> pinned staging");
    if (w.bytes) CUDA_TRY(cudaMemcpyAsync(slot->arena, slot->staging, w.bytes, cudaMemcpyHostToDevice, slot->stream));
    if (timing) {
        CUDA_TRY(cudaStreamSynchronize(slot->stream));
        fprintf(stderr, "[rtc upload] %zu bytes\n", w.bytes);
        lap("staging -> device");
    }
    auto at = [&](size_t off, bool present) -> const void* { return present ? slot->arena + off : nullptr; };
    d.jitter = (const float*)at(o_jitter, !s->jitter.empty());
    d.samples = (const float4*)at(o_samples, !f.samples.empty());
    d.head = (const int4*)at(o_head, !f.head.empty());
    d.rec = (const float4*)at(o_rec, !f.rec.empty());
    d.xform = (const float4*)at(o_xform, !f.xform.empty());
    d.tri = (const float4*)at(o_tri, !f.tri.empty());
    d.bound = (const float4*)at(o_bound, !f.bound.empty());
    d.bvh = (const DevBvhNode*)at(o_bvh, !f.bvh.empty());
    d.linear = (const int*)at(o_linear, !f.linear.empty());
    d.nodes = (const DevNode*)at(o_nodes, !f.nodes.empty());
    d.csg_ops = (const DevCsgOp*)at(o_ops, !f.ops.empty());
    d.materials = (const DevMaterial*)at(o_mat, !f.materials.empty());
    d.patterns = (const DevPattern*)at(o_pat, !f.patterns.empty());
    d.uvs = (const DevUvPattern*)at(o_uv, !f.uvs.empty());
    d.texels = (const float4*)at(o_tex, !f.texels.empty());
    d.small_image = (const float4*)at(o_img, !f.small_image.empty());
    d.n_linear = (int)f.linear.size();
    d.bvh_root = f.bvh_root;
    d.n_prims = f.n_pos;
    d.all_cast_shadow = f.all_cast_shadow;
    d.csg_overflows = &slot->d_counters->overflows;  // reset with the counters before every render / trace
    r.csg_sweep = f.csg_sweep;
    r.small = f.small;
    r.filter_eligible = f.small.filter_ok;
    r.cell_masks_eligible = f.small.cell_masks;
    r.plane_cells_eligible = f.small.plane_cells;
    if ((rc = ensure_frame(slot, (size_t)s->width * s->height))) return rc;
    return 0;
}

double flops_of(const RtcStats& st, uint64_t pixels) {  // SURVEY.md Appendix E
    const double pf[8] = {30, 2, 29, 45, 50, 46, 0, 0};
    double f = 33.0 * st.xforms + 26.0 * st.node_visits;
    for (int i = 0; i < 8; i++) f += pf[i] * st.prim_tests[i];
    f += 36.0 * st.primary_rays + (85.0 + 75.0 + 9.0) * st.shades + 41.0 * st.patterns;
    f += 13.0 * st.shadow_rays + 14.0 * st.cells + 20.0 * st.schlicks + 25.0 * st.refr_dirs + 3.0 * pixels;
    return f;
}

// The device accumulates the secondary rays and the shades; `primary` is what the host knows the launch rendered, and
// every shade_hit casts one shadow ray per light cell (point light: one) — rectangle_light.rs:76-88, point_light.rs:28-34.
void add_counters(RtcStats& st, const DevCounters& c, uint64_t primary, uint64_t shadow_per_shade) {
    st.primary_rays += primary, st.secondary_rays += c.secondary, st.shadow_rays += c.shades * shadow_per_shade, st.shades += c.shades;
    st.node_visits += c.node_visits;
    for (int i = 0; i < 8; i++) st.prim_tests[i] += c.prim_tests[i];
    st.xforms += c.xforms, st.patterns += c.patterns, st.cells += c.cells, st.schlicks += c.schlicks;
    st.refr_dirs += c.refr_dirs, st.capacity_overflows += c.overflows;
}

// Copy the rows of bands [b0, b1) of this shard's band list from the device frame into the caller's full-size
// canvas (band j of the list is frame band `shard + j * n_shards`).
int copy_bands(DeviceSlot* slot, const RtcScene* s, int shard, int n_shards, int b0, int b1, const void* src, void* dst,
               size_t px_bytes) {
    const size_t row = (size_t)s->width * px_bytes;
    const size_t band = row * kBandRows;
    if (b1 <= b0) return 0;
    const int first_band = shard + b0 * n_shards, last_band = shard + (b1 - 1) * n_shards;
    const int last_rows = std::min<int>(kBandRows, (int)s->height - last_band * kBandRows);
    if (n_shards == 1) {  // contiguous rows
        size_t off = (size_t)first_band * band;
        size_t bytes = (size_t)(b1 - b0 - 1) * band + row * last_rows;
        CUDA_TRY(cudaMemcpyAsync((char*)dst + off, (const char*)src + off, bytes, cudaMemcpyDeviceToHost, slot->copy_stream));
        return 0;
    }
    const int full = (last_rows == kBandRows) ? (b1 - b0) : (b1 - b0 - 1);  // every band but possibly the last is full
    size_t off = (size_t)first_band * band;
    if (full > 0)
        CUDA_TRY(cudaMemcpy2DAsync((char*)dst + off, band * n_shards, (const char*)src + off, band * n_shards, band, full,
                                   cudaMemcpyDeviceToHost, slot->copy_stream));
    if (full < b1 - b0) {
        size_t o2 = (size_t)last_band * band;
        CUDA_TRY(cudaMemcpyAsync((char*)dst + o2, (const char*)src + o2, row * last_rows, cudaMemcpyDeviceToHost,
                                 slot->copy_stream));
    }
    return 0;
}

// The same rows from a pinned staging frame into the caller's pageable canvas, by the host's threads.
void host_copy_bands(const RtcScene* s, int shard, int n_shards, int b0, int b1, const char* src, char* dst, size_t px_bytes) {
    const size_t row = (size_t)s->width * px_bytes;
    const size_t band = row * kBandRows;
    if (b1 <= b0) return;
    if (n_shards == 1) {
        const int last_rows = std::min<int>(kBandRows, (int)s->height - (b1 - 1) * kBandRows);
        const size_t off = (size_t)b0 * band, bytes = (size_t)(b1 - b0 - 1) * band + row * last_rows;
        parallel_copy(dst + off, src + off, bytes, (size_t)96 << 10);  // a slice is ~1 MiB: all threads take a piece of it
        return;
    }
    parallel_for((size_t)(b1 - b0), 1, [&](size_t jb, size_t je, int) {
        for (size_t j = jb; j < je; j++) {
            const int frame_band = shard + (b0 + (int)j) * n_shards;
            const int rows = std::min<int>(kBandRows, (int)s->height - frame_band * kBandRows);
            memcpy(dst + (size_t)frame_band * band, src + (size_t)frame_band * band, row * rows);
        }
    });
}
bool is_pageable(const void* p) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        cudaGetLastError();
        return false;  // let the copy itself report what is wrong with the pointer
    }
    return attr.type == cudaMemoryTypeUnregistered;
}
int ensure_stage(DeviceSlot* d, char** stage, size_t* have, size_t bytes) {
    if (bytes <= *have) return 0;
    CUDA_TRY(cudaSetDevice(d->device));
    if (*stage) cudaFreeHost(*stage);
    *stage = nullptr, *have = 0;
    CUDA_TRY(cudaHostAlloc(stage, bytes, cudaHostAllocPortable));
    *have = bytes;
    return 0;
}

// Device frames -> the caller's canvases, for rtc_render and rtc_render_views.  A piece is bands [b0, b1) of a shard's
// band list in views [v0, v1) of the canvases (rtc_render: the one view 0); the device holds view v0's frame at d_rgb / d_u8
// and the following views' frames after it.  With several devices the pieces wait in `pending` until every device has its
// kernels: a device-to-host copy into pageable memory blocks the calling thread, and queued inside the device loop it would
// make the devices run one after the other (ADVICE r1).  One device: a piece's copy is queued right behind its kernel.
// A pageable destination (the reference's Canvas is a Vec): cudaMemcpyAsync into it would block the calling thread slice
// after slice at the driver's single-threaded staging rate (~10 GB/s).  Instead the pieces land in a pinned frame kept
// with the device slot (view v at stage index v - stage_v0), and the host's threads move each one on as soon as its copy
// event has fired, while the device renders and copies the next (c3's 24.9 MB 8-bit canvas into a heap array: 0.71 ms
// end to end instead of 3.07; into pinned memory 0.66).
struct CanvasCopy {
    struct Piece {
        DeviceSlot* slot;
        int shard, b0, b1, v0, v1;
        const float* d_rgb;
        const unsigned char* d_u8;
    };
    RtcScene* s;
    int n_shards;
    float* rgb;
    uint8_t* u8;
    bool stage_rgb, stage_u8;
    int stage_views, stage_v0 = 0;  // views the pinned staging frames hold, and the first of them
    std::vector<Piece> pending;
    struct Unstage {
        cudaEvent_t done;
        Piece p;
    };
    std::vector<Unstage> unstage;
    size_t unstaged = 0;
    std::vector<int> events_used;
    CanvasCopy(RtcScene* s_, int n_shards_, float* rgb_, uint8_t* u8_, bool stage_rgb_, bool stage_u8_, int stage_views_)
        : s(s_), n_shards(n_shards_), rgb(rgb_), u8(u8_), stage_rgb(stage_rgb_), stage_u8(stage_u8_), stage_views(stage_views_),
          events_used(s_->replicas.size(), 0) {}
    size_t frame_px() const { return (size_t)s->width * s->height; }
    int slot_index(DeviceSlot* slot) const {
        for (size_t i = 0; i < s->replicas.size(); i++)
            if (s->replicas[i].slot == slot) return (int)i;
        return 0;
    }
    int nb(int shard) const {
        const int total = ((int)s->height + kBandRows - 1) / kBandRows;
        return shard < total ? (total - shard + n_shards - 1) / n_shards : 0;
    }
    // one plane of a piece: whole views of a one-shard frame are one contiguous copy, anything else goes band by band
    int copy_plane(const Piece& p, const char* src, char* dst, size_t px_bytes) {
        const size_t fb = frame_px() * px_bytes;
        if (p.v1 - p.v0 > 1 && n_shards == 1 && p.b0 == 0 && p.b1 == nb(p.shard)) {
            CUDA_TRY(cudaMemcpyAsync(dst, src, (size_t)(p.v1 - p.v0) * fb, cudaMemcpyDeviceToHost, p.slot->copy_stream));
            return 0;
        }
        for (int v = 0; v < p.v1 - p.v0; v++)
            if (int rc = copy_bands(p.slot, s, p.shard, n_shards, p.b0, p.b1, src + v * fb, dst + v * fb, px_bytes)) return rc;
        return 0;
    }
    int copy_out(const Piece& p) {  // device frames -> canvas or staging frame
        int rc;
        const size_t px = frame_px();
        DeviceSlot* slot = p.slot;
        if (stage_rgb && (rc = ensure_stage(slot, &slot->h_stage_rgb, &slot->h_stage_rgb_bytes, px * 12 * stage_views))) return rc;
        if (stage_u8 && (rc = ensure_stage(slot, &slot->h_stage_u8, &slot->h_stage_u8_bytes, px * 3 * stage_views))) return rc;
        if (rgb && (rc = copy_plane(p, (const char*)p.d_rgb,
                                    stage_rgb ? slot->h_stage_rgb + (p.v0 - stage_v0) * px * 12 : (char*)(rgb + p.v0 * px * 3), 12)))
            return rc;
        if (u8 && (rc = copy_plane(p, (const char*)p.d_u8,
                                   stage_u8 ? slot->h_stage_u8 + (p.v0 - stage_v0) * px * 3 : (char*)(u8 + p.v0 * px * 3), 3)))
            return rc;
        if (stage_rgb || stage_u8) {
            int& used = events_used[slot_index(slot)];
            while ((int)slot->copy_done.size() <= used) {
                cudaEvent_t e;
                CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
                slot->copy_done.push_back(e);
            }
            CUDA_TRY(cudaEventRecord(slot->copy_done[used], slot->copy_stream));
            unstage.push_back({slot->copy_done[used], p});
            used++;
        }
        return 0;
    }
    int queue(const Piece& p) {
        if (s->replicas.size() > 1) {
            pending.push_back(p);
            return 0;
        }
        return copy_out(p);
    }
    int flush_pending() {  // the copy stream of each device already waits for the piece's event
        for (const Piece& p : pending) {
            CUDA_TRY(cudaSetDevice(p.slot->device));
            if (int rc = copy_out(p)) return rc;
        }
        pending.clear();
        return 0;
    }
    void host_plane(const Piece& p, const char* stage, char* dst, size_t px_bytes) {
        const size_t fb = frame_px() * px_bytes;
        const char* src = stage + (p.v0 - stage_v0) * fb;
        dst += p.v0 * fb;
        if (p.v1 - p.v0 > 1 && n_shards == 1 && p.b0 == 0 && p.b1 == nb(p.shard)) {
            parallel_copy(dst, src, (size_t)(p.v1 - p.v0) * fb, (size_t)96 << 10);
            return;
        }
        for (int v = 0; v < p.v1 - p.v0; v++) host_copy_bands(s, p.shard, n_shards, p.b0, p.b1, src + v * fb, dst + v * fb, px_bytes);
    }
    int drain() {  // the host half of the staged copies queued so far
        for (; unstaged < unstage.size(); unstaged++) {
            const Unstage& u = unstage[unstaged];
            CUDA_TRY(cudaSetDevice(u.p.slot->device));
            CUDA_TRY(cudaEventSynchronize(u.done));
            if (stage_rgb) host_plane(u.p, u.p.slot->h_stage_rgb, (char*)rgb, 12);
            if (stage_u8) host_plane(u.p, u.p.slot->h_stage_u8, (char*)u8, 3);
        }
        return 0;
    }
};

// The wavefront renderer's chunking: about a million pixels of the shard at a time (whole bands).
int wave_chunk_bands(int width, int nb) {
    const int per_band = std::max(1, width) * kBandRows;
    int bands = std::max(1, (1 << 20) / per_band);
    while ((nb + bands - 1) / bands > kWaveMaxChunks) bands *= 2;
    return std::min(bands, std::max(nb, 1));
}
int ensure_wave_pool(DeviceSlot* d, int width, int nb) {
    const int chunk_px = wave_chunk_bands(width, nb) * kBandRows * ((width + 7) / 8 * 8);
    const long long want = (long long)chunk_px * d->wave_rays_per_pixel;
    if (want > 0x7fffffffLL / 2) return fail(RTC_ERR_CAPACITY, "wavefront ray pool too large");
    CUDA_TRY(cudaSetDevice(d->device));
    if (!d->d_wave_ints) CUDA_TRY(cudaMalloc(&d->d_wave_ints, kWaveInts * sizeof(int) + 3 * kWaveMaxChunks * sizeof(unsigned long long) + 64));
    if ((int)want > d->wave_capacity) {
        if (d->d_wave_rays) cudaFree(d->d_wave_rays);
        if (d->d_wave_nodes) cudaFree(d->d_wave_nodes);
        d->d_wave_rays = d->d_wave_nodes = nullptr, d->wave_capacity = 0;
        CUDA_TRY(cudaMalloc(&d->d_wave_rays, (size_t)want * 96));
        CUDA_TRY(cudaMalloc(&d->d_wave_nodes, (size_t)want * 64));
        d->wave_capacity = (int)want;
    }
    return 0;
}

int render_impl(RtcScene* s, int depth, int shard0, int n_shards_ext, float* rgb, uint8_t* u8, RtcStats* stats, bool detailed) {
    if (!s) return fail(RTC_ERR_INVALID, "null scene");
    if (!s->committed) return fail(RTC_ERR_STATE, "rtc_render before rtc_scene_commit");
    if (depth < 0 || depth > kMaxFrames - 1)
        return fail(RTC_ERR_CAPACITY, "reflection_recursion_depth must be in [0, " + std::to_string(kMaxFrames - 1) + "]");
    auto t0 = std::chrono::steady_clock::now();
    const int ndev = (int)s->replicas.size();
    const bool external = n_shards_ext > 0;
    if (external && ndev != 1) return fail(RTC_ERR_STATE, "rtc_render_shard needs a scene committed on exactly one device");
    if (external && (shard0 < 0 || shard0 >= n_shards_ext)) return fail(RTC_ERR_INVALID, "bad shard index");
    const int n_shards = external ? n_shards_ext : ndev;
    const int total_bands = ((int)s->height + kBandRows - 1) / kBandRows;
    const bool copy_out = rgb || u8;
    RtcStats st;
    memset(&st, 0, sizeof(st));
    st.n_devices = ndev;
    st.detailed = detailed;
    // (small planes are left to the driver: waking the worker threads costs more than its pageable path loses — c1's 1.2 MB:
    // 0.28 ms through the driver, 0.40 ms staged)
    const size_t frame_px = (size_t)s->width * s->height;
    const bool stage_rgb = rgb && frame_px * 12 >= ((size_t)4 << 20) && is_pageable(rgb);
    const bool stage_u8 = u8 && frame_px * 3 >= ((size_t)4 << 20) && is_pageable(u8);
    CanvasCopy cc(s, n_shards, rgb, u8, stage_rgb, stage_u8, 1);
    auto copy_out_bands = [&](DeviceSlot* slot, int shard, int b0, int b1) -> int {  // device frame -> canvas or staging frame
        return cc.copy_out({slot, shard, b0, b1, 0, 1, slot->d_rgb, slot->d_u8});
    };
    auto drain_unstage = [&]() -> int { return cc.drain(); };
    auto queue_copy = [&](DeviceSlot* slot, int shard, int b0, int b1) -> int {
        return cc.queue({slot, shard, b0, b1, 0, 1, slot->d_rgb, slot->d_u8});
    };
    for (int i = 0; i < ndev; i++) {
        Replica& r = s->replicas[i];
        DeviceSlot* slot = r.slot;
        const int shard = external ? shard0 : i;
        r.small.filter_ok = r.filter_eligible && s->shadow_filter;
        r.small.cell_masks = r.cell_masks_eligible && s->shadow_filter;
        r.small.plane_cells = r.plane_cells_eligible && r.small.cell_masks;
        const int nb = shard < total_bands ? (total_bands - shard + n_shards - 1) / n_shards : 0;
        CUDA_TRY(cudaSetDevice(slot->device));
        CUDA_TRY(cudaMemsetAsync(slot->d_counters, 0, sizeof(DevCounters), slot->stream));
        // Longest-processing-time-first: a frame's cost is concentrated in a few tiles (deep reflection trees: one
        // block there runs ~10x longer than the average), and a long block that starts late is the tail of the
        // launch — the term that limits strong scaling over shards (c3, 1/8 of the frame: the SMs were busy for
        // only 53 % of the launch).  The first render of a (shard, depth) configuration runs in natural order and
        // records how many clock cycles every tile's block took; later renders launch the shard's tiles
        // most-expensive-first from a list kept on the device.  The order changes no pixel.  It needs one
        // copy-free launch, so it is used when the frame stays on the device or is copied in one piece.  Whether it
        // pays depends on the frame, not on its size alone (c3: 1/8 of the 4K frame 13 % faster, 1/4 of it 2 %
        // slower, the whole frame 7 % slower; the whole 1080p mesh frame c4 25 % faster), so the second render is a
        // trial: the learnt order is kept only if that render beats the natural-order one by more than 2 %.
        // tree scenes whose ray trees branch: the streaming kernel (lanes draw pixels from a per-launch counter).  A
        // persistent launch pays its tail once per launch and such frames take far longer than their copy, so they
        // are not sliced
        const bool stream_scene = r.small.n == 0 && (s->stream < 0 ? s->has_branching_materials : s->stream != 0);
        // a frame is cut only as finely as its copy is long: one slice per MiB that leaves the device, at most
        // `render_slices` (c3's 24.9 MB 8-bit canvas: 23 slices, 0.67 ms end to end against 1.10 in one piece; c1's 1.2 MB:
        // 1 slice, 0.22 ms against 0.43 in six).  Slices on one stream cost ~15 us each of launch ramp and tail (6 slices
        // of 4 MiB: 0.74 ms); rotated over three streams (below) they cost next to nothing and can be small
        const size_t copy_bytes = (size_t)s->width * kBandRows * nb * ((rgb ? 12 : 0) + (u8 ? 3 : 0));
        static const int slice_shift = [] {
            const char* env = getenv("RTC_SLICE_BYTES_LOG2");  // tuning aid
            return env ? std::max(16, std::min(30, atoi(env))) : 20;
        }();
        const int n_slices = copy_out && !stream_scene
                                 ? std::max(1, std::min(std::min(s->render_slices, nb), (int)(copy_bytes >> slice_shift)))
                                 : 1;
        const bool use_wave = stream_scene && !detailed && !s->light_is_rect && s->wavefront != 0 && nb > 0;
        const int tiles_x = ((int)s->width + kTileW - 1) / kTileW;
        int rc0;
        if ((rc0 = ensure_tiles(slot, total_bands * tiles_x))) return rc0;
        const long long launch_blocks = (long long)nb * tiles_x;
        const bool order_wanted = !stream_scene && s->adaptive_order && n_slices == 1 && nb > 0 &&
                                  launch_blocks < (long long)s->order_max_waves * 5 * slot->sm_count;
        const bool learnt = r.order_shard == shard && r.order_n_shards == n_shards && r.order_depth == depth &&
                            r.order_filter == s->shadow_filter;
        r.learning = order_wanted && !learnt && r.renders_done > 0;
        // undecided: stage 1 = natural order again, stages 2 and 3 = the learnt order; decided: by the verdict
        r.order_timed = order_wanted && learnt && r.order_verdict == 0 && !detailed;
        r.order_lost_here = order_wanted && learnt && r.order_verdict < 0 && !detailed;
        const bool use_order = order_wanted && learnt && (r.order_verdict > 0 || (r.order_verdict == 0 && r.order_stage >= 2));
        if (r.learning) CUDA_TRY(cudaMemsetAsync(slot->d_tile_cost, 0, (size_t)total_bands * tiles_x * sizeof(unsigned), slot->stream));
        // With a host destination the frame is rendered in a few slices so that the device-to-host copy of one
        // slice overlaps the kernel of the next (the 4K canvases are 124 MB: ~2.3 ms of PCIe against ~2 ms of
        // kernel); left on the device it is one launch.
        while ((int)slot->slice_done.size() < n_slices) {
            cudaEvent_t e;
            CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            slot->slice_done.push_back(e);
        }
        const bool use_stream = stream_scene;
        if (use_stream) CUDA_TRY(cudaMemsetAsync(slot->d_stream_counter, 0, 64 * sizeof(unsigned), slot->stream));
        CUDA_TRY(cudaEventRecord(slot->ev0, slot->stream));
        // The wavefront renderer (dev_wave.cuh): tree scenes with branching ray trees under a point light.  The shard's
        // bands are rendered chunk by chunk through one ray pool; a chunk is also the unit of the device-to-host copy.
        r.wave_chunks = 0;
        if (use_wave) {
            int rc;
            if ((rc = ensure_wave_pool(slot, (int)s->width, nb))) return rc;
            const int chunk_bands = wave_chunk_bands((int)s->width, nb);
            for (int b0 = 0, k = 0; b0 < nb; b0 += chunk_bands, k++) {
                const int b1 = std::min(nb, b0 + chunk_bands);
                DevFrame F{slot->d_rgb, slot->d_u8, shard, n_shards, depth, b1 - b0, b0, nullptr, nullptr, 1, nullptr, 0};
                WavePoolRaw pool{slot->d_wave_rays, slot->d_wave_nodes, slot->wave_capacity, slot->d_wave_ints,
                                 reinterpret_cast<unsigned long long*>(slot->d_wave_ints + kWaveInts) + 3 * k};
                kernel_build(s->strict_fp, r.csg_sweep).wave(r.scene, r.small, F, pool, slot->d_counters, slot->sm_count * 8, slot->stream);
                CUDA_TRY(cudaGetLastError());
                st.launches += 2 + 5 * (depth + 1) + (depth + 1);
                r.wave_chunks = k + 1;
                if (copy_out) {
                    while ((int)slot->slice_done.size() <= k) {
                        cudaEvent_t e;
                        CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
                        slot->slice_done.push_back(e);
                    }
                    CUDA_TRY(cudaEventRecord(slot->slice_done[k], slot->stream));
                    CUDA_TRY(cudaStreamWaitEvent(slot->copy_stream, slot->slice_done[k], 0));
                    if ((rc = queue_copy(slot, shard, b0, b1))) return rc;
                }
            }
        }
        // The slices of a frame are independent launches, so they rotate over three streams: the blocks of slice k + 1
        // fill the SMs as slice k drains instead of waiting for its last block (per slice that tail and the next launch's
        // ramp were ~15 us of mostly idle SMs).  Every stream starts behind ev0 (the counters are reset), the frame ends
        // at ev1 on the first stream behind the others' last slices, each slice's copy waits for its own event.
        static const bool rotate = [] {
            const char* env = getenv("RTC_SLICE_STREAMS");  // tuning aid: 0 = all slices on one stream
            return !env || atoi(env) != 0;
        }();
        cudaStream_t lanes[3] = {slot->stream, slot->slice_stream[0], slot->slice_stream[1]};
        const int n_lanes = rotate && n_slices > 1 && !use_wave ? std::min(3, n_slices) : 1;
        for (int l = 1; l < n_lanes; l++) CUDA_TRY(cudaStreamWaitEvent(lanes[l], slot->ev0, 0));
        int last_on_lane[3] = {-1, -1, -1};
        for (int k = 0; k < n_slices && !use_wave; k++) {
            const int b0 = (int)((int64_t)nb * k / n_slices), b1 = (int)((int64_t)nb * (k + 1) / n_slices);
            if (b1 <= b0) continue;
            cudaStream_t lane = lanes[k % n_lanes];
            DevFrame F{slot->d_rgb, slot->d_u8, shard, n_shards, depth, b1 - b0, b0, use_order ? slot->d_tile_order : nullptr,
                       r.learning ? slot->d_tile_cost : nullptr, s->converge < 0 ? (int)s->has_branching_materials : s->converge,
                       nullptr, 0};
            if (use_stream) {
                F.stream_counter = slot->d_stream_counter + k;
                F.stream_blocks = slot->sm_count * 6;
                F.tile_order = nullptr, F.tile_cost = nullptr;
            }
            kernel_build(s->strict_fp, r.csg_sweep).render(r.scene, r.small, F, slot->d_counters, detailed, lane);
            CUDA_TRY(cudaGetLastError());
            st.launches++;
            if (copy_out) {
                CUDA_TRY(cudaEventRecord(slot->slice_done[k], lane));
                CUDA_TRY(cudaStreamWaitEvent(slot->copy_stream, slot->slice_done[k], 0));
                if (int rc = queue_copy(slot, shard, b0, b1)) return rc;
                last_on_lane[k % n_lanes] = k;
            }
        }
        for (int l = 1; l < n_lanes; l++)
            if (last_on_lane[l] >= 0) CUDA_TRY(cudaStreamWaitEvent(slot->stream, slot->slice_done[last_on_lane[l]], 0));
        CUDA_TRY(cudaEventRecord(slot->ev1, slot->stream));
        CUDA_TRY(cudaMemcpyAsync(slot->h_counters, slot->d_counters, sizeof(DevCounters), cudaMemcpyDeviceToHost, slot->stream));
    }
    if (int rc = cc.flush_pending()) return rc;
    if (int rc = drain_unstage()) return rc;
    const bool timing = getenv("RTC_TIMING") != nullptr;  // tuning aid
    auto since = [&] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); };
    if (timing) fprintf(stderr, "[rtc render] launches queued at      %8.3f ms\n", since());
    for (int i = 0; i < ndev; i++) {
        DeviceSlot* slot = s->replicas[i].slot;
        CUDA_TRY(cudaSetDevice(slot->device));
        CUDA_TRY(cudaStreamSynchronize(slot->stream));
        if (timing) fprintf(stderr, "[rtc render] kernels done at          %8.3f ms\n", since());
        CUDA_TRY(cudaStreamSynchronize(slot->copy_stream));
        if (timing) fprintf(stderr, "[rtc render] copies done at           %8.3f ms\n", since());
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, slot->ev0, slot->ev1));
        st.kernel_ms = std::max(st.kernel_ms, (double)ms);
        Replica& rw = s->replicas[i];
        if (rw.wave_chunks > 0) {
            // the chunks' records: rays that did not fit the pool (the chunk is rendered again, by render_stream — never a
            // silently truncated ray tree), secondary rays, shades
            const int shard = external ? shard0 : i;
            const int nb = shard < total_bands ? (total_bands - shard + n_shards - 1) / n_shards : 0;
            std::vector<unsigned long long> rec(3 * (size_t)rw.wave_chunks);
            CUDA_TRY(cudaMemcpy(rec.data(), reinterpret_cast<unsigned long long*>(slot->d_wave_ints + kWaveInts), rec.size() * 8,
                                cudaMemcpyDeviceToHost));
            const int chunk_bands = wave_chunk_bands((int)s->width, nb);
            DevCounters extra{};
            bool again = false;
            for (int k = 0; k < rw.wave_chunks; k++) {
                if (rec[3 * k] == 0) {
                    extra.secondary += rec[3 * k + 1], extra.shades += rec[3 * k + 2];
                    continue;
                }
                again = true;
                st.wave_overflows++;
                const int b0 = k * chunk_bands, b1 = std::min(nb, b0 + chunk_bands);
                DevFrame F{slot->d_rgb, slot->d_u8, shard, n_shards, depth, b1 - b0, b0, nullptr, nullptr, 1, slot->d_stream_counter + (k % 64),
                           slot->sm_count * 6};
                CUDA_TRY(cudaMemsetAsync(slot->d_stream_counter + (k % 64), 0, sizeof(unsigned), slot->stream));
                kernel_build(s->strict_fp, rw.csg_sweep).render(rw.scene, rw.small, F, slot->d_counters, false, slot->stream);
                CUDA_TRY(cudaGetLastError());
                st.launches++;
                CUDA_TRY(cudaStreamSynchronize(slot->stream));  // one chunk at a time: they may share a counter slot
                if (int rc = copy_out_bands(slot, shard, b0, b1)) return rc;
            }
            if (again) {
                CUDA_TRY(cudaStreamSynchronize(slot->copy_stream));
                if (int rc = drain_unstage()) return rc;
                slot->wave_rays_per_pixel = std::min(64, slot->wave_rays_per_pixel * 2);  // a bigger pool next time
                CUDA_TRY(cudaMemcpy(slot->h_counters, slot->d_counters, sizeof(DevCounters), cudaMemcpyDeviceToHost));  // the re-rendered chunks counted too
            }
            st.secondary_rays += extra.secondary, st.shades += extra.shades;
            st.shadow_rays += extra.shades * (s->light_is_rect ? (uint64_t)s->u_steps * s->v_steps : 1);
        }
        const DevCounters c = *slot->h_counters;  // copied behind ev1 on the render stream (synchronized above)
        {
            // camera.rs:80-81: rows y < h - 1 and columns x < w - 1 of this shard's bands
            const int shard = external ? shard0 : i;
            uint64_t rows = 0;
            for (int b = shard; b < total_bands; b += n_shards)
                rows += (uint64_t)std::max(0, std::min<int>((int)s->height - 1, (b + 1) * kBandRows) - b * kBandRows);
            add_counters(st, c, rows * (uint64_t)(s->width - 1), s->light_is_rect ? (uint64_t)s->u_steps * s->v_steps : 1);
        }
        Replica& r = s->replicas[i];
        r.renders_done++;
        if (r.order_timed) {
            if (r.order_stage <= 1) r.natural_ms = std::min(r.natural_ms, ms);
            if (r.order_stage == 2) r.ordered_ms = ms;
            if (r.order_stage == 3) {
                r.order_verdict = std::min(r.ordered_ms, ms) < 0.98f * r.natural_ms ? 1 : -1;
                r.renders_since_loss = 0;
            }
            r.order_stage++;
            r.order_timed = false;
        } else if (r.order_lost_here && r.order_retrials < 3 && ++r.renders_since_loss >= 32) {
            r.order_retrials++;
            r.order_verdict = 0, r.order_stage = 0, r.natural_ms = 3.4e38f;  // stages 0, 1: natural order; 2, 3: the learnt one
        }
        if (r.learning) {  // sort this shard's tiles by the cycles their blocks took: the launch order from now on
            const int shard = external ? shard0 : i;
            const int tiles_x = ((int)s->width + kTileW - 1) / kTileW;
            std::vector<unsigned> cost((size_t)total_bands * tiles_x);
            CUDA_TRY(cudaMemcpy(cost.data(), slot->d_tile_cost, cost.size() * sizeof(unsigned), cudaMemcpyDeviceToHost));
            std::vector<int> order;
            for (int b = shard; b < total_bands; b += n_shards)
                for (int x = 0; x < tiles_x; x++) order.push_back(b * tiles_x + x);
            std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return cost[a] > cost[b]; });
            if (const char* dump = getenv("RTC_DUMP_TILE_COST")) {  // tuning aid: the learnt costs, in launch order
                if (FILE* fh = fopen(dump, "w")) {
                    for (int id : order) fprintf(fh, "%d %d %u\n", id / tiles_x, id % tiles_x, cost[id]);
                    fclose(fh);
                }
            }
            CUDA_TRY(cudaMemcpy(slot->d_tile_order, order.data(), order.size() * sizeof(int), cudaMemcpyHostToDevice));
            r.order_shard = shard, r.order_n_shards = n_shards, r.order_depth = depth, r.order_filter = s->shadow_filter;
            r.order_verdict = 0, r.order_stage = 1, r.natural_ms = ms, r.order_retrials = 0, r.renders_since_loss = 0;
            r.learning = false;
        }
    }
    st.flops = detailed ? flops_of(st, st.primary_rays) : 0.0;
    st.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (stats) *stats = st;
    if (st.capacity_overflows)
        return fail(RTC_ERR_CAPACITY, "CSG evaluation overflowed its buffers " + std::to_string(st.capacity_overflows) + " times");
    return 0;
}

// rtc_render_views: the device frames of a batch live in a per-device arena of this many bytes (both planes of a chunk of
// whole views); a bigger batch is rendered chunk by chunk through it.  RTC_VIEW_ARENA_BYTES (read at every call) lowers or
// raises it: a test aid that forces several chunks.
constexpr size_t kViewArenaBytes = (size_t)2 << 30;
// ... and a pageable destination is staged through pinned host frames of at most this many bytes per device (or one view's
// planes, when a view alone is bigger): a chunk holds no more views than its staged planes fit in.  Page-locked host memory
// is taken from the whole system and the frames are kept with the pooled device slot, so they are bounded apart from the
// device arena.
constexpr size_t kViewStageBytes = (size_t)256 << 20;
constexpr int kMaxViewsPerLaunch = 65535;  // gridDim.z

int ensure_views(DeviceSlot* d, uint32_t n, size_t frame_bytes) {
    CUDA_TRY(cudaSetDevice(d->device));
    if (n > d->views_capacity) {
        if (d->d_views) cudaFree(d->d_views);
        if (d->h_views) cudaFreeHost(d->h_views);
        d->d_views = nullptr, d->h_views = nullptr, d->views_capacity = 0;
        const uint32_t cap = std::max<uint32_t>(n, 64);
        CUDA_TRY(cudaMalloc(&d->d_views, cap * sizeof(DevView)));
        CUDA_TRY(cudaHostAlloc(&d->h_views, cap * sizeof(DevView), cudaHostAllocDefault));
        d->views_capacity = cap;
    }
    if (frame_bytes > d->view_frames_bytes) {
        if (d->d_view_frames) cudaFree(d->d_view_frames);
        d->d_view_frames = nullptr, d->view_frames_bytes = 0;
        CUDA_TRY(cudaMalloc(&d->d_view_frames, frame_bytes));
        d->view_frames_bytes = frame_bytes;
    }
    return 0;
}

int render_views_impl(RtcScene* s, int depth, uint32_t n_views, const RtcView* views, float* rgb, uint8_t* u8, RtcStats* stats) {
    // the arguments first (no device needed), then the scene's state
    if (!s) return fail(RTC_ERR_INVALID, "null scene");
    if (n_views == 0 || !views) return fail(RTC_ERR_INVALID, "rtc_render_views: n_views must be >= 1 and views non-null");
    for (uint32_t v = 0; v < n_views; v++) {
        const RtcView& w = views[v];
        bool finite = std::isfinite(w.half_width) && std::isfinite(w.half_height) && std::isfinite(w.pixel_size);
        for (float x : w.transform_inverse) finite = finite && std::isfinite(x);
        if (!finite) return fail(RTC_ERR_INVALID, "rtc_render_views: view " + std::to_string(v) + " has a non-finite field");
        if (!(w.pixel_size > 0.f)) return fail(RTC_ERR_INVALID, "rtc_render_views: view " + std::to_string(v) + " has pixel_size <= 0");
    }
    if (depth < 0 || depth > kMaxFrames - 1)
        return fail(RTC_ERR_INVALID, "reflection_recursion_depth must be in [0, " + std::to_string(kMaxFrames - 1) + "]");
    if (!s->committed) return fail(RTC_ERR_STATE, "rtc_render_views before rtc_scene_commit");
    // The tree's boxes are padded for ray origins up to the commit's reach (rtc_commit.cu: "pad"): a camera farther out
    // could lose hits the reference reports.  Small and tree-less scenes test every item exactly: any view goes.
    if (s->replicas[0].scene.bvh_root >= 0)
        for (uint32_t v = 0; v < n_views; v++)
            for (int a = 0; a < 3; a++) {
                const float c = views[v].transform_inverse[a * 4 + 3];
                if (std::fabs(c) > s->reach) {
                    char msg[320];
                    snprintf(msg, sizeof(msg),
                             "rtc_render_views: view %u's camera origin has a coordinate %g beyond the scene's reach %g (the tree is "
                             "padded for coordinates up to it); commit the scene with the farthest camera of the batch",
                             v, (double)c, (double)s->reach);
                    return fail(RTC_ERR_INVALID, msg);
                }
            }
    auto t0 = std::chrono::steady_clock::now();
    const int ndev = (int)s->replicas.size(), n_shards = ndev;
    const int total_bands = ((int)s->height + kBandRows - 1) / kBandRows;
    const bool copy_out = rgb || u8;
    const size_t frame_px = (size_t)s->width * s->height;
    RtcStats st;
    memset(&st, 0, sizeof(st));
    st.n_devices = ndev;
    // both planes of every view of a chunk, as rtc_render's frame holds both
    size_t budget = kViewArenaBytes;
    if (const char* env = getenv("RTC_VIEW_ARENA_BYTES")) budget = (size_t)std::max(1LL, atoll(env));
    const bool stream_scene = s->replicas[0].small.n == 0 && (s->stream < 0 ? s->has_branching_materials : s->stream != 0);
    const int blocks_x = ((int)s->width + 7) / 8;
    const int nb_max = (total_bands + n_shards - 1) / n_shards;
    uint32_t chunk = (uint32_t)std::max<size_t>(1, std::min<size_t>(budget / (frame_px * 15), n_views));
    chunk = std::min<uint32_t>(chunk, kMaxViewsPerLaunch);
    if (stream_scene)  // the pixel stream's index (views x bands x 8x4 blocks x 32) is 32-bit
        chunk = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(chunk, 0xffffffffull / ((uint64_t)nb_max * blocks_x * 64)));
    const bool stage_rgb = rgb && frame_px * 12 * n_views >= ((size_t)4 << 20) && is_pageable(rgb);
    const bool stage_u8 = u8 && frame_px * 3 * n_views >= ((size_t)4 << 20) && is_pageable(u8);
    const size_t staged_per_view = frame_px * ((stage_rgb ? 12 : 0) + (stage_u8 ? 3 : 0));
    if (staged_per_view) chunk = (uint32_t)std::max<size_t>(1, std::min<size_t>(chunk, kViewStageBytes / staged_per_view));
    CanvasCopy cc(s, n_shards, rgb, u8, stage_rgb, stage_u8, (int)chunk);
    static const bool rotate = [] {
        const char* env = getenv("RTC_SLICE_STREAMS");  // tuning aid: 0 = all slices on one stream
        return !env || atoi(env) != 0;
    }();
    static const int slice_shift = [] {
        const char* env = getenv("RTC_SLICE_BYTES_LOG2");  // tuning aid
        return env ? std::max(16, std::min(30, atoi(env))) : 20;
    }();
    std::vector<int> launches_on(ndev, 0);  // slice events used per device
    std::vector<cudaEvent_t> chunk_copied(ndev, nullptr);  // the previous chunk's copies: the arena is free after them
    for (int i = 0; i < ndev; i++) {
        Replica& r = s->replicas[i];
        DeviceSlot* slot = r.slot;
        r.small.filter_ok = r.filter_eligible && s->shadow_filter;
        r.small.cell_masks = r.cell_masks_eligible && s->shadow_filter;
        r.small.plane_cells = r.plane_cells_eligible && r.small.cell_masks;
        if (int rc = ensure_views(slot, n_views, frame_px * 15 * chunk)) return rc;
        for (uint32_t v = 0; v < n_views; v++) {  // the view table, uploaded once per call on the render stream
            DevView& d = slot->h_views[v];
            rows3(views[v].transform_inverse, d.cam_inv);
            d.half_w = views[v].half_width, d.half_h = views[v].half_height, d.pixel_size = views[v].pixel_size, d.pad = 0.f;
        }
        CUDA_TRY(cudaMemcpyAsync(slot->d_views, slot->h_views, n_views * sizeof(DevView), cudaMemcpyHostToDevice, slot->stream));
        CUDA_TRY(cudaMemsetAsync(slot->d_counters, 0, sizeof(DevCounters), slot->stream));
        CUDA_TRY(cudaEventRecord(slot->ev0, slot->stream));
    }
    auto slice_event = [&](DeviceSlot* slot, int& used) -> cudaEvent_t {
        while ((int)slot->slice_done.size() <= used) {
            cudaEvent_t e;
            if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return nullptr;
            slot->slice_done.push_back(e);
        }
        return slot->slice_done[used++];
    };
    for (uint32_t c0 = 0; c0 < n_views; c0 += chunk) {
        const uint32_t c1 = std::min(n_views, c0 + chunk);
        cc.stage_v0 = (int)c0;
        for (int i = 0; i < ndev; i++) {
            Replica& r = s->replicas[i];
            DeviceSlot* slot = r.slot;
            const int shard = i;
            const int nb = shard < total_bands ? (total_bands - shard + n_shards - 1) / n_shards : 0;
            CUDA_TRY(cudaSetDevice(slot->device));
            float* d_rgb = reinterpret_cast<float*>(slot->d_view_frames);
            unsigned char* d_u8 = reinterpret_cast<unsigned char*>(slot->d_view_frames + frame_px * 12 * chunk);
            // The launches of a chunk: left on the device, one.  Copied to host memory, rtc_render's slice rule applied to the
            // whole batch — one slice per MiB copied, at most RTC_OPT_RENDER_SLICES — as runs of whole views, or, when a view
            // is bigger than a slice, that view cut by bands as rtc_render cuts it.  A branching tree scene renders a chunk as
            // one pixel stream (rtc_render does not slice it either).
            struct Launch {
                uint32_t v0, v1;
                int b0, b1;
            };
            std::vector<Launch> plan;
            const size_t view_copy = (size_t)s->width * kBandRows * nb * ((rgb ? 12 : 0) + (u8 ? 3 : 0));
            const int want = copy_out && !stream_scene
                                 ? std::max(1, (int)std::min<size_t>((size_t)s->render_slices, (view_copy * n_views) >> slice_shift))
                                 : 1;
            if (nb == 0) {
            } else if (want <= (int)n_views) {
                const uint32_t per_run = (n_views + want - 1) / want;
                for (uint32_t v = c0; v < c1; v += per_run) plan.push_back({v, std::min(c1, v + per_run), 0, nb});
            } else {
                const int per_view = std::max(1, std::min(std::min(s->render_slices, nb), (int)(view_copy >> slice_shift)));
                for (uint32_t v = c0; v < c1; v++)
                    for (int k = 0; k < per_view; k++) {
                        const int b0 = (int)((int64_t)nb * k / per_view), b1 = (int)((int64_t)nb * (k + 1) / per_view);
                        if (b1 > b0) plan.push_back({v, v + 1, b0, b1});
                    }
            }
            cudaStream_t lanes[3] = {slot->stream, slot->slice_stream[0], slot->slice_stream[1]};
            const int n_lanes = rotate && plan.size() > 1 ? std::min<int>(3, (int)plan.size()) : 1;
            // every lane starts behind the table upload and the counter reset, and behind the previous chunk's copies
            for (int l = 1; l < n_lanes; l++) CUDA_TRY(cudaStreamWaitEvent(lanes[l], slot->ev0, 0));
            if (chunk_copied[i])
                for (int l = 0; l < n_lanes; l++) CUDA_TRY(cudaStreamWaitEvent(lanes[l], chunk_copied[i], 0));
            int last_on_lane[3] = {-1, -1, -1};
            for (size_t k = 0; k < plan.size(); k++) {
                const Launch& L = plan[k];
                cudaStream_t lane = lanes[k % n_lanes];
                const size_t off = (size_t)(L.v0 - c0) * frame_px * 3;
                DevFrame F{d_rgb + off, d_u8 + off, shard, n_shards, depth, L.b1 - L.b0, L.b0, nullptr, nullptr,
                           s->converge < 0 ? (int)s->has_branching_materials : s->converge, nullptr, 0};
                if (stream_scene) {  // one launch at a time on the render stream: one counter does
                    F.stream_counter = slot->d_stream_counter, F.stream_blocks = slot->sm_count * 6;
                    CUDA_TRY(cudaMemsetAsync(slot->d_stream_counter, 0, sizeof(unsigned), lane));
                }
                kernel_build(s->strict_fp, r.csg_sweep).views(r.scene, r.small, F, slot->d_views + L.v0, (int)(L.v1 - L.v0), slot->d_counters, lane);
                CUDA_TRY(cudaGetLastError());
                st.launches++;
                const int idx = launches_on[i];
                cudaEvent_t done = slice_event(slot, launches_on[i]);
                if (!done) return fail(RTC_ERR_CUDA, "cudaEventCreateWithFlags failed");
                CUDA_TRY(cudaEventRecord(done, lane));
                last_on_lane[k % n_lanes] = idx;
                if (copy_out) {
                    CUDA_TRY(cudaStreamWaitEvent(slot->copy_stream, done, 0));
                    if (int rc = cc.queue({slot, shard, L.b0, L.b1, (int)L.v0, (int)L.v1, d_rgb + off, d_u8 + off})) return rc;
                }
            }
            for (int l = 0; l < n_lanes; l++)
                if (l > 0 && last_on_lane[l] >= 0) CUDA_TRY(cudaStreamWaitEvent(slot->stream, slot->slice_done[last_on_lane[l]], 0));
        }
        if (int rc = cc.flush_pending()) return rc;
        if (c1 < n_views) {  // the next chunk reuses the arena (and the staging frames): it waits for this chunk's copies
            if (int rc = cc.drain()) return rc;
            for (int i = 0; i < ndev; i++) {
                DeviceSlot* slot = s->replicas[i].slot;
                CUDA_TRY(cudaSetDevice(slot->device));
                int& used = launches_on[i];
                cudaEvent_t e = slice_event(slot, used);
                if (!e) return fail(RTC_ERR_CUDA, "cudaEventCreateWithFlags failed");
                CUDA_TRY(cudaEventRecord(e, copy_out ? slot->copy_stream : slot->stream));
                chunk_copied[i] = e;
            }
        }
    }
    if (int rc = cc.drain()) return rc;
    for (int i = 0; i < ndev; i++) {
        DeviceSlot* slot = s->replicas[i].slot;
        CUDA_TRY(cudaSetDevice(slot->device));
        CUDA_TRY(cudaEventRecord(slot->ev1, slot->stream));
        CUDA_TRY(cudaMemcpyAsync(slot->h_counters, slot->d_counters, sizeof(DevCounters), cudaMemcpyDeviceToHost, slot->stream));
    }
    for (int i = 0; i < ndev; i++) {
        DeviceSlot* slot = s->replicas[i].slot;
        CUDA_TRY(cudaSetDevice(slot->device));
        CUDA_TRY(cudaStreamSynchronize(slot->stream));
        CUDA_TRY(cudaStreamSynchronize(slot->copy_stream));
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, slot->ev0, slot->ev1));
        st.kernel_ms = std::max(st.kernel_ms, (double)ms);
        uint64_t rows = 0;  // camera.rs:80-81, per view, of this device's bands
        for (int b = i; b < total_bands; b += n_shards)
            rows += (uint64_t)std::max(0, std::min<int>((int)s->height - 1, (b + 1) * kBandRows) - b * kBandRows);
        add_counters(st, *slot->h_counters, (uint64_t)n_views * rows * (uint64_t)(s->width - 1),
                     s->light_is_rect ? (uint64_t)s->u_steps * s->v_steps : 1);
    }
    st.total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    if (stats) *stats = st;
    if (st.capacity_overflows)
        return fail(RTC_ERR_CAPACITY, "CSG evaluation overflowed its buffers " + std::to_string(st.capacity_overflows) + " times");
    return 0;
}

}  // namespace

extern "C" {

const char* rtc_last_error(void) { return g_error.c_str(); }

int rtc_device_count(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) return fail(RTC_ERR_NO_DEVICE, std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e));
    return n;
}

int rtc_scene_create(RtcScene** out) {
    if (!out) return fail(RTC_ERR_INVALID, "null out pointer");
    *out = new RtcScene();
    if (const char* env = getenv("RTC_ADAPTIVE_ORDER")) (*out)->adaptive_order = atoi(env) != 0;  // tuning aids
    if (const char* env = getenv("RTC_SHADOW_FILTER")) (*out)->shadow_filter = atoi(env) != 0;
    if (const char* env = getenv("RTC_ORDER_MAX_WAVES")) (*out)->order_max_waves = atoi(env);
    if (const char* env = getenv("RTC_CONVERGE")) (*out)->converge = atoi(env);
    if (const char* env = getenv("RTC_STREAM")) (*out)->stream = atoi(env);
    if (const char* env = getenv("RTC_RENDER_SLICES")) (*out)->render_slices = std::max(1, std::min(64, atoi(env)));
    if (const char* env = getenv("RTC_WAVEFRONT")) (*out)->wavefront = atoi(env) != 0;
    if (const char* env = getenv("RTC_BVH_BUILDER")) (*out)->bvh_builder = atoi(env) != 0;
    return 0;
}
void rtc_scene_destroy(RtcScene* s) {
    if (!s) return;
    release(s);
    delete s;
}

int rtc_set_camera(RtcScene* s, uint32_t w, uint32_t h, float half_w, float half_h, float pixel_size, const float inv[16]) {
    if (!s || !inv) return fail(RTC_ERR_INVALID, "null argument");
    if (w == 0 || h == 0 || (uint64_t)w * h > (1ull << 31) / 3) return fail(RTC_ERR_INVALID, "bad canvas size");
    s->width = w, s->height = h, s->half_w = half_w, s->half_h = half_h, s->pixel_size = pixel_size;
    memcpy(s->cam_inv, inv, sizeof(s->cam_inv));
    s->have_camera = true;
    s->committed = false;
    return 0;
}
int rtc_set_primitives(RtcScene* s, uint32_t n, const RtcPrim* prims) {
    if (!s || (n && !prims)) return fail(RTC_ERR_INVALID, "null argument");
    if (n >= (1u << 27)) return fail(RTC_ERR_CAPACITY, "too many primitives");
    s->prims.resize(n);
    parallel_copy(s->prims.data(), prims, (size_t)n * sizeof(RtcPrim));
    s->committed = false;
    return 0;
}
int rtc_set_nodes(RtcScene* s, uint32_t n_nodes, const RtcNode* nodes, uint32_t n_refs, const int32_t* refs) {
    if (!s || (n_nodes && !nodes) || (n_refs && !refs)) return fail(RTC_ERR_INVALID, "null argument");
    s->nodes.resize(n_nodes);
    parallel_copy(s->nodes.data(), nodes, (size_t)n_nodes * sizeof(RtcNode));
    s->refs.assign(refs, refs + n_refs);
    s->committed = false;
    return 0;
}
int rtc_map_primitives(RtcScene* s, uint32_t n, RtcPrim** prims) {
    if (!s || !prims) return fail(RTC_ERR_INVALID, "null argument");
    if (n >= (1u << 27)) return fail(RTC_ERR_CAPACITY, "too many primitives");
    s->prims.resize(n);
    *prims = s->prims.data();
    s->committed = false;
    return 0;
}
int rtc_map_nodes(RtcScene* s, uint32_t n_nodes, uint32_t n_refs, RtcNode** nodes, int32_t** refs) {
    if (!s || !nodes || !refs) return fail(RTC_ERR_INVALID, "null argument");
    s->nodes.resize(n_nodes);
    s->refs.resize(n_refs);
    *nodes = s->nodes.data(), *refs = s->refs.data();
    s->committed = false;
    return 0;
}
int rtc_set_materials(RtcScene* s, uint32_t n, const RtcMaterial* m) {
    if (!s || (n && !m)) return fail(RTC_ERR_INVALID, "null argument");
    if (n >= (1u << 23)) return fail(RTC_ERR_CAPACITY, "too many materials");
    s->materials.assign(m, m + n);
    s->committed = false;
    return 0;
}
int rtc_set_patterns(RtcScene* s, uint32_t n, const RtcPattern* p, uint32_t n_uv, const RtcUvPattern* uv) {
    if (!s || (n && !p) || (n_uv && !uv)) return fail(RTC_ERR_INVALID, "null argument");
    s->patterns.assign(p, p + n);
    s->uvs.assign(uv, uv + n_uv);
    s->committed = false;
    return 0;
}
int rtc_set_textures(RtcScene* s, uint32_t n, const RtcTexture* t) {
    if (!s || (n && !t)) return fail(RTC_ERR_INVALID, "null argument");
    s->textures.clear();
    for (uint32_t i = 0; i < n; i++) {
        if (!t[i].rgb && t[i].width * t[i].height) return fail(RTC_ERR_INVALID, "texture without pixels");
        RtcScene::Texture x;
        x.width = t[i].width, x.height = t[i].height;
        x.rgb.assign(t[i].rgb, t[i].rgb + (size_t)t[i].width * t[i].height * 3);
        s->textures.push_back(std::move(x));
    }
    s->committed = false;
    return 0;
}
int rtc_set_point_light(RtcScene* s, const float position[3], const float intensity[3]) {
    if (!s || !position || !intensity) return fail(RTC_ERR_INVALID, "null argument");
    s->light_is_rect = false;
    memcpy(s->light_pos, position, 12);
    memcpy(s->light_rgb, intensity, 12);
    memset(s->corner, 0, 12), memset(s->u_cell, 0, 12), memset(s->v_cell, 0, 12);
    s->u_steps = s->v_steps = 1;
    s->jitter.clear();
    s->have_light = true;
    s->committed = false;
    return 0;
}
int rtc_set_rect_light(RtcScene* s, const float intensity[3], const float corner[3], const float u_cell[3], int32_t u_steps,
                       const float v_cell[3], int32_t v_steps, const float position[3], const float* table, uint32_t table_len,
                       uint64_t seed) {
    if (!s || !intensity || !corner || !u_cell || !v_cell || !position || (table_len && !table))
        return fail(RTC_ERR_INVALID, "null argument");
    if (u_steps < 1 || v_steps < 1 || (int64_t)u_steps * v_steps > (1 << 20)) return fail(RTC_ERR_INVALID, "bad light steps");
    // every intensity_at restarts the table (see the header): identical to the reference's carried-over cursor only
    // when each call consumes whole cycles
    if (table_len && (2 * (int64_t)u_steps * v_steps) % table_len != 0)
        return fail(RTC_ERR_INVALID, "jitter table length " + std::to_string(table_len) + " does not divide 2 * u_steps * v_steps = " +
                                         std::to_string(2 * (int64_t)u_steps * v_steps) +
                                         ": the reference's cyclic table would carry its cursor from one intensity_at to the next "
                                         "in render order, which a parallel render cannot reproduce");
    s->light_is_rect = true;
    memcpy(s->light_rgb, intensity, 12);
    memcpy(s->corner, corner, 12);
    memcpy(s->u_cell, u_cell, 12);
    memcpy(s->v_cell, v_cell, 12);
    memcpy(s->light_pos, position, 12);
    s->u_steps = u_steps, s->v_steps = v_steps;
    s->jitter.assign(table, table + table_len);
    s->seed = seed;
    s->have_light = true;
    s->committed = false;
    return 0;
}
int rtc_set_option(RtcScene* s, int32_t option, int64_t value) {
    if (!s) return fail(RTC_ERR_INVALID, "null scene");
    switch (option) {
        case RTC_OPT_FMA_CONTRACTION: s->strict_fp = value == 0; return 0;  // may change between renders
        case RTC_OPT_BVH_LEAF_SIZE:
            if (value < 0 || value > 16) return fail(RTC_ERR_INVALID, "leaf size must be in [1,16], or 0 = automatic");
            s->leaf_size = (int)value;
            s->committed = false;
            return 0;
        case RTC_OPT_ADAPTIVE_ORDER:
            s->adaptive_order = value != 0;
            return 0;
        case RTC_OPT_SHADOW_FILTER:  // may change between renders
            s->shadow_filter = value != 0;
            return 0;
        case RTC_OPT_RENDER_SLICES:
            if (value < 1 || value > 64) return fail(RTC_ERR_INVALID, "render slices must be in [1,64]");
            s->render_slices = (int)value;
            return 0;
        case RTC_OPT_BVH_BUILDER:
            if (value != 0 && value != 1) return fail(RTC_ERR_INVALID, "bvh builder: 0 (host binned SAH) or 1 (device LBVH)");
            s->bvh_builder = (int)value;
            s->committed = false;
            return 0;
        case RTC_OPT_WAVEFRONT:  // may change between renders
            s->wavefront = value != 0;
            return 0;
        case RTC_OPT_BVH_MIN_PRIMS:
            s->bvh_min_prims = (int)std::max<int64_t>(0, value);
            s->committed = false;
            return 0;
        case RTC_OPT_EXACT_GROUPS:
            if (value != 0 && value != 1) return fail(RTC_ERR_INVALID, "exact groups: 0 (default) or 1");
            s->exact_groups = (int)value;
            s->committed = false;
            return 0;
    }
    return fail(RTC_ERR_INVALID, "unknown option");
}

int rtc_scene_inspect(RtcScene* s, RtcCommitInfo* out) {
    if (!s || !out) return fail(RTC_ERR_INVALID, "null argument");
    if (!s->have_camera) return fail(RTC_ERR_STATE, "camera not set");
    if (!s->have_light) return fail(RTC_ERR_STATE, "World light should be set");
    const auto t0 = std::chrono::steady_clock::now();
    Flattened f;
    int rc = flatten(s, f);
    if (rc) return rc;
    memset(out, 0, sizeof(*out));
    out->host_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    out->n_positions = f.n_pos, out->n_bvh_nodes = (int)f.bvh.size(), out->n_linear = (int)f.linear.size();
    out->n_xforms = (int)f.xform.size() / 3, out->bvh_leaf_size = f.leaf_size, out->bvh_depth = f.bvh_depth;
    out->small_n = f.small.n, out->filter_ok = f.small.filter_ok, out->cell_masks = f.small.cell_masks;
    out->plane_cells = f.small.plane_cells, out->converge = s->has_branching_materials ? 1 : 0, out->lean = f.small.lean;
    out->tol_sphere = f.small.tol_sphere;
    out->exact_groups = s->exact_groups, out->loose_group_boxes = f.loose_group_boxes;
    out->light_ball[0] = f.small.light_ball.x, out->light_ball[1] = f.small.light_ball.y;
    out->light_ball[2] = f.small.light_ball.z, out->light_ball[3] = f.small.light_ball.w;
    // FNV-1a over the padding-free geometry arrays (the tree's two unused link lanes are skipped)
    uint64_t h = 1469598103934665603ull;
    auto mix = [&h](const void* p, size_t bytes) {
        const unsigned char* b = static_cast<const unsigned char*>(p);
        for (size_t i = 0; i < bytes; i++) h = (h ^ b[i]) * 1099511628211ull;
    };
    auto mix_vec = [&](const auto& v) { mix(v.data(), v.size() * sizeof(v[0])); };
    mix_vec(f.head), mix_vec(f.xform), mix_vec(f.tri), mix_vec(f.bound), mix_vec(f.rec), mix_vec(f.linear);
    for (const DevBvhNode& n : f.bvh) mix(&n, offsetof(DevBvhNode, d) + 3 * sizeof(int));
    const int tail[3] = {f.n_pos, f.bvh_root, f.leaf_size};
    mix(tail, sizeof(tail));
    out->digest = h;
    return 0;
}

int rtc_scene_commit(RtcScene* s, int32_t n_devices, const int32_t* device_ids) {
    if (!s) return fail(RTC_ERR_INVALID, "null scene");
    if (!s->have_camera) return fail(RTC_ERR_STATE, "camera not set");
    if (!s->have_light) return fail(RTC_ERR_STATE, "World light should be set");  // world.rs:66
    int visible = rtc_device_count();
    if (visible < 0) return visible;
    if (visible == 0) return fail(RTC_ERR_NO_DEVICE, "no CUDA device is visible; this library has no CPU fallback");
    if (n_devices == 0) n_devices = visible;
    if (n_devices < 0 || n_devices > visible) return fail(RTC_ERR_INVALID, "bad device count");
    release(s);
    Flattened f;
    int rc;
    if (s->bvh_builder == 1) {  // the tree of a big scene is built on the first device of the commit
        const int dev0 = device_ids ? device_ids[0] : 0;
        if (dev0 < 0 || dev0 >= visible) return fail(RTC_ERR_INVALID, "bad device id");
        DeviceSlot* slot = nullptr;
        if ((rc = lease_slot(dev0, &slot))) return rc;
        CUDA_TRY(cudaSetDevice(dev0));
        LbvhContext ctx{slot->stream, &slot->lbvh_scratch, &slot->lbvh_scratch_bytes, &slot->lbvh_pinned, &slot->lbvh_pinned_bytes};
        rc = flatten(s, f, lbvh_build, &ctx);
        return_slot(slot);
    } else {
        rc = flatten(s, f);
    }
    if (rc) return rc;
    s->replicas.resize(n_devices);
    s->replica_devices.resize(n_devices);
    for (int i = 0; i < n_devices; i++) {
        s->replica_devices[i] = device_ids ? device_ids[i] : i;
        if (s->replica_devices[i] < 0 || s->replica_devices[i] >= visible) {
            release(s);
            return fail(RTC_ERR_INVALID, "bad device id");
        }
        if ((rc = upload_replica(s, f, s->replicas[i], s->replica_devices[i]))) {
            release(s);
            return rc;
        }
    }
    s->reach = f.reach;
    s->committed = true;
    return 0;
}

int rtc_shard_bands(uint32_t height, int32_t shard, int32_t n_shards, uint32_t* first_rows) {
    static_assert(RTC_BAND_ROWS == kBandRows, "public band height must match the kernel tile height");
    if (n_shards < 1 || shard < 0 || shard >= n_shards) return fail(RTC_ERR_INVALID, "bad shard index");
    const int total = ((int)height + kBandRows - 1) / kBandRows;
    int n = 0;
    for (int b = shard; b < total; b += n_shards, n++)
        if (first_rows) first_rows[n] = (uint32_t)b * kBandRows;
    return n;
}

int rtc_render(RtcScene* s, int32_t depth, float* rgb, uint8_t* u8, RtcStats* stats) {
    return render_impl(s, depth, 0, 0, rgb, u8, stats, false);
}
int rtc_render_shard(RtcScene* s, int32_t depth, int32_t shard, int32_t n_shards, float* rgb, uint8_t* u8, RtcStats* stats) {
    if (n_shards < 1) return fail(RTC_ERR_INVALID, "n_shards must be >= 1");
    return render_impl(s, depth, shard, n_shards, rgb, u8, stats, false);
}
int rtc_render_detailed(RtcScene* s, int32_t depth, float* rgb, uint8_t* u8, RtcStats* stats) {
    return render_impl(s, depth, 0, 0, rgb, u8, stats, true);
}
int rtc_render_views(RtcScene* s, int32_t depth, uint32_t n_views, const RtcView* views, float* rgb, uint8_t* u8, RtcStats* stats) {
    return render_views_impl(s, depth, n_views, views, rgb, u8, stats);
}

int rtc_trace_rays(RtcScene* s, uint32_t n, const float* origins, const float* directions, int32_t depth, float* out_rgb,
                   float* out_t, int32_t* out_prim) {
    if (!s || !origins || !directions || !out_rgb) return fail(RTC_ERR_INVALID, "null argument");
    if (!s->committed) return fail(RTC_ERR_STATE, "rtc_trace_rays before rtc_scene_commit");
    if (depth < 0 || depth > kMaxFrames - 1) return fail(RTC_ERR_CAPACITY, "depth out of range");
    if (n == 0) return 0;
    Replica& rep = s->replicas[0];
    rep.small.filter_ok = rep.filter_eligible && s->shadow_filter;
    rep.small.cell_masks = rep.cell_masks_eligible && s->shadow_filter;
    rep.small.plane_cells = rep.plane_cells_eligible && rep.small.cell_masks;
    struct {
        int device;
        cudaStream_t stream;
        DevCounters* d_counters;
        DevScene& scene;
        SmallScene& small;
    } r{rep.slot->device, rep.slot->stream, rep.slot->d_counters, rep.scene, rep.small};
    CUDA_TRY(cudaSetDevice(r.device));
    struct Buffers {  // freed on every exit path
        float *o = nullptr, *d = nullptr, *rgb = nullptr, *t = nullptr;
        int* pos = nullptr;
        ~Buffers() { cudaFree(o), cudaFree(d), cudaFree(rgb), cudaFree(t), cudaFree(pos); }
    } b;
    size_t b3 = (size_t)n * 3 * sizeof(float);
    CUDA_TRY(cudaMalloc(&b.o, b3));
    CUDA_TRY(cudaMalloc(&b.d, b3));
    CUDA_TRY(cudaMalloc(&b.rgb, b3));
    CUDA_TRY(cudaMalloc(&b.t, (size_t)n * sizeof(float)));
    CUDA_TRY(cudaMalloc(&b.pos, (size_t)n * sizeof(int)));
    CUDA_TRY(cudaMemcpyAsync(b.o, origins, b3, cudaMemcpyHostToDevice, r.stream));
    CUDA_TRY(cudaMemcpyAsync(b.d, directions, b3, cudaMemcpyHostToDevice, r.stream));
    CUDA_TRY(cudaMemsetAsync(r.d_counters, 0, sizeof(DevCounters), r.stream));
    kernel_build(s->strict_fp, rep.csg_sweep).trace(r.scene, r.small, (int)n, b.o, b.d, depth, b.rgb, b.t, b.pos, r.d_counters, r.stream);
    CUDA_TRY(cudaGetLastError());
    std::vector<int> pos(n);
    CUDA_TRY(cudaMemcpyAsync(out_rgb, b.rgb, b3, cudaMemcpyDeviceToHost, r.stream));
    if (out_t) CUDA_TRY(cudaMemcpyAsync(out_t, b.t, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, r.stream));
    CUDA_TRY(cudaMemcpyAsync(pos.data(), b.pos, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, r.stream));
    unsigned long long overflows = 0;
    CUDA_TRY(cudaMemcpyAsync(&overflows, &r.d_counters->overflows, sizeof(overflows), cudaMemcpyDeviceToHost, r.stream));
    CUDA_TRY(cudaStreamSynchronize(r.stream));
    if (overflows) return fail(RTC_ERR_CAPACITY, "CSG evaluation overflowed its buffers " + std::to_string(overflows) + " times");
    if (out_prim)
        for (uint32_t i = 0; i < n; i++) out_prim[i] = pos[i] >= 0 ? s->pos_to_prim[pos[i]] : -1;
    return 0;
}

void* rtc_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocPortable) != cudaSuccess) {
        g_error = "cudaHostAlloc failed";
        return nullptr;
    }
    return p;
}
void rtc_host_free(void* p) {
    if (p) cudaFreeHost(p);
}
int rtc_host_register(void* ptr, size_t bytes) {
    CUDA_TRY(cudaHostRegister(ptr, bytes, cudaHostRegisterPortable));
    return 0;
}
int rtc_host_unregister(void* ptr) {
    CUDA_TRY(cudaHostUnregister(ptr));
    return 0;
}

int rtc_flush_l2(RtcScene* s) {
    if (!s || !s->committed) return fail(RTC_ERR_STATE, "scene not committed");
    for (Replica& rep : s->replicas) {
        DeviceSlot* r = rep.slot;
        CUDA_TRY(cudaSetDevice(r->device));
        if (!r->d_flush) {
            r->flush_bytes = 256u << 20;  // > 126 MB L2
            CUDA_TRY(cudaMalloc(&r->d_flush, r->flush_bytes));
        }
        CUDA_TRY(cudaMemsetAsync(r->d_flush, 0x5a, r->flush_bytes, r->stream));
        CUDA_TRY(cudaStreamSynchronize(r->stream));
    }
    return 0;
}

int rtc_measure_fp32_peak(int32_t device, double* tflops, double* sm_clock_mhz) {
    if (!tflops) return fail(RTC_ERR_INVALID, "null argument");
    CUDA_TRY(cudaSetDevice(device));
    int sms = 0, khz = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
    CUDA_TRY(cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, device));
    if (sm_clock_mhz) *sm_clock_mhz = khz / 1000.0;
    float* d = nullptr;
    CUDA_TRY(cudaMalloc(&d, 64));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    const int blocks = sms * 16, iters = 32768;
    double best = 0;
    for (int rep = 0; rep < 4; rep++) {
        CUDA_TRY(cudaEventRecord(e0, 0));
        fast::launch_fma_peak(d, blocks, iters, 0);
        CUDA_TRY(cudaEventRecord(e1, 0));
        CUDA_TRY(cudaEventSynchronize(e1));
        float ms = 0;
        CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
        double fl = (double)blocks * 256 * 8 * 2 * iters;
        if (rep > 0) best = std::max(best, fl / (ms * 1e-3) / 1e12);
    }
    *tflops = best;
    cudaEventDestroy(e0), cudaEventDestroy(e1), cudaFree(d);
    return 0;
}

}  // extern "C"
