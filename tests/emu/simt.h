// simt.h — TEST INFRASTRUCTURE ONLY: the SIMT execution model for the host harness of the kernels (emu_kernels.cpp).
// A launch runs every thread of a block as a host thread, so shared memory, barriers and warp collectives are used by
// as many threads as on the GPU and ThreadSanitizer sees their accesses.
//
// - Launch: blocks of blockDim.x host threads (threadIdx / blockIdx are thread_local).  Blocks run one after another,
//   because __shared__ arrays are statics and the dynamic block is one array; a kernel that uses neither may run a few
//   blocks at once (`concurrent`), so its global atomics and pixel counters really interleave.  Before every block the
//   shared memory, static and dynamic, is filled with a NaN pattern; under AddressSanitizer the dynamic block is poisoned
//   beyond the bytes the launch asked for.  Every thread is joined before launch() returns.
// - __syncthreads: a barrier of the block's threads that have not exited.
// - Warp collectives (__ballot_sync, __any_sync, __shfl_sync, __reduce_add_sync, __syncwarp): a rendezvous of the lanes
//   of the warp that have not exited.  The device code calls every collective converged, with the full mask; a lane
//   arriving with another mask, at another collective or at another call site, and a rendezvous that does not complete
//   within the timeout (a lane waits at a barrier or another collective), abort with where every lane of the warp was.
// - __activemask: all live lanes, the caller alone, or a seeded random set that includes the caller (emu_set_activemask).
// - atomicAdd / atomicMax: relaxed __atomic builtins, as CUDA's; clock64: a per-thread counter; __stcs: a plain store.
#pragma once
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <mutex>
#include <thread>
#include <vector>

#include "shim.h"

#if defined(__SANITIZE_ADDRESS__)
#include <sanitizer/asan_interface.h>
#endif

// static __shared__ arrays go to one section, so that the launch can fill all of them before a block
#undef __shared__
#define __shared__ static __attribute__((section("rtc_emu_shared")))
extern "C" char __start_rtc_emu_shared[] __attribute__((weak)), __stop_rtc_emu_shared[] __attribute__((weak));

namespace simt {
struct Dim {
    unsigned x = 0, y = 0, z = 0;
};
}  // namespace simt
static thread_local simt::Dim threadIdx, blockIdx;
static simt::Dim blockDim, gridDim;

namespace simt {
constexpr unsigned kFull = 0xffffffffu;
enum Op { kBallot, kAny, kShfl, kReduceAdd, kSyncWarp, kSyncThreads };
static const char* const kOpName[] = {"__ballot_sync", "__any_sync", "__shfl_sync", "__reduce_add_sync", "__syncwarp", "__syncthreads"};
static double g_timeout_s = 120.0;  // a rendezvous that has not completed by then never will

struct Where {
    int op = -1;  // -1 running, -2 exited
    const char* file = "";
    int line = 0;
};
struct Warp {
    unsigned live = 0, arrived = 0;  // lanes that have not exited; lanes waiting at the current rendezvous
    unsigned long long gen = 0;
    int op = -1;
    const char* file = "";
    int line = 0;
    unsigned val[32], arg[32], out[32];
    Where at[32];
    std::condition_variable cv;
};
struct Block {
    std::mutex m;
    int n = 0, live = 0, bar_arrived = 0;
    unsigned long long bar_gen = 0;
    std::condition_variable bar_cv;
    Warp warp[32];
    void reset(int threads) {
        n = live = threads, bar_arrived = 0;
        for (int w = 0; w * 32 < threads; w++) {
            const int lanes = threads - w * 32 < 32 ? threads - w * 32 : 32;
            warp[w].live = lanes == 32 ? kFull : (1u << lanes) - 1u;
            warp[w].arrived = 0, warp[w].op = -1;
            for (Where& a : warp[w].at) a = Where{};
        }
    }
};
struct Thread {
    Block* block;
    int tid;
};
static thread_local Thread t_self{nullptr, 0};

[[noreturn]] static void report(Warp& w, int warp, const char* what) {
    fprintf(stderr, "simt: %s (block %u,%u,%u warp %d)\n", what, blockIdx.x, blockIdx.y, blockIdx.z, warp);
    for (int l = 0; l < 32; l++) {
        const Where& a = w.at[l];
        if (!(w.live >> l & 1u) && a.op != -2) continue;
        fprintf(stderr, "  lane %2d: %s", l, a.op == -2 ? "exited" : a.op == -1 ? "running" : kOpName[a.op]);
        if (a.op >= 0) fprintf(stderr, " at %s:%d", a.file, a.line);
        fprintf(stderr, "\n");
    }
    fflush(stderr);
    abort();
}

static void complete(Warp& w) {
    unsigned ballot = 0, sum = 0;
    for (int l = 0; l < 32; l++)
        if (w.arrived >> l & 1u) ballot |= (w.val[l] != 0) << l, sum += w.val[l];
    for (int l = 0; l < 32; l++) {
        if (!(w.arrived >> l & 1u)) continue;
        switch (w.op) {
            case kBallot: w.out[l] = ballot; break;
            case kAny: w.out[l] = ballot != 0; break;
            case kReduceAdd: w.out[l] = sum; break;
            case kShfl: {
                const unsigned src = w.arg[l] & 31u;
                if (!(w.arrived >> src & 1u)) report(w, (int)(&w - t_self.block->warp), "__shfl_sync from a lane that is not there");
                w.out[l] = w.val[src];
                break;
            }
            default: w.out[l] = 0;
        }
        w.at[l] = Where{};
    }
    w.arrived = 0, w.op = -1, w.gen++;
    w.cv.notify_all();
}

template <class Done>
static void wait(std::unique_lock<std::mutex>& lk, std::condition_variable& cv, Done done, Warp& w, int warp, const char* what) {
    const auto deadline = std::chrono::steady_clock::now() + std::chrono::duration<double>(g_timeout_s);
    while (!done())
        if (cv.wait_until(lk, deadline) == std::cv_status::timeout && !done()) report(w, warp, what);
}

static unsigned collective(int op, unsigned mask, unsigned v, unsigned arg, const char* file, int line) {
    Block& b = *t_self.block;
    const int warp = t_self.tid >> 5, lane = t_self.tid & 31;
    Warp& w = b.warp[warp];
    std::unique_lock<std::mutex> lk(b.m);
    w.at[lane] = Where{op, file, line};
    if (mask != kFull) report(w, warp, "a warp collective with a partial mask");
    if (w.arrived == 0) {
        w.op = op, w.file = file, w.line = line;
    } else if (w.op != op || w.file != file || w.line != line) {
        if (w.op != op || strcmp(w.file, file) != 0 || w.line != line) report(w, warp, "lanes of a warp at different collectives");
    }
    w.val[lane] = v, w.arg[lane] = arg, w.arrived |= 1u << lane;
    if (w.arrived == w.live) {
        complete(w);
        return w.out[lane];
    }
    const unsigned long long gen = w.gen;
    wait(lk, w.cv, [&] { return w.gen != gen; }, w, warp, "a warp collective that does not complete");
    return w.out[lane];
}

static void syncthreads(const char* file, int line) {
    Block& b = *t_self.block;
    const int warp = t_self.tid >> 5, lane = t_self.tid & 31;
    std::unique_lock<std::mutex> lk(b.m);
    b.warp[warp].at[lane] = Where{kSyncThreads, file, line};
    if (++b.bar_arrived == b.live) {
        b.bar_arrived = 0, b.bar_gen++;
        b.bar_cv.notify_all();
    } else {
        const unsigned long long gen = b.bar_gen;
        wait(lk, b.bar_cv, [&] { return b.bar_gen != gen; }, b.warp[warp], warp, "a __syncthreads that does not complete");
    }
    b.warp[warp].at[lane] = Where{};
}

// the thread leaves the kernel: barriers and rendezvous wait for it no longer
static void exit_thread() {
    Block& b = *t_self.block;
    const int warp = t_self.tid >> 5, lane = t_self.tid & 31;
    std::lock_guard<std::mutex> lk(b.m);
    Warp& w = b.warp[warp];
    w.live &= ~(1u << lane), w.at[lane].op = -2;
    if (w.arrived && w.arrived == w.live) complete(w);
    if (--b.live > 0 && b.bar_arrived == b.live) {
        b.bar_arrived = 0, b.bar_gen++;
        b.bar_cv.notify_all();
    }
}

// __activemask: 0 every live lane, 1 the caller alone, 2 a seeded random set of live lanes that includes the caller
static int g_activemask_mode = 0;
static unsigned g_activemask_seed = 1;
static unsigned activemask() {
    const int lane = t_self.tid & 31;
    if (g_activemask_mode == 1) return 1u << lane;
    unsigned live;
    {
        std::lock_guard<std::mutex> lk(t_self.block->m);
        live = t_self.block->warp[t_self.tid >> 5].live;
    }
    if (g_activemask_mode == 0) return live;
    static thread_local unsigned x = 0;
    if (x == 0) x = g_activemask_seed * 2246822519u + (unsigned)t_self.tid * 3266489917u + 1u;
    x ^= x << 13, x ^= x >> 17, x ^= x << 5;
    return (live & x) | 1u << lane;
}

// The dynamic shared-memory block of every launch and its capacity
static float4* g_smem = nullptr;
static size_t g_smem_cap = 0;

static void fill_shared(size_t dyn_bytes) {
    const uint32_t nan = 0x7FBADBADu;  // a signalling-looking NaN no kernel writes
    for (char* p = __start_rtc_emu_shared; p && p + 4 <= __stop_rtc_emu_shared; p += 4) memcpy(p, &nan, 4);
    if (!g_smem) return;
#if defined(__SANITIZE_ADDRESS__)
    __asan_unpoison_memory_region(g_smem, g_smem_cap);
#endif
    for (size_t i = 0; i < g_smem_cap / 4; i++) memcpy(reinterpret_cast<char*>(g_smem) + 4 * i, &nan, 4);
#if defined(__SANITIZE_ADDRESS__)
    if (dyn_bytes < g_smem_cap) __asan_poison_memory_region(reinterpret_cast<char*>(g_smem) + dyn_bytes, g_smem_cap - dyn_bytes);
#else
    (void)dyn_bytes;
#endif
}

// A barrier of the host threads that run one sequence of blocks (between blocks, outside the kernel's view)
struct Gate {
    std::mutex m;
    std::condition_variable cv;
    int n, arrived = 0;
    unsigned long long gen = 0;
    explicit Gate(int n_) : n(n_) {}
    void arrive() {
        std::unique_lock<std::mutex> lk(m);
        if (++arrived == n) {
            arrived = 0, gen++;
            cv.notify_all();
            return;
        }
        const unsigned long long g = gen;
        cv.wait(lk, [&] { return gen != g; });
    }
};

// Runs body() as every thread of a grid.x * grid.y * grid.z grid of `threads`-thread blocks, `concurrent` blocks at a
// time (1 for kernels with shared memory); dyn_bytes: the dynamic shared memory the launch asks for.
template <class Body>
void launch(Dim grid, int threads, size_t dyn_bytes, int concurrent, Body body) {
    if (dyn_bytes > g_smem_cap || threads < 1 || threads > 1024 || concurrent < 1) abort();
    const unsigned long long n_blocks = (unsigned long long)grid.x * grid.y * grid.z;
    if (n_blocks == 0) return;
    if ((unsigned long long)concurrent > n_blocks) concurrent = (int)n_blocks;
    blockDim = Dim{(unsigned)threads, 1, 1}, gridDim = grid;
    std::vector<Block> blocks((size_t)concurrent);
    std::vector<Gate*> gates;
    for (int g = 0; g < concurrent; g++) gates.push_back(new Gate(threads));
    if (concurrent == 1) fill_shared(dyn_bytes);
    std::vector<std::thread> pool;
    for (int g = 0; g < concurrent; g++)
        for (int t = 0; t < threads; t++)
            pool.emplace_back([&, g, t] {
                Block& b = blocks[(size_t)g];
                for (unsigned long long id = (unsigned long long)g; id < n_blocks; id += (unsigned long long)concurrent) {
                    if (t == 0) {
                        b.reset(threads);
                        if (concurrent == 1 && id > 0) fill_shared(dyn_bytes);
                    }
                    gates[(size_t)g]->arrive();  // the block is set up
                    t_self = Thread{&b, t};
                    threadIdx = Dim{(unsigned)t, 0, 0};
                    blockIdx = Dim{(unsigned)(id % grid.x), (unsigned)(id / grid.x % grid.y), (unsigned)(id / grid.x / grid.y)};
                    body();
                    exit_thread();
                    gates[(size_t)g]->arrive();  // every thread has left the block
                }
            });
    for (std::thread& th : pool) th.join();
    for (Gate* g : gates) delete g;
#if defined(__SANITIZE_ADDRESS__)
    if (g_smem) __asan_unpoison_memory_region(g_smem, g_smem_cap);
#endif
}
}  // namespace simt

template <typename T>
static inline T simt_shfl(unsigned mask, T v, int src, const char* file, int line) {
    static_assert(sizeof(T) == 4, "32-bit shuffles only");
    unsigned u, r;
    memcpy(&u, &v, 4);
    r = simt::collective(simt::kShfl, mask, u, (unsigned)src, file, line);
    T out;
    memcpy(&out, &r, 4);
    return out;
}
#define __ballot_sync(mask, p) simt::collective(simt::kBallot, (mask), (p) ? 1u : 0u, 0u, __FILE__, __LINE__)
#define __any_sync(mask, p) ((int)simt::collective(simt::kAny, (mask), (p) ? 1u : 0u, 0u, __FILE__, __LINE__))
#define __reduce_add_sync(mask, v) simt::collective(simt::kReduceAdd, (mask), (unsigned)(v), 0u, __FILE__, __LINE__)
#define __shfl_sync(mask, v, src) simt_shfl((mask), (v), (src), __FILE__, __LINE__)
#define __syncwarp(...) simt_syncwarp(__FILE__, __LINE__ __VA_OPT__(, ) __VA_ARGS__)
#define __syncthreads() simt::syncthreads(__FILE__, __LINE__)
static inline void simt_syncwarp(const char* file, int line, unsigned mask = simt::kFull) {
    simt::collective(simt::kSyncWarp, mask, 0u, 0u, file, line);
}
static inline unsigned __activemask() { return simt::activemask(); }

static inline unsigned atomicAdd(unsigned* p, unsigned v) { return __atomic_fetch_add(p, v, __ATOMIC_RELAXED); }
static inline int atomicAdd(int* p, int v) { return __atomic_fetch_add(p, v, __ATOMIC_RELAXED); }
static inline unsigned long long atomicAdd(unsigned long long* p, unsigned long long v) { return __atomic_fetch_add(p, v, __ATOMIC_RELAXED); }
static inline unsigned atomicMax(unsigned* p, unsigned v) {
    unsigned old = __atomic_load_n(p, __ATOMIC_RELAXED);
    while (old < v && !__atomic_compare_exchange_n(p, &old, v, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {
    }
    return old;
}
static inline long long clock64() {
    static thread_local long long c = 0;
    return c += 1000;
}
template <typename T>
static inline void __stcs(T* p, const T& v) {
    *p = v;
}
