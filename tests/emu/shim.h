// shim.h — TEST INFRASTRUCTURE ONLY: the CUDA keywords and the thread-independent intrinsics of the device code, for the
// host harnesses of tests/emu (emu_nearest.cpp, emu_color.cpp, emu_kernels.cpp).  Include after rtc_internal.h (whose CUDA
// headers define the keywords for the host compiler) and before the device code.  Warp collectives, barriers, atomics and
// the launch model are the harness's: one lane per "warp" in emu_color.cpp, real 32-lane warps in simt.h.
#pragma once
#include <math.h>
#include <string.h>

#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstring>

#undef __device__
#undef __forceinline__
#undef __noinline__
#undef __shared__
#undef __global__
#undef __launch_bounds__
#undef __grid_constant__
#define __device__
#define __forceinline__ inline
#define __noinline__ __attribute__((noinline))
#define __global__
#define __launch_bounds__(...)
#define __grid_constant__
#define RTC_EXTERN_SHARED extern  // dev_small.cuh: the dynamic block is the harness's array rtc::emu::rtc_smem

template <typename T>
static inline T __ldg(const T* p) {
    return *p;
}
static inline float __fmaf_rn(float a, float b, float c) { return std::fmaf(a, b, c); }
static inline int __float_as_int(float f) {
    int i;
    memcpy(&i, &f, 4);
    return i;
}
static inline float __int_as_float(int i) {
    float f;
    memcpy(&f, &i, 4);
    return f;
}
static inline unsigned __float_as_uint(float f) {
    unsigned i;
    memcpy(&i, &f, 4);
    return i;
}
static inline float __uint_as_float(unsigned i) {
    float f;
    memcpy(&f, &i, 4);
    return f;
}
// cvt.rzi.s32.f32 / cvt.rzi.u32.f32 saturate to the destination's range and turn NaN into 0 (the oracle's sat_i32 does
// the same).  A plain C cast is undefined there, and x86 gives INT_MIN for every out-of-range value: even_floor would
// then call 2^31 and beyond even.
static inline int __float2int_rz(float f) {
    if (f != f) return 0;
    if (f >= 2147483648.0f) return 2147483647;
    if (f <= -2147483648.0f) return (-2147483647 - 1);
    return (int)f;
}
static inline unsigned __float2uint_rz(float f) {
    if (!(f > 0.0f)) return 0u;  // NaN and everything at or below zero
    if (f >= 4294967296.0f) return 4294967295u;
    return (unsigned)f;
}
static inline int min(int a, int b) { return a < b ? a : b; }
static inline unsigned min(unsigned a, unsigned b) { return a < b ? a : b; }
static inline long long min(long long a, long long b) { return a < b ? a : b; }
static inline int max(int a, int b) { return a > b ? a : b; }
static inline unsigned max(unsigned a, unsigned b) { return a > b ? a : b; }
[[noreturn]] static inline void __trap() { abort(); }
static inline int __popc(unsigned v) { return __builtin_popcount(v); }
static inline int __ffs(int v) { return __builtin_ffs(v); }

// rsqrtf and __fdividef.  Mode 0: correctly rounded (the default).  Otherwise within the envelopes the CUDA
// programming guide documents for them (2 ulp; __fdividef also 0 for 2^126 < |y| < 2^128): 1 the rounded value 2 ulp
// lower, 2 2 ulp higher, 3 a seeded pseudo-random 0-2 ulp either way.  The shadow filter's bounds must cover these, so
// frames do not depend on the mode.  rcp_estimate (dev_math.cuh) is host-only 1 / m here in every mode.
static int g_approx_mode = 0;
static unsigned g_approx_seed = 1;
extern "C" void emu_set_approx(int mode, unsigned seed) { g_approx_mode = mode, g_approx_seed = seed ? seed : 1; }
static inline float emu_ulps(float v, int n) {
    for (; n > 0; n--) v = nextafterf(v, INFINITY);
    for (; n < 0; n++) v = nextafterf(v, -INFINITY);
    return v;
}
static inline float emu_approx(float v) {
    if (g_approx_mode == 0 || !std::isfinite(v) || v == 0.0f) return v;
    if (g_approx_mode == 1) return emu_ulps(v, -2);
    if (g_approx_mode == 2) return emu_ulps(v, 2);
    static thread_local unsigned x = 0;
    if (x == 0) x = g_approx_seed * 2654435761u + (unsigned)(uintptr_t)&x;  // per thread
    x ^= x << 13, x ^= x >> 17, x ^= x << 5;
    return emu_ulps(v, (int)(x % 5u) - 2);
}
static inline float rsqrtf(float a) { return emu_approx(1.0f / std::sqrt(a)); }
static inline float __fdividef(float a, float b) {
    if (g_approx_mode != 0 && std::fabs(b) > 0x1p126f && std::isfinite(b)) return 0.0f;
    return emu_approx(a / b);
}
