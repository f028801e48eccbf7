// Shared device/host helpers for the oflib_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <atomic>

#include "../../include/oflib_b200.h"

namespace ofk {

// ------------------------------------------------------------------------------------------------ host-side plumbing
void set_error(const char* fmt, ...);
extern std::atomic<unsigned long long> g_launches;
extern std::atomic<unsigned long long> g_paths[4];   // see ofk_rt_path_count
extern std::atomic<unsigned long long> g_consistency_paths[2];   // ofk_consistency: TMA kernel, rows kernel
int staged_copy(void* dst, const void* src, size_t bytes, bool to_device, cudaStream_t user);   // staging.cu
unsigned long long c3_ws_mixed_count();               // combine3_ws.cu
unsigned long long warp_ws_mixed_count();             // warp_t_ws.cu
unsigned long long forward_s_stat(int which);         // forward_s.cu

#define OFK_CHECK_ARG(cond, ...)                \
    do {                                        \
        if (!(cond)) {                          \
            ofk::set_error(__VA_ARGS__);        \
            return OFK_EINVAL;                  \
        }                                       \
    } while (0)

#define OFK_CUDA(call)                                                                       \
    do {                                                                                     \
        cudaError_t e_ = (call);                                                             \
        if (e_ != cudaSuccess) {                                                             \
            ofk::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, \
                           __LINE__);                                                        \
            return OFK_ECUDA;                                                                \
        }                                                                                    \
    } while (0)

// every kernel launch goes through this so launches are counted and launch errors surface immediately
#define OFK_LAUNCHED()                                                                          \
    do {                                                                                        \
        ofk::g_launches.fetch_add(1, std::memory_order_relaxed);                                \
        cudaError_t e_ = cudaPeekAtLastError();                                                 \
        if (e_ != cudaSuccess) {                                                                \
            ofk::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(e_), __FILE__, \
                           __LINE__);                                                           \
            return OFK_ECUDA;                                                                   \
        }                                                                                       \
    } while (0)

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static inline cudaStream_t as_stream(ofk_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

int sm_count();  // cached multiprocessor count of the current device

// ------------------------------------------------------------------------------------------------ device helpers
#ifdef __CUDACC__

// OpenCV's remap coordinate quantisation (INTER_BITS = 5): X float32 -> integer tap + 5-bit fraction.
// cvRound == round-half-even == cvt.rni; the integer part saturates to int16 like saturate_cast<short>.
struct QCoord {
    int i;  // integer tap (left / top)
    int f;  // fraction in 1/32
};
__device__ __forceinline__ QCoord quantise(float X) {
    int s = __float2int_rn(X * 32.0f);
    QCoord q;
    q.i = max(-32768, min(32767, s >> 5));
    q.f = s & 31;
    return q;
}

// Same quantisation without the XU-pipe conversion: adding 1.5*2^23 rounds X*32 to an integer (round-half-even, one
// rounding because X*32 is exact) in the mantissa. Valid for |X| < 2^16; callers test that and fall back to quantise().
#define OFK_FAST_COORD_LIMIT 65536.0f
__device__ __forceinline__ QCoord quantise_fast(float X) {
    const int bits = __float_as_int(__fmaf_rn(X, 32.0f, 12582912.0f)) - 0x4B400000;
    QCoord q;
    q.i = bits >> 5;
    q.f = bits & 31;
    return q;
}

// "every tap with a non-zero weight lies inside the frame" for the sampling position (X, Y): the valid-area test of
// valid_geom_vec4 (warp_t.cu) and of ofk_track's status (track_device.cuh).
__device__ __forceinline__ unsigned strict_in_frame(float X, float Y, int H, int W) {
    // clamping keeps the fast quantiser in range; a clamped coordinate is an integer outside [0, W-1] -> invalid
    X = fminf(fmaxf(X, -2.0f), (float)(W + 1));
    Y = fminf(fmaxf(Y, -2.0f), (float)(H + 1));
    const QCoord qx = quantise_fast(X), qy = quantise_fast(Y);
    const bool ok = qx.i >= 0 && qy.i >= 0 && (qx.i + 1 < W || (qx.f == 0 && qx.i < W)) &&
                    (qy.i + 1 < H || (qy.f == 0 && qy.i < H));
    return ok ? 1u : 0u;
}

// Absolute sampling coordinate: float32(sign*flow) + float32(grid), one rounding, as numpy's in-place
// `field *= -1; field += arange` (utils.py:233-235).
__device__ __forceinline__ float sample_coord(float flow_component, float sign, int grid) {
    return __fadd_rn(sign * flow_component, static_cast<float>(grid));
}

// The four bilinear weights in units of 1/1024 (exact integers).
struct QWeights {
    int w00, w01, w10, w11;
};
__device__ __forceinline__ QWeights qweights(int a, int b) {
    QWeights w;
    w.w00 = (32 - a) * (32 - b);
    w.w01 = a * (32 - b);
    w.w10 = (32 - a) * b;
    w.w11 = a * b;
    return w;
}

__device__ __forceinline__ bool mask_rule_pass(int S, int rule) {
    return rule == OFK_RULE_STRICT ? (S == 1024) : (rule == OFK_RULE_GT_HALF ? (S > 512) : (S >= 512));
}

// streaming (read-once / write-once) accesses: keep them out of L1 so the gathered payload stays resident
__device__ __forceinline__ float4 ld_stream_f4(const float4* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}
__device__ __forceinline__ float2 ld_stream_f2(const float2* p) {
    float2 v;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ uint32_t ld_stream_u32(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ void st_stream_f4(float4* p, float4 v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
                 "f"(v.w)
                 : "memory");
}
__device__ __forceinline__ void st_stream_u32(uint32_t* p, uint32_t v) {
    asm volatile("st.global.L1::no_allocate.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

#endif  // __CUDACC__

}  // namespace ofk
