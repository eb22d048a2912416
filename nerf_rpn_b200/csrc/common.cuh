// Shared host/device helpers for libnerf_rpn_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <atomic>
#include "../../include/nerf_rpn_b200.h"

namespace nrpn {

extern thread_local int g_last_cuda_error;
extern std::atomic<unsigned long long> g_launch_count;

inline int cuda_fail(cudaError_t e) {
    g_last_cuda_error = (int)e;
    return NRPN_ERR_CUDA;
}

// Every kernel launch goes through this so that nrpn_launch_count() is an honest count.
#define NRPN_LAUNCH_CHECK()                                         \
    do {                                                            \
        ::nrpn::g_launch_count.fetch_add(1, std::memory_order_relaxed); \
        cudaError_t e__ = cudaGetLastError();                       \
        if (e__ != cudaSuccess) return ::nrpn::cuda_fail(e__);      \
    } while (0)

#define NRPN_CUDA_TRY(expr)                                         \
    do {                                                            \
        cudaError_t e__ = (expr);                                   \
        if (e__ != cudaSuccess) return ::nrpn::cuda_fail(e__);      \
    } while (0)

inline int num_sms() {
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return 148;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) sms = 148;
    }
    return sms;
}

// 16-bit activation format of a launch: 0 = bf16 (default, BASELINE config 2), 1 = fp16 (same tensor-core rate, 11-bit
// significand: the higher-parity mode of DESIGN.md section 4).  Storage is 2 bytes either way; only conversions differ.
#ifdef __CUDACC__
__device__ __forceinline__ uint32_t pack_act2(float a, float b, int fp16) {
    if (fp16) { __half2 v = __floats2half2_rn(a, b); return *reinterpret_cast<uint32_t*>(&v); }
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float load_act(const __nv_bfloat16* p, int fp16) {
    return fp16 ? __half2float(*reinterpret_cast<const __half*>(p)) : __bfloat162float(*p);
}
__device__ __forceinline__ void store_act(__nv_bfloat16* p, float v, int fp16) {
    if (fp16) *reinterpret_cast<__half*>(p) = __float2half_rn(v);
    else *p = __float2bfloat16(v);
}
__device__ __forceinline__ float2 unpack_act2(uint32_t u, int fp16) {
    if (fp16) return __half22float2(*reinterpret_cast<const __half2*>(&u));
    return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u));
}
// max that propagates NaN, as torch's max-pooling does (fmaxf drops it): one max.NaN instruction
__device__ __forceinline__ float max_nan(float a, float b) {
    float r;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}
#endif

template <typename T>
__host__ __device__ inline T ceil_div(T a, T b) { return (a + b - 1) / b; }

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Monotone map float -> uint32 (larger float => larger key); -0 < +0, NaNs sort to the ends.
__host__ __device__ inline uint32_t float_to_ordered(float f) {
#ifdef __CUDA_ARCH__
    uint32_t u = __float_as_uint(f);
#else
    union { float f; uint32_t u; } c; c.f = f; uint32_t u = c.u;
#endif
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

}  // namespace nrpn
