// Shared helpers for libhicgat_sm100.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "hicgat.h"

namespace hicgat {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);

#define HICGAT_REQUIRE(cond, ...)        \
    do {                                 \
        if (!(cond)) {                   \
            hicgat::set_error(__VA_ARGS__); \
            return HICGAT_ERR_INVALID;   \
        }                                \
    } while (0)

#define HICGAT_CHECK_LAUNCH(name)                                                   \
    do {                                                                            \
        cudaError_t e__ = cudaGetLastError();                                       \
        if (e__ != cudaSuccess) {                                                   \
            hicgat::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__)); \
            return HICGAT_ERR_CUDA;                                                 \
        }                                                                           \
        hicgat::count_launch();                                                     \
    } while (0)

#define HICGAT_CUDA(call)                                                          \
    do {                                                                           \
        cudaError_t e__ = (call);                                                  \
        if (e__ != cudaSuccess) {                                                  \
            hicgat::set_error("%s failed: %s", #call, cudaGetErrorString(e__));    \
            return HICGAT_ERR_CUDA;                                                \
        }                                                                          \
    } while (0)

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// (heads, channels per head) of GATConv that both message-passing paths take: exactly the instantiations of
// HICGAT_DISPATCH_HQ in conv.cu, whose logit kernel the dense path shares.  H*C/128 is 1, 2, 4 or 8.
static inline bool gat_shape_supported(int H, int C) {
    return (H == 1 && (C == 128 || C == 256 || C == 512)) || (H == 2 && (C == 128 || C == 256 || C == 512)) ||
           (H == 4 && (C == 128 || C == 256));
}

// ---------------------------------------------------------------- packed fp32x2 (Blackwell FADD2/FMUL2/FFMA2)
typedef unsigned long long f2;  // two f32 in one 64-bit register pair

__device__ __forceinline__ f2 f2_pack(float lo, float hi) {
    f2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void f2_unpack(f2 v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f2 f2_add(f2 a, f2 b) {
    f2 r;
    asm("add.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f2 f2_sub(f2 a, f2 b) {
    f2 r;
    asm("sub.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f2 f2_mul(f2 a, f2 b) {
    f2 r;
    asm("mul.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f2 f2_fma(f2 a, f2 b, f2 c) {
    f2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ float f2_hsum(f2 v) {
    float a, b;
    f2_unpack(v, a, b);
    return a + b;
}
__device__ __forceinline__ float rsqrt_approx(float x) {
    float r;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// streaming 128-bit load: read-only path, do not allocate in L1 (each target element is used once)
__device__ __forceinline__ float4 ldg_stream_f4(const float* p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::128B.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

}  // namespace hicgat
