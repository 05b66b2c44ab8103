// Shared helpers for the mvoc_b200 CUDA kernels (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/mvoc_b200.h"

namespace mvoc {

// Error text for mvoc_last_error(); thread-local, set by the failing call.
void set_error(const char* fmt, ...);
int check_launch(const char* what);

#define MVOC_REQUIRE(cond, code, ...)      \
    do {                                   \
        if (!(cond)) {                     \
            ::mvoc::set_error(__VA_ARGS__); \
            return (code);                 \
        }                                  \
    } while (0)

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize, bytes) on `kernel`, once per device: `done` is the call site's
// record of the devices already set.  MVOC_ERR_CUDA with `what` in the message on failure.
int set_max_dynamic_smem(const void* kernel, int bytes, bool (&done)[64], const char* what);

// ---- 4-D 16-bit TMA tensor maps (tensormap.cu) ----------------------------
// dims and box innermost first, element strides of dims 1..3, zero fill out of bounds.  The stride of a dimension of
// extent 1 is ignored and the packed value (previous stride x previous extent) is encoded; the stride of any other
// dimension must be a positive multiple of 8 elements (16 bytes), else MVOC_ERR_UNSUPPORTED.  Messages name `what`
// (the entry point) and `operand`.  check_map4 applies that rule without touching the driver.  `elem_stride` is the
// TMA traversal stride of dims 1 and 2: 1 loads every element of the box; 2 loads every other one, so a box of
// {c, 2 b1, 2 b2, b3} delivers c x b1 x b2 x b3 elements (the input rows of a stride-2 convolution).
int check_map4(const int64_t (&dims)[4], const int64_t (&str)[3], const char* what, const char* operand);
int make_map4(CUtensorMap* m, const void* base, int dtype, const int64_t (&dims)[4], const int64_t (&str)[3],
              const int (&box)[4], int elem_stride, CUtensorMapSwizzle swz, const char* what, const char* operand);

// Operands of the tensor-core attention entry points (attn_tc.cu): q, k, v, o non-null and 16-byte aligned, dtype
// bf16 / fp16, D == head_dim, the n_st strides non-negative multiples of 8 elements.
int check_attn_operands(const void* q, const void* k, const void* v, const void* o, int dtype, int D, int head_dim,
                        const int64_t* st, int n_st, const char* what);

inline int num_sms() {
    static int n = 0;
    if (n == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
    }
    return n;
}

// ---- storage <-> fp32 ----------------------------------------------------
template <typename T> struct Elem;
template <> struct Elem<__nv_bfloat16> {
    static __device__ __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
    static __device__ __forceinline__ __nv_bfloat16 from_f(float v) { return __float2bfloat16_rn(v); }
};
template <> struct Elem<__half> {
    static __device__ __forceinline__ float to_f(__half v) { return __half2float(v); }
    static __device__ __forceinline__ __half from_f(float v) { return __float2half_rn(v); }
};
template <> struct Elem<float> {
    static __device__ __forceinline__ float to_f(float v) { return v; }
    static __device__ __forceinline__ float from_f(float v) { return v; }
};

// 16-byte vector of 8 16-bit elements.
struct __align__(16) Vec16 {
    uint32_t w[4];
};

template <typename T>
__device__ __forceinline__ void unpack8(const Vec16& v, float (&f)[8]) {
    const T* p = reinterpret_cast<const T*>(&v);
#pragma unroll
    for (int i = 0; i < 8; ++i) f[i] = Elem<T>::to_f(p[i]);
}
// Two fp32 values rounded to nearest into a 16-bit pair, `lo` in the low half.
template <typename T> __device__ __forceinline__ uint32_t pack2_rn(float lo, float hi);
template <> __device__ __forceinline__ uint32_t pack2_rn<__nv_bfloat16>(float lo, float hi) {
    __nv_bfloat162 b = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&b);
}
template <> __device__ __forceinline__ uint32_t pack2_rn<__half>(float lo, float hi) {
    __half2 b = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&b);
}
template <typename T>
__device__ __forceinline__ Vec16 pack8(const float (&f)[8]) {
    Vec16 v;
    T* p = reinterpret_cast<T*>(&v);
#pragma unroll
    for (int i = 0; i < 8; ++i) p[i] = Elem<T>::from_f(f[i]);
    return v;
}

// Streaming 128-bit global accesses (data touched once: keep it out of L1).
__device__ __forceinline__ Vec16 ld_stream16(const void* p) {
    Vec16 v;
    // not .nc: several kernels update the same tensor in place
    asm volatile("ld.global.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.w[0]), "=r"(v.w[1]), "=r"(v.w[2]), "=r"(v.w[3])
                 : "l"(p));
    return v;
}
__device__ __forceinline__ Vec16 ld_global16(const void* p) {
    Vec16 v;
    asm volatile("ld.global.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(v.w[0]), "=r"(v.w[1]), "=r"(v.w[2]), "=r"(v.w[3])
                 : "l"(p));
    return v;
}
__device__ __forceinline__ void st_stream16(void* p, const Vec16& v) {
    asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.w[0]),
                 "r"(v.w[1]), "r"(v.w[2]), "r"(v.w[3])
                 : "memory");
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// SiLU with ONE MUFU op per element: x * sigmoid(x) = 0.5 x (1 + tanh(x / 2)); tanh.approx has an absolute
// error of ~2^-11, far below the bf16 rounding of the result.
__device__ __forceinline__ float silu_f(float x) {
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * x));
    return 0.5f * x * (1.0f + t);
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

}  // namespace mvoc
