// common.cuh -- shared helpers for libmergerec_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/mergerec_b200.h"

#ifndef __CUDA_ARCH_LIST__
#define __CUDA_ARCH_LIST__ 1000
#endif

namespace mr {

void set_error(const char* fmt, ...);
int sm_count();

#define MR_REQUIRE(cond, ...)               \
    do {                                    \
        if (!(cond)) {                      \
            ::mr::set_error(__VA_ARGS__);   \
            return MR_ERR_INVALID_ARG;      \
        }                                   \
    } while (0)

#define MR_CUDA_LAUNCH_CHECK(name)                                              \
    do {                                                                        \
        cudaError_t e__ = cudaGetLastError();                                   \
        if (e__ != cudaSuccess) {                                               \
            ::mr::set_error("%s: %s", name, cudaGetErrorString(e__));           \
            return (int)e__;                                                    \
        }                                                                       \
    } while (0)

// x rounded to TF32 (nearest, ties away): the hi part of the 3xTF32 split, and of x - hi its lo part
__device__ __forceinline__ float rna_tf32(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

// ---- streaming 128-bit global accesses (read-once data: keep it out of L1) --------------------
__device__ __forceinline__ float4 ldg_stream4(const float* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ float ldg_stream1(const float* p) {
    float r;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream4(float* p, float4 v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y),
                 "f"(v.z), "f"(v.w)
                 : "memory");
}

__device__ __forceinline__ bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
inline bool host_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// ---- torch.sum(dim=0) order over K addends (reference: ATen CPU reduce; SURVEY.md 7.3-1) ------
// sequential: s = 0; s += p_k.   interleaved (trailing n mod 32 columns, K >= 5): four partial sums.
template <int K>
__device__ __forceinline__ float sum_seq(const float (&p)[K]) {
    float s = 0.0f;
#pragma unroll
    for (int k = 0; k < K; ++k) s = __fadd_rn(s, p[k]);
    return s;
}
template <int K>
__device__ __forceinline__ float sum_inter4(const float (&p)[K]) {
    float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
    constexpr int full = K / 4;
#pragma unroll
    for (int i = 0; i < full; ++i) {
        a0 = __fadd_rn(a0, p[4 * i + 0]);
        a1 = __fadd_rn(a1, p[4 * i + 1]);
        a2 = __fadd_rn(a2, p[4 * i + 2]);
        a3 = __fadd_rn(a3, p[4 * i + 3]);
    }
#pragma unroll
    for (int r = 4 * full; r < K; ++r) a0 = __fadd_rn(a0, p[r]);
    return __fadd_rn(__fadd_rn(__fadd_rn(a0, a1), a2), a3);
}
template <int K>
__device__ __forceinline__ float torch_sum_dim0(const float (&p)[K], bool tail) {
    if (K >= 5 && tail) return sum_inter4<K>(p);
    return sum_seq<K>(p);
}

// Dispatch a runtime K in [1, MR_MAX_K] to a template instantiation.
#define MR_DISPATCH_K(K, ...)                          \
    switch (K) {                                       \
        case 1: { constexpr int KK = 1; __VA_ARGS__; } break;   \
        case 2: { constexpr int KK = 2; __VA_ARGS__; } break;   \
        case 3: { constexpr int KK = 3; __VA_ARGS__; } break;   \
        case 4: { constexpr int KK = 4; __VA_ARGS__; } break;   \
        case 5: { constexpr int KK = 5; __VA_ARGS__; } break;   \
        case 6: { constexpr int KK = 6; __VA_ARGS__; } break;   \
        case 7: { constexpr int KK = 7; __VA_ARGS__; } break;   \
        case 8: { constexpr int KK = 8; __VA_ARGS__; } break;   \
        case 9: { constexpr int KK = 9; __VA_ARGS__; } break;   \
        case 10: { constexpr int KK = 10; __VA_ARGS__; } break; \
        case 11: { constexpr int KK = 11; __VA_ARGS__; } break; \
        case 12: { constexpr int KK = 12; __VA_ARGS__; } break; \
        case 13: { constexpr int KK = 13; __VA_ARGS__; } break; \
        case 14: { constexpr int KK = 14; __VA_ARGS__; } break; \
        case 15: { constexpr int KK = 15; __VA_ARGS__; } break; \
        case 16: { constexpr int KK = 16; __VA_ARGS__; } break; \
        default: ::mr::set_error("K=%d outside [1,%d]", K, MR_MAX_K); return MR_ERR_INVALID_ARG; \
    }

template <int K>
struct PtrPack {
    const float* p[K];
};

}  // namespace mr
