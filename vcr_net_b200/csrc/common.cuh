// Shared helpers for the vcr_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <float.h>

#define VCR_OK 0
#define VCR_ERR_INVALID (-1)      // bad pointer / size / alignment
#define VCR_ERR_UNSUPPORTED (-2)  // shape outside what the kernel was built for
#define VCR_ERR_LAUNCH (-3)       // cudaGetLastError() != cudaSuccess after the launch
#define VCR_ERR_WORKSPACE (-4)    // workspace too small

#define VCR_API extern "C" __attribute__((visibility("default")))

// every kernel launch of the library bumps this counter (bench.py reports it as gpu_launches)
extern unsigned long long g_vcr_launches;

#define VCR_CHECK_LAUNCH()                                   \
    do {                                                     \
        cudaError_t e__ = cudaGetLastError();                \
        if (e__ != cudaSuccess) return VCR_ERR_LAUNCH;       \
        __atomic_fetch_add(&g_vcr_launches, 1ull, __ATOMIC_RELAXED); \
    } while (0)

#define VCR_REQUIRE(cond)                  \
    do {                                   \
        if (!(cond)) return VCR_ERR_INVALID; \
    } while (0)

static inline int vcr_cdiv(long long a, long long b) { return (int)((a + b - 1) / b); }

__device__ __forceinline__ float leaky(float v, float slope) { return v >= 0.f ? v : v * slope; }

// Length of item b of a ragged batch (the *_ragged entry points): len[b] clamped to [lo, n_max], so that an out-of-range
// length stays in bounds; n_max when len is null (a uniform batch).
__device__ __forceinline__ int vcr_item_len(const int* len, int b, int n_max, int lo) {
    return len != nullptr ? min(max(__ldg(len + b), lo), n_max) : n_max;
}

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
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
