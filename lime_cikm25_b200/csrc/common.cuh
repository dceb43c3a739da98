// Shared device/host helpers for liblime_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "lime_b200.h"

namespace lime {

// ---- error plumbing -------------------------------------------------------------------------
void set_error(const char *fmt, ...);
void count_launch();

#define LIME_CHECK_ARG(cond, ...)                                                            \
    do {                                                                                       \
        if (!(cond)) {                                                                         \
            ::lime::set_error(__VA_ARGS__);                                                    \
            return 1;                                                                          \
        }                                                                                      \
    } while (0)

// call after every kernel launch: picks up launch-configuration errors without synchronising
#define LIME_LAUNCH_CHECK(name)                                                              \
    do {                                                                                       \
        ::lime::count_launch();                                                                \
        cudaError_t e__ = cudaGetLastError();                                                  \
        if (e__ != cudaSuccess) {                                                              \
            ::lime::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__));         \
            return 2;                                                                          \
        }                                                                                      \
    } while (0)

#define LIME_CUDA(call)                                                                      \
    do {                                                                                       \
        cudaError_t e__ = (call);                                                              \
        if (e__ != cudaSuccess) {                                                              \
            ::lime::set_error("%s failed: %s", #call, cudaGetErrorString(e__));                \
            return 3;                                                                          \
        }                                                                                      \
    } while (0)

inline cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }

int num_sms();

// ---- warp helpers ---------------------------------------------------------------------------
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
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ long long warp_sum_ll(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Stateless counter-based generator of the training dropouts: (seed, element index) -> 32 random bits via two rounds of a
// 64-bit mix; forward and backward evaluate the same mask.  drop_scale = keep / (1 - p).
__device__ __forceinline__ uint32_t mix_bits(uint64_t seed, uint64_t idx) {
    uint64_t z = seed + 0x9E3779B97F4A7C15ull * (idx + 1);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z = z ^ (z >> 31);
    return (uint32_t)(z >> 32);
}
__device__ __forceinline__ float drop_scale(uint64_t seed, uint64_t idx, float p) {
    const float u = (float)mix_bits(seed, idx) * (1.0f / 4294967296.0f);
    return u >= p ? 1.0f / (1.0f - p) : 0.0f;
}

// FreshnessEncoder.bucketize (newsEncoders.py:53-58), bit-exact with the reference's fp32 op
// sequence AS ATen EXECUTES IT ON CUDA (the reference asserts a GPU, config.py:212):
// clamp(min=1) -> log -> "divide" by the CPU 0-dim tensor torch.log(torch.tensor(86400.)) =
// 0x4135de2e, which ATen's CUDA div kernel turns into a multiplication by the fp32 reciprocal
// (BinaryDivTrueKernel.cu: iter.is_cpu_scalar(2) -> a * (1/b)) -> multiply by fp32(num_buckets/7)
// (python double rounded to fp32, as tensor * python-float does) -> truncate -> clamp(max).
// The CPU path of the same reference performs a true division and differs on 57 of 20,654
// knife-edge inputs at B = 50 (none at B = 10, 20): tests/test_gpu_kernels.py.  No fast-math here.
__device__ __forceinline__ int bucketize_seconds(float x, float scale, int num_buckets) {
    x = fmaxf(x, 1.0f);
    if (x != x) x = 1.0f;  // torch.clamp propagates NaN; a NaN age has no bucket -> treat as 1 s
    const float log_day = __uint_as_float(0x4135de2eu);
    const float inv_log_day = __fdiv_rn(1.0f, log_day);
    float scaled = __fmul_rn(logf(x), inv_log_day);
    float prod = __fmul_rn(scaled, scale);
    long long b = (long long)prod;  // truncation toward zero, like Tensor.long()
    if (b > num_buckets - 1) b = num_buckets - 1;
    if (b < 0) b = 0;
    return (int)b;
}

}  // namespace lime
