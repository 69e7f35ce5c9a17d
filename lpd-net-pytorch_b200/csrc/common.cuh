// Shared helpers of the lpd_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <math.h>
#include "../../include/lpd_b200.h"

namespace lpd {

// thread-local text of the last CUDA failure (read through lpd_last_cuda_error)
extern thread_local char g_last_error[512];

inline int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
    snprintf(g_last_error, sizeof(g_last_error), "%s: %s (%s:%d)", what, cudaGetErrorString(e), file, line);
    return LPD_ECUDA;
}

#define LPD_CUDA_CHECK(expr)                                                        \
    do {                                                                            \
        cudaError_t _e = (expr);                                                    \
        if (_e != cudaSuccess) return ::lpd::cuda_fail(_e, #expr, __FILE__, __LINE__); \
    } while (0)

// after a kernel launch: launch-configuration errors only (asynchronous, no sync)
#define LPD_LAUNCH_CHECK()                                                          \
    do {                                                                            \
        cudaError_t _e = cudaGetLastError();                                        \
        if (_e != cudaSuccess) return ::lpd::cuda_fail(_e, "kernel launch", __FILE__, __LINE__); \
    } while (0)

#define LPD_REQUIRE(cond)                                                           \
    do {                                                                            \
        if (!(cond)) {                                                              \
            snprintf(::lpd::g_last_error, sizeof(::lpd::g_last_error),              \
                     "invalid argument: %s (%s:%d)", #cond, __FILE__, __LINE__);    \
            return LPD_EINVAL;                                                      \
        }                                                                           \
    } while (0)

// the tensor-core kernels are built for sm_100a only: LPD_EUNSUPPORTED on any other device
inline int require_sm100() {
    int dev = 0, major = 0;
    LPD_CUDA_CHECK(cudaGetDevice(&dev));
    LPD_CUDA_CHECK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    return major == 10 ? LPD_OK : LPD_EUNSUPPORTED;
}

// SMs of the current device (a persistent kernel launches at most one CTA per SM)
inline int sm_count(int* sms) {
    int dev = 0;
    LPD_CUDA_CHECK(cudaGetDevice(&dev));
    LPD_CUDA_CHECK(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev));
    return LPD_OK;
}

// the activations a fused epilogue applies as act(v) = max(v, v * neg_slope)
inline bool act_is_slope(int act, float slope) {
    return act == LPD_ACT_NONE || act == LPD_ACT_RELU || (act == LPD_ACT_LEAKY && slope >= 0.f && slope <= 1.f);
}
// neg_slope: 1 -> identity, 0 -> ReLU, 0 < s < 1 -> LeakyReLU(s)
inline float act_neg_slope(int act, float slope) { return act == LPD_ACT_NONE ? 1.f : (act == LPD_ACT_RELU ? 0.f : slope); }

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
inline long long ceil_div_ll(long long a, long long b) { return (a + b - 1) / b; }

// opt in to > 48 KB dynamic shared memory once per kernel symbol
template <typename K>
inline cudaError_t allow_smem(K kernel, size_t bytes) {
    return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

__device__ __forceinline__ float apply_act(float v, int act, float slope) {
    switch (act) {
        case LPD_ACT_RELU: return fmaxf(v, 0.f);
        case LPD_ACT_LEAKY: return v > 0.f ? v : v * slope;
        case LPD_ACT_SIGMOID: return 1.f / (1.f + expf(-v));
        default: return v;
    }
}

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

}  // namespace lpd
