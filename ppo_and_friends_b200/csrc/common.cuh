// Shared helpers for libppoaf_b200.so (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <utility>

#include "../../include/ppoaf_b200.h"

namespace ppoaf {

void set_error(const char* fmt, ...);

#define PPOAF_CHECK_ARG(cond, ...)                 \
    do {                                           \
        if (!(cond)) {                             \
            ::ppoaf::set_error(__VA_ARGS__);       \
            return 1;                              \
        }                                          \
    } while (0)

#define PPOAF_CHECK_LAUNCH(name)                                                   \
    do {                                                                           \
        cudaError_t e__ = cudaGetLastError();                                      \
        if (e__ != cudaSuccess) {                                                  \
            ::ppoaf::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__)); \
            return 2;                                                              \
        }                                                                          \
    } while (0)

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

int sm_count();  // cached; 148 on B200

__host__ __device__ inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }
inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// ---- streaming 128-bit global access (read-once data: bypass L1 allocation) -------------------
__device__ __forceinline__ float4 ldg_stream_f4(const float4* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream_f4(float4* p, const float4& v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y),
                 "f"(v.z), "f"(v.w)
                 : "memory");
}
__device__ __forceinline__ int4 ldg_stream_i4(const int4* p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream_i4(int4* p, const int4& v) {
    asm volatile("st.global.L1::no_allocate.v4.s32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y),
                 "r"(v.z), "r"(v.w)
                 : "memory");
}

// ---- warp / block reductions ------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// Block-wide sum of `v`; result valid in every thread.  `scratch` holds >= 32 T's.
template <typename T>
__device__ __forceinline__ T block_sum(T v, T* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();
    if (lane == 0) scratch[warp] = v;
    __syncthreads();
    T r = (threadIdx.x < nwarps) ? scratch[threadIdx.x] : T(0);
    if (warp == 0) {
        r = warp_sum(r);
        if (lane == 0) scratch[0] = r;
    }
    __syncthreads();
    r = scratch[0];
    return r;
}

// (n, mean, M2) triple and Chan's parallel merge (reference utils/stats.py:73-94 states the same
// algebra on (count, mean, variance)).
struct Moments {
    double n, mean, m2;
};
__host__ __device__ inline Moments merge_moments(const Moments& a, const Moments& b) {
    if (b.n == 0.0) return a;
    if (a.n == 0.0) return b;
    Moments r;
    r.n = a.n + b.n;
    const double d = b.mean - a.mean;
    r.mean = a.mean + d * (b.n / r.n);
    r.m2 = a.m2 + b.m2 + d * d * a.n * b.n / r.n;
    return r;
}
__device__ __forceinline__ Moments shfl_xor_moments(const Moments& m, int o) {
    Moments r;
    r.n = __shfl_xor_sync(kFull, m.n, o);
    r.mean = __shfl_xor_sync(kFull, m.mean, o);
    r.m2 = __shfl_xor_sync(kFull, m.m2, o);
    return r;
}

__device__ __forceinline__ float fast_tanh(float x) {
    // tanh(x) = 1 - 2 / (exp(2x) + 1); ex2/rcp based, absolute error ~2e-7 (the epilogues' hot math)
    const float t = __expf(2.f * x);
    return 1.f - __fdividef(2.f, t + 1.f);
}
// ---- hidden-layer activations beyond relu / leaky relu / tanh (ids and formulas: ppoaf_b200.h) ----
// Each is written as torch's CUDA kernel writes it (accurate libm, float32), so NaN and +-Inf come out where torch's do.
// SiLU, GELU and Mish cannot recover act'(z) from their output: the update's forward stores it (act_fwd_grad).
// The three helpers are called, not inlined, so each epilogue carries one call site instead of eight functions.
__host__ __device__ __forceinline__ bool act_stores_derivative(int act) {
    return act >= PPOAF_ACT_SILU && act <= PPOAF_ACT_MISH;
}
constexpr float kSeluScale = 1.0507009873554804934193349852946f;
constexpr float kSeluScaleAlpha = float(1.0507009873554804934193349852946 * 1.6732632423543772848170429916717);
constexpr float kSqrtHalf = 0.70710678118654752440f;
constexpr float kInvSqrt2Pi = 0.39894228040143267794f;
constexpr float kGeluTanhBeta = 0.79788456080286535588f;     // sqrt(2 / pi)
constexpr float kGeluTanhKappa = 0.044715f;

static __device__ __noinline__ float act_fwd_ext(float x, int act) {
    switch (act) {
        case PPOAF_ACT_ELU: return x > 0.f ? x : expm1f(x);
        case PPOAF_ACT_SELU: return x > 0.f ? kSeluScale * x : kSeluScaleAlpha * expm1f(x);
        case PPOAF_ACT_SIGMOID: return 1.f / (1.f + expf(-x));
        case PPOAF_ACT_SOFTPLUS: return x > 20.f ? x : log1pf(expf(x));
        case PPOAF_ACT_SILU: return x / (1.f + expf(-x));
        case PPOAF_ACT_GELU: return 0.5f * x * (1.f + erff(x * kSqrtHalf));
        case PPOAF_ACT_GELU_TANH: return 0.5f * x * (1.f + tanhf(kGeluTanhBeta * (x + kGeluTanhKappa * (x * x * x))));
        case PPOAF_ACT_MISH: return x * tanhf(log1pf(expf(x)));
        default: return x;
    }
}
// act'(z) from the output y (ids 4-7; torch's elu_backward / sigmoid_backward / softplus_backward in terms of y)
static __device__ __noinline__ float act_bwd_ext(float y, int act) {
    switch (act) {
        case PPOAF_ACT_ELU: return y > 0.f ? 1.f : y + 1.f;
        case PPOAF_ACT_SELU: return y > 0.f ? kSeluScale : y + kSeluScaleAlpha;
        case PPOAF_ACT_SIGMOID: return y * (1.f - y);
        case PPOAF_ACT_SOFTPLUS: return -expm1f(-y);
        default: return y;                          // ids 8-11: y is the stored act'(z)
    }
}
// ids 8-11: the output (.x) and act'(z) (.y) at once (torch's silu_backward, gelu_backward and mish_backward formulas)
static __device__ __noinline__ float2 act_fwd_grad(float x, int act) {
    switch (act) {
        case PPOAF_ACT_SILU: {
            const float e = 1.f + expf(-x), s = 1.f / e;
            return make_float2(x / e, s * (1.f + x * (1.f - s)));
        }
        case PPOAF_ACT_GELU: {
            const float cdf = 0.5f * (1.f + erff(x * kSqrtHalf));
            return make_float2(x * cdf, cdf + x * (expf(-0.5f * x * x) * kInvSqrt2Pi));
        }
        case PPOAF_ACT_GELU_TANH: {
            const float x2 = x * x;
            const float t = tanhf(kGeluTanhBeta * (x + kGeluTanhKappa * (x2 * x)));
            const float left = 0.5f * x, right = 1.f + t;
            return make_float2(left * right,
                               0.5f * right + left * (1.f - t * t) * kGeluTanhBeta * (1.f + 3.f * kGeluTanhKappa * x2));
        }
        default: {                                  // PPOAF_ACT_MISH
            const float t = tanhf(log1pf(expf(x))), s = 1.f / (1.f + expf(-x));
            return make_float2(x * t, t + x * s * (1.f - t * t));
        }
    }
}

// EXT = false: the grouped GEMM's kernel for ids 0-3, which must not carry the code of the others (mlp.cuh)
template <bool EXT = true>
__device__ __forceinline__ void act_fwd4(float (&o)[4], int act) {
    if (act == PPOAF_ACT_TANH) {
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = fast_tanh(o[j]);
    } else if (act == PPOAF_ACT_RELU) {
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = o[j] > 0.f ? o[j] : 0.f;
    } else if (act == PPOAF_ACT_LEAKY_RELU) {
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = o[j] > 0.f ? o[j] : 0.01f * o[j];
    } else if (EXT && act >= PPOAF_ACT_ELU) {
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = act_fwd_ext(o[j], act);
    }
}
// y: the activation output of the layer (ids 1-7) or its stored act'(z) (ids 8-11)
template <bool EXT = true>
__device__ __forceinline__ void act_bwd4(float (&o)[4], const float (&y)[4], int act) {
    if (act == PPOAF_ACT_TANH) {
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] *= 1.f - y[j] * y[j];
    } else if (act == PPOAF_ACT_RELU) {
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = y[j] > 0.f ? o[j] : 0.f;
    } else if (act == PPOAF_ACT_LEAKY_RELU) {
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = y[j] > 0.f ? o[j] : 0.01f * o[j];
    } else if (EXT && act >= PPOAF_ACT_ELU) {
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] *= act_bwd_ext(y[j], act);
    }
}


// ---- programmatic dependent launch (PDL) ---------------------------------------------------------------------
// The minibatch step is a chain of dependent launches.  Launched with the programmatic-serialization attribute, a
// kernel's CTAs may become resident while the previous kernel is still draining: they run their set-up (barrier
// initialisation, problem lookup, index arithmetic) and block in pdl_wait() until the previous kernel has completed
// and its writes are visible.  NOTHING that another kernel of the chain produces may be read, and nothing it reads
// may be written, before pdl_wait().  pdl_trigger() lets the next kernel's CTAs start arriving; it is always
// issued AFTER pdl_wait(), so whatever a kernel reads early can only race with its immediate predecessor (every
// older kernel has completed), which is what the "static operand" flags of the callers are defined against.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

bool pdl_enabled();    // step.cu: PPOAF_PDL=0 turns the attribute off (plain stream order)

template <typename... KArgs, typename... Args>
inline cudaError_t launch_chain(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

}  // namespace ppoaf
