// Shared plumbing of libmw_b200.so: the 16-bit storage type, scalar device math several kernels share (GELU, LayerNorm rows),
// error strings, launch counting, device guards.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <atomic>
#include <cstdlib>
#include <mutex>

#include "../../include/mw_b200.h"

// ---- 16-bit storage type of activations, K/V caches and weight matrices.
// Default fp16: it is the reference's own GPU compute type (compute_type="float16", /root/reference/transcribe_colab.ipynb:119),
// Whisper checkpoints are published in fp16 (so weights are exact), and its 11-bit significand puts the engine's logit noise
// 8x below bf16's - which is what lets greedy ids match the fp32 oracle (DESIGN.md section 2).  Accumulation, the residual
// stream, softmax statistics and logits are fp32 either way.  -DMW_STORAGE_BF16 builds the bf16 variant for A/B runs.
#ifdef MW_STORAGE_BF16
typedef __nv_bfloat16 mw_h;
typedef __nv_bfloat162 mw_h2;
#define MW_STORAGE_NAME "bf16"
#define MW_MMA_SYNC_TYPE "bf16"
#define MW_UMMA_FMT 1u
__device__ __forceinline__ mw_h f2h(float v) { return __float2bfloat16(v); }
__device__ __forceinline__ float h2f(mw_h v) { return __bfloat162float(v); }
__device__ __forceinline__ mw_h2 f2h2(float a, float b) { return __floats2bfloat162_rn(a, b); }
__device__ __forceinline__ float2 h22f2(mw_h2 v) { return __bfloat1622float2(v); }
__device__ __forceinline__ mw_h2 f2h2_bounded(float a, float b) { return __floats2bfloat162_rn(a, b); }
#else
typedef __half mw_h;
typedef __half2 mw_h2;
#define MW_STORAGE_NAME "fp16"
#define MW_MMA_SYNC_TYPE "f16"
#define MW_UMMA_FMT 0u
// saturating: a value beyond the fp16 range becomes +-65504, never inf (which would turn into NaN downstream)
__device__ __forceinline__ mw_h f2h(float v) { return __float2half_rn(fminf(fmaxf(v, -65504.0f), 65504.0f)); }
__device__ __forceinline__ float h2f(mw_h v) { return __half2float(v); }
__device__ __forceinline__ mw_h2 f2h2(float a, float b) {
    return __floats2half2_rn(fminf(fmaxf(a, -65504.0f), 65504.0f), fminf(fmaxf(b, -65504.0f), 65504.0f));
}
__device__ __forceinline__ float2 h22f2(mw_h2 v) { return __half22float2(v); }
// for values known to lie inside the fp16 range (softmax probabilities, convex combinations of stored values): no clamp
__device__ __forceinline__ mw_h2 f2h2_bounded(float a, float b) { return __floats2half2_rn(a, b); }
#endif

namespace mw {

// ---- scalar device math shared by several kernels

// GELU, 0.5 v (1 + erf(v / sqrt 2)), in two forms that differ in the last bits; each kernel keeps the form it was validated
// with.  gelu_erff uses the library erff: the mma.sync decode projections, the LayerNorm + GELU kernels and wav2vec2.
__device__ __forceinline__ float gelu_erff(float v) { return 0.5f * v * (1.0f + erff(v * 0.70710678118654752f)); }

// gelu_as7126 takes erf from Abramowitz & Stegun 7.1.26 (|error| < 1.5e-7, far below the 16-bit rounding of the value that
// is stored): one MUFU.RCP, one MUFU.EX2 and seven FMAs instead of erff's ~25 instructions - the tcgen05 GEMM's fc1 epilogue
// was issue-bound on erff.  The two tcgen05 GEMMs (gemm.cu, decode_gemm.cu) use it.
__device__ __forceinline__ float gelu_as7126(float v) {
    const float x = fabsf(v) * 0.70710678118654752f;
    const float t = __fdividef(1.0f, fmaf(0.3275911f, x, 1.0f));
    float p = fmaf(1.061405429f, t, -1.453152027f);
    p = fmaf(p, t, 1.421413741f);
    p = fmaf(p, t, -0.284496736f);
    p = fmaf(p, t, 0.254829592f);
    const float e = p * t * exp2f(-1.4426950408889634f * x * x);      // 1 - erf(|x|)
    return 0.5f * v * (1.0f + copysignf(1.0f - e, v));
}

__device__ __forceinline__ float warp_sum(float s) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    return s;
}

__device__ __forceinline__ float sum4(float4 v) { return (v.x + v.y) + (v.z + v.w); }

// LayerNorm of a row of d = 128 nv floats held by one warp: lane l holds float4 i * 32 + l of the row in v[i], i < nv <= MAXV,
// and s = the sum over i of sum4(v[i]), in order.  layernorm_kernel (elementwise.cu) and the fused projection
// skinny_gemm_ln_kernel (decoder.cu) both normalise with these, so the 16-bit operands they produce are the same bits.
template <int MAXV>
__device__ __forceinline__ void ln_stats(float s, const float4 (&v)[MAXV], int nv, int d, float& mean, float& rstd) {
    mean = warp_sum(s) / (float)d;
    float q = 0.0f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i)
        if (i < nv) {
            const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, e = v[i].w - mean;
            q += (a * a + b * b) + (c * c + e * e);
        }
    rstd = rsqrtf(warp_sum(q) / (float)d + 1e-5f);
}

__device__ __forceinline__ float4 ln_apply(float4 v, float mean, float rstd, float4 g, float4 b) {
    return make_float4((v.x - mean) * rstd * g.x + b.x, (v.y - mean) * rstd * g.y + b.y, (v.z - mean) * rstd * g.z + b.z,
                       (v.w - mean) * rstd * g.w + b.w);
}

__device__ __forceinline__ uint2 pack_h16x4(float4 y) {
    mw_h2 h0 = f2h2(y.x, y.y), h1 = f2h2(y.z, y.w);
    uint2 u;
    u.x = *reinterpret_cast<uint32_t*>(&h0);
    u.y = *reinterpret_cast<uint32_t*>(&h1);
    return u;
}

// ---- host-side plumbing

void set_error(const char* fmt, ...);
extern std::atomic<uint64_t> g_launches;

// Launches enqueued while this thread captures a CUDA graph are not launches yet: they are tallied per graph
// (t_captured) and added to g_launches each time the graph is replayed.
extern thread_local bool t_capturing;
extern thread_local uint64_t t_captured;
inline void count_launch(int n = 1) {
    if (t_capturing) t_captured += (uint64_t)n;
    else g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed);
}

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        // always set: on a fresh host thread this is what binds the primary context, which the driver-API tensor-map
        // encoder needs (a thread whose first call into the library is mw_generate got CUDA_ERROR_INVALID_CONTEXT)
        cudaSetDevice(dev);
        if (prev == dev) prev = -1;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

#define MW_CUDA_CHECK(expr)                                                                      \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess) {                                                                 \
            mw::set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__, cudaGetErrorString(_e)); \
            return MW_ERR_CUDA;                                                                  \
        }                                                                                        \
    } while (0)

#define MW_LAUNCH_CHECK()                                                                        \
    do {                                                                                         \
        cudaError_t _e = cudaGetLastError();                                                     \
        if (_e != cudaSuccess) {                                                                 \
            mw::set_error("kernel launch failed at %s:%d: %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
            return MW_ERR_CUDA;                                                                  \
        }                                                                                        \
        mw::count_launch();                                                                      \
    } while (0)

#define MW_REQUIRE(cond, ...)                                                                    \
    do {                                                                                         \
        if (!(cond)) { mw::set_error(__VA_ARGS__); return MW_ERR_INVALID; }                      \
    } while (0)

inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// cudaFuncSetAttribute is per device and must have completed before ANY thread launches the kernel there
// (several host threads drive replicas concurrently): a mutex-guarded per-device flag.
struct PerDeviceOnce {
    std::mutex mu;
    bool done[64] = {};
    template <typename Fn>
    cudaError_t run(Fn&& fn) {
        int dev = 0;
        cudaGetDevice(&dev);
        dev &= 63;
        std::lock_guard<std::mutex> lock(mu);
        if (done[dev]) return cudaSuccess;
        cudaError_t e = fn();
        if (e == cudaSuccess) done[dev] = true;
        return e;
    }
};
inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

}  // namespace mw
