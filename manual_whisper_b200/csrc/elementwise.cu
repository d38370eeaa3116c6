// Small bandwidth-bound kernels around the tensor-core work: LayerNorm (fp32 residual stream -> bf16 GEMM
// operand) and the feature re-layout mw_encode needs (f32 [B, n_mels, frames] -> bf16 time-major).
#include "mw_common.cuh"
#include "kernels.cuh"

namespace mw {

namespace {

// one warp per row; d % 128 == 0, d <= 128 * MAXV.  MODE 0: LN -> h16; 1: GELU(LN) -> h16; 2: GELU(LN) -> f32;
// 3: LN -> h16 AND f32 written back over x (post-LayerNorm encoders: the normalised row is both the next GEMM operand and
// the residual stream)
template <int MAXV, int MODE = 0>
__global__ void __launch_bounds__(256)
layernorm_kernel(const float* x /* MODE 3 writes it back: no __restrict__ */, const float* __restrict__ gamma,
                 const float* __restrict__ beta, void* out_v, int rows, int d) {
    mw_h* out = reinterpret_cast<mw_h*>(out_v);
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    const float4* xr = reinterpret_cast<const float4*>(x + (int64_t)row * d);
    const int nv = d >> 7;   // float4 per lane
    float4 v[MAXV];
    float s = 0.0f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i)
        if (i < nv) {
            v[i] = xr[i * 32 + lane];
            s += sum4(v[i]);
        }
    float mean, rstd;
    ln_stats(s, v, nv, d, mean, rstd);
    const float4* g4 = reinterpret_cast<const float4*>(gamma);
    const float4* b4 = reinterpret_cast<const float4*>(beta);
    uint2* o2 = reinterpret_cast<uint2*>(out + (int64_t)row * d);
#pragma unroll
    for (int i = 0; i < MAXV; ++i)
        if (i < nv) {
            float4 y = ln_apply(v[i], mean, rstd, __ldg(g4 + i * 32 + lane), __ldg(b4 + i * 32 + lane));
            if (MODE == 1 || MODE == 2) y = make_float4(gelu_erff(y.x), gelu_erff(y.y), gelu_erff(y.z), gelu_erff(y.w));
            if (MODE == 2) {
                reinterpret_cast<float4*>(reinterpret_cast<float*>(out_v) + (int64_t)row * d)[i * 32 + lane] = y;
                continue;
            }
            if (MODE == 3)      // the row is held in registers: writing it back in place is safe
                reinterpret_cast<float4*>(const_cast<float*>(x) + (int64_t)row * d)[i * 32 + lane] = y;
            o2[i * 32 + lane] = pack_h16x4(y);
        }
}

// f32 [B, C, F] -> bf16 [B, F+2, C] with zero rows 0 and F+1
__global__ void __launch_bounds__(256)
features_to_time_major_kernel(const float* __restrict__ in, mw_h* __restrict__ out, int C, int F) {
    __shared__ float tile[32][33];
    const int b = blockIdx.z;
    const int f0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 32 x 8
    const float* src = in + (int64_t)b * C * F;
    mw_h* dst = out + (int64_t)b * (F + 2) * C;
    for (int i = ty; i < 32; i += 8) {
        const int c = c0 + i, f = f0 + tx;
        tile[i][tx] = (c < C && f < F) ? src[(int64_t)c * F + f] : 0.0f;
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int f = f0 + i, c = c0 + tx;
        if (f < F && c < C) dst[(int64_t)(f + 1) * C + c] = f2h(tile[tx][i]);
    }
    if (blockIdx.x == 0 && ty == 0) {
        const int c = c0 + tx;
        if (c < C) {
            dst[c] = f2h(0.0f);
            dst[(int64_t)(F + 1) * C + c] = f2h(0.0f);
        }
    }
}

// frame RMS for the energy VAD front end: one warp per frame of `frame` samples
__global__ void __launch_bounds__(256)
frame_rms_kernel(const float* __restrict__ audio, int64_t n, int frame, float* __restrict__ out, int64_t n_frames) {
    const int64_t f = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (f >= n_frames) return;
    const float* a = audio + f * frame;
    float s = 0.0f;
    for (int i = lane; i < frame; i += 32) { const float v = a[i]; s = fmaf(v, v, s); }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) out[f] = sqrtf(s / (float)frame + 1e-12f);
}

}  // namespace

mw_status layernorm_launch(const float* x, const float* gamma, const float* beta, void* out_bf16, int rows, int d,
                           cudaStream_t st) {
    MW_REQUIRE(x && gamma && beta && out_bf16, "layernorm: null pointer");
    MW_REQUIRE(d % 128 == 0 && d >= 128 && d <= 2048, "layernorm: d=%d must be a multiple of 128 in [128, 2048]", d);
    if (rows <= 0) return MW_OK;
    const int grid = ceil_div(rows, 8);
    if (d <= 512) layernorm_kernel<4, 0><<<grid, 256, 0, st>>>(x, gamma, beta, out_bf16, rows, d);
    else if (d <= 1280) layernorm_kernel<10, 0><<<grid, 256, 0, st>>>(x, gamma, beta, out_bf16, rows, d);
    else layernorm_kernel<16, 0><<<grid, 256, 0, st>>>(x, gamma, beta, out_bf16, rows, d);
    MW_LAUNCH_CHECK();
    return MW_OK;
}

mw_status layernorm_dual_launch(float* x_inout, const float* gamma, const float* beta, void* out_h16, int rows, int d,
                                cudaStream_t st) {
    MW_REQUIRE(x_inout && gamma && beta && out_h16, "layernorm_dual: null pointer");
    MW_REQUIRE(d % 128 == 0 && d >= 128 && d <= 2048, "layernorm_dual: d=%d must be a multiple of 128 in [128, 2048]", d);
    if (rows <= 0) return MW_OK;
    const int grid = ceil_div(rows, 8);
    if (d <= 512) layernorm_kernel<4, 3><<<grid, 256, 0, st>>>(x_inout, gamma, beta, out_h16, rows, d);
    else if (d <= 1280) layernorm_kernel<10, 3><<<grid, 256, 0, st>>>(x_inout, gamma, beta, out_h16, rows, d);
    else layernorm_kernel<16, 3><<<grid, 256, 0, st>>>(x_inout, gamma, beta, out_h16, rows, d);
    MW_LAUNCH_CHECK();
    return MW_OK;
}

mw_status layernorm_act_launch(const float* x, const float* gamma, const float* beta, void* out, int rows, int d, int mode,
                               cudaStream_t st) {
    MW_REQUIRE(x && gamma && beta && out, "layernorm_act: null pointer");
    MW_REQUIRE(d % 128 == 0 && d >= 128 && d <= 512, "layernorm_act: d=%d must be a multiple of 128 in [128, 512]", d);
    MW_REQUIRE(mode == 1 || mode == 2, "layernorm_act: mode must be 1 or 2");
    if (rows <= 0) return MW_OK;
    const int grid = ceil_div(rows, 8);
    if (mode == 1) layernorm_kernel<4, 1><<<grid, 256, 0, st>>>(x, gamma, beta, out, rows, d);
    else layernorm_kernel<4, 2><<<grid, 256, 0, st>>>(x, gamma, beta, out, rows, d);
    MW_LAUNCH_CHECK();
    return MW_OK;
}

mw_status features_to_time_major_launch(const float* in, void* out_bf16, int B, int C, int F, cudaStream_t st) {
    dim3 grid(ceil_div(F, 32), ceil_div(C, 32), B);
    features_to_time_major_kernel<<<grid, 256, 0, st>>>(in, (mw_h*)out_bf16, C, F);
    MW_LAUNCH_CHECK();
    return MW_OK;
}

}  // namespace mw

extern "C" mw_status mw_layernorm(const float* d_x, const float* d_gamma, const float* d_beta, void* d_out_bf16,
                                  int rows, int d, void* stream) {
    return mw::layernorm_launch(d_x, d_gamma, d_beta, d_out_bf16, rows, d, (cudaStream_t)stream);
}

extern "C" mw_status mw_layernorm_mode(float* d_x, const float* d_gamma, const float* d_beta, void* d_out, int rows, int d, int mode,
                                       void* stream) {
    // shape and mode first, then the pointers: a rejected call touches no memory
    MW_REQUIRE(mode >= 0 && mode <= 3, "mw_layernorm_mode: mode=%d must be 0..3", mode);
    const int max_d = (mode == 1 || mode == 2) ? 512 : 2048;
    MW_REQUIRE(rows >= 0 && d % 128 == 0 && d >= 128 && d <= max_d,
               "mw_layernorm_mode: rows=%d d=%d (mode %d needs d %% 128 == 0 in [128, %d])", rows, d, mode, max_d);
    MW_REQUIRE(d_x && d_gamma && d_beta && d_out, "mw_layernorm_mode: null pointer");
    const cudaStream_t st = (cudaStream_t)stream;
    if (mode == 0) return mw::layernorm_launch(d_x, d_gamma, d_beta, d_out, rows, d, st);
    if (mode == 3) return mw::layernorm_dual_launch(d_x, d_gamma, d_beta, d_out, rows, d, st);
    return mw::layernorm_act_launch(d_x, d_gamma, d_beta, d_out, rows, d, mode, st);
}

extern "C" mw_status mw_frame_rms(const float* d_audio, int64_t n, int frame, float* d_out, void* stream) {
    MW_REQUIRE(d_audio && d_out && frame > 0 && n >= 0, "mw_frame_rms: bad argument");
    const int64_t n_frames = n / frame;
    if (n_frames == 0) return MW_OK;
    mw::frame_rms_kernel<<<(unsigned)((n_frames + 7) / 8), 256, 0, (cudaStream_t)stream>>>(d_audio, n, frame, d_out, n_frames);
    MW_LAUNCH_CHECK();
    return MW_OK;
}
