// Forced alignment on the GPU (SURVEY.md §8f row 3; /root/reference/transcribe.py:127-135 -> whisperx.load_align_model /
// whisperx.align): the wav2vec2-CTC acoustic model (Hugging Face Wav2Vec2ForCTC, layer-norm feature extractor,
// stable-layer-norm encoder: transformers/models/wav2vec2/modeling_wav2vec2.py:275-300, 326-368, 422-436, 612-655, 742-800)
// and the CTC trellis + backtrack of whisperx/alignment.py.
//
// Data flow of mw_w2v_emissions for n windows (S = longest window of the call, T_l = frames after conv layer l):
//   conv0 (1 -> C, k=10, s=5) + LayerNorm(C) + GELU, fused, fp32 math            -> bf16 [n, T_0, C]
//   conv l=1..6 (k=3/2, s=2): implicit GEMM on the tcgen05 kernel - A row t is the k*C contiguous elements at time-major
//     row s*t of the previous layer (overlapping-row TMA map, nothing materialised) -> f32, then LayerNorm + GELU -> bf16
//   feature projection: LayerNorm(C) -> GEMM C -> d                               -> x f32 [n*T, d]
//   positional conv (k=128, 16 groups of 64 channels): x is re-laid out group-major with zero rows outside each
//     window's valid frames, then one implicit GEMM per group (K = 128 taps x 64 channels) with bias, GELU and the
//     residual add fused in the epilogue
//   24 x { LN -> QKV GEMM -> flash attention with per-window key lengths -> out GEMM (+res) -> LN -> fc1 (GELU) -> fc2 (+res) }
//   LN -> lm_head GEMM -> log_softmax                                              -> f32 [n, T_n, vocab]
// Every op before the positional conv is local in time (valid convs, per-frame norms), so padding a window to S samples
// leaves its first frames(len) frames untouched; the positional conv and attention are told each window's length.
//
// variant 1 = wav2vec2-base (what whisperx loads for en/fr/de/es/it; modeling_wav2vec2.py:302-323, 592-609, 658-727):
//   conv0 has no bias and is followed by GroupNorm(C groups) - per-channel statistics over the window's OWN frames, the one
//     op that is global in time: a statistics pass over conv0 (deterministic two-level sum), then conv0 is recomputed,
//     normalised and GELU'd; conv 1..6: GEMM with GELU in the epilogue, no bias, no norm
//   positional conv groups of 48 channels (768 / 16): weight rows padded to 64 per group, result added by a small kernel
//   post-LayerNorm encoder: LN right after the positional conv, then per layer x = LN(x + attn(x)); x = LN(x + ffn(x)); no
//     final LN - LayerNorm writes the fp32 residual stream and the 16-bit GEMM operand at once (layernorm_dual_launch)
#include "gemm.cuh"
#include "kernels.cuh"
#include <stdlib.h>
#include <vector>
#include <algorithm>

struct mw_w2v {
    mw_w2v_config cfg{};
    std::vector<const void*> w;
    int64_t workspace_bytes = 0;
    std::vector<void*> allocations;
    int vocab_pad = 0;
    int T_max[7] = {};                    // frames after each conv layer at max_samples
    mw_h* act_a = nullptr;       // [B, T_0, C]  conv0 / even layers' output
    mw_h* act_b = nullptr;       // [B, T_1, C]  odd layers' output
    float* conv_f32 = nullptr;            // [B, T_1, C]  GEMM output ahead of LayerNorm
    float* feat = nullptr;                // [B*T, C]     last conv layer after LN + GELU (fp32: feeds a LayerNorm)
    float* x = nullptr;                   // [B*T, d]     fp32 residual stream
    mw_h* xg = nullptr;          // [B, G, T + pos_kernel, 64] group-major, zero padded
    mw_h* ln = nullptr;          // [B*T, max(d, C)]
    mw_h* qkv = nullptr;         // [B*T, 3d]
    mw_h* att = nullptr;         // [B*T, d]
    mw_h* mlp = nullptr;         // [B*T, ffn]
    float* logits = nullptr;              // [B*T, vocab_pad]
    int* d_frames = nullptr;              // [B] valid frames per window of the current call
    // variant 1 (wav2vec2-base)
    float* gn_partial = nullptr;          // [B, ceil(T_0 / 64), C, 2] per-CTA sums of conv0 and conv0^2
    float* gn_stats = nullptr;            // [B, C, 2] mean, rstd
    float* pos_tmp = nullptr;             // [B*T, G*64] positional conv output before bias / GELU / residual

    const void* gw(int id) const { return w[id]; }
    const void* lw(int layer, int id) const { return w[MW_A_GLOBAL_COUNT + layer * MW_EL_COUNT + id]; }
};

namespace mw {
namespace {

constexpr int CONV_K[7] = {10, 3, 3, 3, 3, 2, 2};
constexpr int CONV_S[7] = {5, 2, 2, 2, 2, 2, 2};

__host__ __device__ inline int conv_frames(int64_t n, int upto = 7) {
    int64_t t = n;
    const int k[7] = {10, 3, 3, 3, 3, 2, 2}, s[7] = {5, 2, 2, 2, 2, 2, 2};
    for (int i = 0; i < upto; ++i) t = t >= k[i] ? (t - k[i]) / s[i] + 1 : 0;
    return (int)t;
}

__global__ void w2v_frames_kernel(const int* __restrict__ lens, int n, int* __restrict__ frames) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) frames[i] = conv_frames(max(lens[i], 400));
}

// conv0 + LayerNorm + GELU: one warp per output frame, lane owns channel pairs 2*lane + 64 p; 64 frames per CTA
template <int NP>
__global__ void __launch_bounds__(256)
w2v_conv0_kernel(const float* __restrict__ audio, int64_t n_audio, const int64_t* __restrict__ offs, const int* __restrict__ lens,
                 const float* __restrict__ w, const float* __restrict__ bias, const float* __restrict__ gamma,
                 const float* __restrict__ beta, mw_h* __restrict__ out, int T0) {
    constexpr int C = 64 * NP;
    __shared__ float sw[10][C];
    __shared__ float sb[C], sg[C], sbe[C];
    for (int i = threadIdx.x; i < 10 * C; i += 256) sw[i % 10][i / 10] = w[i];
    for (int i = threadIdx.x; i < C; i += 256) { sb[i] = bias[i]; sg[i] = gamma[i]; sbe[i] = beta[i]; }
    __syncthreads();
    const int b = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int64_t off = offs[b];
    const int len = lens[b];
    const float* a = audio + off;
    for (int it = 0; it < 8; ++it) {
        const int t = blockIdx.x * 64 + it * 8 + warp;
        if (t >= T0) break;                                  // warp-uniform
        float xs = 0.0f;
        if (lane < 10) {
            const int i = 5 * t + lane;
            if (i < len && off + i < n_audio) xs = a[i];
        }
        float xk[10];
#pragma unroll
        for (int k = 0; k < 10; ++k) xk[k] = __shfl_sync(0xffffffffu, xs, k);
        float v[NP][2];
        float s = 0.0f;
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            const int c = 2 * lane + 64 * p;
            float a0 = sb[c], a1 = sb[c + 1];
#pragma unroll
            for (int k = 0; k < 10; ++k) {
                const float2 wk = *reinterpret_cast<const float2*>(&sw[k][c]);
                a0 = fmaf(wk.x, xk[k], a0);
                a1 = fmaf(wk.y, xk[k], a1);
            }
            v[p][0] = a0; v[p][1] = a1;
            s += a0 + a1;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        const float mean = s / (float)C;
        float q = 0.0f;
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            const float d0 = v[p][0] - mean, d1 = v[p][1] - mean;
            q += d0 * d0 + d1 * d1;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
        const float rstd = rsqrtf(q / (float)C + 1e-5f);
        mw_h* o = out + ((int64_t)b * T0 + t) * C;
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            const int c = 2 * lane + 64 * p;
            const float y0 = gelu_erff((v[p][0] - mean) * rstd * sg[c] + sbe[c]);
            const float y1 = gelu_erff((v[p][1] - mean) * rstd * sg[c + 1] + sbe[c + 1]);
            *reinterpret_cast<mw_h2*>(o + c) = f2h2(y0, y1);
        }
    }
}

// ---- wav2vec2-base: conv0 (no bias) + GroupNorm(C groups) + GELU.  MODE 0: per-CTA partial sums of conv0 and conv0^2 over
// the window's own frames; MODE 1: conv0 recomputed, (v - mean_c) rstd_c gamma_c + beta_c, GELU -> h16 time-major.
template <int NP, int MODE>
__global__ void __launch_bounds__(256)
w2v_conv0_gn_kernel(const float* __restrict__ audio, int64_t n_audio, const int64_t* __restrict__ offs, const int* __restrict__ lens,
                    const float* __restrict__ w, const float* __restrict__ gamma, const float* __restrict__ beta,
                    float* __restrict__ partial, const float* __restrict__ stats, mw_h* __restrict__ out, int T0, int n_blk) {
    constexpr int C = 64 * NP;
    __shared__ float sw[10][C];
    __shared__ float red[4][2 * C];         // MODE 0: sums of warp pairs (w, w+4); MODE 1: red[0] = scale | shift per channel
    for (int i = threadIdx.x; i < 10 * C; i += 256) sw[i % 10][i / 10] = w[i];
    const int b = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (MODE == 1) {
        for (int c = threadIdx.x; c < C; c += 256) {
            const float mean = stats[((int64_t)b * C + c) * 2], rstd = stats[((int64_t)b * C + c) * 2 + 1];
            red[0][c] = rstd * gamma[c];                       // scale
            red[0][C + c] = beta[c] - mean * rstd * gamma[c];  // shift
        }
    }
    __syncthreads();
    const int64_t off = offs[b];
    const int len = lens[b];
    const int T0b = conv_frames(max(len, 400), 1);             // this window's own frames (shorter windows are zero-padded to 400)
    const float* a = audio + off;
    float ps[NP][2], pq[NP][2];
#pragma unroll
    for (int p = 0; p < NP; ++p) { ps[p][0] = ps[p][1] = pq[p][0] = pq[p][1] = 0.0f; }
    for (int it = 0; it < 8; ++it) {
        const int t = blockIdx.x * 64 + it * 8 + warp;
        if (t >= T0) break;                                  // warp-uniform
        float xs = 0.0f;
        if (lane < 10) {
            const int i = 5 * t + lane;
            if (i < len && off + i < n_audio) xs = a[i];
        }
        float xk[10];
#pragma unroll
        for (int k = 0; k < 10; ++k) xk[k] = __shfl_sync(0xffffffffu, xs, k);
        mw_h* o = out + ((int64_t)b * T0 + t) * C;
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            const int c = 2 * lane + 64 * p;
            float a0 = 0.0f, a1 = 0.0f;
#pragma unroll
            for (int k = 0; k < 10; ++k) {
                const float2 wk = *reinterpret_cast<const float2*>(&sw[k][c]);
                a0 = fmaf(wk.x, xk[k], a0);
                a1 = fmaf(wk.y, xk[k], a1);
            }
            if (MODE == 0) {
                if (t < T0b) { ps[p][0] += a0; ps[p][1] += a1; pq[p][0] = fmaf(a0, a0, pq[p][0]); pq[p][1] = fmaf(a1, a1, pq[p][1]); }
            } else {
                const float y0 = t < T0b ? gelu_erff(fmaf(a0, red[0][c], red[0][C + c])) : 0.0f;
                const float y1 = t < T0b ? gelu_erff(fmaf(a1, red[0][c + 1], red[0][C + c + 1])) : 0.0f;
                *reinterpret_cast<mw_h2*>(o + c) = f2h2(y0, y1);
            }
        }
    }
    if (MODE == 0) {
        __syncthreads();
#pragma unroll
        for (int round = 0; round < 2; ++round) {             // warps 4..7 park their sums, warps 0..3 fold them in
            if ((warp >= 4) == (round == 0)) {
#pragma unroll
                for (int p = 0; p < NP; ++p) {
                    const int c = 2 * lane + 64 * p;
                    float* r = red[warp & 3];
                    if (round == 1) { ps[p][0] += r[c]; ps[p][1] += r[c + 1]; pq[p][0] += r[C + c]; pq[p][1] += r[C + c + 1]; }
                    r[c] = ps[p][0]; r[c + 1] = ps[p][1];
                    r[C + c] = pq[p][0]; r[C + c + 1] = pq[p][1];
                }
            }
            __syncthreads();
        }
        float* dst = partial + ((int64_t)b * n_blk + blockIdx.x) * 2 * C;
        for (int i = threadIdx.x; i < 2 * C; i += 256)
            dst[i] = (red[0][i] + red[1][i]) + (red[2][i] + red[3][i]);       // fixed order
    }
}

// per (window, channel): mean and rstd from the per-CTA partial sums, summed in block order in double (deterministic)
__global__ void w2v_gn_finalize_kernel(const float* __restrict__ partial, const int* __restrict__ lens, float* __restrict__ stats,
                                       int C, int n_blk) {
    const int b = blockIdx.x;
    const int T0b = conv_frames(max(lens[b], 400), 1);
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        double s = 0.0, q = 0.0;
        const float* p = partial + (int64_t)b * n_blk * 2 * C;
        for (int k = 0; k < n_blk; ++k) { s += p[(int64_t)k * 2 * C + c]; q += p[(int64_t)k * 2 * C + C + c]; }
        const double mean = s / (double)T0b;
        const double var = fmax(q / (double)T0b - mean * mean, 0.0);
        stats[((int64_t)b * C + c) * 2] = (float)mean;
        stats[((int64_t)b * C + c) * 2 + 1] = (float)(1.0 / sqrt(var + 1e-5));
    }
}

// x f32 [n, T, d] -> h16 [n, G, T + kp, gw] (gw = d / G channels per group): row t' holds frame t' - kp/2, zero outside the
// window's valid frames
__global__ void __launch_bounds__(256)
w2v_group_major_kernel(const float* __restrict__ x, const int* __restrict__ frames, mw_h* __restrict__ xg, int T, int d,
                       int kp, int gw) {
    const int tp = blockIdx.x, b = blockIdx.y;
    const int t = tp - kp / 2;
    const bool valid = t >= 0 && t < min(frames[b], T);
    const int G = d / gw;
    const float* src = x + ((int64_t)b * T + t) * d;
    for (int c = threadIdx.x; c < d; c += 256) {
        const int g = c / gw, ci = c - g * gw;
        xg[(((int64_t)b * G + g) * (T + kp) + tp) * gw + ci] = f2h(valid ? src[c] : 0.0f);
    }
}

// groups narrower than 64 channels: x[r, g*gw + c] += GELU(tmp[r, g*64 + c] + bias[g*gw + c])
__global__ void __launch_bounds__(256)
w2v_pos_add_kernel(const float* __restrict__ tmp, const float* __restrict__ bias, float* __restrict__ x, int64_t rows, int d, int gw) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= rows * d) return;
    const int64_t r = i / d;
    const int c = (int)(i - r * d), g = c / gw, ci = c - g * gw;
    const int G = d / gw;
    x[i] += gelu_erff(tmp[r * (int64_t)(G * 64) + g * 64 + ci] + bias[c]);
}

// logits f32 [n*T, ldl] -> log_softmax over the first V columns, written to the caller's [frames_c, V] block of window c
__global__ void __launch_bounds__(128)
w2v_log_softmax_kernel(const float* __restrict__ logits, int ldl, int V, int T, const int* __restrict__ frames,
                       float* __restrict__ out, int64_t window_stride) {
    const int t = blockIdx.x, b = blockIdx.y;
    if (t >= frames[b]) return;
    const float* l = logits + ((int64_t)b * T + t) * ldl;
    __shared__ float red[4];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float m = -INFINITY;
    for (int v = threadIdx.x; v < V; v += 128) m = fmaxf(m, l[v]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) red[warp] = m;
    __syncthreads();
    m = fmaxf(fmaxf(red[0], red[1]), fmaxf(red[2], red[3]));
    __syncthreads();
    float s = 0.0f;
    for (int v = threadIdx.x; v < V; v += 128) s += expf(l[v] - m);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) red[warp] = s;
    __syncthreads();
    const float lse = m + logf((red[0] + red[1]) + (red[2] + red[3]));
    float* o = out + (int64_t)b * window_stride + (int64_t)t * V;
    for (int v = threadIdx.x; v < V; v += 128) o[v] = l[v] - lse;
}

// ---- CTC forced alignment ------------------------------------------------------------------------------------------
// best non-blank log-probability per frame (the score of a '*' wildcard token), one warp per (window, frame)
__global__ void __launch_bounds__(256)
ctc_wild_kernel(const float* __restrict__ em, int64_t window_stride, int V, const int* __restrict__ frames, int blank,
                float* __restrict__ wild, int max_frames) {
    const int b = blockIdx.y, t = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (t >= frames[b] || t >= max_frames) return;
    const float* e = em + (int64_t)b * window_stride + (int64_t)t * V;
    float m = -INFINITY;
    for (int v = lane; v < V; v += 32)
        if (v != blank) m = fmaxf(m, e[v]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0) wild[(int64_t)b * max_frames + t] = m;
}

// One CTA per window.  trellis[t][j] = best score with tokens[0..j] entered after t frames (whisperx get_trellis): a frame
// either stays on token j (scores blank) or enters it (scores tokens[j]); column 0 accumulates blank from frame 1 on.
// Rows live in shared memory (double-buffered) and are spilled to the global trellis for the backtrack, which thread 0
// walks afterwards exactly as whisperx.backtrack does ('changed > stayed' decides, ties stay).
__global__ void __launch_bounds__(256)
ctc_align_kernel(const float* __restrict__ em, int64_t window_stride, int V, const int* __restrict__ frames,
                 const int* __restrict__ tokens, int max_tokens, const int* __restrict__ n_tokens, int blank,
                 float* __restrict__ trellis_ws, const float* __restrict__ wild_ws, int max_frames,
                 int* __restrict__ frame_token, float* __restrict__ frame_score, int* __restrict__ ok) {
    extern __shared__ float rows[];
    const int b = blockIdx.x, tid = threadIdx.x;
    const int T = min(frames[b], max_frames), N = n_tokens[b];
    int* ftok = frame_token + (int64_t)b * max_frames;
    float* fsc = frame_score + (int64_t)b * max_frames;
    if (N <= 0 || N > max_tokens || T <= 0 || N > T) {
        for (int t = tid; t < max_frames; t += 256) { ftok[t] = 0; fsc[t] = 0.0f; }
        if (tid == 0) ok[b] = 0;
        return;
    }
    const float* e0 = em + (int64_t)b * window_stride;
    const int* tok = tokens + (int64_t)b * max_tokens;
    const float* wild = wild_ws + (int64_t)b * max_frames;
    float* tr = trellis_ws + (int64_t)b * max_frames * max_tokens;
    float* prev = rows;
    float* cur = rows + max_tokens;
    for (int j = tid; j < N; j += 256) {
        prev[j] = j == 0 ? 0.0f : -INFINITY;
        tr[j] = prev[j];
    }
    __syncthreads();
    for (int t = 0; t + 1 < T; ++t) {
        const float* e = e0 + (int64_t)t * V;
        const float eb = e[blank];
        for (int j = tid; j < N; j += 256) {
            float v;
            if (j == 0) {
                v = prev[0] + e[V + blank];                     // cumsum of emission[1.., blank]
            } else {
                const int k = tok[j];
                const float et = k < 0 ? wild[t] : e[k];
                v = fmaxf(prev[j] + eb, prev[j - 1] + et);
            }
            cur[j] = v;
            tr[(int64_t)(t + 1) * max_tokens + j] = v;
        }
        __syncthreads();
        float* tmp = prev; prev = cur; cur = tmp;
    }
    if (tid != 0) return;
    __threadfence_block();
    int t = T - 1, j = N - 1, good = 1;
    ftok[t] = j;
    fsc[t] = expf(e0[(int64_t)t * V + blank]);
    while (j > 0) {
        if (t <= 0) { good = 0; break; }
        const float* e = e0 + (int64_t)(t - 1) * V;
        const float p_stay = e[blank];
        const int k = tok[j];
        const float p_change = k < 0 ? wild[t - 1] : e[k];
        const float stayed = tr[(int64_t)(t - 1) * max_tokens + j] + p_stay;
        const float changed = tr[(int64_t)(t - 1) * max_tokens + j - 1] + p_change;
        --t;
        if (changed > stayed) { --j; fsc[t] = expf(p_change); }
        else fsc[t] = expf(p_stay);
        ftok[t] = j;
    }
    while (t > 0) {
        ftok[t - 1] = j;
        fsc[t - 1] = expf(e0[(int64_t)(t - 1) * V + blank]);
        --t;
    }
    for (int tt = T; tt < max_frames; ++tt) { ftok[tt] = N - 1; fsc[tt] = 0.0f; }
    ok[b] = good;
}

mw_status w2v_alloc(mw_w2v* m, void** ptr, int64_t bytes) {
    MW_CUDA_CHECK(cudaMalloc(ptr, (size_t)bytes));
    m->allocations.push_back(*ptr);
    m->workspace_bytes += bytes;
    MW_CUDA_CHECK(cudaMemset(*ptr, 0, (size_t)bytes));      // padding rows must stay finite (masked keys still meet P = 0)
    return MW_OK;
}

}  // namespace
}  // namespace mw

extern "C" int32_t mw_w2v_frames(int64_t n_samples) { return mw::conv_frames(n_samples); }

extern "C" mw_status mw_w2v_create(const mw_w2v_config* cfg, const mw_weight_table* weights, mw_w2v** out_model) {
    MW_REQUIRE(cfg && weights && out_model, "mw_w2v_create: null argument");
    MW_REQUIRE(cfg->d_model == cfg->n_heads * 64, "mw_w2v_create: d_head must be 64 (d_model=%d n_heads=%d)", cfg->d_model, cfg->n_heads);
    MW_REQUIRE(cfg->d_model % 128 == 0 && cfg->ffn % 128 == 0, "mw_w2v_create: d_model and ffn must be multiples of 128");
    MW_REQUIRE(cfg->conv_dim == 128 || cfg->conv_dim == 256 || cfg->conv_dim == 512, "mw_w2v_create: conv_dim must be 128, 256 or 512");
    MW_REQUIRE(cfg->variant == 0 || cfg->variant == 1, "mw_w2v_create: variant must be 0 (XLSR family) or 1 (wav2vec2-base)");
    MW_REQUIRE(cfg->pos_groups > 0 && cfg->d_model % cfg->pos_groups == 0, "mw_w2v_create: d_model must be a multiple of pos_groups");
    {
        const int gw = cfg->d_model / cfg->pos_groups;
        MW_REQUIRE(gw == 64 || (cfg->variant == 1 && gw % 8 == 0 && gw < 64 && (cfg->pos_kernel * gw) % 64 == 0),
                   "mw_w2v_create: d_model / pos_groups = %d is not supported (64; or a multiple of 8 below 64 for variant 1)", gw);
    }
    MW_REQUIRE(cfg->pos_kernel >= 2 && cfg->pos_kernel % 2 == 0, "mw_w2v_create: pos_kernel must be even");
    MW_REQUIRE(cfg->max_batch > 0 && cfg->max_samples >= 400 && cfg->vocab > 1 && cfg->n_layers > 0, "mw_w2v_create: bad sizes");
    const int expect = MW_A_GLOBAL_COUNT + cfg->n_layers * MW_EL_COUNT;
    MW_REQUIRE(weights->n == expect, "mw_w2v_create: weight table has %d entries, expected %d", weights->n, expect);
    for (int i = 0; i < expect; ++i) MW_REQUIRE(weights->ptrs[i] != nullptr, "mw_w2v_create: weight %d is null", i);
    mw::DeviceGuard guard(cfg->device);
    mw_w2v* m = new mw_w2v();
    m->cfg = *cfg;
    m->w.assign(weights->ptrs, weights->ptrs + expect);
    m->vocab_pad = (cfg->vocab + 31) / 32 * 32;
    for (int l = 0; l < 7; ++l) m->T_max[l] = mw::conv_frames(cfg->max_samples, l + 1);
    const int64_t B = cfg->max_batch, C = cfg->conv_dim, d = cfg->d_model, T = m->T_max[6];
    mw_status s = MW_OK;
    auto A = [&](void** p, int64_t bytes) { if (s == MW_OK) s = mw::w2v_alloc(m, p, bytes); };
    A((void**)&m->act_a, B * m->T_max[0] * C * 2);
    A((void**)&m->act_b, B * m->T_max[1] * C * 2);
    A((void**)&m->conv_f32, B * m->T_max[1] * C * 4);
    A((void**)&m->feat, B * T * C * 4);
    A((void**)&m->x, B * T * d * 4);
    A((void**)&m->xg, B * (T + cfg->pos_kernel) * d * 2);
    A((void**)&m->ln, B * T * std::max(d, C) * 2);
    A((void**)&m->qkv, B * T * 3 * d * 2);
    A((void**)&m->att, B * T * d * 2);
    A((void**)&m->mlp, B * T * cfg->ffn * 2);
    A((void**)&m->logits, B * T * m->vocab_pad * 4);
    A((void**)&m->d_frames, B * 4);
    if (cfg->variant == 1) {
        A((void**)&m->gn_partial, B * ((m->T_max[0] + 63) / 64) * 2 * C * 4);
        A((void**)&m->gn_stats, B * C * 2 * 4);
        if (d / cfg->pos_groups != 64) A((void**)&m->pos_tmp, B * T * cfg->pos_groups * 64 * 4);
    }
    if (s != MW_OK) { mw_w2v_destroy(m); return s; }
    *out_model = m;
    return MW_OK;
}

extern "C" void mw_w2v_destroy(mw_w2v* m) {
    if (!m) return;
    mw::DeviceGuard guard(m->cfg.device);
    for (void* p : m->allocations) cudaFree(p);
    delete m;
}

extern "C" int64_t mw_w2v_workspace_bytes(const mw_w2v* m) { return m ? m->workspace_bytes : 0; }

extern "C" mw_status mw_w2v_emissions(mw_w2v* m, const float* d_audio, int64_t n_audio, const int64_t* d_offsets,
                                      const int32_t* d_lengths, const int32_t* h_lengths, int n, float* d_out,
                                      int64_t out_window_stride, void* stream) {
    using namespace mw;
    MW_REQUIRE(m && d_audio && d_offsets && d_lengths && h_lengths && d_out, "mw_w2v_emissions: null argument");
    const mw_w2v_config& c = m->cfg;
    MW_REQUIRE(n > 0 && n <= c.max_batch, "mw_w2v_emissions: n=%d outside 1..max_batch=%d", n, c.max_batch);
    int S = 400;
    for (int i = 0; i < n; ++i) {
        MW_REQUIRE(h_lengths[i] >= 0 && h_lengths[i] <= c.max_samples, "mw_w2v_emissions: window %d has %d samples, max_samples=%d",
                   i, h_lengths[i], c.max_samples);
        S = std::max(S, (int)h_lengths[i]);
    }
    int Tl[7];
    for (int l = 0; l < 7; ++l) Tl[l] = conv_frames(S, l + 1);
    const int T = Tl[6], C = c.conv_dim, d = c.d_model;
    MW_REQUIRE(out_window_stride >= (int64_t)T * c.vocab, "mw_w2v_emissions: out_window_stride too small for %d frames", T);
    DeviceGuard guard(c.device);
    cudaStream_t st = (cudaStream_t)stream;
    mw_status s;
    w2v_frames_kernel<<<ceil_div(n, 128), 128, 0, st>>>(d_lengths, n, m->d_frames);
    MW_LAUNCH_CHECK();
    const bool base = c.variant == 1;
    if (base) {
        const int n_blk = ceil_div(Tl[0], 64);
        dim3 grid(n_blk, n);
        const float* w0 = (const float*)m->gw(MW_A_CONV0_W);
        const float* g0 = (const float*)m->gw(MW_A_CONV0_LN_G);
        const float* be0 = (const float*)m->gw(MW_A_CONV0_LN_B);
#define MW_GN(np)                                                                                                              \
        w2v_conv0_gn_kernel<np, 0><<<grid, 256, 0, st>>>(d_audio, n_audio, d_offsets, d_lengths, w0, g0, be0, m->gn_partial,    \
                                                         nullptr, m->act_a, Tl[0], n_blk);                                      \
        MW_LAUNCH_CHECK();                                                                                                      \
        w2v_gn_finalize_kernel<<<n, 256, 0, st>>>(m->gn_partial, d_lengths, m->gn_stats, C, n_blk);                             \
        MW_LAUNCH_CHECK();                                                                                                      \
        w2v_conv0_gn_kernel<np, 1><<<grid, 256, 0, st>>>(d_audio, n_audio, d_offsets, d_lengths, w0, g0, be0, nullptr,          \
                                                         m->gn_stats, m->act_a, Tl[0], n_blk);                                  \
        MW_LAUNCH_CHECK();
        if (C == 512) { MW_GN(8) } else if (C == 256) { MW_GN(4) } else { MW_GN(2) }
#undef MW_GN
    } else {
        dim3 grid(ceil_div(Tl[0], 64), n);
        const float* w0 = (const float*)m->gw(MW_A_CONV0_W);
        const float* b0 = (const float*)m->gw(MW_A_CONV0_B);
        const float* g0 = (const float*)m->gw(MW_A_CONV0_LN_G);
        const float* be0 = (const float*)m->gw(MW_A_CONV0_LN_B);
        if (C == 512) w2v_conv0_kernel<8><<<grid, 256, 0, st>>>(d_audio, n_audio, d_offsets, d_lengths, w0, b0, g0, be0, m->act_a, Tl[0]);
        else if (C == 256) w2v_conv0_kernel<4><<<grid, 256, 0, st>>>(d_audio, n_audio, d_offsets, d_lengths, w0, b0, g0, be0, m->act_a, Tl[0]);
        else w2v_conv0_kernel<2><<<grid, 256, 0, st>>>(d_audio, n_audio, d_offsets, d_lengths, w0, b0, g0, be0, m->act_a, Tl[0]);
        MW_LAUNCH_CHECK();
    }
    const mw_h* in = m->act_a;
    for (int l = 1; l < 7; ++l) {
        GemmArgs a;
        a.a = in; a.a_row_stride = (int64_t)CONV_S[l] * C; a.a_batch_stride = (int64_t)Tl[l - 1] * C;
        a.w = m->gw(MW_A_CONV0_W + 4 * l); a.w_row_stride = (int64_t)CONV_K[l] * C;
        void* out = l == 6 ? (void*)m->feat : (void*)((l & 1) ? m->act_b : m->act_a);
        if (base) {      // conv (no bias) + GELU in the GEMM epilogue, no norm; the last layer stays fp32 (it feeds a LayerNorm)
            a.out = out; a.out_batch_rows = Tl[l]; a.ld_out = C;
            a.batch = n; a.M = Tl[l]; a.N = C; a.K = CONV_K[l] * C; a.gelu = true; a.out_f32 = l == 6;
            if ((s = gemm_launch(a, st)) != MW_OK) return s;
            in = (const mw_h*)out;
            continue;
        }
        a.bias = (const float*)m->gw(MW_A_CONV0_W + 4 * l + 1);
        a.out = m->conv_f32; a.out_batch_rows = Tl[l]; a.ld_out = C;
        a.batch = n; a.M = Tl[l]; a.N = C; a.K = CONV_K[l] * C; a.out_f32 = true;
        if ((s = gemm_launch(a, st)) != MW_OK) return s;
        if ((s = layernorm_act_launch(m->conv_f32, (const float*)m->gw(MW_A_CONV0_W + 4 * l + 2),
                                      (const float*)m->gw(MW_A_CONV0_W + 4 * l + 3), out, n * Tl[l], C, l == 6 ? 2 : 1, st)) != MW_OK)
            return s;
        in = (const mw_h*)out;
    }
    const int rows = n * T;
    if ((s = layernorm_launch(m->feat, (const float*)m->gw(MW_A_FP_LN_G), (const float*)m->gw(MW_A_FP_LN_B), m->ln, rows, C, st)) != MW_OK) return s;
    {
        GemmArgs a;
        a.a = m->ln; a.a_row_stride = C; a.w = m->gw(MW_A_FP_W); a.w_row_stride = C;
        a.bias = (const float*)m->gw(MW_A_FP_B);
        a.out = m->x; a.ld_out = d; a.M = rows; a.N = d; a.K = C; a.out_f32 = true;
        if ((s = gemm_launch(a, st)) != MW_OK) return s;
    }
    {   // x += GELU(pos_conv(x) + bias): one implicit GEMM per 64-channel group over the group-major copy
        const int kp = c.pos_kernel, G = c.pos_groups, gw = d / G;
        w2v_group_major_kernel<<<dim3(T + kp, n), 256, 0, st>>>(m->x, m->d_frames, m->xg, T, d, kp, gw);
        MW_LAUNCH_CHECK();
        for (int g = 0; g < G; ++g) {
            GemmArgs a;
            a.a = m->xg + (int64_t)g * (T + kp) * gw; a.a_row_stride = gw; a.a_batch_stride = (int64_t)G * (T + kp) * gw;
            a.w = (const mw_h*)m->gw(MW_A_POS_W) + (int64_t)g * 64 * kp * gw; a.w_row_stride = (int64_t)kp * gw;
            a.batch = n; a.M = T; a.N = 64; a.K = kp * gw; a.out_f32 = true;
            if (gw == 64) {
                a.bias = (const float*)m->gw(MW_A_POS_B) + g * 64;
                a.residual = m->x + g * 64; a.res_batch_rows = T; a.ld_res = d;
                a.out = m->x + g * 64; a.out_batch_rows = T; a.ld_out = d;
                a.gelu = true;
            } else {     // narrower groups: 64 padded output columns per group into a scratch buffer, added below
                a.out = m->pos_tmp + g * 64; a.out_batch_rows = T; a.ld_out = (int64_t)G * 64;
            }
            if ((s = gemm_launch(a, st)) != MW_OK) return s;
        }
        if (gw != 64) {
            const int64_t tot = (int64_t)rows * d;
            w2v_pos_add_kernel<<<(unsigned)ceil_div64(tot, 256), 256, 0, st>>>(m->pos_tmp, (const float*)m->gw(MW_A_POS_B), m->x, rows, d, gw);
            MW_LAUNCH_CHECK();
        }
    }
    { const char* e = getenv("MW_W2V_STOP"); if (e && e[0] == 'p') return MW_OK; }      // debug: x = projection + pos conv
    if (base)      // post-LayerNorm encoder: the encoder LayerNorm comes right after the positional embedding
        if ((s = layernorm_dual_launch(m->x, (const float*)m->gw(MW_A_ENC_LN_G), (const float*)m->gw(MW_A_ENC_LN_B), m->ln, rows, d, st)) != MW_OK) return s;
    for (int l = 0; l < c.n_layers; ++l) {
        if (!base && (s = layernorm_launch(m->x, (const float*)m->lw(l, MW_EL_LN1_G), (const float*)m->lw(l, MW_EL_LN1_B), m->ln, rows, d, st)) != MW_OK) return s;
        {
            GemmArgs a;
            a.a = m->ln; a.a_row_stride = d; a.w = m->lw(l, MW_EL_WQKV); a.w_row_stride = d;
            a.bias = (const float*)m->lw(l, MW_EL_BQKV);
            a.out = m->qkv; a.ld_out = 3 * d; a.M = rows; a.N = 3 * d; a.K = d;
            if ((s = gemm_launch(a, st)) != MW_OK) return s;
        }
        if ((s = attention_launch(m->qkv, m->att, n, T, c.n_heads, st, m->d_frames)) != MW_OK) return s;
        {
            GemmArgs a;
            a.a = m->att; a.a_row_stride = d; a.w = m->lw(l, MW_EL_WO); a.w_row_stride = d;
            a.bias = (const float*)m->lw(l, MW_EL_BO);
            a.residual = m->x; a.ld_res = d;
            a.out = m->x; a.ld_out = d; a.M = rows; a.N = d; a.K = d; a.out_f32 = true;
            if ((s = gemm_launch(a, st)) != MW_OK) return s;
        }
        if (base) {      // x = LN(x + attn(x)): written back as the residual stream and as the fc1 operand
            if ((s = layernorm_dual_launch(m->x, (const float*)m->lw(l, MW_EL_LN1_G), (const float*)m->lw(l, MW_EL_LN1_B), m->ln, rows, d, st)) != MW_OK) return s;
        } else if ((s = layernorm_launch(m->x, (const float*)m->lw(l, MW_EL_LN2_G), (const float*)m->lw(l, MW_EL_LN2_B), m->ln, rows, d, st)) != MW_OK) return s;
        {
            GemmArgs a;
            a.a = m->ln; a.a_row_stride = d; a.w = m->lw(l, MW_EL_W1); a.w_row_stride = d;
            a.bias = (const float*)m->lw(l, MW_EL_B1);
            a.out = m->mlp; a.ld_out = c.ffn; a.M = rows; a.N = c.ffn; a.K = d; a.gelu = true;
            if ((s = gemm_launch(a, st)) != MW_OK) return s;
        }
        {
            GemmArgs a;
            a.a = m->mlp; a.a_row_stride = c.ffn; a.w = m->lw(l, MW_EL_W2); a.w_row_stride = c.ffn;
            a.bias = (const float*)m->lw(l, MW_EL_B2);
            a.residual = m->x; a.ld_res = d;
            a.out = m->x; a.ld_out = d; a.M = rows; a.N = d; a.K = c.ffn; a.out_f32 = true;
            if ((s = gemm_launch(a, st)) != MW_OK) return s;
        }
        if (base && (s = layernorm_dual_launch(m->x, (const float*)m->lw(l, MW_EL_LN2_G), (const float*)m->lw(l, MW_EL_LN2_B), m->ln, rows, d, st)) != MW_OK) return s;
    }
    if (!base && (s = layernorm_launch(m->x, (const float*)m->gw(MW_A_ENC_LN_G), (const float*)m->gw(MW_A_ENC_LN_B), m->ln, rows, d, st)) != MW_OK) return s;
    {
        GemmArgs a;
        a.a = m->ln; a.a_row_stride = d; a.w = m->gw(MW_A_LM_W); a.w_row_stride = d;
        a.bias = (const float*)m->gw(MW_A_LM_B);
        a.out = m->logits; a.ld_out = m->vocab_pad; a.M = rows; a.N = m->vocab_pad; a.K = d; a.out_f32 = true;
        if ((s = gemm_launch(a, st)) != MW_OK) return s;
    }
    w2v_log_softmax_kernel<<<dim3(T, n), 128, 0, st>>>(m->logits, m->vocab_pad, c.vocab, T, m->d_frames, d_out, out_window_stride);
    MW_LAUNCH_CHECK();
    return MW_OK;
}

extern "C" mw_status mw_ctc_align(const float* d_emissions, int64_t window_stride, int vocab, const int32_t* d_frames,
                                  const int32_t* d_tokens, int max_tokens, const int32_t* d_n_tokens, int n, int blank,
                                  int32_t* d_frame_token, float* d_frame_score, int max_frames, int32_t* d_ok,
                                  float* d_workspace, void* stream) {
    using namespace mw;
    MW_REQUIRE(d_emissions && d_frames && d_tokens && d_n_tokens && d_frame_token && d_frame_score && d_ok && d_workspace,
               "mw_ctc_align: null argument");
    MW_REQUIRE(n > 0 && vocab > 1 && blank >= 0 && blank < vocab, "mw_ctc_align: bad n/vocab/blank");
    MW_REQUIRE(max_tokens > 0 && max_tokens <= 4096 && max_frames > 0, "mw_ctc_align: max_tokens must be in 1..4096, max_frames positive");
    MW_REQUIRE(window_stride >= (int64_t)max_frames * vocab, "mw_ctc_align: window_stride smaller than max_frames * vocab");
    cudaStream_t st = (cudaStream_t)stream;
    float* wild = d_workspace + (int64_t)n * max_frames * max_tokens;
    ctc_wild_kernel<<<dim3(ceil_div(max_frames, 8), n), 256, 0, st>>>(d_emissions, window_stride, vocab, d_frames, blank, wild, max_frames);
    MW_LAUNCH_CHECK();
    ctc_align_kernel<<<n, 256, 2 * max_tokens * sizeof(float), st>>>(d_emissions, window_stride, vocab, d_frames, d_tokens, max_tokens,
                                                                     d_n_tokens, blank, d_workspace, wild, max_frames, d_frame_token,
                                                                     d_frame_score, d_ok);
    MW_LAUNCH_CHECK();
    return MW_OK;
}

// test hook: copy one of the model's internal buffers of the last mw_w2v_emissions call to the caller (device to device).
// which: 0 = conv stack output feat f32 [n*T, C], 1 = residual stream x f32 [n*T, d], 2 = GroupNorm statistics f32 [n, C, 2],
// 3 = conv0 output h16 [n, T_0, C]
extern "C" mw_status mw_w2v_debug_copy(mw_w2v* m, int which, void* d_dst, int64_t nbytes, void* stream) {
    MW_REQUIRE(m && d_dst && nbytes > 0, "mw_w2v_debug_copy: bad argument");
    const void* src = which == 0 ? (const void*)m->feat : which == 1 ? (const void*)m->x : which == 2 ? (const void*)m->gn_stats
                                                                                         : (const void*)m->act_a;
    MW_REQUIRE(src != nullptr, "mw_w2v_debug_copy: buffer %d is not allocated for this variant", which);
    MW_CUDA_CHECK(cudaMemcpyAsync(d_dst, src, (size_t)nbytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return MW_OK;
}
