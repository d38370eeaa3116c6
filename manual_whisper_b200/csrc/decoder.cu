// Batched autoregressive decoder (S3: ctranslate2.models.Whisper.generate, SURVEY.md §8 a8/a9, A.8).
//
// Per chunk, once:   cross K/V projection of the encoder output for every layer (tcgen05 GEMM).
// Per step (R = B*beam rows, one token each), replayed as a CUDA graph:
//   embed -> L x { LN -> qkv skinny GEMM -> self-attention over the KV cache (appends k,v)
//                  -> out-proj (+residual) -> LN -> cross-q GEMM -> cross-attention over the chunk's K/V
//                  -> out-proj (+residual) -> LN -> fc1 (GELU) -> fc2 (+residual) }
//   -> LN -> logits = h E^T (skinny GEMM over the tied embedding) -> select (suppress / timestamp rules,
//   log-softmax, argmax or beam candidates) entirely on device; ids reach the host once at the end.
//
// The step is HBM-bound: every weight byte and every cross-K/V byte is streamed exactly once per step.
// "Skinny" GEMMs put the weight rows on the M side of mma.sync.m16n8k16 (bf16, fp32 accumulate) so each
// weight element is loaded once as a 16-byte vector and reused for all R rows.
#include "model.cuh"
#include "gemm.cuh"
#include "kernels.cuh"
#include "ptx_sm100.cuh"

#include <algorithm>
#include <stdlib.h>
#include <vector>

namespace mw {

struct DecCtl {
    int pos;        // position of the token being fed this step
    int step;       // steps executed so far (prefill + generated)
    int n_done;     // rows (greedy) or chunks (beam) finished
    int pad;
};

struct GenOptsDev {
    int eot, timestamp_begin, with_timestamps, max_initial_ts;
    int forced_eot_len, beam, max_new, max_fin;
    float length_penalty;
    int n_prefill;      // forced steps before sampling starts
    int vocab, pad;
};

constexpr int MAX_BEAM = 8;
constexpr int NCAND = 2 * MAX_BEAM;

}  // namespace mw

struct DecoderState {
    int R_max = 0, max_new = 0;
    mw_h* kv_cross = nullptr;   // [L][B*T][2d]
    mw_h* k_self = nullptr;     // [L][R][ctx][d]
    mw_h* v_self = nullptr;
    float* x = nullptr;                  // [R, d]
    mw_h* ln = nullptr;         // [R, d]
    mw_h* qkv = nullptr;        // [R, 3d]
    mw_h* qx = nullptr;         // [R, d]
    mw_h* att = nullptr;        // [R, d]
    mw_h* mlp = nullptr;        // [R, ffn]
    float* logits = nullptr;             // [R, V]
    int* cur_tok = nullptr;              // [R]
    mw::DecCtl* ctl = nullptr;
    mw::GenOptsDev* opts = nullptr;
    int* prompt = nullptr;               // [ctx]
    uint8_t* sup_mask = nullptr;         // [V] 1 = always masked
    uint8_t* begin_mask = nullptr;       // [V] 1 = masked at the first generated step
    // per-row generation state (double-buffered where beam search re-parents rows)
    int* tokens[2] = {nullptr, nullptr}; // [R][max_new]
    int* gen_len = nullptr;              // [R]
    int* done = nullptr;                 // [R]
    float* cum = nullptr;                // [R]
    int* last_ts[2] = {nullptr, nullptr};// [R] most recent timestamp token or -1
    int* self_idx[2] = {nullptr, nullptr};   // [R][ctx] physical cache row holding position p (beam search)
    // beam search
    float* cand_val = nullptr;           // [R][NCAND]
    int* cand_idx = nullptr;             // [R][NCAND]
    float* row_lse = nullptr;            // [R]
    int* fin_count = nullptr;            // [B]
    float* fin_score = nullptr;          // [B][MAX_BEAM]
    int* fin_len = nullptr;              // [B][MAX_BEAM]
    int* fin_tok = nullptr;              // [B][MAX_BEAM][max_new]
    int* active = nullptr;               // [B]
    // host side
    mw::DecCtl* h_ctl = nullptr;         // pinned [2]
    cudaStream_t cap_stream = nullptr;
    int parts_epoch = 0;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    // step graphs are specific to (rows, beam): a small cache keeps the last few shapes (full batches and the short
    // last batch of a recording alternate) so they are not re-captured on every call
    bool solo = false;                   // mw_set_solo: this replica decodes alone on its GPU (latency mode, see sk_choose)
    struct Graphs { int R = 0, beam = 0; bool solo = false; int n_prefill = 0, n_gen[2] = {0, 0}; uint64_t last_use = 0; cudaGraphExec_t prefill = nullptr, gen[2] = {nullptr, nullptr}; };
    static constexpr int GRAPH_CACHE = 4;
    Graphs graph_cache[GRAPH_CACHE];
    uint64_t graph_clock = 0;
    Graphs graphs;                       // the entry selected by ensure_graphs for the current call (non-owning copy)
};

namespace mw {

namespace {

// ------------------------------------------------------------------------------------------------
// skinny GEMM: out[r, n] = sum_k X[r, k] W[n, k] (+bias) (gelu) (+resid);  R small, N x K streamed once.
// A CTA owns 32 rows of X and WT 16-row weight tiles.  Lane (g, q) = (lane / 4, lane % 4) holds the mma.sync fragments of
// weight rows g, g + 8 and X rows t * 8 + g (t < 4), columns q * 8 .. q * 8 + 7 of each 32-wide K block.  Every warp sums
// its share of K, parks the sums in a shared-memory slot, and the slots are summed in order.
// ------------------------------------------------------------------------------------------------
constexpr int SK_FLAG_GELU = 1, SK_FLAG_F32 = 2;

__device__ __forceinline__ void mma_h16_16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                               uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32." MW_MMA_SYNC_TYPE "." MW_MMA_SYNC_TYPE ".f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// A weight load: a weight byte is read once per step, so its line is marked evict_first in L2.  `volatile` keeps the loads
// in program order ahead of the MMAs, so a kernel's whole weight slice is in flight before the first MMA waits.
__device__ __forceinline__ uint4 ldg_stream(const void* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.u32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p), "l"(ptx::l2_policy_evict_first()));
    return r;
}

// Weight prefetch: a decode step is a serial chain of short kernels whose weights arrive cold from HBM (one DRAM round trip
// per launch with nothing else in flight).  Every projection kernel therefore asks L2 for the NEXT projection's weight
// matrix once its own weights have arrived (`pf`, `pf_lines` 128-byte lines, spread over the grid's threads), so the next
// kernel's stream starts from L2; the cross-attention kernel does the same for its output projection.
// With several batches in flight, the other batches stream cross-attention K/V and self-attention K/V through L2 between
// the prefetch and the load that consumes it.  Those streams are loaded evict_first and the prefetch marks its lines
// evict_last, so L2 gives up the streamed lines first and the prefetched weights are still there when they are read.
// The consuming load (ldg_stream) is evict_first, and a hinted access re-marks a resident line (the PTX ISA's
// evict_unchanged priority exists to opt out of that), so a weight line is demoted once it has been read and evict_last
// lines do not pile up: at any time they are at most the next matrix of each batch in flight.
__device__ __forceinline__ void l2_prefetch_slice(const char* pf, int pf_lines) {
    if (!pf) return;
    const int nthr = gridDim.x * gridDim.y * blockDim.x;
    for (int i = (blockIdx.y * gridDim.x + blockIdx.x) * blockDim.x + threadIdx.x; i < pf_lines; i += nthr)
        ptx::prefetch_l2_evict_last(pf + (int64_t)i * 128);
}

// The weight fragments of WT tiles (rows n0 + 16 wt + g and + 8, clamped to N - 1) x KB blocks from column k0 (q * 8 included)
template <int WT, int KB>
__device__ __forceinline__ void sk_load_w(uint4 (&alo)[WT][KB], uint4 (&ahi)[WT][KB], const mw_h* W, int ldw, int N, int n0,
                                          int g, int k0) {
#pragma unroll
    for (int wt = 0; wt < WT; ++wt) {
        const mw_h* wa = W + (int64_t)min(n0 + wt * 16 + g, N - 1) * ldw + k0;
        const mw_h* wb = W + (int64_t)min(n0 + wt * 16 + g + 8, N - 1) * ldw + k0;
#pragma unroll
        for (int i = 0; i < KB; ++i) {
            alo[wt][i] = ldg_stream(wa + i * 32);
            ahi[wt][i] = ldg_stream(wb + i * 32);
        }
    }
}

// The MMAs of loaded K block i against the four X fragments x_frag(t) (rows t * 8 + g).  x_frag reads X from global memory
// or from shared memory; it is inlined, so the choice is made at compile time.
template <int WT, int KB, typename XFrag>
__device__ __forceinline__ void sk_mma_block(float (&c)[WT][4][4], const uint4 (&alo)[WT][KB], const uint4 (&ahi)[WT][KB], int i,
                                             XFrag x_frag) {
    uint4 b[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) b[t] = x_frag(t);
#pragma unroll
    for (int wt = 0; wt < WT; ++wt)
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            mma_h16_16816(c[wt][t], alo[wt][i].x, ahi[wt][i].x, alo[wt][i].y, ahi[wt][i].y, b[t].x, b[t].y);
            mma_h16_16816(c[wt][t], alo[wt][i].z, ahi[wt][i].z, alo[wt][i].w, ahi[wt][i].w, b[t].z, b[t].w);
        }
}

// The accumulators into a reduction slot at their fragment positions (rows t * 8 + 2q, + 1; columns 16 wt + g, + 8)
template <int WT>
__device__ __forceinline__ void sk_park(float (&slot)[32][WT * 16 + 1], const float (&c)[WT][4][4], int g, int q) {
#pragma unroll
    for (int wt = 0; wt < WT; ++wt)
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            slot[t * 8 + 2 * q][wt * 16 + g] = c[wt][t][0];
            slot[t * 8 + 2 * q + 1][wt * 16 + g] = c[wt][t][1];
            slot[t * 8 + 2 * q][wt * 16 + g + 8] = c[wt][t][2];
            slot[t * 8 + 2 * q + 1][wt * 16 + g + 8] = c[wt][t][3];
        }
}

// Output (r0 + rl, n0 + nl): reduction slots 0 .. NS-1 summed in order (+bias) (GELU) (+resid), stored f32 or 16-bit
template <int NS, int LD>
__device__ __forceinline__ void sk_output(float (*red)[32][LD], int rl, int nl, int r0, int n0, int R, int N,
                                          const float* __restrict__ bias, const float* resid, void* out, int ldo, int flags) {
    const int r = r0 + rl, n = n0 + nl;
    float v = 0.0f;
#pragma unroll
    for (int w = 0; w < NS; ++w) v += red[w][rl][nl];
    if (r < R && n < N) {
        if (bias) v += __ldg(bias + n);
        if (flags & SK_FLAG_GELU) v = gelu_erff(v);
        const int64_t oi = (int64_t)r * ldo + n;
        if (resid) v += resid[oi];
        if (flags & SK_FLAG_F32) reinterpret_cast<float*>(out)[oi] = v;
        else reinterpret_cast<mw_h*>(out)[oi] = f2h(v);
    }
}

// Any K % 32 == 0: grid (ceil(N/16), ceil(R/32)), 256 threads; warp w owns K blocks w, w+8, ...  At most 64 registers, so
// 4 CTAs fit an SM (the cache policy of the weight loads would otherwise take it to 70 and 3 CTAs).
__global__ void __launch_bounds__(256, 4)
skinny_gemm_kernel(const mw_h* __restrict__ X, int ldx, const mw_h* __restrict__ W, int ldw,
                   const float* __restrict__ bias, const float* resid, void* out, int ldo, int R, int N, int K,
                   int flags) {
    __shared__ float red[8][32][17];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, q = lane & 3;
    const int n0 = blockIdx.x * 16, r0 = blockIdx.y * 32;
    const mw_h* wa = W + (int64_t)min(n0 + g, N - 1) * ldw + q * 8;
    const mw_h* wb = W + (int64_t)min(n0 + g + 8, N - 1) * ldw + q * 8;
    const mw_h* xr[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) xr[t] = X + (int64_t)min(r0 + t * 8 + g, R - 1) * ldx + q * 8;
    float c[1][4][4] = {};
    const int nkb = K >> 5;
#pragma unroll 2
    for (int kb = warp; kb < nkb; kb += 8) {
        const int k = kb << 5;
        const uint4 alo[1][1] = {{ldg_stream(wa + k)}}, ahi[1][1] = {{ldg_stream(wb + k)}};
        sk_mma_block(c, alo, ahi, 0, [&](int t) { return __ldg(reinterpret_cast<const uint4*>(xr[t] + k)); });
    }
    sk_park(red[warp], c, g, q);
    __syncthreads();
#pragma unroll
    for (int o = threadIdx.x; o < 512; o += 256) sk_output<8>(red, o >> 4, o & 15, r0, n0, R, N, bias, resid, out, ldo, flags);
}

// Main version: a CTA owns 16 weight rows and the whole K; its NW warps split K into contiguous runs of KB
// 32-element blocks and issue EVERY weight load (ld.global.nc, L1 no-allocate) before touching
// anything else, so a kernel's whole matrix is in flight at once.
template <int KB, int NW, int WT>
__global__ void __launch_bounds__(NW * 32, WT == 2 ? 2 : 1)
skinny_gemm_rows16_kernel(const mw_h* __restrict__ X, int ldx, const mw_h* __restrict__ W, int ldw,
                          const float* __restrict__ bias, const float* resid, void* out, int ldo, int R, int N, int K,
                          int flags, const char* pf, int pf_lines) {
    // WT = 16-row weight tiles per CTA.  Every CTA re-reads the whole X block [32, K] from L2, so with one tile the L2->SM
    // traffic is 3x the HBM traffic and caps several batches in flight at ~3.3 TB/s of weights; two tiles halve the X share.
    __shared__ float red[NW][32][WT * 16 + 1];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, q = lane & 3;
    const int n0 = blockIdx.x * (16 * WT), r0 = blockIdx.y * 32;
    const int k_start = warp * (KB * 32) + q * 8;
    uint4 alo[WT][KB], ahi[WT][KB];
    sk_load_w(alo, ahi, W, ldw, N, n0, g, k_start);
    // the whole weight slice is in flight before the first X load is issued
    const mw_h* xr[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) xr[t] = X + (int64_t)min(r0 + t * 8 + g, R - 1) * ldx + k_start;
    float c[WT][4][4] = {};
#pragma unroll
    for (int i = 0; i < KB; ++i)
        sk_mma_block(c, alo, ahi, i, [&](int t) { return __ldg(reinterpret_cast<const uint4*>(xr[t] + i * 32)); });
    l2_prefetch_slice(pf, pf_lines);
    sk_park(red[warp], c, g, q);
    __syncthreads();
    for (int o = threadIdx.x; o < 32 * 16 * WT; o += NW * 32)
        sk_output<NW>(red, o / (16 * WT), o % (16 * WT), r0, n0, R, N, bias, resid, out, ldo, flags);
}

// LayerNorm folded into the projection that consumes it (QKV, cross-attention Q, fc1).  A decode step is a serial chain of
// ~350 graph nodes and a node costs >= 3.3 us however little it does (scripts/gpu_chain_floor.py), so the 96 stand-alone
// LayerNorm launches of a large-v3 step were 0.7 ms of a 3.9 ms single-stream step.  Here every CTA normalises its 32 rows
// itself - warp per row, with the ln_stats / ln_apply / pack_h16x4 of layernorm_kernel (mw_common.cuh), so the 16-bit
// operand is bit-identical to the stand-alone kernel's - into shared memory, and the MMAs read it from there.
// The price is L2 traffic (each CTA reads the fp32 rows instead of the 16-bit copy), not HBM traffic.
template <int KB, int NW, int WT>
__global__ void __launch_bounds__(NW * 32, WT == 2 ? 2 : 1)
skinny_gemm_ln_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                      const mw_h* __restrict__ W, int ldw, const float* __restrict__ bias, mw_h* __restrict__ out, int ldo,
                      int R, int N, int flags, const char* pf, int pf_lines) {
    constexpr int K = KB * NW * 32, MAXV = K / 128, XS = K + 32;      // row pitch K + 32: conflict-free 16-byte fragment reads
    static_assert(K % 128 == 0, "LayerNorm rows are walked in 128-element steps");
    extern __shared__ __align__(16) unsigned char ln_smem[];
    mw_h* xs = reinterpret_cast<mw_h*>(ln_smem);                                        // [32][XS]
    float (*red)[32][WT * 16 + 1] = reinterpret_cast<float (*)[32][WT * 16 + 1]>(ln_smem);   // aliased once the MMAs are done
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, q = lane & 3;
    const int n0 = blockIdx.x * (16 * WT), r0 = blockIdx.y * 32;
    // ---- LayerNorm of rows r0 .. r0+31, two rows per warp at a time (their loads are in flight together)
    const float4* g4 = reinterpret_cast<const float4*>(gamma);
    const float4* b4 = reinterpret_cast<const float4*>(beta);
    for (int rl0 = warp; rl0 < 32; rl0 += 2 * NW) {
        float4 v[2][MAXV];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const float4* xr = reinterpret_cast<const float4*>(x + (int64_t)min(r0 + rl0 + h * NW, R - 1) * K);
#pragma unroll
            for (int i = 0; i < MAXV; ++i) v[h][i] = xr[i * 32 + lane];
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int rl = rl0 + h * NW;
            if (rl >= 32 || r0 + rl >= R) break;      // rows past the batch: their products are never stored (warp-uniform)
            float s = 0.0f, mean, rstd;
#pragma unroll
            for (int i = 0; i < MAXV; ++i) s += sum4(v[h][i]);
            ln_stats(s, v[h], MAXV, K, mean, rstd);
            uint2* o2 = reinterpret_cast<uint2*>(xs + rl * XS);
#pragma unroll
            for (int i = 0; i < MAXV; ++i)
                o2[i * 32 + lane] = pack_h16x4(ln_apply(v[h][i], mean, rstd, __ldg(g4 + i * 32 + lane), __ldg(b4 + i * 32 + lane)));
        }
    }
    // ---- the projection, as skinny_gemm_rows16_kernel with the X fragments read from shared memory
    const int k_start = warp * (KB * 32) + q * 8;
    uint4 alo[WT][KB], ahi[WT][KB];
    sk_load_w(alo, ahi, W, ldw, N, n0, g, k_start);
    __syncthreads();
    float c[WT][4][4] = {};
#pragma unroll
    for (int i = 0; i < KB; ++i)
        sk_mma_block(c, alo, ahi, i, [&](int t) { return *reinterpret_cast<const uint4*>(xs + (t * 8 + g) * XS + k_start + i * 32); });
    l2_prefetch_slice(pf, pf_lines);
    __syncthreads();          // every warp has read its X fragments: the reduction buffer may overwrite them
    sk_park(red[warp], c, g, q);
    __syncthreads();
    for (int o = threadIdx.x; o < 32 * 16 * WT; o += NW * 32)         // 16-bit output, no residual
        sk_output<NW>(red, o / (16 * WT), o % (16 * WT), r0, n0, R, N, bias, nullptr, out, ldo, flags & SK_FLAG_GELU);
}

// K = 5120-class shapes (16 warps): the same two-tile idea needs 160 weight registers, so K is walked in two halves of
// KB blocks per warp (weights of one half in flight at a time) and the 16 warps reduce through 8 shared-memory slots.
template <int KB, int NW, int WT>
__global__ void __launch_bounds__(NW * 32, 1)
skinny_gemm_rows32_khalf_kernel(const mw_h* __restrict__ X, int ldx, const mw_h* __restrict__ W, int ldw,
                                const float* __restrict__ bias, const float* resid, void* out, int ldo, int R, int N, int K,
                                int flags, const char* pf, int pf_lines) {
    static_assert(NW == 16, "two rounds through 8 reduction slots");
    // WT = 2 weight tiles per CTA; WT = 1 (a lone batch, mw_set_solo) doubles the CTAs and halves the bytes each waits for -
    // per output element the K order and the reduction are the same, so both give the same bits
    __shared__ float red[NW / 2][32][WT * 16 + 1];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = lane >> 2, q = lane & 3;
    const int n0 = blockIdx.x * (16 * WT), r0 = blockIdx.y * 32;
    float c[WT][4][4] = {};
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int k_start = h * (NW * KB * 32) + warp * (KB * 32) + q * 8;
        uint4 alo[WT][KB], ahi[WT][KB];
        sk_load_w(alo, ahi, W, ldw, N, n0, g, k_start);
        // this half's weights are in flight before its X loads are issued
#pragma unroll
        for (int i = 0; i < KB; ++i)
            sk_mma_block(c, alo, ahi, i, [&](int t) {
                return __ldg(reinterpret_cast<const uint4*>(X + (int64_t)min(r0 + t * 8 + g, R - 1) * ldx + k_start + i * 32));
            });
    }
    l2_prefetch_slice(pf, pf_lines);
    // warps 8..15 park their partial sums, warps 0..7 fold them in (same fragment positions), then the usual 8-slot reduce
    const int slot = warp & 7;
#pragma unroll
    for (int round = 0; round < 2; ++round) {
        if ((warp >= 8) == (round == 0)) {
#pragma unroll
            for (int wt = 0; wt < WT; ++wt)
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    float* r0p = &red[slot][t * 8 + 2 * q][wt * 16 + g];
                    float* r1p = &red[slot][t * 8 + 2 * q + 1][wt * 16 + g];
                    if (round == 1) { c[wt][t][0] += r0p[0]; c[wt][t][1] += r1p[0]; c[wt][t][2] += r0p[8]; c[wt][t][3] += r1p[8]; }
                    r0p[0] = c[wt][t][0]; r1p[0] = c[wt][t][1]; r0p[8] = c[wt][t][2]; r1p[8] = c[wt][t][3];
                }
        }
        __syncthreads();
    }
    for (int o = threadIdx.x; o < 32 * 16 * WT; o += NW * 32)
        sk_output<NW / 2>(red, o / (16 * WT), o % (16 * WT), r0, n0, R, N, bias, resid, out, ldo, flags);
}

// The tuned shapes (KB, NW) of the mma.sync kernels, K = KB * NW * 32 (the d_model and ffn widths of the Whisper sizes and
// the test dims): rows16 with one weight tile serves all of them; the K-halved kernel replaces it where sk_k_halved holds,
// and where sk_two_tiles holds rows16 and the fused LayerNorm projection run with two tiles.  Other K: the generic kernel.
#define MW_SK(X)                                \
    X(5, 8)     /* 1280  (large) */             \
    X(10, 16)   /* 5120  (large ffn) */         \
    X(4, 8)     /* 1024  (medium) */            \
    X(8, 16)    /* 4096  (medium ffn) */        \
    X(3, 8)     /* 768   (small) */             \
    X(6, 16)    /* 3072  (small ffn) */         \
    X(2, 8)     /* 512   (base / test ffn) */   \
    X(4, 16)    /* 2048  (base ffn) */          \
    X(3, 4)     /* 384   (tiny) */              \
    X(6, 8)     /* 1536  (tiny ffn) */          \
    X(1, 4)     /* 128   (test dims) */         \
    X(1, 8)     /* 256 */

// two weight tiles fit the registers
constexpr bool sk_two_tiles(int KB, int NW) { return NW <= 8 && KB <= 5; }
// the 16-warp shapes, as two halves of KB / 2 blocks per warp
constexpr bool sk_k_halved(int KB, int NW) { return NW == 16 && KB % 2 == 0 && KB / 2 <= 5; }

// warps per CTA of the tuned entry for K, 0 when K has none
int sk_table_warps(int K) {
#define MW_SK_WARPS(kb, nw) if (K == kb * nw * 32) return nw;
    MW_SK(MW_SK_WARPS)
#undef MW_SK_WARPS
    return 0;
}

// The kernels of a decode-step projection.  A caller asks for SK_ROUTE (the step's own routing) or forces one kernel
// (mw_step_projection_h16); sk_choose answers with the kernel that runs, or SK_NONE.
enum SkKernel { SK_ROUTE, SK_ROWS16_WT1, SK_ROWS16_WT2, SK_KHALF_WT1, SK_KHALF_WT2, SK_GENERIC, SK_LN_FUSED, SK_DECODE_GEMM, SK_NONE };
const char* const SK_NAME[SK_NONE] = {"routed", "rows16", "two-tile rows16", "K-halved", "K-halved", "generic",
                                      "fused LayerNorm (16-bit output)", "decode GEMM"};

// rows from which the tcgen05 decode GEMM takes over the projections the step routes to it
constexpr int DG_MIN_ROWS = 96;

// The kernel for out[R, N] = X[R, K] W[N, K]^T (row pitches ldx, ldw) as `path` asks, X = LayerNorm(x) when `ln`; SK_NONE
// when a forced kernel does not exist for K (or, SK_LN_FUSED, for fp32 output).  The step's routing:
//  * R >= DG_MIN_ROWS rows (merged greedy batches): the weight-stationary tcgen05 kernel (decode_gemm.cu) streams W once
//    for all rows; the mma.sync kernels re-read it per 32-row block (from L2 after the first block) and stay in charge of
//    the 32-row batches they were tuned on and of beam search, where they measured faster (DESIGN.md section 4: a decode
//    step is a chain of ~360 latency-bound launches, so bytes saved do not buy time unless the launch is also shorter).
//    The step passes allow_dg = (beam <= 1) for the layer projections; the vocabulary projection (enqueue_logits) keeps
//    it, so at R >= 96 rows it runs on the decode GEMM in beam search as well.
//  * LayerNorm: with `solo` (mw_set_solo: the replica decodes alone on its GPU) ONE launch where the fused kernel applies
//    (16-bit output, two tiles, rows that do not go to the decode GEMM).  Otherwise the stand-alone LayerNorm, then the
//    projection as routed without `solo`.  Both give the same bits; which is faster depends on what else the GPU is doing -
//    measured on large-v3, ms per 32-row step, fused / separate: one batch in flight 3.71 / 3.88 (96 graph nodes fewer),
//    two 2.78 / 2.75, four 2.33 / 2.20, eight 2.30 / 2.09.  With several batches in flight a node's fixed cost is hidden by
//    the other batches anyway, and every CTA now holds its SM slot (and 84 KB of shared memory) for the ~1 us it spends
//    normalising 32 rows before it asks for its weights.  (It is not the extra L2->SM traffic: reading the 16-bit operand
//    twice in the plain kernels costs nothing at eight streams.)
//  * the K-halved kernel with one weight tile for a lone batch (3.87 -> 3.76 ms per single-stream step), else two; two-tile
//    rows16 where it fits, else one tile; the generic kernel for K outside MW_SK.
SkKernel sk_choose(int ldx, int ldw, int R, int N, int K, int flags, SkKernel path, bool allow_dg, bool solo, bool ln) {
    const bool to_dg = allow_dg && R >= DG_MIN_ROWS && decode_gemm_supported(ldx, ldw, R, N, K);
    const int nw = sk_table_warps(K), kb = nw ? K / (nw * 32) : 0;
    const bool two_tiles = nw && sk_two_tiles(kb, nw), k_halved = nw && sk_k_halved(kb, nw);
    if (ln && (path == SK_LN_FUSED || (path == SK_ROUTE && solo && !to_dg)) && two_tiles && !(flags & SK_FLAG_F32))
        return SK_LN_FUSED;
    if (ln) solo = false;
    switch (path) {
        case SK_ROUTE:
            if (to_dg) return SK_DECODE_GEMM;
            if (k_halved) return solo ? SK_KHALF_WT1 : SK_KHALF_WT2;
            return two_tiles ? SK_ROWS16_WT2 : nw ? SK_ROWS16_WT1 : SK_GENERIC;
        case SK_GENERIC: return path;
        case SK_ROWS16_WT1: return nw ? path : SK_NONE;
        case SK_ROWS16_WT2: return two_tiles ? path : SK_NONE;
        case SK_KHALF_WT1: case SK_KHALF_WT2: return k_halved ? path : SK_NONE;
        default: return SK_NONE;
    }
}

mw_status sk_missing(const char* who, SkKernel path, int K) {
    set_error("%s: no %s kernel for K=%d", who, SK_NAME[path], K);
    return MW_ERR_UNSUPPORTED;
}

// kernel k of a tuned shape; x, gamma, beta: the fp32 rows and the LayerNorm of SK_LN_FUSED
template <int KB, int NW>
mw_status launch_tuned(SkKernel k, const void* X, int ldx, const void* W, int ldw, const float* bias, const float* resid, void* out,
                       int ldo, int R, int N, int K, int flags, cudaStream_t st, const char* pf, int pf_lines, const float* x,
                       const float* gamma, const float* beta) {
    const dim3 grid(ceil_div(N, k == SK_ROWS16_WT1 || k == SK_KHALF_WT1 ? 16 : 32), ceil_div(R, 32)), block(NW * 32);
    const mw_h* Xh = (const mw_h*)X;
    const mw_h* Wh = (const mw_h*)W;
    if (k == SK_ROWS16_WT1)
        skinny_gemm_rows16_kernel<KB, NW, 1><<<grid, block, 0, st>>>(Xh, ldx, Wh, ldw, bias, resid, out, ldo, R, N, K, flags, pf, pf_lines);
    if constexpr (sk_two_tiles(KB, NW)) {
        if (k == SK_ROWS16_WT2)
            skinny_gemm_rows16_kernel<KB, NW, 2><<<grid, block, 0, st>>>(Xh, ldx, Wh, ldw, bias, resid, out, ldo, R, N, K, flags, pf,
                                                                        pf_lines);
        if (k == SK_LN_FUSED) {
            constexpr int xs_bytes = 32 * (KB * NW * 32 + 32) * 2, red_bytes = NW * 32 * (2 * 16 + 1) * 4;
            constexpr int smem = xs_bytes > red_bytes ? xs_bytes : red_bytes;
            static PerDeviceOnce attr_once;
            MW_CUDA_CHECK(attr_once.run([&] { return cudaFuncSetAttribute(skinny_gemm_ln_kernel<KB, NW, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); }));
            skinny_gemm_ln_kernel<KB, NW, 2><<<grid, block, smem, st>>>(x, gamma, beta, Wh, ldw, bias, (mw_h*)out, ldo, R, N, flags, pf,
                                                                       pf_lines);
        }
    }
    if constexpr (sk_k_halved(KB, NW)) {
        if (k == SK_KHALF_WT1)
            skinny_gemm_rows32_khalf_kernel<KB / 2, NW, 1><<<grid, block, 0, st>>>(Xh, ldx, Wh, ldw, bias, resid, out, ldo, R, N, K, flags,
                                                                                  pf, pf_lines);
        if (k == SK_KHALF_WT2)
            skinny_gemm_rows32_khalf_kernel<KB / 2, NW, 2><<<grid, block, 0, st>>>(Xh, ldx, Wh, ldw, bias, resid, out, ldo, R, N, K, flags,
                                                                                  pf, pf_lines);
    }
    MW_LAUNCH_CHECK();
    return MW_OK;
}

// kernel k of sk_choose.  `next_w` / `next_bytes`: the weight matrix of the projection that follows this one in the step
// (prefetched into L2)
mw_status sk_launch(SkKernel k, const void* X, int ldx, const void* W, int ldw, const float* bias, const float* resid, void* out,
                    int ldo, int R, int N, int K, int flags, cudaStream_t st, const void* next_w, int64_t next_bytes,
                    const float* x = nullptr, const float* gamma = nullptr, const float* beta = nullptr) {
    if (k == SK_DECODE_GEMM) return decode_gemm_launch(X, ldx, W, ldw, bias, resid, out, ldo, R, N, K, flags, st);
    const char* pf = (const char*)next_w;
    const int pf_lines = pf ? (int)(next_bytes / 128) : 0;
#define MW_SK_LAUNCH(kb, nw) \
    if (k != SK_GENERIC && K == kb * nw * 32) \
        return launch_tuned<kb, nw>(k, X, ldx, W, ldw, bias, resid, out, ldo, R, N, K, flags, st, pf, pf_lines, x, gamma, beta);
    MW_SK(MW_SK_LAUNCH)
#undef MW_SK_LAUNCH
    dim3 grid(ceil_div(N, 16), ceil_div(R, 32));
    skinny_gemm_kernel<<<grid, 256, 0, st>>>((const mw_h*)X, ldx, (const mw_h*)W, ldw, bias, resid, out, ldo, R, N, K, flags);
    MW_LAUNCH_CHECK();
    return MW_OK;
}

mw_status skinny_gemm(const void* X, int ldx, const void* W, int ldw, const float* bias, const float* resid, void* out,
                      int ldo, int R, int N, int K, int flags, cudaStream_t st, bool allow_dg = true,
                      const void* next_w = nullptr, int64_t next_bytes = 0, bool solo = false, SkKernel path = SK_ROUTE) {
    const SkKernel k = sk_choose(ldx, ldw, R, N, K, flags, path, allow_dg, solo, false);
    if (k == SK_NONE) return sk_missing("skinny gemm", path, K);
    return sk_launch(k, X, ldx, W, ldw, bias, resid, out, ldo, R, N, K, flags, st, next_w, next_bytes);
}

// ------------------------------------------------------------------------------------------------
__global__ void embed_kernel(const int* __restrict__ cur_tok, const mw_h* __restrict__ emb,
                             const float* __restrict__ pos_emb, const DecCtl* __restrict__ ctl, float* __restrict__ x, int d) {
    const int r = blockIdx.x;
    const int tok = cur_tok[r];
    const int pos = ctl->pos;
    for (int i = threadIdx.x; i < d; i += blockDim.x)
        x[(int64_t)r * d + i] = h2f(emb[(int64_t)tok * d + i]) + pos_emb[(int64_t)pos * d + i];
}

// LayerNorm + projection (the routing: sk_choose): the fused kernel, or the stand-alone LayerNorm into `ln_buf` and the projection
mw_status skinny_gemm_ln(const float* x, const float* gamma, const float* beta, void* ln_buf, const void* W, const float* bias,
                         void* out, int ldo, int R, int N, int K, int flags, cudaStream_t st, bool allow_dg, const void* next_w,
                         int64_t next_bytes, bool solo, SkKernel path = SK_ROUTE) {
    const SkKernel k = sk_choose(K, K, R, N, K, flags, path, allow_dg, solo, true);
    if (k == SK_NONE) return sk_missing("skinny gemm", path, K);
    if (k != SK_LN_FUSED) {
        mw_status r = layernorm_launch(x, gamma, beta, ln_buf, R, K, st);
        if (r != MW_OK) return r;
    }
    return sk_launch(k, ln_buf, K, W, K, bias, nullptr, out, ldo, R, N, K, flags, st, next_w, next_bytes, x, gamma, beta);
}

// ------------------------------------------------------------------------------------------------
// decode attention: one CTA (128 threads) per (head, row); keys streamed once, 16 bytes per lane,
// 8 lanes per key.  SELF: appends this step's k,v to the cache first and reads pos+1 keys.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void h16x8_to_float(const uint4& u, float (&f)[8]) {
    const mw_h2* h = reinterpret_cast<const mw_h2*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 t = h22f2(h[i]);
        f[2 * i] = t.x;
        f[2 * i + 1] = t.y;
    }
}

template <bool SELF>
__global__ void __launch_bounds__(128)
decode_attn_kernel(const mw_h* __restrict__ q, int ldq,
                   mw_h* kbase, mw_h* vbase, int64_t key_stride, int64_t keys_per_seq,
                   const int* __restrict__ idx_table, int ctx, const DecCtl* __restrict__ ctl, int n_keys_fixed,
                   int rows_per_seq, const mw_h* __restrict__ knew, const mw_h* __restrict__ vnew,
                   int ld_new, mw_h* __restrict__ out, int ldo, int causal_rows = 0) {
    extern __shared__ float sc[];          // scores [n_keys] + reduction scratch
    __shared__ float red[4][64];
    __shared__ float red_s[8];
    const int h = blockIdx.x, r = blockIdx.y;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    constexpr int UNR = SELF ? 4 : 8;             // independent 16-byte loads in flight per thread
    const int lg = lane & 7, kq = lane >> 3;      // 8 lanes per key, 4 keys per warp instruction
    const int seq0 = r / rows_per_seq;
    int n_keys = n_keys_fixed;
    if (!SELF && causal_rows > 0) n_keys = (r % causal_rows) + 1;     // batched prefill: row (b, p) sees keys 0..p
    if (SELF) {
        const int pos = ctl->pos;
        n_keys = pos + 1;
        // append this row's k, v at position pos into its own physical cache row
        if (tid < 16) {
            const int part = tid >> 3, c8 = tid & 7;
            const mw_h* src = (part ? vnew : knew) + (int64_t)r * ld_new + h * 64 + c8 * 8;
            mw_h* dst = (part ? vbase : kbase) + ((int64_t)r * keys_per_seq + pos) * key_stride + h * 64 + c8 * 8;
            *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(src);
        }
        __syncthreads();
    }
    const int* idx = (SELF && idx_table) ? idx_table + (int64_t)r * ctx : nullptr;
    // The self K/V cache is read once per step and is larger than L2 with several batches in flight, so its lines go first
    // (ld.global.cs: evict-first in L1 and L2).  It is a coherent load because this kernel appends to the cache; the
    // batched prefill reads activations and keeps the default policy.
    auto kv_load = [](const mw_h* p) { return SELF ? __ldcs(reinterpret_cast<const uint4*>(p)) : *reinterpret_cast<const uint4*>(p); };
    float qf[8];
    {
        const uint4 u = *reinterpret_cast<const uint4*>(q + (int64_t)r * ldq + h * 64 + lg * 8);
        h16x8_to_float(u, qf);
#pragma unroll
        for (int i = 0; i < 8; ++i) qf[i] *= 0.125f;
    }
    // ---- scores
    float mx = -INFINITY;
    for (int kbase0 = warp * 4; kbase0 < n_keys; kbase0 += 16 * UNR) {   // warp-uniform trip count (shuffles inside)
        const int key0 = kbase0 + kq;
        uint4 kv[UNR];
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int key = key0 + 16 * u;
            if (key < n_keys) {
                const int seq = idx ? ((key == n_keys - 1) ? r : idx[key]) : (SELF ? r : seq0);
                kv[u] = kv_load(kbase + ((int64_t)seq * keys_per_seq + key) * key_stride + h * 64 + lg * 8);
            }
        }
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int key = key0 + 16 * u;
            float s = 0.0f;
            if (key < n_keys) {
                float kf[8];
                h16x8_to_float(kv[u], kf);
#pragma unroll
                for (int i = 0; i < 8; ++i) s = fmaf(qf[i], kf[i], s);
            }
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            s += __shfl_xor_sync(0xffffffffu, s, 4);
            if (key < n_keys) {
                if (lg == 0) sc[key] = s;
                mx = fmaxf(mx, s);
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 0) red_s[warp] = mx;
    __syncthreads();
    mx = fmaxf(fmaxf(red_s[0], red_s[1]), fmaxf(red_s[2], red_s[3]));
    float sum = 0.0f;
    for (int key = tid; key < n_keys; key += 128) {
        const float p = __expf(sc[key] - mx);
        sc[key] = p;
        sum += p;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) red_s[4 + warp] = sum;
    __syncthreads();
    sum = (red_s[4] + red_s[5]) + (red_s[6] + red_s[7]);
    // ---- P.V
    float acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.0f;
    for (int kbase0 = warp * 4; kbase0 < n_keys; kbase0 += 16 * UNR) {
        const int key0 = kbase0 + kq;
        uint4 vv[UNR];
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int key = key0 + 16 * u;
            if (key < n_keys) {
                const int seq = idx ? ((key == n_keys - 1) ? r : idx[key]) : (SELF ? r : seq0);
                vv[u] = kv_load(vbase + ((int64_t)seq * keys_per_seq + key) * key_stride + h * 64 + lg * 8);
            }
        }
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int key = key0 + 16 * u;
            if (key < n_keys) {
                const float p = sc[key];
                float vf[8];
                h16x8_to_float(vv[u], vf);
#pragma unroll
                for (int i = 0; i < 8; ++i) acc[i] = fmaf(p, vf[i], acc[i]);
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], 8);
        acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], 16);
    }
    if (kq == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) red[warp][lg * 8 + i] = acc[i];
    }
    __syncthreads();
    if (tid < 64) {
        const float v = ((red[0][tid] + red[1][tid]) + (red[2][tid] + red[3][tid])) / sum;
        out[(int64_t)r * ldo + h * 64 + tid] = f2h(v);
    }
}

// ------------------------------------------------------------------------------------------------
// Greedy cross-attention (the dominant kernel of the decode step): one CTA per (head, row) streams the chunk's K and
// V exactly once, in a SINGLE pass: every 8-lane group keeps its own online-softmax state (running max, sum and an
// 8-dim slice of the output) over the keys it owns, so K and V loads are interleaved with no mid-kernel barrier and
// no score buffer; the 16 partial states of the CTA are merged at the end (log-sum-exp).  Same lane mapping as
// decode_attn_kernel: 16 bytes per lane, 8 lanes per key, 4 keys per warp instruction.
// ------------------------------------------------------------------------------------------------
// UNR = independent K/V loads in flight per lane.  4 (95 registers, 5 CTAs/SM) is right when rows x heads fill the GPU (32
// rows of large-v3 = 640 CTAs = one wave); when they do not (the 17-row shard of an 8-GPU job: 340 CTAs for 740 slots, 35 us
// for bytes that need 21) UNR = 8 doubles the bytes in flight per CTA instead.  A group's keys are visited in the same order
// either way, so the result is bit-identical and a sharded job decodes the ids of the single-GPU one.
template <int UNR>
__global__ void __launch_bounds__(128)
cross_attn_stream_kernel(const mw_h* __restrict__ q, int ldq, const mw_h* __restrict__ kbase,
                         const mw_h* __restrict__ vbase, int64_t key_stride, int n_keys,
                         mw_h* __restrict__ out, int ldo, const char* pf, int pf_lines) {
    __shared__ float part_acc[16][64];
    __shared__ float part_m[16], part_l[16];
    const int h = blockIdx.x, r = blockIdx.y;
    const int key_lo = 0, key_hi = n_keys;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int lg = lane & 7, kq = lane >> 3;
    const mw_h* kp = kbase + (int64_t)r * n_keys * key_stride + h * 64 + lg * 8;
    const mw_h* vp = vbase + (int64_t)r * n_keys * key_stride + h * 64 + lg * 8;
    const uint64_t pol = ptx::l2_policy_evict_first();     // K/V are read once per step: let them go before the prefetched weights
    float qf[8];
    {
        const uint4 u = *reinterpret_cast<const uint4*>(q + (int64_t)r * ldq + h * 64 + lg * 8);
        h16x8_to_float(u, qf);
#pragma unroll
        for (int i = 0; i < 8; ++i) qf[i] *= 0.125f;
    }
    float m = -INFINITY, l = 0.0f, acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.0f;
    for (int kbase0 = key_lo + warp * 4; kbase0 < key_hi; kbase0 += 16 * UNR) {   // warp-uniform trip count (shuffles inside)
        const int key0 = kbase0 + kq;
        uint4 kv[UNR], vv[UNR];
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int key = key0 + 16 * u;
            if (key < key_hi) {
                kv[u] = ptx::ldg_nc_hint(kp + (int64_t)key * key_stride, pol);
                vv[u] = ptx::ldg_nc_hint(vp + (int64_t)key * key_stride, pol);
            }
        }
        float sv[UNR];
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            sv[u] = 0.0f;
            if (key0 + 16 * u < key_hi) {
                float kf[8];
                h16x8_to_float(kv[u], kf);
#pragma unroll
                for (int i = 0; i < 8; ++i) sv[u] = fmaf(qf[i], kf[i], sv[u]);
            }
        }
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            sv[u] += __shfl_xor_sync(0xffffffffu, sv[u], 1);
            sv[u] += __shfl_xor_sync(0xffffffffu, sv[u], 2);
            sv[u] += __shfl_xor_sync(0xffffffffu, sv[u], 4);
        }
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            if (key0 + 16 * u < key_hi) {
                const float sc = sv[u];
                if (sc > m) {                       // uniform over the 8 lanes of the key; rare after the first keys
                    const float scale = __expf(m - sc);      // exp(-inf) = 0 on the first key
                    l *= scale;
#pragma unroll
                    for (int i = 0; i < 8; ++i) acc[i] *= scale;
                    m = sc;
                }
                const float p = __expf(sc - m);
                l += p;
                float vf[8];
                h16x8_to_float(vv[u], vf);
#pragma unroll
                for (int i = 0; i < 8; ++i) acc[i] = fmaf(p, vf[i], acc[i]);
            }
        }
    }
    l2_prefetch_slice(pf, pf_lines);       // this CTA's K/V stream is done: ask L2 for a slice of the output projection's weights
    const int grp = warp * 4 + kq;
#pragma unroll
    for (int i = 0; i < 8; ++i) part_acc[grp][lg * 8 + i] = acc[i];
    if (lg == 0) { part_m[grp] = m; part_l[grp] = l; }
    __syncthreads();
    if (tid < 64) {
        float M = -INFINITY;
#pragma unroll
        for (int g = 0; g < 16; ++g) M = fmaxf(M, part_m[g]);
        float num = 0.0f, den = 0.0f;
#pragma unroll
        for (int g = 0; g < 16; ++g) {
            const float w = (part_m[g] == -INFINITY) ? 0.0f : __expf(part_m[g] - M);     // groups that saw no key
            num = fmaf(w, part_acc[g][tid], num);
            den = fmaf(w, part_l[g], den);
        }
        out[(int64_t)r * ldo + h * 64 + tid] = f2h(num / den);
    }
}

// ------------------------------------------------------------------------------------------------
// Grouped cross-attention for beam search: the G hypotheses of one chunk attend to the SAME encoder K/V, so one CTA
// per (head, chunk) streams K and V once and serves all G queries (CTranslate2 instead tiles the encoder output
// beam_size times, SURVEY.md Appendix C).  Same lane mapping as decode_attn_kernel: 16 bytes per lane, 8 lanes per key.
// ------------------------------------------------------------------------------------------------
template <int G>
__global__ void __launch_bounds__(128, 5)
cross_attn_grouped_kernel(const mw_h* __restrict__ q, int ldq, const mw_h* __restrict__ kbase,
                          const mw_h* __restrict__ vbase, int64_t key_stride, int n_keys,
                          mw_h* __restrict__ out, int ldo) {
    extern __shared__ float sc[];          // [G][n_keys] scores, then probabilities
    __shared__ float red[4][G][64];
    __shared__ float red_s[G][8];
    constexpr int UNR = 4;
    const int h = blockIdx.x, b = blockIdx.y;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int lg = lane & 7, kq = lane >> 3;
    float qf[G][8];
#pragma unroll
    for (int g = 0; g < G; ++g) {
        const uint4 u = *reinterpret_cast<const uint4*>(q + (int64_t)(b * G + g) * ldq + h * 64 + lg * 8);
        h16x8_to_float(u, qf[g]);
#pragma unroll
        for (int i = 0; i < 8; ++i) qf[g][i] *= 0.125f;
    }
    const mw_h* kb = kbase + (int64_t)b * n_keys * key_stride + h * 64 + lg * 8;
    const mw_h* vb = vbase + (int64_t)b * n_keys * key_stride + h * 64 + lg * 8;
    const uint64_t pol = ptx::l2_policy_evict_first();     // K and V are read once per step, as in cross_attn_stream_kernel
    // Scores: every lane forms 8-dim partial dots for all G queries; a 3-round reduce-scatter over the 8 lanes of a key
    // (4 + 2 + 1 shuffles instead of 3 per query) leaves lane lg with the complete score of query lg.
    const bool b2 = lg & 4, b1 = lg & 2, b0 = lg & 1;
    float mx = -INFINITY;                  // running max of query lg over the keys this lane group sees
    for (int kbase0 = warp * 4; kbase0 < n_keys; kbase0 += 16 * UNR) {
        const int key0 = kbase0 + kq;
        uint4 kv[UNR];
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int key = key0 + 16 * u;
            if (key < n_keys) kv[u] = ptx::ldg_nc_hint(kb + (int64_t)key * key_stride, pol);
        }
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int key = key0 + 16 * u;
            float v[8];
#pragma unroll
            for (int g = 0; g < 8; ++g) v[g] = 0.0f;
            if (key < n_keys) {
                float kf[8];
                h16x8_to_float(kv[u], kf);
#pragma unroll
                for (int g = 0; g < G; ++g) {
#pragma unroll
                    for (int i = 0; i < 8; ++i) v[g] = fmaf(qf[g][i], kf[i], v[g]);
                }
            }
            float w[4], x2[2];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float send = b2 ? v[i] : v[i + 4];
                const float keep = b2 ? v[i + 4] : v[i];
                w[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
            }
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const float send = b1 ? w[i] : w[i + 2];
                const float keep = b1 ? w[i + 2] : w[i];
                x2[i] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
            }
            const float send = b0 ? x2[0] : x2[1];
            const float keep = b0 ? x2[1] : x2[0];
            const float sc_q = keep + __shfl_xor_sync(0xffffffffu, send, 1);      // score of query lg for this key
            if (key < n_keys && lg < G) {
                sc[lg * n_keys + key] = sc_q;
                mx = fmaxf(mx, sc_q);
            }
        }
    }
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 8));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 16));
    if (kq == 0 && lg < G) red_s[lg][warp] = mx;
    __syncthreads();
#pragma unroll
    for (int g = 0; g < G; ++g) {
        const float m = fmaxf(fmaxf(red_s[g][0], red_s[g][1]), fmaxf(red_s[g][2], red_s[g][3]));
        float a = 0.0f;
        for (int key = tid; key < n_keys; key += 128) {
            const float p = __expf(sc[g * n_keys + key] - m);
            sc[g * n_keys + key] = p;
            a += p;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
        if (lane == 0) red_s[g][4 + warp] = a;
    }
    __syncthreads();
    float acc[G][8];
#pragma unroll
    for (int g = 0; g < G; ++g)
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[g][i] = 0.0f;
    for (int kbase0 = warp * 4; kbase0 < n_keys; kbase0 += 16 * UNR) {
        const int key0 = kbase0 + kq;
        uint4 vv[UNR];
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int key = key0 + 16 * u;
            if (key < n_keys) vv[u] = ptx::ldg_nc_hint(vb + (int64_t)key * key_stride, pol);
        }
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int key = key0 + 16 * u;
            if (key < n_keys) {
                float vf[8];
                h16x8_to_float(vv[u], vf);
#pragma unroll
                for (int g = 0; g < G; ++g) {
                    const float p = sc[g * n_keys + key];
#pragma unroll
                    for (int i = 0; i < 8; ++i) acc[g][i] = fmaf(p, vf[i], acc[g][i]);
                }
            }
        }
    }
#pragma unroll
    for (int g = 0; g < G; ++g) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            acc[g][i] += __shfl_xor_sync(0xffffffffu, acc[g][i], 8);
            acc[g][i] += __shfl_xor_sync(0xffffffffu, acc[g][i], 16);
        }
        if (kq == 0) {
#pragma unroll
            for (int i = 0; i < 8; ++i) red[warp][g][lg * 8 + i] = acc[g][i];
        }
    }
    __syncthreads();
    for (int o = tid; o < G * 64; o += 128) {
        const int g = o >> 6, dcol = o & 63;
        const float v = ((red[0][g][dcol] + red[1][g][dcol]) + (red[2][g][dcol] + red[3][g][dcol])) / ((red_s[g][4] + red_s[g][5]) + (red_s[g][6] + red_s[g][7]));
        out[(int64_t)(b * G + g) * ldo + h * 64 + dcol] = f2h(v);
    }
}

template <int G>
mw_status launch_cross_grouped(const mw_h* q, int ldq, const mw_h* k, const mw_h* v, int64_t key_stride,
                               int n_keys, mw_h* out, int ldo, int n_heads, int B, cudaStream_t st) {
    const size_t smem = (size_t)G * n_keys * sizeof(float);
    MW_REQUIRE(smem <= 96 * 1024, "cross attention: %zu bytes of scores exceed shared memory", smem);
    static PerDeviceOnce attr_once;
    MW_CUDA_CHECK(attr_once.run([&] { return cudaFuncSetAttribute(cross_attn_grouped_kernel<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024); }));
    cross_attn_grouped_kernel<G><<<dim3(n_heads, B), 128, smem, st>>>(q, ldq, k, v, key_stride, n_keys, out, ldo);
    MW_LAUNCH_CHECK();
    return MW_OK;
}

// ------------------------------------------------------------------------------------------------
// logit rules (SURVEY.md A.8; timestamp rules as transformers/generation/logits_process.py:1996-2043)
// ------------------------------------------------------------------------------------------------
struct RowRule {
    int gen_len, last_is_ts, pen_is_ts, ts_floor;   // ts_floor: timestamps below this id are masked (0 = none)
    int first_step;
};

__device__ __forceinline__ RowRule make_rule(const int* toks, int gen_len, int last_ts, const GenOptsDev& o) {
    RowRule rr;
    rr.gen_len = gen_len;
    rr.first_step = gen_len == 0;
    rr.last_is_ts = 0; rr.pen_is_ts = 1; rr.ts_floor = 0;
    if (o.with_timestamps) {
        const int tb = o.timestamp_begin;
        rr.last_is_ts = gen_len >= 1 && toks[gen_len - 1] >= tb;
        rr.pen_is_ts = gen_len < 2 || toks[gen_len - 2] >= tb;
        if (last_ts >= 0) rr.ts_floor = (rr.last_is_ts && !rr.pen_is_ts) ? last_ts : last_ts + 1;
    }
    return rr;
}

__device__ __forceinline__ bool is_masked(int i, const RowRule& rr, const GenOptsDev& o, const uint8_t* sup, const uint8_t* beg) {
    if (sup[i]) return true;
    if (rr.first_step && beg[i]) return true;
    if (o.with_timestamps) {
        const int tb = o.timestamp_begin;
        if (rr.last_is_ts) {
            if (rr.pen_is_ts) { if (i >= tb) return true; }
            else if (i < o.eot) return true;
        }
        if (i >= tb && i < rr.ts_floor) return true;
        if (rr.first_step) {
            if (i < tb) return true;
            if (o.max_initial_ts >= 0 && i > tb + o.max_initial_ts) return true;
        }
    }
    return false;
}

struct ValIdx { float v; int i; };
__device__ __forceinline__ ValIdx better(ValIdx a, ValIdx b) {    // larger value, then lower index
    return (b.v > a.v || (b.v == a.v && b.i < a.i)) ? b : a;
}
__device__ __forceinline__ ValIdx warp_best(ValIdx a) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        ValIdx b;
        b.v = __shfl_xor_sync(0xffffffffu, a.v, o);
        b.i = __shfl_xor_sync(0xffffffffu, a.i, o);
        a = better(a, b);
    }
    return a;
}
__device__ __forceinline__ float warp_sum(float a) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
    return a;
}

constexpr int SEL_THREADS = 512;

// Row statistics shared by greedy and beam selection.  Applies the masks IN PLACE to logits (masked -> -inf),
// including the "timestamp mass beats every text token" rule, and returns max/argmax + logsumexp.
__device__ void row_rules_and_stats(float* lg, int V, const RowRule& rr, const GenOptsDev& o, const uint8_t* sup,
                                    const uint8_t* beg, ValIdx& best_out, float& lse_out) {
    __shared__ ValIdx s_txt[SEL_THREADS / 32], s_ts[SEL_THREADS / 32];
    __shared__ float s_sum[2][SEL_THREADS / 32];
    __shared__ ValIdx b_all, b_txt, b_ts;
    __shared__ float f_sum_all, f_sum_ts;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int tb = o.timestamp_begin;
    ValIdx m_txt{-INFINITY, 0x7fffffff}, m_ts{-INFINITY, 0x7fffffff};
    // four independent loads per thread per trip: the row is 207 KB and a one-load-at-a-time loop is pure latency
    constexpr int UNR = 4;
    for (int i0 = tid; i0 < V; i0 += UNR * SEL_THREADS) {
        float v[UNR];
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int i = i0 + u * SEL_THREADS;
            v[u] = i < V ? lg[i] : -INFINITY;
        }
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int i = i0 + u * SEL_THREADS;
            if (i >= V) break;
            if (is_masked(i, rr, o, sup, beg)) { v[u] = -INFINITY; lg[i] = v[u]; }
            ValIdx c{v[u], i};
            if (o.with_timestamps && i >= tb) m_ts = better(m_ts, c);
            else m_txt = better(m_txt, c);
        }
    }
    m_txt = warp_best(m_txt);
    m_ts = warp_best(m_ts);
    if (lane == 0) { s_txt[warp] = m_txt; s_ts[warp] = m_ts; }
    __syncthreads();
    if (tid == 0) {
        ValIdx a = s_txt[0], b = s_ts[0];
        for (int w = 1; w < SEL_THREADS / 32; ++w) { a = better(a, s_txt[w]); b = better(b, s_ts[w]); }
        b_txt = a; b_ts = b; b_all = better(a, b);
    }
    __syncthreads();
    const float gm = b_all.v;
    float sum_all = 0.0f, sum_ts = 0.0f;
    for (int i0 = tid; i0 < V; i0 += UNR * SEL_THREADS) {
        float v[UNR];
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int i = i0 + u * SEL_THREADS;
            v[u] = i < V ? lg[i] : -INFINITY;
        }
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int i = i0 + u * SEL_THREADS;
            const float e = __expf(v[u] - gm);      // exp(-inf) = 0
            sum_all += e;
            if (o.with_timestamps && i >= tb) sum_ts += e;
        }
    }
    sum_all = warp_sum(sum_all);
    sum_ts = warp_sum(sum_ts);
    if (lane == 0) { s_sum[0][warp] = sum_all; s_sum[1][warp] = sum_ts; }
    __syncthreads();
    if (tid == 0) {
        float a = 0.0f, b = 0.0f;
        for (int w = 0; w < SEL_THREADS / 32; ++w) { a += s_sum[0][w]; b += s_sum[1][w]; }
        f_sum_all = a; f_sum_ts = b;
    }
    __syncthreads();
    bool force_ts = false;
    if (o.with_timestamps && f_sum_ts > 0.0f) {
        const float lse_ts = gm + logf(f_sum_ts);
        force_ts = lse_ts > b_txt.v;
    }
    if (force_ts) {
        for (int i = tid; i < tb; i += SEL_THREADS) lg[i] = -INFINITY;
        best_out = b_ts;
        lse_out = gm + logf(f_sum_ts);
    } else {
        best_out = b_all;
        lse_out = gm + logf(f_sum_all);
    }
    __syncthreads();
}

// greedy: one CTA per row
__global__ void __launch_bounds__(SEL_THREADS)
select_greedy_kernel(float* logits, int V, const GenOptsDev* __restrict__ opts, const uint8_t* __restrict__ sup,
                     const uint8_t* __restrict__ beg, int* tokens, int* gen_len, int* done, float* cum, int* last_ts,
                     int* cur_tok, DecCtl* ctl, int max_new) {
    const int r = blockIdx.x;
    const GenOptsDev o = *opts;
    float* lg = logits + (int64_t)r * V;
    int* toks = tokens + (int64_t)r * max_new;
    const int gl = gen_len[r];
    const bool was_done = done[r] != 0;
    const RowRule rr = make_rule(toks, gl, last_ts[r], o);
    ValIdx best; float lse;
    row_rules_and_stats(lg, V, rr, o, sup, beg, best, lse);
    if (threadIdx.x == 0) {
        int t = best.i;
        if (!was_done) {
            if (o.forced_eot_len > 0 && gl >= o.forced_eot_len) t = o.eot;
            else cum[r] += best.v - lse;
            if (t == o.eot || gl >= max_new) {
                done[r] = 1;
                atomicAdd(&ctl->n_done, 1);
                t = o.eot;
            } else {
                toks[gl] = t;
                gen_len[r] = gl + 1;
                if (o.with_timestamps && t >= o.timestamp_begin) last_ts[r] = t;
            }
        } else {
            t = o.eot;
        }
        cur_tok[r] = t;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) { ctl->pos += 1; ctl->step += 1; }
}

// prefill / teacher forcing: next input token comes from a list; forced[step+1] for every row, or per-row lists
__global__ void advance_forced_kernel(const int* __restrict__ forced, int per_row_stride, int n_forced, int* cur_tok,
                                      DecCtl* ctl, int R) {
    // single CTA: every thread reads ctl->step before thread 0 advances it
    const int next = ctl->step + 1;
    if (next < n_forced)
        for (int r = threadIdx.x; r < R; r += blockDim.x) cur_tok[r] = forced[(int64_t)r * per_row_stride + next];
    __syncthreads();
    if (threadIdx.x == 0) { ctl->pos += 1; ctl->step += 1; }
}

// ------------------------------------------------------------------------------------------------
// beam search (definition: oracle/generate.py docstring)
// stage 1, one CTA per row: rules + log-softmax stats + the row's top-2k candidates
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(SEL_THREADS)
beam_candidates_kernel(float* logits, int V, const GenOptsDev* __restrict__ opts, const uint8_t* __restrict__ sup,
                       const uint8_t* __restrict__ beg, const int* __restrict__ tokens, const int* __restrict__ gen_len,
                       const int* __restrict__ last_ts, float* cand_val, int* cand_idx, float* row_lse, int max_new,
                       DecCtl* ctl) {
    __shared__ ValIdx s_c[SEL_THREADS / 32];
    __shared__ ValIdx s_pick;
    const int r = blockIdx.x;
    const GenOptsDev o = *opts;
    float* lg = logits + (int64_t)r * V;
    const int* toks = tokens + (int64_t)r * max_new;
    const int chunk = r / o.beam;
    const RowRule rr = make_rule(toks, gen_len[chunk], last_ts[r], o);
    ValIdx best; float lse;
    row_rules_and_stats(lg, V, rr, o, sup, beg, best, lse);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nc = 2 * o.beam;
    // thread-local sorted top-NCAND of its strided elements (static indices keep the list in registers)
    ValIdx loc[NCAND];
#pragma unroll
    for (int j = 0; j < NCAND; ++j) loc[j] = ValIdx{-INFINITY, 0x7fffffff};
    constexpr int UNR = 4;      // independent loads per trip (same element order per thread as a plain strided loop)
    for (int i0 = tid; i0 < V; i0 += UNR * SEL_THREADS) {
        float v[UNR];
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            const int i = i0 + u * SEL_THREADS;
            v[u] = i < V ? lg[i] : -INFINITY;
        }
#pragma unroll
        for (int u = 0; u < UNR; ++u) {
            ValIdx c{v[u], i0 + u * SEL_THREADS};
            if (c.v == -INFINITY) continue;
            if (c.v > loc[NCAND - 1].v || (c.v == loc[NCAND - 1].v && c.i < loc[NCAND - 1].i)) {
                loc[NCAND - 1] = c;
#pragma unroll
                for (int j = NCAND - 1; j > 0; --j) {
                    const bool up = loc[j].v > loc[j - 1].v || (loc[j].v == loc[j - 1].v && loc[j].i < loc[j - 1].i);
                    if (up) { ValIdx t = loc[j - 1]; loc[j - 1] = loc[j]; loc[j] = t; }
                }
            }
        }
    }
    int head = 0;
    for (int k = 0; k < nc; ++k) {
        ValIdx mine = ValIdx{-INFINITY, 0x7fffffff};
#pragma unroll
        for (int j = 0; j < NCAND; ++j) if (j == head) mine = loc[j];
        ValIdx w = warp_best(mine);
        if (lane == 0) s_c[warp] = w;
        __syncthreads();
        if (tid == 0) {
            ValIdx a = s_c[0];
            for (int ww = 1; ww < SEL_THREADS / 32; ++ww) a = better(a, s_c[ww]);
            s_pick = a;
            cand_val[(int64_t)r * NCAND + k] = a.v;
            cand_idx[(int64_t)r * NCAND + k] = (a.v == -INFINITY) ? 0 : a.i;
        }
        __syncthreads();
        if (s_pick.v != -INFINITY && mine.i == s_pick.i && mine.v == s_pick.v) ++head;
        __syncthreads();
    }
    if (tid == 0) row_lse[r] = lse;
    // The step counters advance HERE: no CTA of this kernel reads them, and the kernel boundary orders the write before
    // every CTA of beam_update_kernel (which used to advance them itself while its other CTAs were still reading pos).
    if (blockIdx.x == 0 && tid == 0) { ctl->pos += 1; ctl->step += 1; }
}

// stage 2, one thread per chunk: merge the k rows' candidates, walk them in order, re-parent the beams
__global__ void beam_update_kernel(const GenOptsDev* __restrict__ opts, const float* __restrict__ cand_val,
                                   const int* __restrict__ cand_idx, const float* __restrict__ row_lse,
                                   const int* __restrict__ tok_in, int* tok_out, int* gen_len, float* cum,
                                   const int* __restrict__ last_ts_in, int* last_ts_out,
                                   const int* __restrict__ idx_in, int* idx_out, int ctx,
                                   int* fin_count, float* fin_score, int* fin_len, int* fin_tok, int* active,
                                   int* cur_tok, DecCtl* ctl, int B, int max_new) {
    const GenOptsDev o = *opts;
    const int k = o.beam, nc = 2 * k;
    const int b = blockIdx.x;
    const int pos = ctl->pos - 1;      // position fed this step (beam_candidates_kernel already advanced the counter); new token goes to pos+1
    __shared__ float s_val[MAX_BEAM * NCAND];
    __shared__ int s_flat[MAX_BEAM * NCAND];
    __shared__ int s_parent[MAX_BEAM], s_tok[MAX_BEAM];
    __shared__ float s_cum[MAX_BEAM];
    __shared__ int s_live, s_active;
    const int tid = threadIdx.x;
    const int gl = gen_len[b];
    if (tid == 0) {
        s_active = active[b];
        s_live = 0;
        if (s_active) {
            // gather k*nc candidates: value = cum[parent] + (logit - lse[parent]); flat = parent*V + token
            int n = 0;
            for (int j = 0; j < k; ++j) {
                const int r = b * k + j;
                const float cj = cum[r];
                for (int c = 0; c < nc; ++c) {
                    const float lv = cand_val[(int64_t)r * NCAND + c];
                    float v = (cj == -INFINITY || lv == -INFINITY) ? -INFINITY : cj + (lv - row_lse[r]);
                    s_val[n] = v;
                    s_flat[n] = j * o.vocab + cand_idx[(int64_t)r * NCAND + c];
                    ++n;
                }
            }
            // selection sort of the top nc by (value desc, flat asc)
            int live = 0;
            int nfin = fin_count[b];
            for (int pick = 0; pick < nc && live < k; ++pick) {
                int bi = -1;
                for (int i = 0; i < n; ++i) {
                    if (s_flat[i] < 0) continue;
                    if (bi < 0 || s_val[i] > s_val[bi] || (s_val[i] == s_val[bi] && s_flat[i] < s_flat[bi])) bi = i;
                }
                if (bi < 0 || s_val[bi] == -INFINITY) break;
                const float val = s_val[bi];
                const int pj = s_flat[bi] / o.vocab, t = s_flat[bi] - pj * o.vocab;
                s_flat[bi] = -1;
                if (t == o.eot) {
                    if (nfin < o.max_fin) {
                        const int len = gl + 1;
                        fin_score[b * MAX_BEAM + nfin] = (o.length_penalty != 0.0f) ? val / powf((float)len, o.length_penalty) : val;
                        fin_len[b * MAX_BEAM + nfin] = gl;
                        const int* src = tok_in + (int64_t)(b * k + pj) * max_new;
                        int* dst = fin_tok + ((int64_t)b * MAX_BEAM + nfin) * max_new;
                        for (int i = 0; i < gl; ++i) dst[i] = src[i];
                        ++nfin;
                    }
                    continue;
                }
                s_parent[live] = pj; s_tok[live] = t; s_cum[live] = val;
                ++live;
            }
            fin_count[b] = nfin;
            s_live = live;
            if (nfin >= o.max_fin || live == 0) {
                s_active = 0;
                active[b] = 0;
                atomicAdd(&ctl->n_done, 1);
            }
        }
    }
    __syncthreads();
    const int live = s_live;
    // re-parent: token histories, timestamps state, cache index tables
    for (int j = 0; j < k; ++j) {
        const int row = b * k + j;
        int* dst = tok_out + (int64_t)row * max_new;
        int* idst = idx_out + (int64_t)row * ctx;
        if (j < live) {
            const int prow = b * k + s_parent[j];
            const int* src = tok_in + (int64_t)prow * max_new;
            const int* isrc = idx_in + (int64_t)prow * ctx;
            for (int i = tid; i < gl; i += blockDim.x) dst[i] = src[i];
            // positions 0..pos were written in rows named by the parent's table (its own row for position pos)
            for (int i = tid; i <= pos; i += blockDim.x) idst[i] = (i == pos) ? prow : isrc[i];
            if (tid == 0) {
                dst[gl] = s_tok[j];
                cum[row] = s_cum[j];
                cur_tok[row] = s_tok[j];
                const int lt = last_ts_in[prow];
                last_ts_out[row] = (o.with_timestamps && s_tok[j] >= o.timestamp_begin) ? s_tok[j] : lt;
            }
        } else {
            const int* src = tok_in + (int64_t)row * max_new;
            const int* isrc = idx_in + (int64_t)row * ctx;
            for (int i = tid; i < gl; i += blockDim.x) dst[i] = src[i];
            for (int i = tid; i <= pos; i += blockDim.x) idst[i] = (i == pos) ? row : isrc[i];
            if (tid == 0) {
                if (s_active || live > 0) cum[row] = -INFINITY;    // dead slot of a still-running chunk
                cur_tok[row] = o.eot;
                last_ts_out[row] = last_ts_in[row];
            }
        }
    }
    __syncthreads();
    if (tid == 0 && live > 0) gen_len[b] = gl + 1;
}

// after the last step: chunks still active contribute their live beams (best first) as hypotheses
__global__ void beam_finalize_kernel(const GenOptsDev* __restrict__ opts, const int* __restrict__ tok, const int* __restrict__ gen_len,
                                     const float* __restrict__ cum, int* fin_count, float* fin_score, int* fin_len,
                                     int* fin_tok, const int* __restrict__ active, int max_new) {
    const GenOptsDev o = *opts;
    const int b = blockIdx.x;
    if (threadIdx.x != 0) return;
    int nfin = fin_count[b];
    if (active[b] || nfin == 0) {
        const int gl = gen_len[b];
        for (int j = 0; j < o.beam && nfin < o.max_fin; ++j) {
            const int row = b * o.beam + j;
            const float c = cum[row];
            if (c == -INFINITY) continue;
            fin_score[b * MAX_BEAM + nfin] = (o.length_penalty != 0.0f) ? c / powf((float)max(gl, 1), o.length_penalty) : c;
            fin_len[b * MAX_BEAM + nfin] = gl;
            const int* src = tok + (int64_t)row * max_new;
            int* dst = fin_tok + ((int64_t)b * MAX_BEAM + nfin) * max_new;
            for (int i = 0; i < gl; ++i) dst[i] = src[i];
            ++nfin;
        }
        fin_count[b] = nfin;
    }
    // stable sort by score desc (insertion sort on at most MAX_BEAM entries; tokens swapped through indices)
    int order[MAX_BEAM];
    for (int i = 0; i < nfin; ++i) order[i] = i;
    for (int i = 1; i < nfin; ++i) {
        const int oi = order[i];
        int j = i - 1;
        while (j >= 0 && fin_score[b * MAX_BEAM + order[j]] < fin_score[b * MAX_BEAM + oi]) { order[j + 1] = order[j]; --j; }
        order[j + 1] = oi;
    }
    // publish the order in fin_len's upper half: store rank -> slot mapping in cand-free area (reuse active[] is not safe)
    // simplest: write ranks into fin_len as (len | slot << 16) is ambiguous; instead permute scores/lengths in place and
    // remember the slot permutation inside the first token slots' companion array below.
    float sc[MAX_BEAM]; int ln[MAX_BEAM];
    for (int i = 0; i < nfin; ++i) { sc[i] = fin_score[b * MAX_BEAM + order[i]]; ln[i] = fin_len[b * MAX_BEAM + order[i]]; }
    for (int i = 0; i < nfin; ++i) {
        fin_score[b * MAX_BEAM + i] = sc[i];
        fin_len[b * MAX_BEAM + i] = ln[i] | (order[i] << 16);    // low 16 bits: length, high bits: source slot
    }
}

}  // namespace

// ================================================================================================
// host side
// ================================================================================================

mw_status decoder_state_create(mw_model* m) {
    const mw_model_config& c = m->cfg;
    DecoderState* s = new DecoderState();
    m->dec = s;
    const int64_t B = c.max_batch, R = (int64_t)c.max_batch * c.max_beam, T = c.n_audio_ctx, d = c.d_model, L = c.dec_layers;
    const int64_t ctx = c.n_text_ctx, V = c.vocab;
    s->R_max = (int)R;
    s->max_new = (int)(ctx / 2);
    mw_status st = MW_OK;
    auto A = [&](void** p, int64_t bytes, bool zero) { if (st == MW_OK) st = model_alloc(m, p, bytes, zero); };
    A((void**)&s->kv_cross, L * B * T * 2 * d * 2, false);
    A((void**)&s->k_self, L * R * ctx * d * 2, false);
    A((void**)&s->v_self, L * R * ctx * d * 2, false);
    A((void**)&s->x, R * d * 4, false);
    A((void**)&s->ln, R * d * 2, false);
    A((void**)&s->qkv, R * 3 * d * 2, false);
    A((void**)&s->qx, R * d * 2, false);
    A((void**)&s->att, R * d * 2, false);
    A((void**)&s->mlp, R * c.ffn * 2, false);
    A((void**)&s->logits, R * V * 4, false);
    A((void**)&s->cur_tok, R * 4, true);
    A((void**)&s->ctl, sizeof(DecCtl), true);
    A((void**)&s->opts, sizeof(GenOptsDev), true);
    A((void**)&s->prompt, R * ctx * 4, true);
    A((void**)&s->sup_mask, V, true);
    A((void**)&s->begin_mask, V, true);
    for (int i = 0; i < 2; ++i) {
        A((void**)&s->tokens[i], R * s->max_new * 4, true);
        A((void**)&s->last_ts[i], R * 4, true);
        A((void**)&s->self_idx[i], R * ctx * 4, true);
    }
    A((void**)&s->gen_len, R * 4, true);
    A((void**)&s->done, R * 4, true);
    A((void**)&s->cum, R * 4, true);
    A((void**)&s->cand_val, R * NCAND * 4, true);
    A((void**)&s->cand_idx, R * NCAND * 4, true);
    A((void**)&s->row_lse, R * 4, true);
    A((void**)&s->fin_count, B * 4, true);
    A((void**)&s->fin_score, B * MAX_BEAM * 4, true);
    A((void**)&s->fin_len, B * MAX_BEAM * 4, true);
    A((void**)&s->fin_tok, B * MAX_BEAM * s->max_new * 4, true);
    A((void**)&s->active, B * 4, true);
    if (st != MW_OK) return st;
    MW_CUDA_CHECK(cudaMallocHost((void**)&s->h_ctl, 2 * sizeof(DecCtl)));
    MW_CUDA_CHECK(cudaStreamCreateWithFlags(&s->cap_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) MW_CUDA_CHECK(cudaEventCreateWithFlags(&s->ev[i], cudaEventDisableTiming));
    MW_CUDA_CHECK(cudaFuncSetAttribute(decode_attn_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    return MW_OK;
}

static void destroy_graph_entry(DecoderState::Graphs& g) {
    if (g.prefill) cudaGraphExecDestroy(g.prefill);
    for (int i = 0; i < 2; ++i) if (g.gen[i]) cudaGraphExecDestroy(g.gen[i]);
    g = DecoderState::Graphs();
}
static void destroy_graphs(DecoderState* s) {
    for (auto& g : s->graph_cache) destroy_graph_entry(g);
    s->graphs = DecoderState::Graphs();
}

void decoder_state_destroy(mw_model* m) {
    DecoderState* s = m->dec;
    if (!s) return;
    destroy_graphs(s);
    if (s->h_ctl) cudaFreeHost(s->h_ctl);
    if (s->cap_stream) cudaStreamDestroy(s->cap_stream);
    for (int i = 0; i < 2; ++i) if (s->ev[i]) cudaEventDestroy(s->ev[i]);
    delete s;
    m->dec = nullptr;
}

namespace {

mw_status cross_kv_project(mw_model* m, const void* d_enc, int B, cudaStream_t st) {
    const mw_model_config& c = m->cfg;
    DecoderState* s = m->dec;
    const int64_t T = c.n_audio_ctx, d = c.d_model;
    for (int l = 0; l < c.dec_layers; ++l) {
        GemmArgs a;
        a.a = d_enc; a.a_row_stride = d; a.w = m->dlw(l, MW_DL_WXKV); a.w_row_stride = d;
        a.bias = (const float*)m->dlw(l, MW_DL_BXKV);
        a.out = s->kv_cross + (int64_t)l * c.max_batch * T * 2 * d; a.ld_out = 2 * d;
        a.M = (int)(B * T); a.N = (int)(2 * d); a.K = (int)d;
        mw_status r = gemm_launch(a, st);
        if (r != MW_OK) return r;
    }
    return MW_OK;
}

// one decoder step up to (and excluding) the logits; `beam_phase` selects the self-index table to read
enum { PART_EMBED = 1, PART_LN = 2, PART_GEMM = 4, PART_SELF = 8, PART_CROSS = 16, PART_LOGITS = 32, PART_SELECT = 64, PART_ALL = 127 };

mw_status enqueue_layers(mw_model* m, int R, int beam, int idx_phase, cudaStream_t st, int parts = PART_ALL) {
    const mw_model_config& c = m->cfg;
    DecoderState* s = m->dec;
    const int d = c.d_model, ctx = c.n_text_ctx, T = c.n_audio_ctx;
    mw_status r;
    if (parts & PART_EMBED) {
        embed_kernel<<<R, 128, 0, st>>>(s->cur_tok, (const mw_h*)m->gw(MW_DEC_EMB), (const float*)m->gw(MW_DEC_POS), s->ctl, s->x, d);
        MW_LAUNCH_CHECK();
    }
    const int* idx = beam > 1 ? s->self_idx[idx_phase] : nullptr;
    for (int l = 0; l < c.dec_layers; ++l) {
        auto W = [&](int id) { return m->dlw(l, id); };
        auto F = [&](int id) { return (const float*)m->dlw(l, id); };
        const bool LN = parts & PART_LN, GM = parts & PART_GEMM;
        const bool dg = beam <= 1;
        const int64_t dd = (int64_t)d * d * 2, df = (int64_t)d * c.ffn * 2;          // bytes of a d x d / d x ffn weight matrix
        const void* next_qkv = l + 1 < c.dec_layers ? m->dlw(l + 1, MW_DL_WQKV) : nullptr;
        const char* pf_xo = GM ? (const char*)W(MW_DL_WXO) : nullptr;
        if (LN && GM) {
            if ((r = skinny_gemm_ln(s->x, F(MW_DL_LN1_G), F(MW_DL_LN1_B), s->ln, W(MW_DL_WQKV), F(MW_DL_BQKV), s->qkv, 3 * d, R, 3 * d, d, 0,
                                    st, dg, W(MW_DL_WO), dd, s->solo)) != MW_OK) return r;
        } else {
            if (LN && (r = layernorm_launch(s->x, F(MW_DL_LN1_G), F(MW_DL_LN1_B), s->ln, R, d, st)) != MW_OK) return r;
            if (GM && (r = skinny_gemm(s->ln, d, W(MW_DL_WQKV), d, F(MW_DL_BQKV), nullptr, s->qkv, 3 * d, R, 3 * d, d, 0, st, dg, W(MW_DL_WO), dd)) != MW_OK) return r;
        }
        if (parts & PART_SELF) {
            mw_h* kc = s->k_self + (int64_t)l * s->R_max * ctx * d;
            mw_h* vc = s->v_self + (int64_t)l * s->R_max * ctx * d;
            dim3 grid(c.n_heads, R);
            decode_attn_kernel<true><<<grid, 128, ctx * sizeof(float), st>>>(s->qkv, 3 * d, kc, vc, d, ctx, idx, ctx, s->ctl, 0, 1, s->qkv + d,
                                                                            s->qkv + 2 * d, 3 * d, s->att, d, 0);
            MW_LAUNCH_CHECK();
        }
        if (GM && (r = skinny_gemm(s->att, d, W(MW_DL_WO), d, F(MW_DL_BO), s->x, s->x, d, R, d, d, SK_FLAG_F32, st, dg, W(MW_DL_WXQ), dd)) != MW_OK) return r;
        if (LN && GM) {
            if ((r = skinny_gemm_ln(s->x, F(MW_DL_LNX_G), F(MW_DL_LNX_B), s->ln, W(MW_DL_WXQ), F(MW_DL_BXQ), s->qx, d, R, d, d, 0, st, dg,
                                    nullptr, 0, s->solo)) != MW_OK) return r;
        } else {
            if (LN && (r = layernorm_launch(s->x, F(MW_DL_LNX_G), F(MW_DL_LNX_B), s->ln, R, d, st)) != MW_OK) return r;
            if (GM && (r = skinny_gemm(s->ln, d, W(MW_DL_WXQ), d, F(MW_DL_BXQ), nullptr, s->qx, d, R, d, d, 0, st, dg)) != MW_OK) return r;
        }
        if (parts & PART_CROSS) {
            mw_h* kv = s->kv_cross + (int64_t)l * c.max_batch * T * 2 * d;
            if (beam > 1) {
                const int Bc = R / beam;
#define MW_XG(g) case g: r = launch_cross_grouped<g>(s->qx, d, kv, kv + d, 2 * d, T, s->att, d, c.n_heads, Bc, st); break
                switch (beam) {
                    MW_XG(2); MW_XG(3); MW_XG(4); MW_XG(5); MW_XG(6); MW_XG(7); MW_XG(8);
                    default: r = MW_ERR_UNSUPPORTED; set_error("beam_size %d unsupported", beam);
                }
#undef MW_XG
                if (r != MW_OK) return r;
            } else {
                dim3 grid(c.n_heads, R);
                // under-filled grid (fewer CTAs than 3 per SM): more loads in flight per CTA, same arithmetic
                if ((int)(grid.x * grid.y) <= 3 * device_sm_count())
                    cross_attn_stream_kernel<8><<<grid, 128, 0, st>>>(s->qx, d, kv, kv + d, 2 * d, T, s->att, d, pf_xo, (int)(dd / 128));
                else
                    cross_attn_stream_kernel<4><<<grid, 128, 0, st>>>(s->qx, d, kv, kv + d, 2 * d, T, s->att, d, pf_xo, (int)(dd / 128));
                MW_LAUNCH_CHECK();
            }
        }
        if (GM && (r = skinny_gemm(s->att, d, W(MW_DL_WXO), d, F(MW_DL_BXO), s->x, s->x, d, R, d, d, SK_FLAG_F32, st, dg, W(MW_DL_W1), df)) != MW_OK) return r;
        if (LN && GM) {
            if ((r = skinny_gemm_ln(s->x, F(MW_DL_LN2_G), F(MW_DL_LN2_B), s->ln, W(MW_DL_W1), F(MW_DL_B1), s->mlp, c.ffn, R, c.ffn, d,
                                    SK_FLAG_GELU, st, dg, W(MW_DL_W2), df, s->solo)) != MW_OK) return r;
        } else {
            if (LN && (r = layernorm_launch(s->x, F(MW_DL_LN2_G), F(MW_DL_LN2_B), s->ln, R, d, st)) != MW_OK) return r;
            if (GM && (r = skinny_gemm(s->ln, d, W(MW_DL_W1), d, F(MW_DL_B1), nullptr, s->mlp, c.ffn, R, c.ffn, d, SK_FLAG_GELU, st, dg, W(MW_DL_W2), df)) != MW_OK) return r;
        }
        if (GM && (r = skinny_gemm(s->mlp, c.ffn, W(MW_DL_W2), c.ffn, F(MW_DL_B2), s->x, s->x, d, R, d, c.ffn, SK_FLAG_F32, st, dg, next_qkv, 3 * dd, s->solo)) != MW_OK) return r;
    }
    return MW_OK;
}

mw_status enqueue_logits(mw_model* m, int R, cudaStream_t st) {
    const mw_model_config& c = m->cfg;
    DecoderState* s = m->dec;
    mw_status r;
    if ((r = layernorm_launch(s->x, (const float*)m->gw(MW_DEC_LN_G), (const float*)m->gw(MW_DEC_LN_B), s->ln, R, c.d_model, st)) != MW_OK) return r;
    return skinny_gemm(s->ln, c.d_model, m->gw(MW_DEC_EMB), c.d_model, nullptr, nullptr, s->logits, c.vocab, R, c.vocab,
                       c.d_model, SK_FLAG_F32, st);
}

mw_status enqueue_select(mw_model* m, int B, int beam, int phase, cudaStream_t st) {
    const mw_model_config& c = m->cfg;
    DecoderState* s = m->dec;
    const int R = B * beam;
    if (beam <= 1) {
        select_greedy_kernel<<<R, SEL_THREADS, 0, st>>>(s->logits, c.vocab, s->opts, s->sup_mask, s->begin_mask, s->tokens[0], s->gen_len,
                                                       s->done, s->cum, s->last_ts[0], s->cur_tok, s->ctl, s->max_new);
        MW_LAUNCH_CHECK();
        return MW_OK;
    }
    beam_candidates_kernel<<<R, SEL_THREADS, 0, st>>>(s->logits, c.vocab, s->opts, s->sup_mask, s->begin_mask, s->tokens[phase],
                                                      s->gen_len, s->last_ts[phase], s->cand_val, s->cand_idx, s->row_lse, s->max_new,
                                                      s->ctl);
    MW_LAUNCH_CHECK();
    beam_update_kernel<<<B, 128, 0, st>>>(s->opts, s->cand_val, s->cand_idx, s->row_lse, s->tokens[phase], s->tokens[phase ^ 1],
                                          s->gen_len, s->cum, s->last_ts[phase], s->last_ts[phase ^ 1], s->self_idx[phase],
                                          s->self_idx[phase ^ 1], c.n_text_ctx, s->fin_count, s->fin_score, s->fin_len, s->fin_tok,
                                          s->active, s->cur_tok, s->ctl, B, s->max_new);
    MW_LAUNCH_CHECK();
    return MW_OK;
}

template <typename Fn>
mw_status capture_graph(DecoderState* s, cudaGraphExec_t* out, int* n_nodes, Fn&& enqueue) {
    cudaGraph_t graph = nullptr;
    MW_CUDA_CHECK(cudaStreamBeginCapture(s->cap_stream, cudaStreamCaptureModeThreadLocal));
    t_capturing = true;                      // captured launches are counted when the graph is replayed
    t_captured = 0;
    mw_status r = enqueue(s->cap_stream);
    t_capturing = false;
    *n_nodes = (int)t_captured;
    cudaError_t e = cudaStreamEndCapture(s->cap_stream, &graph);
    if (r != MW_OK) { if (graph) cudaGraphDestroy(graph); return r; }
    if (e != cudaSuccess) { set_error("graph capture failed: %s", cudaGetErrorString(e)); return MW_ERR_CUDA; }
    e = cudaGraphInstantiate(out, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) { set_error("graph instantiate failed: %s", cudaGetErrorString(e)); return MW_ERR_CUDA; }
    return MW_OK;
}

// ------------------------------------------------------------------------------------------------
// Batched prefill: the prompt tokens 0..P-2 of all chunks go through the decoder in ONE pass (M = B*(P-1) rows) on
// the tensor-core GEMM / flash-attention kernels of the encoder, instead of P-1 single-token steps.  What it leaves
// behind is exactly what the step graph expects: self K/V of positions 0..P-2 in the cache (physical row b*beam,
// shared by the beams through the index table), pos = step = P-1 and the last prompt token as the next input.
// Matters for the reference's own call, which passes an initial_prompt (/root/reference/transcribe.py:40,111).
// ------------------------------------------------------------------------------------------------
__global__ void embed_prefill_kernel(const int* __restrict__ prompt, const mw_h* __restrict__ emb,
                                     const float* __restrict__ pos_emb, float* __restrict__ x, int Pm, int d) {
    const int r = blockIdx.x, p = r % Pm;
    const int tok = prompt[p];
    for (int i = threadIdx.x; i < d; i += blockDim.x)
        x[(int64_t)r * d + i] = h2f(emb[(int64_t)tok * d + i]) + pos_emb[(int64_t)p * d + i];
}

__global__ void kv_scatter_kernel(const mw_h* __restrict__ qkv, mw_h* __restrict__ kc, mw_h* __restrict__ vc,
                                  int Pm, int d, int ctx, int beam) {
    const int r = blockIdx.x, b = r / Pm, p = r - b * Pm;
    const uint4* src = reinterpret_cast<const uint4*>(qkv + (int64_t)r * 3 * d + d);
    uint4* dk = reinterpret_cast<uint4*>(kc + ((int64_t)(b * beam) * ctx + p) * d);
    uint4* dv = reinterpret_cast<uint4*>(vc + ((int64_t)(b * beam) * ctx + p) * d);
    const int nv = d / 8;
    for (int i = threadIdx.x; i < nv; i += blockDim.x) { dk[i] = src[i]; dv[i] = src[nv + i]; }
}

__global__ void prefill_finish_kernel(const int* __restrict__ prompt, int Pm, int* cur_tok, DecCtl* ctl, int* idx0, int* idx1,
                                      int R, int ctx, int beam) {
    for (int r = threadIdx.x; r < R; r += blockDim.x) {
        cur_tok[r] = prompt[Pm];
        if (idx0) {
            const int phys = (r / beam) * beam;
            for (int p = 0; p < Pm; ++p) { idx0[(int64_t)r * ctx + p] = phys; idx1[(int64_t)r * ctx + p] = phys; }
        }
    }
    if (threadIdx.x == 0) { ctl->pos = Pm; ctl->step = Pm; }
}

mw_status batched_prefill(mw_model* m, int B, int beam, int Pm, cudaStream_t st) {
    const mw_model_config& c = m->cfg;
    DecoderState* s = m->dec;
    const int d = c.d_model, ctx = c.n_text_ctx, T = c.n_audio_ctx, M = B * Pm, R = B * beam;
    mw_status r;
    embed_prefill_kernel<<<M, 128, 0, st>>>(s->prompt, (const mw_h*)m->gw(MW_DEC_EMB), (const float*)m->gw(MW_DEC_POS), m->x, Pm, d);
    MW_LAUNCH_CHECK();
    auto gemm = [&](const void* A, int K, const void* W, const float* bias, const float* res, void* out, int N, bool gelu, bool f32) {
        GemmArgs a;
        a.a = A; a.a_row_stride = K; a.w = W; a.w_row_stride = K; a.bias = bias;
        a.residual = res; a.ld_res = N; a.out = out; a.ld_out = N; a.M = M; a.N = N; a.K = K; a.gelu = gelu; a.out_f32 = f32;
        return gemm_launch(a, st);
    };
    for (int l = 0; l < c.dec_layers; ++l) {
        auto W = [&](int id) { return m->dlw(l, id); };
        auto F = [&](int id) { return (const float*)m->dlw(l, id); };
        mw_h* kc = s->k_self + (int64_t)l * s->R_max * ctx * d;
        mw_h* vc = s->v_self + (int64_t)l * s->R_max * ctx * d;
        if ((r = layernorm_launch(m->x, F(MW_DL_LN1_G), F(MW_DL_LN1_B), m->ln, M, d, st)) != MW_OK) return r;
        if ((r = gemm(m->ln, d, W(MW_DL_WQKV), F(MW_DL_BQKV), nullptr, m->qkv, 3 * d, false, false)) != MW_OK) return r;
        kv_scatter_kernel<<<M, 128, 0, st>>>(m->qkv, kc, vc, Pm, d, ctx, beam);
        MW_LAUNCH_CHECK();
        {   // causal self-attention straight from the packed q|k|v rows of this pass
            dim3 grid(c.n_heads, M);
            decode_attn_kernel<false><<<grid, 128, Pm * sizeof(float), st>>>(m->qkv, 3 * d, m->qkv + d, m->qkv + 2 * d, 3 * d, Pm, nullptr,
                                                                            ctx, s->ctl, Pm, Pm, nullptr, nullptr, 0, m->att, d, Pm);
            MW_LAUNCH_CHECK();
        }
        if ((r = gemm(m->att, d, W(MW_DL_WO), F(MW_DL_BO), m->x, m->x, d, false, true)) != MW_OK) return r;
        if ((r = layernorm_launch(m->x, F(MW_DL_LNX_G), F(MW_DL_LNX_B), m->ln, M, d, st)) != MW_OK) return r;
        if ((r = gemm(m->ln, d, W(MW_DL_WXQ), F(MW_DL_BXQ), nullptr, m->att, d, false, false)) != MW_OK) return r;     // cross q
        {
            mw_h* kv = s->kv_cross + (int64_t)l * c.max_batch * T * 2 * d;
            if ((r = attention_launch_general(m->att, d, 0, kv, 2 * d, 0, d, m->ln, d, B, Pm, T, c.n_heads, st)) != MW_OK) return r;
        }
        if ((r = gemm(m->ln, d, W(MW_DL_WXO), F(MW_DL_BXO), m->x, m->x, d, false, true)) != MW_OK) return r;
        if ((r = layernorm_launch(m->x, F(MW_DL_LN2_G), F(MW_DL_LN2_B), m->ln, M, d, st)) != MW_OK) return r;
        if ((r = gemm(m->ln, d, W(MW_DL_W1), F(MW_DL_B1), nullptr, m->mlp, c.ffn, true, false)) != MW_OK) return r;
        if ((r = gemm(m->mlp, c.ffn, W(MW_DL_W2), F(MW_DL_B2), m->x, m->x, d, false, true)) != MW_OK) return r;
    }
    prefill_finish_kernel<<<1, 256, 0, st>>>(s->prompt, Pm, s->cur_tok, s->ctl, beam > 1 ? s->self_idx[0] : nullptr,
                                             beam > 1 ? s->self_idx[1] : nullptr, R, ctx, beam);
    MW_LAUNCH_CHECK();
    return MW_OK;
}

std::atomic<int> g_step_parts{PART_ALL};
std::atomic<int> g_step_parts_epoch{0};

mw_status ensure_graphs(mw_model* m, int B, int beam) {
    DecoderState* s = m->dec;
    const int R = B * beam;
    if (s->parts_epoch != g_step_parts_epoch.load()) {      // the kept classes changed: cached graphs are stale
        destroy_graphs(s);
        s->parts_epoch = g_step_parts_epoch.load();
    }
    DecoderState::Graphs* slot = nullptr;
    for (auto& g : s->graph_cache)
        if (g.prefill && g.R == R && g.beam == beam && g.solo == s->solo) { g.last_use = ++s->graph_clock; s->graphs = g; return MW_OK; }
    slot = &s->graph_cache[0];                // a free slot, else the least recently used one
    for (auto& g : s->graph_cache) {
        if (!g.prefill) { slot = &g; break; }
        if (g.last_use < slot->last_use) slot = &g;
    }
    destroy_graph_entry(*slot);
    s->graphs = DecoderState::Graphs();
    mw_status r;
    // prefill step: layers + forced advance.  With beam search the prefill rows are their own ancestors, so the
    // identity index table (phase 0) is used.
    r = capture_graph(s, &s->graphs.prefill, &s->graphs.n_prefill, [&](cudaStream_t st) -> mw_status {
        mw_status q = enqueue_layers(m, R, beam, 0, st);
        if (q != MW_OK) return q;
        advance_forced_kernel<<<1, 256, 0, st>>>(s->prompt, 0, 1 << 30, s->cur_tok, s->ctl, R);
        MW_LAUNCH_CHECK();
        return MW_OK;
    });
    if (r != MW_OK) { destroy_graph_entry(s->graphs); return r; }
    for (int phase = 0; phase < (beam > 1 ? 2 : 1); ++phase) {
        // measurement only (mw_debug_step_parts; ids are then meaningless): kernel classes kept in the step graph
        const int step_parts = g_step_parts.load();
        r = capture_graph(s, &s->graphs.gen[phase], &s->graphs.n_gen[phase], [&](cudaStream_t st) -> mw_status {
            mw_status q = enqueue_layers(m, R, beam, phase, st, step_parts);
            if (q != MW_OK) return q;
            if ((q = enqueue_logits(m, R, st)) != MW_OK) return q;
            return enqueue_select(m, B, beam, phase, st);
        });
        if (r != MW_OK) { destroy_graph_entry(s->graphs); return r; }
    }
    s->graphs.R = R;
    s->graphs.beam = beam;
    s->graphs.solo = s->solo;
    s->graphs.last_use = ++s->graph_clock;
    *slot = s->graphs;
    return MW_OK;
}

__global__ void fill_identity_idx_kernel(int* idx, int R, int ctx) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < R * ctx) idx[i] = i / ctx;
}
__global__ void init_beam_state_kernel(float* cum, int* last_ts0, int* last_ts1, int* active, int B, int beam) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < B * beam) {
        cum[r] = (r % beam == 0) ? 0.0f : -INFINITY;
        last_ts0[r] = -1;
        last_ts1[r] = -1;
    }
    if (r < B) active[r] = 1;
}

mw_status reset_state(mw_model* m, int B, int beam, const int32_t* h_prompt, int prompt_len, const mw_gen_options* opt,
                      int n_prefill, int max_new, cudaStream_t st) {
    const mw_model_config& c = m->cfg;
    DecoderState* s = m->dec;
    const int R = B * beam;
    GenOptsDev o{};
    o.eot = opt ? opt->eot : 0;
    o.timestamp_begin = opt ? opt->timestamp_begin : c.vocab;
    o.with_timestamps = opt ? opt->with_timestamps : 0;
    o.max_initial_ts = opt ? opt->max_initial_timestamp_index : -1;
    o.forced_eot_len = opt ? opt->forced_eot_len : 0;
    o.beam = beam;
    o.max_new = max_new;
    o.max_fin = opt ? std::max(1, std::min((int)MAX_BEAM, (int)lroundf(beam * opt->patience))) : 1;
    o.length_penalty = opt ? opt->length_penalty : 1.0f;
    o.n_prefill = n_prefill;
    o.vocab = c.vocab;
    MW_CUDA_CHECK(cudaMemcpyAsync(s->opts, &o, sizeof(o), cudaMemcpyHostToDevice, st));
    if (opt) {
        std::vector<uint8_t> sup(c.vocab, 0), beg(c.vocab, 0);
        for (int i = 0; i < opt->n_suppress; ++i) {
            const int t = opt->h_suppress[i];
            MW_REQUIRE(t >= 0 && t < c.vocab, "mw_generate: suppress id %d outside the vocabulary", t);
            sup[t] = 1;
        }
        for (int i = 0; i < opt->n_suppress_begin; ++i) {
            const int t = opt->h_suppress_begin[i];
            MW_REQUIRE(t >= 0 && t < c.vocab, "mw_generate: begin-suppress id %d outside the vocabulary", t);
            beg[t] = 1;
        }
        MW_CUDA_CHECK(cudaMemcpyAsync(s->sup_mask, sup.data(), c.vocab, cudaMemcpyHostToDevice, st));
        MW_CUDA_CHECK(cudaMemcpyAsync(s->begin_mask, beg.data(), c.vocab, cudaMemcpyHostToDevice, st));
        MW_CUDA_CHECK(cudaStreamSynchronize(st));     // sup/beg are stack-lifetime host vectors
    }
    MW_CUDA_CHECK(cudaMemsetAsync(s->ctl, 0, sizeof(DecCtl), st));
    MW_CUDA_CHECK(cudaMemsetAsync(s->gen_len, 0, R * 4, st));
    MW_CUDA_CHECK(cudaMemsetAsync(s->done, 0, R * 4, st));
    MW_CUDA_CHECK(cudaMemsetAsync(s->cum, 0, R * 4, st));
    MW_CUDA_CHECK(cudaMemsetAsync(s->fin_count, 0, B * 4, st));
    init_beam_state_kernel<<<ceil_div(R, 256), 256, 0, st>>>(s->cum, s->last_ts[0], s->last_ts[1], s->active, B, beam);
    MW_LAUNCH_CHECK();
    if (beam > 1) {
        for (int i = 0; i < 2; ++i) {
            fill_identity_idx_kernel<<<ceil_div(R * c.n_text_ctx, 256), 256, 0, st>>>(s->self_idx[i], R, c.n_text_ctx);
            MW_LAUNCH_CHECK();
        }
    }
    if (h_prompt && prompt_len > 0) {
        MW_CUDA_CHECK(cudaMemcpyAsync(s->prompt, h_prompt, prompt_len * 4, cudaMemcpyHostToDevice, st));
        std::vector<int> first(R, h_prompt[0]);
        MW_CUDA_CHECK(cudaMemcpyAsync(s->cur_tok, first.data(), R * 4, cudaMemcpyHostToDevice, st));
        MW_CUDA_CHECK(cudaStreamSynchronize(st));
    }
    return MW_OK;
}

}  // namespace
}  // namespace mw

using namespace mw;

extern "C" mw_status mw_generate(mw_model* m, const void* d_enc, int B, const int32_t* h_prompt, int prompt_len,
                                 const mw_gen_options* opt, int32_t* h_out_ids, int32_t* h_out_len, float* h_out_scores,
                                 void* stream) {
    MW_REQUIRE(m && d_enc && h_prompt && opt && h_out_ids && h_out_len && h_out_scores, "mw_generate: null argument");
    const mw_model_config& c = m->cfg;
    DecoderState* s = m->dec;
    const int beam = opt->beam_size < 1 ? 1 : opt->beam_size;
    MW_REQUIRE(B > 0 && B <= c.max_batch, "mw_generate: B=%d outside 1..max_batch=%d", B, c.max_batch);
    MW_REQUIRE(beam <= c.max_beam && beam <= MAX_BEAM, "mw_generate: beam_size=%d exceeds the model's max_beam=%d", beam, c.max_beam);
    MW_REQUIRE(prompt_len >= 1 && prompt_len < c.n_text_ctx, "mw_generate: prompt_len=%d outside 1..%d", prompt_len, c.n_text_ctx - 1);
    MW_REQUIRE(opt->max_length >= 2 && opt->max_length <= c.n_text_ctx, "mw_generate: max_length=%d outside 2..%d", opt->max_length, c.n_text_ctx);
    for (int i = 0; i < prompt_len; ++i)
        MW_REQUIRE(h_prompt[i] >= 0 && h_prompt[i] < c.vocab, "mw_generate: prompt token %d outside the vocabulary", h_prompt[i]);
    MW_REQUIRE(opt->eot >= 0 && opt->eot < c.vocab, "mw_generate: eot outside the vocabulary");
    const int nh = std::max(1, std::min(opt->num_hypotheses, beam));
    const int max_new = std::max(0, std::min(opt->max_length / 2, opt->max_length - prompt_len));
    const int out_stride = std::max(max_new, 1);
    MW_REQUIRE(max_new <= s->max_new, "mw_generate: max_new=%d exceeds workspace", max_new);
    mw::DeviceGuard guard(c.device);
    cudaStream_t st = (cudaStream_t)stream;
    const int R = B * beam;
    for (int i = 0; i < B * nh; ++i) { h_out_len[i] = 0; h_out_scores[i] = 0.0f; }
    if (max_new == 0) return MW_OK;
    mw_status r;
    if ((r = cross_kv_project(m, d_enc, B, st)) != MW_OK) return r;
    if ((r = reset_state(m, B, beam, h_prompt, prompt_len, opt, prompt_len - 1, max_new, st)) != MW_OK) return r;
    if ((r = ensure_graphs(m, B, beam)) != MW_OK) return r;
    const int Pm = prompt_len - 1;
    const char* force_stepwise = getenv("MW_STEPWISE_PREFILL");      // test hook: compare the two prefill paths
    if (Pm >= 4 && Pm <= c.n_audio_ctx && !(force_stepwise && force_stepwise[0] == '1')) {
        if ((r = batched_prefill(m, B, beam, Pm, st)) != MW_OK) return r;       // long prompts (initial_prompt): one pass
    } else {
        for (int i = 0; i < Pm; ++i) {
            MW_CUDA_CHECK(cudaGraphLaunch(s->graphs.prefill, st));
            count_launch(s->graphs.n_prefill);        // nodes counted when the graph was captured
        }
    }
    // generation: the finished counter is polled one window late so the stream never drains
    const int window = 8;
    const int n_target = beam > 1 ? B : R;
    int pending = -1, w = 0;
    bool stop = false;
    for (int step = 0; step < max_new && !stop; ++step) {
        MW_CUDA_CHECK(cudaGraphLaunch(s->graphs.gen[beam > 1 ? (step & 1) : 0], st));
        count_launch(s->graphs.n_gen[beam > 1 ? (step & 1) : 0]);
        if ((step + 1) % window == 0 && step + 1 < max_new) {
            MW_CUDA_CHECK(cudaMemcpyAsync(&s->h_ctl[w & 1], s->ctl, sizeof(DecCtl), cudaMemcpyDeviceToHost, st));
            MW_CUDA_CHECK(cudaEventRecord(s->ev[w & 1], st));
            if (pending >= 0) {
                MW_CUDA_CHECK(cudaEventSynchronize(s->ev[pending & 1]));
                if (s->h_ctl[pending & 1].n_done >= n_target) stop = true;
            }
            pending = w;
            ++w;
        }
    }
    // ---- results
    if (beam <= 1) {
        std::vector<int> len(R), toks((size_t)R * s->max_new);
        std::vector<float> cum(R);
        std::vector<int> done(R);
        MW_CUDA_CHECK(cudaMemcpyAsync(len.data(), s->gen_len, R * 4, cudaMemcpyDeviceToHost, st));
        MW_CUDA_CHECK(cudaMemcpyAsync(cum.data(), s->cum, R * 4, cudaMemcpyDeviceToHost, st));
        MW_CUDA_CHECK(cudaMemcpyAsync(done.data(), s->done, R * 4, cudaMemcpyDeviceToHost, st));
        MW_CUDA_CHECK(cudaMemcpyAsync(toks.data(), s->tokens[0], (size_t)R * s->max_new * 4, cudaMemcpyDeviceToHost, st));
        MW_CUDA_CHECK(cudaStreamSynchronize(st));
        for (int b = 0; b < B; ++b) {
            const int n = std::min(len[b], max_new);
            h_out_len[b * nh] = n;
            for (int i = 0; i < n; ++i) h_out_ids[(size_t)b * nh * out_stride + i] = toks[(size_t)b * s->max_new + i];
            const int length = n + (done[b] ? 1 : 0);
            h_out_scores[b * nh] = (opt->length_penalty != 0.0f) ? cum[b] / powf((float)std::max(length, 1), opt->length_penalty) : cum[b];
        }
        return MW_OK;
    }
    const int final_phase = 0;   // both token buffers hold the live histories of their own phase; pick the current one
    (void)final_phase;
    {
        // the buffer written by the last executed step is tokens[(steps & 1)]: step i reads phase i&1 and writes (i&1)^1
        MW_CUDA_CHECK(cudaMemcpyAsync(&s->h_ctl[0], s->ctl, sizeof(DecCtl), cudaMemcpyDeviceToHost, st));
        MW_CUDA_CHECK(cudaStreamSynchronize(st));
        const int gen_steps = s->h_ctl[0].step - (prompt_len - 1);
        const int cur = gen_steps & 1;
        beam_finalize_kernel<<<B, 32, 0, st>>>(s->opts, s->tokens[cur], s->gen_len, s->cum, s->fin_count, s->fin_score,
                                               s->fin_len, s->fin_tok, s->active, s->max_new);
        MW_LAUNCH_CHECK();
        std::vector<int> cnt(B), flen((size_t)B * MAX_BEAM), ftok((size_t)B * MAX_BEAM * s->max_new);
        std::vector<float> fsc((size_t)B * MAX_BEAM);
        MW_CUDA_CHECK(cudaMemcpyAsync(cnt.data(), s->fin_count, B * 4, cudaMemcpyDeviceToHost, st));
        MW_CUDA_CHECK(cudaMemcpyAsync(flen.data(), s->fin_len, (size_t)B * MAX_BEAM * 4, cudaMemcpyDeviceToHost, st));
        MW_CUDA_CHECK(cudaMemcpyAsync(fsc.data(), s->fin_score, (size_t)B * MAX_BEAM * 4, cudaMemcpyDeviceToHost, st));
        MW_CUDA_CHECK(cudaMemcpyAsync(ftok.data(), s->fin_tok, (size_t)B * MAX_BEAM * s->max_new * 4, cudaMemcpyDeviceToHost, st));
        MW_CUDA_CHECK(cudaStreamSynchronize(st));
        for (int b = 0; b < B; ++b) {
            for (int hyp = 0; hyp < nh && hyp < cnt[b]; ++hyp) {
                const int packed = flen[(size_t)b * MAX_BEAM + hyp];
                const int n = std::min(packed & 0xffff, max_new), slot = packed >> 16;
                h_out_len[b * nh + hyp] = n;
                h_out_scores[b * nh + hyp] = fsc[(size_t)b * MAX_BEAM + hyp];
                for (int i = 0; i < n; ++i)
                    h_out_ids[((size_t)b * nh + hyp) * out_stride + i] = ftok[((size_t)b * MAX_BEAM + slot) * s->max_new + i];
            }
        }
    }
    return MW_OK;
}

extern "C" mw_status mw_decoder_logits(mw_model* m, const void* d_enc, int B, const int32_t* h_tokens, int n,
                                       float* d_logits, void* stream) {
    MW_REQUIRE(m && d_enc && h_tokens && d_logits, "mw_decoder_logits: null argument");
    const mw_model_config& c = m->cfg;
    DecoderState* s = m->dec;
    MW_REQUIRE(B > 0 && B <= c.max_batch && B <= s->R_max, "mw_decoder_logits: B=%d outside 1..%d", B, c.max_batch);
    MW_REQUIRE(n >= 1 && n <= c.n_text_ctx, "mw_decoder_logits: n=%d outside 1..%d", n, c.n_text_ctx);
    for (int i = 0; i < B * n; ++i)
        MW_REQUIRE(h_tokens[i] >= 0 && h_tokens[i] < c.vocab, "mw_decoder_logits: token %d outside the vocabulary", h_tokens[i]);
    mw::DeviceGuard guard(c.device);
    cudaStream_t st = (cudaStream_t)stream;
    mw_status r;
    if ((r = cross_kv_project(m, d_enc, B, st)) != MW_OK) return r;
    if ((r = reset_state(m, B, 1, nullptr, 0, nullptr, 0, 0, st)) != MW_OK) return r;
    // per-row forced token lists: prompt buffer holds [B][n]
    MW_CUDA_CHECK(cudaMemcpyAsync(s->prompt, h_tokens, (size_t)B * n * 4, cudaMemcpyHostToDevice, st));
    std::vector<int> first(B);
    for (int b = 0; b < B; ++b) first[b] = h_tokens[(size_t)b * n];
    MW_CUDA_CHECK(cudaMemcpyAsync(s->cur_tok, first.data(), B * 4, cudaMemcpyHostToDevice, st));
    MW_CUDA_CHECK(cudaStreamSynchronize(st));
    for (int i = 0; i < n; ++i) {
        if ((r = enqueue_layers(m, B, 1, 0, st)) != MW_OK) return r;
        if ((r = enqueue_logits(m, B, st)) != MW_OK) return r;
        MW_CUDA_CHECK(cudaMemcpy2DAsync(d_logits + (size_t)i * c.vocab, (size_t)n * c.vocab * 4, s->logits, (size_t)c.vocab * 4,
                                        (size_t)c.vocab * 4, B, cudaMemcpyDeviceToDevice, st));
        advance_forced_kernel<<<1, 256, 0, st>>>(s->prompt, n, n, s->cur_tok, s->ctl, B);
        MW_LAUNCH_CHECK();
    }
    return MW_OK;
}

extern "C" mw_status mw_detect_language(mw_model* m, const void* d_enc, int B, int32_t sot, int32_t first_lang,
                                        int32_t n_langs, float* h_probs, void* stream) {
    MW_REQUIRE(m && d_enc && h_probs, "mw_detect_language: null argument");
    const mw_model_config& c = m->cfg;
    DecoderState* s = m->dec;
    MW_REQUIRE(B > 0 && B <= c.max_batch, "mw_detect_language: B=%d outside 1..%d", B, c.max_batch);
    MW_REQUIRE(sot >= 0 && sot < c.vocab && first_lang >= 0 && n_langs > 0 && first_lang + n_langs <= c.vocab,
               "mw_detect_language: token ids outside the vocabulary");
    mw::DeviceGuard guard(c.device);
    cudaStream_t st = (cudaStream_t)stream;
    mw_status r;
    if ((r = cross_kv_project(m, d_enc, B, st)) != MW_OK) return r;
    if ((r = reset_state(m, B, 1, &sot, 1, nullptr, 0, 0, st)) != MW_OK) return r;
    if ((r = enqueue_layers(m, B, 1, 0, st)) != MW_OK) return r;
    if ((r = enqueue_logits(m, B, st)) != MW_OK) return r;
    std::vector<float> lg((size_t)B * n_langs);
    MW_CUDA_CHECK(cudaMemcpy2DAsync(lg.data(), (size_t)n_langs * 4, s->logits + first_lang, (size_t)c.vocab * 4,
                                    (size_t)n_langs * 4, B, cudaMemcpyDeviceToHost, st));
    MW_CUDA_CHECK(cudaStreamSynchronize(st));
    for (int b = 0; b < B; ++b) {
        float mx = -INFINITY;
        for (int i = 0; i < n_langs; ++i) mx = std::max(mx, lg[(size_t)b * n_langs + i]);
        double sum = 0.0;
        for (int i = 0; i < n_langs; ++i) sum += exp((double)lg[(size_t)b * n_langs + i] - mx);
        for (int i = 0; i < n_langs; ++i) h_probs[(size_t)b * n_langs + i] = (float)(exp((double)lg[(size_t)b * n_langs + i] - mx) / sum);
    }
    return MW_OK;
}

// ---- measurement hook (bench.py "roofline"): times one hot decode kernel in isolation with CUDA events on the
// caller's stream, cycling through the layers so consecutive launches never re-read L2-resident data.
//   which = 0 : cross-attention decode kernel, R = B rows        (bytes/launch = B*T*2d*2)
//   which = 1 : skinny GEMM on the fc1 weights, R = B rows       (bytes/launch = ffn*d*2)
//   which = 2 : skinny GEMM on the self-attention out-proj       (bytes/launch = d*d*2)
extern "C" mw_status mw_bench_kernel(mw_model* m, int which, int B, int iters, float* h_ms_avg, void* stream) {
    MW_REQUIRE(m && h_ms_avg && iters > 0, "mw_bench_kernel: bad argument");
    const mw_model_config& c = m->cfg;
    DecoderState* s = m->dec;
    MW_REQUIRE(B > 0 && B <= c.max_batch * (which == 0 ? 1 : c.max_beam), "mw_bench_kernel: B outside 1..max_batch (x max_beam for the GEMMs)");
    mw::DeviceGuard guard(c.device);
    cudaStream_t st = (cudaStream_t)stream;
    const int d = c.d_model, T = c.n_audio_ctx;
    cudaEvent_t e0, e1;
    MW_CUDA_CHECK(cudaEventCreate(&e0));
    MW_CUDA_CHECK(cudaEventCreate(&e1));
    auto one = [&](int l) -> mw_status {
        if (which == 0) {
            mw_h* kv = s->kv_cross + (int64_t)l * c.max_batch * T * 2 * d;
            dim3 grid(c.n_heads, B);
            cross_attn_stream_kernel<4><<<grid, 128, 0, st>>>(s->qx, d, kv, kv + d, 2 * d, T, s->att, d, nullptr, 0);
            MW_LAUNCH_CHECK();
            return MW_OK;
        }
        if (which == 1)
            return skinny_gemm(s->ln, d, m->dlw(l, MW_DL_W1), d, (const float*)m->dlw(l, MW_DL_B1), nullptr, s->mlp, c.ffn, B,
                               c.ffn, d, SK_FLAG_GELU, st);
        return skinny_gemm(s->att, d, m->dlw(l, MW_DL_WO), d, (const float*)m->dlw(l, MW_DL_BO), nullptr, s->qx, d, B, d, d, 0, st);
    };
    mw_status r;
    for (int i = 0; i < 3; ++i) if ((r = one(i % c.dec_layers)) != MW_OK) return r;
    MW_CUDA_CHECK(cudaEventRecord(e0, st));
    for (int i = 0; i < iters; ++i) if ((r = one(i % c.dec_layers)) != MW_OK) return r;
    MW_CUDA_CHECK(cudaEventRecord(e1, st));
    MW_CUDA_CHECK(cudaEventSynchronize(e1));
    float ms = 0.f;
    MW_CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *h_ms_avg = ms / iters;
    return MW_OK;
}

// ---- measurement hook: average ms of one decode step restricted to the kernel classes in `parts`
// (1 embed, 2 LayerNorm, 4 skinny GEMMs, 8 self-attention, 16 cross-attention, 32 logits GEMM), replayed as a CUDA graph.
extern "C" mw_status mw_bench_step(mw_model* m, int B, int parts, int iters, float* h_ms_avg, void* stream) {
    MW_REQUIRE(m && h_ms_avg && iters > 0, "mw_bench_step: bad argument");
    const mw_model_config& c = m->cfg;
    DecoderState* s = m->dec;
    MW_REQUIRE(B > 0 && B <= c.max_batch, "mw_bench_step: B outside 1..max_batch");
    mw::DeviceGuard guard(c.device);
    cudaStream_t st = (cudaStream_t)stream;
    MW_CUDA_CHECK(cudaMemsetAsync(s->ctl, 0, sizeof(DecCtl), st));
    MW_CUDA_CHECK(cudaMemsetAsync(s->cur_tok, 0, B * 4, st));
    cudaGraphExec_t g = nullptr;
    int n_nodes = 0;
    mw_status r = capture_graph(s, &g, &n_nodes, [&](cudaStream_t cs) -> mw_status {
        mw_status q = enqueue_layers(m, B, 1, 0, cs, parts);
        if (q != MW_OK) return q;
        if ((parts & PART_LOGITS) && (q = enqueue_logits(m, B, cs)) != MW_OK) return q;
        return MW_OK;
    });
    if (r != MW_OK) return r;
    cudaEvent_t e0, e1;
    MW_CUDA_CHECK(cudaEventCreate(&e0));
    MW_CUDA_CHECK(cudaEventCreate(&e1));
    for (int i = 0; i < 2; ++i) MW_CUDA_CHECK(cudaGraphLaunch(g, st));
    MW_CUDA_CHECK(cudaEventRecord(e0, st));
    for (int i = 0; i < iters; ++i) MW_CUDA_CHECK(cudaGraphLaunch(g, st));
    count_launch((iters + 2) * n_nodes);
    MW_CUDA_CHECK(cudaEventRecord(e1, st));
    MW_CUDA_CHECK(cudaEventSynchronize(e1));
    float ms = 0.f;
    MW_CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaGraphExecDestroy(g);
    *h_ms_avg = ms / iters;
    return MW_OK;
}

// ---- measurement hook (bench.py "in_step" attribution): keep only the kernel classes in `parts` (mask of mw_bench_step) in
// the decode-step graphs captured from now on, process-wide; 127 restores the real step.  Decoded ids are meaningless while a
// class is missing: the difference in step time with and without a class is its in-step cost under real concurrency.
extern "C" mw_status mw_set_solo(mw_model* m, int solo) {
    MW_REQUIRE(m && m->dec, "mw_set_solo: null model");
    m->dec->solo = solo != 0;          // step graphs are cached per mode (ensure_graphs)
    return MW_OK;
}

extern "C" void mw_debug_step_parts(int parts) {
    mw::g_step_parts.store(parts);
    mw::g_step_parts_epoch.fetch_add(1);
}

// ---- test entry points (include/mw_b200.h): the decode step's kernels on caller buffers, the launch path named by an argument.
// Shapes and the path are checked before any pointer, and all of it before anything is launched, so a rejected call touches
// no memory.
extern "C" mw_status mw_step_projection_h16(const void* d_x_h16, const float* d_x_f32, const float* d_gamma, const float* d_beta,
                                            const void* d_w, const float* d_bias, const float* d_resid, void* d_out, int R, int N,
                                            int K, int flags, int path, void* stream) {
    MW_REQUIRE(R >= 1 && R <= 65535 * 32 && N >= 1 && K >= 32 && K % 32 == 0,
               "mw_step_projection_h16: R=%d N=%d K=%d (K a multiple of 32)", R, N, K);
    MW_REQUIRE(flags >= 0 && flags <= 3, "mw_step_projection_h16: flags=%d (1 = GELU, 2 = fp32 out)", flags);
    MW_REQUIRE(path >= MW_STEP_PATH_GREEDY && path <= MW_STEP_PATH_LN_SEPARATE, "mw_step_projection_h16: unknown path %d", path);
    const bool ln = d_gamma || d_beta;
    const bool ln_path = path == MW_STEP_PATH_LN_FUSED || path == MW_STEP_PATH_LN_SEPARATE;
    const bool forced = path >= MW_STEP_PATH_ROWS16_WT1 && !ln_path;
    MW_REQUIRE(ln || !ln_path, "mw_step_projection_h16: path %d is a LayerNorm path: gamma and beta are required", path);
    MW_REQUIRE(!ln || !forced, "mw_step_projection_h16: path %d forces one projection kernel on x_h16: no LayerNorm", path);
    MW_REQUIRE(!ln || !d_resid, "mw_step_projection_h16: a LayerNorm projection takes no residual");
    MW_REQUIRE(!ln || (K % 128 == 0 && K <= 2048), "mw_step_projection_h16: LayerNorm over K=%d (a multiple of 128 up to 2048)", K);
    // LN_SEPARATE is the beam routing, whose LayerNorm is never fused
    const SkKernel kernel_of_path[] = {SK_ROUTE, SK_ROUTE, SK_ROUTE, SK_ROUTE, SK_ROWS16_WT1, SK_ROWS16_WT2, SK_KHALF_WT1,
                                       SK_KHALF_WT2, SK_GENERIC, SK_LN_FUSED, SK_ROUTE};
    const SkKernel p = kernel_of_path[path];
    const bool allow_dg = path == MW_STEP_PATH_GREEDY || path == MW_STEP_PATH_GREEDY_SOLO;
    const bool solo = path == MW_STEP_PATH_GREEDY_SOLO || path == MW_STEP_PATH_BEAM_SOLO;
    if (sk_choose(K, K, R, N, K, flags, p, allow_dg, solo, ln) == SK_NONE) return sk_missing("mw_step_projection_h16", p, K);
    MW_REQUIRE(d_x_h16 && d_w && d_out && (!ln || (d_x_f32 && d_gamma && d_beta)), "mw_step_projection_h16: null pointer");
    MW_REQUIRE((uintptr_t)d_x_h16 % 16 == 0 && (uintptr_t)d_w % 16 == 0 && (uintptr_t)d_x_f32 % 16 == 0,
               "mw_step_projection_h16: x and W must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    if (ln)
        return skinny_gemm_ln(d_x_f32, d_gamma, d_beta, const_cast<void*>(d_x_h16), d_w, d_bias, d_out, N, R, N, K, flags, st,
                              allow_dg, nullptr, 0, solo, p);
    return skinny_gemm(d_x_h16, K, d_w, K, d_bias, d_resid, d_out, N, R, N, K, flags, st, allow_dg, nullptr, 0, solo, p);
}

extern "C" mw_status mw_step_self_attention_h16(const void* d_qkv, void* d_k_cache, void* d_v_cache, const int32_t* d_idx, int R,
                                                int n_heads, int ctx, int pos, void* d_out, void* stream) {
    MW_REQUIRE(R >= 1 && R <= 65535 && n_heads >= 1 && n_heads <= 65535 && ctx >= 1 && ctx <= 12 * 1024 && pos >= 0 && pos < ctx,
               "mw_step_self_attention_h16: R=%d n_heads=%d ctx=%d pos=%d", R, n_heads, ctx, pos);
    MW_REQUIRE(d_qkv && d_k_cache && d_v_cache && d_out, "mw_step_self_attention_h16: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const int d = n_heads * 64;
    const mw_h* qkv = (const mw_h*)d_qkv;
    DecCtl h_ctl = {pos, 0, 0, 0};
    DecCtl* ctl = nullptr;
    MW_CUDA_CHECK(cudaMalloc((void**)&ctl, sizeof(DecCtl)));
    cudaError_t e = cudaMemcpyAsync(ctl, &h_ctl, sizeof(DecCtl), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) {
        decode_attn_kernel<true><<<dim3(n_heads, R), 128, ctx * sizeof(float), st>>>(qkv, 3 * d, (mw_h*)d_k_cache, (mw_h*)d_v_cache, d, ctx,
                                                                                     (const int*)d_idx, ctx, ctl, 0, 1, qkv + d, qkv + 2 * d,
                                                                                     3 * d, (mw_h*)d_out, d, 0);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) { count_launch(); e = cudaStreamSynchronize(st); }      // h_ctl is read by the copy until then
    cudaFree(ctl);
    if (e != cudaSuccess) { set_error("mw_step_self_attention_h16: %s", cudaGetErrorString(e)); return MW_ERR_CUDA; }
    return MW_OK;
}

extern "C" mw_status mw_step_prefill_attention_h16(const void* d_qkv, int B, int P, int n_heads, void* d_out, void* stream) {
    MW_REQUIRE(B >= 1 && P >= 1 && P <= 16 * 1024 && (int64_t)B * P <= 65535 && n_heads >= 1,
               "mw_step_prefill_attention_h16: B=%d P=%d n_heads=%d", B, P, n_heads);
    MW_REQUIRE(d_qkv && d_out, "mw_step_prefill_attention_h16: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    static PerDeviceOnce attr_once;
    MW_CUDA_CHECK(attr_once.run([] { return cudaFuncSetAttribute(decode_attn_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024); }));
    const int d = n_heads * 64;
    mw_h* qkv = (mw_h*)const_cast<void*>(d_qkv);       // read only: the kernel writes the cache only when SELF
    decode_attn_kernel<false><<<dim3(n_heads, B * P), 128, P * sizeof(float), st>>>(qkv, 3 * d, qkv + d, qkv + 2 * d, 3 * d, P, nullptr,
                                                                                   0, nullptr, P, P, nullptr, nullptr, 0, (mw_h*)d_out, d, P);
    MW_LAUNCH_CHECK();
    return MW_OK;
}

extern "C" mw_status mw_step_cross_attention_h16(const void* d_q, const void* d_kv, int B, int G, int T, int n_heads, int unr,
                                                 void* d_out, void* stream) {
    MW_REQUIRE(B >= 1 && B <= 65535 && T >= 1 && n_heads >= 1 && n_heads <= 65535,
               "mw_step_cross_attention_h16: B=%d T=%d n_heads=%d", B, T, n_heads);
    MW_REQUIRE(G >= 1 && G <= MAX_BEAM, "mw_step_cross_attention_h16: G=%d outside 1..%d", G, MAX_BEAM);
    MW_REQUIRE(G > 1 || unr == 4 || unr == 8, "mw_step_cross_attention_h16: unr=%d (4 or 8)", unr);
    MW_REQUIRE(d_q && d_kv && d_out, "mw_step_cross_attention_h16: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const int d = n_heads * 64;
    const mw_h* q = (const mw_h*)d_q;
    const mw_h* kv = (const mw_h*)d_kv;
    mw_h* out = (mw_h*)d_out;
    if (G == 1) {
        if (unr == 8) cross_attn_stream_kernel<8><<<dim3(n_heads, B), 128, 0, st>>>(q, d, kv, kv + d, 2 * d, T, out, d, nullptr, 0);
        else cross_attn_stream_kernel<4><<<dim3(n_heads, B), 128, 0, st>>>(q, d, kv, kv + d, 2 * d, T, out, d, nullptr, 0);
        MW_LAUNCH_CHECK();
        return MW_OK;
    }
#define MW_XG(g) case g: return launch_cross_grouped<g>(q, d, kv, kv + d, 2 * d, T, out, d, n_heads, B, st)
    switch (G) { MW_XG(2); MW_XG(3); MW_XG(4); MW_XG(5); MW_XG(6); MW_XG(7); default: MW_XG(8); }
#undef MW_XG
}
