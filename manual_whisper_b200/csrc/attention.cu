// Encoder self-attention (non-causal, d_head = 64) as a flash-style kernel on tcgen05 tensor cores.
// Replaces CTranslate2's batched-cuBLAS + softmax attention inside ctranslate2.models.Whisper.encode
// (SURVEY.md §8 a6, A.7).
//
// One CTA = one (batch, head, 128-query tile); 128 threads, thread i owns query row i.
//   S = Q K_j^T        tcgen05.mma 128x64x64   (Q, K_j: TMA, K-major SWIZZLE_128B)        -> TMEM cols [0,64)
//   softmax            thread reads its S row (64 fp32) with tcgen05.ld, max / exp2 in registers, writes the
//                      un-normalised P (16-bit) into 128B-swizzled shared memory (A operand of the next MMA)
//   O += P V_j         tcgen05.mma 128x64x64   (V_j: TMA tile [keys, d] used MN-major)      -> TMEM cols [64,128)
// Round 2: O is ACCUMULATED IN TMEM across key blocks instead of being read back and rescaled in registers every block.  The
// exponent reference of a row is only moved - and its O row rescaled through tcgen05.ld/st - when a block's maximum exceeds it
// by more than 2^8 ("lazy rescale": after the first blocks it practically never happens; P <= 256 fits 16-bit storage with the
// same relative rounding).
// The kernel is bound by per-warp instruction latency (time ~ 1 / resident CTAs: 1843 / 1044 / 796 us at 1 / 2 / 3 CTAs per
// SM; removing every exponential changes nothing - profiles/ncu_attention_r2.txt), so everything is arranged for FOUR CTAs per
// SM, the most 128 TMEM columns each allow: one K and one V buffer (48 KB of shared memory; K_{j+1} is requested as soon as
// S_j is complete, V_j as soon as P V_{j-1} is), P leaves for shared memory 8 columns at a time (124 registers, no spill), and
// the exponent arguments and row sums run as packed fp32 pairs (FFMA2 / FADD2).  796 -> 588 us at the large-v3 shape
// (627 TFLOP/s; cuDNN SDPA: 797), bit-identical output.
#include "gemm.cuh"
#include "ptx_sm100.cuh"

namespace mw {
using namespace ptx;

namespace {

constexpr int TQ = 128;   // queries per CTA
constexpr int TK = 64;    // keys per block
constexpr int DH = 64;
constexpr int Q_BYTES = TQ * DH * 2;       // 16 KB
constexpr int KV_BYTES = TK * DH * 2;      // 8 KB
constexpr int P_BYTES = TQ * TK * 2;       // 16 KB: 128 rows x 128 bytes (one swizzle row per query)
constexpr int ATT_SMEM = Q_BYTES + 2 * KV_BYTES + P_BYTES + 128 + 1024;   // one K and one V buffer; + barriers + alignment slack
constexpr float RESCALE_LOG2 = 8.0f;       // a row's exponent reference moves only when a block maximum exceeds it by 2^8
constexpr int ATT_TMEM_COLS = 128;         // S: cols [0,64)   O: cols [64,128)

__device__ __forceinline__ float ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__global__ void __launch_bounds__(128, 4)
attention_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_kv,
                         mw_h* __restrict__ out, int Tq, int Tk_max, int colq0, int colk0, int colv0, int out_ld,
                         float scale_log2e, const int* __restrict__ kv_lens) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    unsigned char* sQ = smem;
    unsigned char* sK = smem + Q_BYTES;                 // one K buffer
    unsigned char* sV = sK + KV_BYTES;                  // one V buffer
    unsigned char* sP = sV + KV_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(sP + P_BYTES);
    uint64_t* bar_q = bars;
    uint64_t* bar_k = bars + 1;
    uint64_t* bar_v = bars + 2;
    uint64_t* bar_s = bars + 3;
    uint64_t* bar_o = bars + 4;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 5);

    const int tid = threadIdx.x, warp = tid >> 5;
    const int q0 = blockIdx.x * TQ;
    const int h = blockIdx.y, b = blockIdx.z;
    // ragged self-attention (forced-alignment windows of different lengths): keys >= kv_lens[b] are masked exactly like the
    // tail of the last key block, and query tiles that lie wholly in the padding are skipped
    const int Tk = kv_lens ? min(Tk_max, max(__ldg(kv_lens + b), 1)) : Tk_max;
    if (kv_lens && q0 >= Tk) return;
    const int n_blocks = (Tk + TK - 1) / TK;
    const int col_q = colq0 + h * DH, col_k = colk0 + h * DH, col_v = colv0 + h * DH;

    if (tid == 0) {
        prefetch_tensormap(&tmap_q);
        prefetch_tensormap(&tmap_kv);
        for (int i = 0; i < 5; ++i) mbar_init(&bars[i], 1);
        fence_barrier_init();
        fence_proxy_async();
    }
    if (warp == 0) {
        tmem_alloc(tmem_slot, ATT_TMEM_COLS);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t tmem_s = tmem_base;
    const uint32_t tmem_o = tmem_base + 64;
    const uint32_t lane_off = (uint32_t)(warp * 32) << 16;

    constexpr uint32_t idesc_s = make_idesc_h16(128, TK, 0);
    constexpr uint32_t idesc_o = make_idesc_h16(128, DH, 1);   // B (=V) is MN-major

    auto issue_s = [&](int j) {        // thread 0: S = Q K_j^T into TMEM cols [0,64)
        mbar_wait(bar_k, j & 1);
        tc_fence_after();
        const uint64_t dq = make_desc_sw128(smem_u32(sQ), 1024, 0);
        const uint64_t dk = make_desc_sw128(smem_u32(sK), 1024, 0);
#pragma unroll
        for (int k = 0; k < DH / 16; ++k) umma_h16(tmem_s, dq + 2 * k, dk + 2 * k, idesc_s, k ? 1u : 0u);
        umma_commit(bar_s);
    };

    if (tid == 0) {
        mbar_arrive_expect_tx(bar_q, Q_BYTES);
        tma_load_3d(sQ, &tmap_q, bar_q, col_q, q0, b);
        mbar_arrive_expect_tx(bar_k, KV_BYTES);
        tma_load_3d(sK, &tmap_kv, bar_k, col_k, 0, b);
        mbar_arrive_expect_tx(bar_v, KV_BYTES);
        tma_load_3d(sV, &tmap_kv, bar_v, col_v, 0, b);
        mbar_wait(bar_q, 0);
        issue_s(0);
    }
    __syncwarp();

    float m_used = -INFINITY, l_run = 0.0f;       // exponent reference of this row (raw score units), running sum of P
    const uint32_t prow = smem_u32(sP) + tid * 128;

    for (int j = 0; j < n_blocks; ++j) {
        mbar_wait(bar_s, j & 1);                  // S_j is in TMEM, so the K buffer is free
        tc_fence_after();
        if (tid == 0 && j + 1 < n_blocks) {
            mbar_arrive_expect_tx(bar_k, KV_BYTES);
            tma_load_3d(sK, &tmap_kv, bar_k, col_k, (j + 1) * TK, b);
        }
        __syncwarp();
        uint32_t r0[32], r1[32];
        tmem_ld32(tmem_s + lane_off, r0);
        tmem_ld32(tmem_s + lane_off + 32, r1);
        tmem_ld_wait();
        if (j > 0) {
            mbar_wait(bar_o, (j - 1) & 1);        // P V_{j-1} is done: O holds blocks 0..j-1, sP and the V buffer are free
            tc_fence_after();
            if (tid == 0) {
                mbar_arrive_expect_tx(bar_v, KV_BYTES);
                tma_load_3d(sV, &tmap_kv, bar_v, col_v, j * TK, b);
            }
            __syncwarp();
        }

        const int n_valid = min(TK, Tk - j * TK);    // >= 1
        if (n_valid < TK) {       // last, partial block only: masked keys contribute exp2(-inf) = 0
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                if (i >= n_valid) r0[i] = 0xff800000u;
                if (32 + i >= n_valid) r1[i] = 0xff800000u;
            }
        }
        float mx0 = -INFINITY, mx1 = -INFINITY, mx2 = -INFINITY, mx3 = -INFINITY;   // four chains for ILP
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
            mx0 = fmaxf(mx0, __uint_as_float(r0[i]));
            mx1 = fmaxf(mx1, __uint_as_float(r0[i + 1]));
            mx2 = fmaxf(mx2, __uint_as_float(r1[i]));
            mx3 = fmaxf(mx3, __uint_as_float(r1[i + 1]));
        }
        const float mx = fmaxf(fmaxf(mx0, mx1), fmaxf(mx2, mx3));
        // lazy rescale, decided per warp (tcgen05.ld/st are warp-wide): move the exponent reference only when some row of
        // the warp would otherwise produce P > 2^8
        const bool need = __any_sync(0xffffffffu, (mx - m_used) * scale_log2e > RESCALE_LOG2);
        if (need) {
            const float m_new = fmaxf(m_used, mx);
            const float alpha = ex2((m_used - m_new) * scale_log2e);       // m_used = -inf on the first block -> 0
            l_run *= alpha;
            m_used = m_new;
            if (j > 0) {
#pragma unroll
                for (int q8 = 0; q8 < 8; ++q8) {
                    uint32_t o0[8];
                    tmem_ld8(tmem_o + lane_off + q8 * 8, o0);
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < 8; ++i) o0[i] = __float_as_uint(__uint_as_float(o0[i]) * alpha);
                    tmem_st8(tmem_o + lane_off + q8 * 8, o0);
                }
                tmem_st_wait();
            }
        }
        const float mb = m_used * scale_log2e;
        // exponent arguments and the four partial row sums as packed fp32 pairs (FFMA2 / FADD2: the same bits as the scalar
        // form at half the issue slots - this kernel is bound by per-warp instruction latency, profiles/ncu_attention_r2.txt);
        // P leaves for shared memory 8 columns at a time so that only four packed words are live
        const uint64_t sc2 = pack2(scale_log2e, scale_log2e), nmb2 = pack2(-mb, -mb);
        uint64_t ls01 = pack2(0.0f, 0.0f), ls23 = pack2(0.0f, 0.0f);
#pragma unroll
        for (int g = 0; g < 8; ++g) {
            uint32_t packed[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int i = (g & 3) * 8 + 2 * e;
                float t0, t1;
                unpack2(fma2(pack2(__uint_as_float(g < 4 ? r0[i] : r1[i]), __uint_as_float(g < 4 ? r0[i + 1] : r1[i + 1])), sc2, nmb2), t0, t1);
                const float p0 = ex2(t0), p1 = ex2(t1);
                if (i & 2) ls23 = add2(ls23, pack2(p0, p1)); else ls01 = add2(ls01, pack2(p0, p1));
                mw_h2 hh = f2h2_bounded(p0, p1);      // p <= 2^8
                packed[e] = *reinterpret_cast<uint32_t*>(&hh);
            }
            const int chunk = g ^ (tid & 7);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(prow + chunk * 16), "r"(packed[0]), "r"(packed[1]), "r"(packed[2]),
                         "r"(packed[3]) : "memory");
        }
        float ls0, ls1, ls2, ls3;
        unpack2(ls01, ls0, ls1);
        unpack2(ls23, ls2, ls3);
        l_run += (ls0 + ls1) + (ls2 + ls3);
        fence_proxy_async();      // generic-proxy smem writes -> visible to the tensor core's async proxy
        tc_fence_before();
        __syncthreads();          // P complete, rescaled O rows stored, every thread holds its S_j row
        if (tid == 0) {
            if (j + 1 < n_blocks) issue_s(j + 1);
            mbar_wait(bar_v, j & 1);
            tc_fence_after();
#pragma unroll
            for (int k = 0; k < TK / 16; ++k) {
                const uint64_t dp = make_desc_sw128(smem_u32(sP) + k * 32, 1024, 0);
                const uint64_t dv = make_desc_sw128(smem_u32(sV) + k * 2048, 1024, KV_BYTES);
                umma_h16(tmem_o, dp, dv, idesc_o, (j | k) ? 1u : 0u);
            }
            umma_commit(bar_o);
        }
        __syncwarp();
    }

    mbar_wait(bar_o, (n_blocks - 1) & 1);
    tc_fence_after();
    const int q = q0 + tid;
    {
        uint32_t r0[32], r1[32];
        tmem_ld32(tmem_o + lane_off, r0);
        tmem_ld32(tmem_o + lane_off + 32, r1);
        tmem_ld_wait();
        if (q < Tq) {
            const float inv = 1.0f / l_run;
            uint4* o4 = reinterpret_cast<uint4*>(out + ((int64_t)b * Tq + q) * out_ld + h * DH);
#pragma unroll
            for (int g = 0; g < 8; ++g) {
                uint32_t w[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int c = 8 * g + 2 * i;
                    const float a0 = __uint_as_float(c < 32 ? r0[c] : r1[c - 32]) * inv;
                    const float a1 = __uint_as_float(c + 1 < 32 ? r0[c + 1] : r1[c + 1 - 32]) * inv;
                    mw_h2 hh = f2h2_bounded(a0, a1);      // convex combination of V rows
                    w[i] = *reinterpret_cast<uint32_t*>(&hh);
                }
                o4[g] = make_uint4(w[0], w[1], w[2], w[3]);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem_base, ATT_TMEM_COLS);
    }
}

}  // namespace

// General form: queries [B, Tq, ldq] (head h at column colq0 + 64 h) attend to keys/values [B, Tk, ldkv] (columns
// colk0 + 64 h / colv0 + 64 h); out [B*Tq, out_ld].  The encoder's self-attention and the decoder's batched-prefill
// cross-attention are both instances.
mw_status attention_launch_general(const void* d_q, int64_t ldq, int colq0, const void* d_kv, int64_t ldkv, int colk0, int colv0,
                                   void* d_out, int out_ld, int B, int Tq, int Tk, int n_heads, cudaStream_t st,
                                   const int* d_kv_lens) {
    MW_REQUIRE(d_q && d_kv && d_out && B > 0 && Tq > 0 && Tk > 0 && n_heads > 0, "attention: bad arguments");
    CUtensorMap tm_q, tm_kv;
    {
        uint64_t dims[3] = {(uint64_t)ldq, (uint64_t)Tq, (uint64_t)B};
        uint64_t str[2] = {(uint64_t)ldq * 2, (uint64_t)Tq * ldq * 2};
        uint32_t box[3] = {DH, TQ, 1};
        mw_status s = encode_tensor_map(&tm_q, d_q, 3, dims, str, box, true);
        if (s != MW_OK) return s;
    }
    {
        uint64_t dims[3] = {(uint64_t)ldkv, (uint64_t)Tk, (uint64_t)B};
        uint64_t str[2] = {(uint64_t)ldkv * 2, (uint64_t)Tk * ldkv * 2};
        uint32_t box[3] = {DH, TK, 1};
        mw_status s = encode_tensor_map(&tm_kv, d_kv, 3, dims, str, box, true);
        if (s != MW_OK) return s;
    }
    static PerDeviceOnce attr_once;
    MW_CUDA_CHECK(attr_once.run([&] { return cudaFuncSetAttribute(attention_tcgen05_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ATT_SMEM); }));
    dim3 grid(ceil_div(Tq, TQ), n_heads, B);
    const float scale_log2e = 0.125f * 1.4426950408889634f;   // d_head^-0.5 * log2(e)
    attention_tcgen05_kernel<<<grid, 128, ATT_SMEM, st>>>(tm_q, tm_kv, (mw_h*)d_out, Tq, Tk, colq0, colk0, colv0, out_ld,
                                                          scale_log2e, d_kv_lens);
    MW_LAUNCH_CHECK();
    return MW_OK;
}

mw_status attention_launch(const void* d_qkv, void* d_out, int B, int T, int n_heads, cudaStream_t st, const int* d_lens) {
    const int d = n_heads * DH;
    return attention_launch_general(d_qkv, 3 * d, 0, d_qkv, 3 * d, d, 2 * d, d_out, d, B, T, T, n_heads, st, d_lens);
}

}  // namespace mw

extern "C" mw_status mw_attention_h16(const void* d_qkv, void* d_out, int B, int T, int n_heads, void* stream) {
    return mw::attention_launch(d_qkv, d_out, B, T, n_heads, (cudaStream_t)stream, nullptr);
}

extern "C" mw_status mw_attention_general_h16(const void* d_q, int64_t ldq, int colq0, const void* d_kv, int64_t ldkv, int colk0,
                                               int colv0, void* d_out, int out_ld, int B, int Tq, int Tk, int n_heads,
                                               const int32_t* d_kv_lens, void* stream) {
    // shapes and column ranges first, then the pointers: a rejected call touches no memory
    MW_REQUIRE(B > 0 && Tq > 0 && Tk > 0 && n_heads > 0, "mw_attention_general_h16: bad shape B=%d Tq=%d Tk=%d n_heads=%d",
               B, Tq, Tk, n_heads);
    const int64_t w = (int64_t)mw::DH * n_heads;
    MW_REQUIRE(ldq % 8 == 0 && ldkv % 8 == 0 && out_ld % 8 == 0 && colq0 % 8 == 0 && colk0 % 8 == 0 && colv0 % 8 == 0,
               "mw_attention_general_h16: leading dimensions and column offsets must be multiples of 8");
    MW_REQUIRE(colq0 >= 0 && colq0 + w <= ldq && colk0 >= 0 && colk0 + w <= ldkv && colv0 >= 0 && colv0 + w <= ldkv && w <= out_ld,
               "mw_attention_general_h16: %d heads do not fit: colq0=%d ldq=%lld colk0=%d colv0=%d ldkv=%lld out_ld=%d", n_heads,
               colq0, (long long)ldq, colk0, colv0, (long long)ldkv, out_ld);
    MW_REQUIRE(!d_kv_lens || Tq == Tk, "mw_attention_general_h16: kv_lens needs Tq == Tk (Tq=%d Tk=%d)", Tq, Tk);
    MW_REQUIRE(d_q && d_kv && d_out, "mw_attention_general_h16: null pointer");
    return mw::attention_launch_general(d_q, ldq, colq0, d_kv, ldkv, colk0, colv0, d_out, out_ld, B, Tq, Tk, n_heads,
                                        (cudaStream_t)stream, d_kv_lens);
}
