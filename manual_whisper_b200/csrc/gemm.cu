// Persistent warp-specialised bf16 GEMM on the 5th-gen tensor cores (tcgen05.mma, accumulators in TMEM,
// operands staged by TMA into 128B-swizzled shared memory).  It is the engine behind every large
// matrix product of the encoder (SURVEY.md §8 a6: conv stem as implicit GEMM, QKV / out / MLP
// projections) and the cross-attention K/V projection (a8), replacing CTranslate2's cuBLAS/cuDNN calls.
//
//   warp 0      : TMA producer   (one lane)      smem ring: full[s] / empty[s]
//   warp 1      : MMA issuer     (one lane) + TMEM allocator
//   warps 2..9  : epilogue       TMEM -> registers -> bias / GELU / residual -> global
//                                two TMEM accumulator buffers: tmem_full[2] / tmem_empty[2]
//
// Tile = 128 x BLOCK_N x 64; one tcgen05.mma is 128 x BLOCK_N x 16.  Tiles are walked n-fastest so the
// CTAs resident at one time share A rows and all of W through L2.
#include "gemm.cuh"
#include "ptx_sm100.cuh"

#include <mutex>

namespace mw {

using namespace ptx;

namespace {

#ifdef MW_STORAGE_BF16
constexpr CUtensorMapDataType MW_TMA_DTYPE = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
#else
constexpr CUtensorMapDataType MW_TMA_DTYPE = CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
#endif
constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;
constexpr int NUM_EPI_WARPS = 8;
constexpr int NUM_THREADS = 32 * (2 + NUM_EPI_WARPS);

struct GemmParams {
    int batch, M, N, K;
    const float* bias;
    const float* residual;
    int64_t res_batch_rows, ld_res;
    void* out;
    int64_t out_batch_rows, out_row_off, ld_out;
    int gelu, out_f32;
};

template <int BLOCK_N, int STAGES>
struct SmemLayout {
    static constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;
    static constexpr int B_BYTES = BLOCK_N * BLOCK_K * 2;
    static constexpr int BAR_OFF = STAGES * (A_BYTES + B_BYTES);
    static constexpr int TOTAL = BAR_OFF + (2 * STAGES + 4) * 8 + 16 + 1024;  // +1024: manual alignment slack
};

#ifndef MW_GEMM_MINBLOCKS
#define MW_GEMM_MINBLOCKS 1
#endif
#ifndef MW_GEMM_STAGES256
#define MW_GEMM_STAGES256 4
#endif
template <int BLOCK_N, int STAGES>
__global__ void __launch_bounds__(NUM_THREADS, MW_GEMM_MINBLOCKS)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_w,
                    const GemmParams p) {
    using L = SmemLayout<BLOCK_N, STAGES>;
    extern __shared__ unsigned char smem_raw[];
    // SWIZZLE_128B operands need 1024-byte aligned stage buffers
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    unsigned char* smem_a = smem;
    unsigned char* smem_b = smem + STAGES * L::A_BYTES;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tmem_full = empty_bar + STAGES;
    uint64_t* tmem_empty = tmem_full + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int tiles_m = (p.M + BLOCK_M - 1) / BLOCK_M;
    const int tiles_n = (p.N + BLOCK_N - 1) / BLOCK_N;
    const int num_tiles = p.batch * tiles_m * tiles_n;
    const int num_kb = (p.K + BLOCK_K - 1) / BLOCK_K;
    constexpr uint32_t TMEM_COLS = 2 * BLOCK_N;   // 256 or 512: a power of two >= 32

    if (threadIdx.x == 0) {
        prefetch_tensormap(&tmap_a);
        prefetch_tensormap(&tmap_w);
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], NUM_EPI_WARPS); }
        fence_barrier_init();
        fence_proxy_async();
    }
    if (warp == 1) {
        tmem_alloc(tmem_slot, TMEM_COLS);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================= TMA producer =================
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                const int tn = tile % tiles_n;
                const int tm = (tile / tiles_n) % tiles_m;
                const int b = tile / (tiles_n * tiles_m);
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    mbar_arrive_expect_tx(&full_bar[stage], L::A_BYTES + L::B_BYTES);
                    tma_load_3d(smem_a + stage * L::A_BYTES, &tmap_a, &full_bar[stage], kb * BLOCK_K, tm * BLOCK_M, b);
                    tma_load_2d(smem_b + stage * L::B_BYTES, &tmap_w, &full_bar[stage], kb * BLOCK_K, tn * BLOCK_N);
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer =================
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc_h16(BLOCK_M, BLOCK_N);
            int stage = 0; uint32_t phase = 0;
            int acc = 0; uint32_t acc_phase = 0;
            for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
                mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint64_t da = make_desc_sw128(smem_u32(smem_a + stage * L::A_BYTES), 1024, 0);
                    const uint64_t db = make_desc_sw128(smem_u32(smem_b + stage * L::B_BYTES), 1024, 0);
#pragma unroll
                    for (int k = 0; k < BLOCK_K / 16; ++k) {
                        // +32 bytes per 16-element K step inside the 128-byte swizzle row (address field is >>4)
                        umma_h16(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) ? 1u : 0u);
                    }
                    umma_commit(&empty_bar[stage]);          // frees the smem slot when these MMAs retire
                    if (++stage == STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit(&tmem_full[acc]);                // accumulator ready for the epilogue
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        // ================= epilogue =================
        const int we = warp - 2;
        const int q = warp & 3;                 // TMEM lane quadrant this warp may read
        const int half = we >> 2;               // which half of the tile's columns
        constexpr int COLS_PER_WARP = BLOCK_N / 2;
        int acc = 0; uint32_t acc_phase = 0;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
            const int tn = tile % tiles_n;
            const int tm = (tile / tiles_n) % tiles_m;
            const int b = tile / (tiles_n * tiles_m);
            const int m = tm * BLOCK_M + q * 32 + lane;
            const bool row_ok = m < p.M;
            const int64_t out_row = (int64_t)b * p.out_batch_rows + p.out_row_off + m;
            const int64_t res_row = (int64_t)b * p.res_batch_rows + m;
            const int nbase = tn * BLOCK_N + half * COLS_PER_WARP;
            // the residual tile does not depend on the accumulator: fetch the first chunk while the MMAs still run
            float4 res_next[8];
            const bool use_res = p.residual != nullptr && row_ok;
            if (use_res && nbase < p.N) {
                const float4* r4 = reinterpret_cast<const float4*>(p.residual + res_row * p.ld_res + nbase);
#pragma unroll
                for (int j = 0; j < 8; ++j) res_next[j] = r4[j];
            }
            mbar_wait(&tmem_full[acc], acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * BLOCK_N + half * COLS_PER_WARP;
#pragma unroll 1
            for (int c = 0; c < COLS_PER_WARP; c += 32) {
                const int n0 = nbase + c;
                if (n0 >= p.N) break;            // warp-uniform
                uint32_t r[32];
                tmem_ld32(taddr + c, r);
                float4 res_cur[8];
                if (use_res) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) res_cur[j] = res_next[j];
                    if (c + 32 < COLS_PER_WARP && n0 + 32 < p.N) {      // one chunk ahead
                        const float4* r4 = reinterpret_cast<const float4*>(p.residual + res_row * p.ld_res + n0 + 32);
#pragma unroll
                        for (int j = 0; j < 8; ++j) res_next[j] = r4[j];
                    }
                }
                tmem_ld_wait();
                if (row_ok) {
                    float v[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
                    if (p.bias) {
                        const float4* b4 = reinterpret_cast<const float4*>(p.bias + n0);
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float4 bb = __ldg(b4 + j);
                            v[4 * j] += bb.x; v[4 * j + 1] += bb.y; v[4 * j + 2] += bb.z; v[4 * j + 3] += bb.w;
                        }
                    }
                    if (p.gelu) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] = gelu_as7126(v[j]);
                    }
                    if (use_res) {
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            v[4 * j] += res_cur[j].x; v[4 * j + 1] += res_cur[j].y; v[4 * j + 2] += res_cur[j].z; v[4 * j + 3] += res_cur[j].w;
                        }
                    }
                    if (p.out_f32) {
                        float4* o4 = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + out_row * p.ld_out + n0);
#pragma unroll
                        for (int j = 0; j < 8; ++j) o4[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                    } else {
                        uint4* o4 = reinterpret_cast<uint4*>(reinterpret_cast<mw_h*>(p.out) + out_row * p.ld_out + n0);
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            mw_h2 h0 = f2h2(v[8 * j], v[8 * j + 1]);
                            mw_h2 h1 = f2h2(v[8 * j + 2], v[8 * j + 3]);
                            mw_h2 h2 = f2h2(v[8 * j + 4], v[8 * j + 5]);
                            mw_h2 h3 = f2h2(v[8 * j + 6], v[8 * j + 7]);
                            uint4 u;
                            u.x = *reinterpret_cast<uint32_t*>(&h0); u.y = *reinterpret_cast<uint32_t*>(&h1);
                            u.z = *reinterpret_cast<uint32_t*>(&h2); u.w = *reinterpret_cast<uint32_t*>(&h3);
                            o4[j] = u;
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[acc]);
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    });
    return fn;
}

template <int BLOCK_N, int STAGES>
mw_status launch_cfg(const CUtensorMap& ta, const CUtensorMap& tw, const GemmParams& p, cudaStream_t st) {
    using L = SmemLayout<BLOCK_N, STAGES>;
    static PerDeviceOnce attr_once;
    auto kern = gemm_tcgen05_kernel<BLOCK_N, STAGES>;
    MW_CUDA_CHECK(attr_once.run([&] { return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL); }));
    const int tiles = p.batch * ceil_div(p.M, BLOCK_M) * ceil_div(p.N, BLOCK_N);
    const int grid = tiles < device_sm_count() ? tiles : device_sm_count();
    kern<<<grid, NUM_THREADS, L::TOTAL, st>>>(ta, tw, p);
    MW_LAUNCH_CHECK();
    return MW_OK;
}

}  // namespace

int device_sm_count() {
    static std::atomic<int> cache[64] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    int n = cache[dev & 63].load();
    if (!n) {
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (n <= 0) n = 148;
        cache[dev & 63].store(n);
    }
    return n;
}

mw_status encode_tensor_map(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                            const uint64_t* strides_bytes, const uint32_t* box, bool swizzle128) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) { set_error("cuTensorMapEncodeTiled entry point not available"); return MW_ERR_CUDA; }
    cuuint64_t gdim[5]; cuuint64_t gstr[4]; cuuint32_t bx[5]; cuuint32_t es[5];
    for (int i = 0; i < rank; ++i) { gdim[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
    for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i];
    CUresult r = fn(map, MW_TMA_DTYPE, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bx, es,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed (CUresult %d) rank %d dims [%llu,%llu,%llu] stride0 %llu box [%u,%u]",
                  (int)r, rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
                  (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 1 ? strides_bytes[0] : 0),
                  box[0], rank > 1 ? box[1] : 0);
        return MW_ERR_CUDA;
    }
    return MW_OK;
}

mw_status gemm_launch(const GemmArgs& a, cudaStream_t st) {
    MW_REQUIRE(a.a && a.w && a.out, "gemm: null pointer");
    MW_REQUIRE(a.M > 0 && a.N > 0 && a.K > 0 && a.batch > 0, "gemm: bad shape M=%d N=%d K=%d batch=%d", a.M, a.N, a.K, a.batch);
    MW_REQUIRE(a.N % 32 == 0, "gemm: N=%d must be a multiple of 32", a.N);
    MW_REQUIRE(a.K % 8 == 0 && a.a_row_stride % 8 == 0 && a.w_row_stride % 8 == 0 && (a.batch == 1 || a.a_batch_stride % 8 == 0),
               "gemm: K and operand strides must be multiples of 8 elements (TMA 16-byte rule)");
    MW_REQUIRE(a.ld_out % 8 == 0 && (!a.residual || a.ld_res % 4 == 0), "gemm: ld_out/ld_res alignment");
    MW_REQUIRE(((uintptr_t)a.a % 16 == 0) && ((uintptr_t)a.w % 16 == 0) && ((uintptr_t)a.out % 16 == 0), "gemm: pointers must be 16-byte aligned");
    const int block_n = (a.N % 256 == 0 || a.N > 1024) ? 256 : 128;
    CUtensorMap ta, tw;
    {
        uint64_t dims[3] = {(uint64_t)a.K, (uint64_t)a.M, (uint64_t)a.batch};
        uint64_t str[2] = {(uint64_t)a.a_row_stride * 2, (uint64_t)(a.batch > 1 ? a.a_batch_stride : (int64_t)a.a_row_stride * a.M) * 2};
        uint32_t box[3] = {BLOCK_K, BLOCK_M, 1};
        mw_status s = encode_tensor_map(&ta, a.a, 3, dims, str, box, true);
        if (s != MW_OK) return s;
    }
    {
        uint64_t dims[2] = {(uint64_t)a.K, (uint64_t)a.N};
        uint64_t str[1] = {(uint64_t)a.w_row_stride * 2};
        uint32_t box[2] = {BLOCK_K, (uint32_t)block_n};
        mw_status s = encode_tensor_map(&tw, a.w, 2, dims, str, box, true);
        if (s != MW_OK) return s;
    }
    GemmParams p;
    p.batch = a.batch; p.M = a.M; p.N = a.N; p.K = a.K;
    p.bias = a.bias; p.residual = a.residual; p.res_batch_rows = a.res_batch_rows; p.ld_res = a.ld_res;
    p.out = a.out; p.out_batch_rows = a.out_batch_rows; p.out_row_off = a.out_row_off; p.ld_out = a.ld_out;
    p.gelu = a.gelu ? 1 : 0; p.out_f32 = a.out_f32 ? 1 : 0;
    if (block_n == 256) return launch_cfg<256, MW_GEMM_STAGES256>(ta, tw, p, st);
    return launch_cfg<128, 6>(ta, tw, p, st);
}

}  // namespace mw

extern "C" mw_status mw_gemm_h16(const void* d_a, const void* d_w, const float* d_bias, const float* d_residual,
                                  void* d_out, int M, int N, int K, int gelu, int out_f32, void* stream) {
    mw::GemmArgs a;
    a.a = d_a; a.a_row_stride = K; a.a_batch_stride = (int64_t)M * K;
    a.w = d_w; a.w_row_stride = K;
    a.bias = d_bias; a.residual = d_residual; a.res_batch_rows = 0; a.ld_res = N;
    a.out = d_out; a.out_batch_rows = 0; a.out_row_off = 0; a.ld_out = N;
    a.batch = 1; a.M = M; a.N = N; a.K = K; a.gelu = gelu != 0; a.out_f32 = out_f32 != 0;
    return mw::gemm_launch(a, (cudaStream_t)stream);
}

extern "C" mw_status mw_gemm_general_h16(const void* d_a, int64_t a_row_stride, int64_t a_batch_stride, const void* d_w,
                                          int64_t w_row_stride, const float* d_bias, const float* d_resid, int64_t res_batch_rows,
                                          int64_t ld_res, void* d_out, int64_t out_batch_rows, int64_t out_row_off, int64_t ld_out,
                                          int batch, int M, int N, int K, int gelu, int out_f32, void* stream) {
    // shapes and strides first, then the pointers: a rejected call touches no memory
    MW_REQUIRE(batch > 0 && M > 0 && N > 0 && K > 0 && N % 32 == 0 && K % 8 == 0,
               "mw_gemm_general_h16: bad shape batch=%d M=%d N=%d K=%d (N %% 32 == 0, K %% 8 == 0)", batch, M, N, K);
    MW_REQUIRE(a_row_stride > 0 && a_row_stride % 8 == 0 && a_batch_stride >= 0 && a_batch_stride % 8 == 0 &&
               w_row_stride >= K && w_row_stride % 8 == 0,
               "mw_gemm_general_h16: operand strides must be positive multiples of 8 (a_row_stride=%lld a_batch_stride=%lld "
               "w_row_stride=%lld, K=%d)", (long long)a_row_stride, (long long)a_batch_stride, (long long)w_row_stride, K);
    MW_REQUIRE(ld_out >= N && ld_out % 8 == 0 && out_row_off >= 0 && out_batch_rows >= 0 &&
               (batch == 1 || out_batch_rows >= out_row_off + M),
               "mw_gemm_general_h16: bad output geometry ld_out=%lld out_batch_rows=%lld out_row_off=%lld (N=%d M=%d)",
               (long long)ld_out, (long long)out_batch_rows, (long long)out_row_off, N, M);
    MW_REQUIRE(!d_resid || (ld_res >= N && ld_res % 4 == 0 && res_batch_rows >= 0),
               "mw_gemm_general_h16: bad residual geometry ld_res=%lld res_batch_rows=%lld", (long long)ld_res,
               (long long)res_batch_rows);
    MW_REQUIRE(d_a && d_w && d_out, "mw_gemm_general_h16: null pointer");
    MW_REQUIRE((uintptr_t)d_bias % 16 == 0 && (uintptr_t)d_resid % 16 == 0,
               "mw_gemm_general_h16: bias and residual must be 16-byte aligned");
    mw::GemmArgs a;
    a.a = d_a; a.a_row_stride = a_row_stride; a.a_batch_stride = a_batch_stride;
    a.w = d_w; a.w_row_stride = w_row_stride;
    a.bias = d_bias; a.residual = d_resid; a.res_batch_rows = res_batch_rows; a.ld_res = ld_res;
    a.out = d_out; a.out_batch_rows = out_batch_rows; a.out_row_off = out_row_off; a.ld_out = ld_out;
    a.batch = batch; a.M = M; a.N = N; a.K = K; a.gelu = gelu != 0; a.out_f32 = out_f32 != 0;
    return mw::gemm_launch(a, (cudaStream_t)stream);
}
