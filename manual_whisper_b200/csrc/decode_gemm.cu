// Weight-stationary decode-time GEMM on the 5th-gen tensor cores (SURVEY.md §8 a8: the per-step projections of
// ctranslate2.models.Whisper.generate, /root/reference/transcribe.py:123).
//
//   out[r, n] = sum_k X[r, k] W[n, k]  (+bias[n]) (gelu) (+resid[r, n]),   R <= 256 rows, W streamed ONCE for all rows.
//
// "Swap-AB": the 128 weight rows of a tile are the M side of tcgen05.mma (A operand, TMA -> 128B-swizzled smem), the R
// activation rows are the N side (B operand, one TMA box of RB rows), the fp32 accumulator D[128, RB] lives in TMEM.
// A d x d projection has only 10 such tiles, so K is split over the CTAs of a thread-block cluster (cluster dims
// (1, ks, 1)); the partial accumulators are reduce-scattered through distributed shared memory in a fixed order
// (deterministic), each CTA finishing a slice of the rows with the fused bias / GELU / residual epilogue.  The epilogue
// is transposed for free: TMEM lane = weight row n, so for one activation row the 32 lanes of a warp write 32
// consecutive n.
//
//   warp 0: TMA producer (one lane)   warp 1: MMA issuer (one lane) + TMEM allocator   warps 2..5: epilogue
#include "gemm.cuh"
#include "ptx_sm100.cuh"

namespace mw {

using namespace ptx;

namespace {

constexpr int DG_M = 128, DG_K = 64, DG_THREADS = 192;
constexpr int DG_FLAG_GELU = 1, DG_FLAG_F32 = 2;

struct DgParams {
    int R, N, nkb, ks;
    const float* bias;
    const float* resid;
    void* out;
    int64_t ldo;
    int flags;
    unsigned long long* dbg;      // phase timestamps of CTA (0,0) (scripts/gpu_dg_phases.py), normally null
};

__device__ __forceinline__ unsigned long long dg_now() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define DG_STAMP(i) do { if (p.dbg && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 64) p.dbg[i] = dg_now(); } while (0)

// Shared-memory layout for a row block of RB rows (RB = R rounded up to 16, the tcgen05.mma N granularity at M = 128).
//   ring   : STAGES x (W tile 16 KB + X tile RB x 128 B), every stage 1024-byte aligned (RB % 16 == 0 -> X tile % 2048 == 0)
//   reduce : split-K reduce-scatter buffer [src CTA][cpd / 4][128 weight rows] float4 (cpd = rows finished per CTA).  RB <= 128:
//            its own region, so only ONE blocking cluster barrier is needed; larger: it aliases the operand ring (free once
//            every CTA's MMAs have retired, which costs a second barrier).
struct DgLayout {
    int rb, stages, x_bytes, ring, red, bar_off, total;
    bool alias;
};
constexpr int DG_W_BYTES = DG_M * DG_K * 2;
__host__ __device__ constexpr DgLayout dg_layout(int R) {
    DgLayout l{};
    l.rb = (R + 15) & ~15;
    l.stages = 4;
    l.x_bytes = l.rb * DG_K * 2;
    l.ring = l.stages * (DG_W_BYTES + l.x_bytes);
    l.alias = l.rb > 128;
    const int cpd_max = l.rb / 8 > 8 ? ((l.rb / 8 + 7) & ~7) : 8;          // rows per destination CTA at ks = 8
    const int need = 8 * 128 * cpd_max * 4;
    l.red = l.alias ? 0 : need;
    l.bar_off = l.ring + l.red;
    l.total = l.bar_off + (2 * l.stages + 1) * 8 + 16 + 1024;
    return l;
}

__device__ __forceinline__ float dg_finish(const DgParams& p, int64_t oi, float v, float bias) {
    v += bias;
    if (p.flags & DG_FLAG_GELU) v = gelu_as7126(v);
    if (p.resid) v += p.resid[oi];
    return v;
}
__device__ __forceinline__ void dg_store(const DgParams& p, int row, int n, float v, float bias) {
    const int64_t oi = (int64_t)row * p.ldo + n;
    v = dg_finish(p, oi, v, bias);
    if (p.flags & DG_FLAG_F32) reinterpret_cast<float*>(p.out)[oi] = v;
    else reinterpret_cast<mw_h*>(p.out)[oi] = f2h(v);
}
// four consecutive n of one row; the widest store the row's alignment allows (warp-uniform)
__device__ __forceinline__ void dg_store4(const DgParams& p, int row, int n, const float (&acc)[4], const float (&bias)[4]) {
    const int64_t oi = (int64_t)row * p.ldo + n;
    if (n + 3 >= p.N) {
        for (int i = 0; i < 4; ++i) if (n + i < p.N) dg_store(p, row, n + i, acc[i], bias[i]);
        return;
    }
    float v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = dg_finish(p, oi + i, acc[i], bias[i]);
    if (p.flags & DG_FLAG_F32) {
        float* o = reinterpret_cast<float*>(p.out) + oi;
        if ((reinterpret_cast<uintptr_t>(o) & 15) == 0) *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
        else if ((reinterpret_cast<uintptr_t>(o) & 7) == 0) {
            *reinterpret_cast<float2*>(o) = make_float2(v[0], v[1]);
            *reinterpret_cast<float2*>(o + 2) = make_float2(v[2], v[3]);
        } else { o[0] = v[0]; o[1] = v[1]; o[2] = v[2]; o[3] = v[3]; }
    } else {
        mw_h* o = reinterpret_cast<mw_h*>(p.out) + oi;
        const mw_h2 a = f2h2(v[0], v[1]), b = f2h2(v[2], v[3]);
        if ((reinterpret_cast<uintptr_t>(o) & 7) == 0) {
            uint2 u;
            u.x = *reinterpret_cast<const uint32_t*>(&a); u.y = *reinterpret_cast<const uint32_t*>(&b);
            *reinterpret_cast<uint2*>(o) = u;
        } else if ((reinterpret_cast<uintptr_t>(o) & 3) == 0) {
            *reinterpret_cast<mw_h2*>(o) = a; *reinterpret_cast<mw_h2*>(o + 2) = b;
        } else { o[0] = f2h(v[0]); o[1] = f2h(v[1]); o[2] = f2h(v[2]); o[3] = f2h(v[3]); }
    }
}

__device__ __forceinline__ void st_cluster_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared::cluster.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, 128;" ::: "memory"); }     // the 4 epilogue warps

template <int KS>
__global__ void __launch_bounds__(DG_THREADS, 1)
decode_gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmap_w, const __grid_constant__ CUtensorMap tmap_x,
                           const DgParams p) {
    const DgLayout L = dg_layout(p.R);
    const int RB = L.rb, STAGES = L.stages;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    unsigned char* smem_w = smem;
    unsigned char* smem_x = smem + STAGES * DG_W_BYTES;
    float* red = reinterpret_cast<float*>(smem + (L.alias ? 0 : L.ring));
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + L.bar_off);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* tmem_full = empty_bar + STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

    DG_STAMP(0);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tile_m = blockIdx.x, split = blockIdx.y;
    const int kb0 = (int)((int64_t)split * p.nkb / KS), kb1 = (int)((int64_t)(split + 1) * p.nkb / KS);
    const uint32_t TMEM_COLS = RB <= 32 ? 32u : RB <= 64 ? 64u : RB <= 128 ? 128u : 256u;      // power of two >= 32

    if (threadIdx.x == 0) {
        prefetch_tensormap(&tmap_w);
        prefetch_tensormap(&tmap_x);
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        mbar_init(tmem_full, 1);
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
    // phase 1 of the cluster barrier only has to prove that every peer CTA is running before its shared memory is written:
    // arrive now, wait (by then for free) just before the scatter
    if (KS > 1 && !L.alias) cluster_arrive();
    DG_STAMP(1);

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int kb = kb0; kb < kb1; ++kb) {
                mbar_wait(&empty_bar[stage], phase ^ 1);
                mbar_arrive_expect_tx(&full_bar[stage], DG_W_BYTES + L.x_bytes);
                tma_load_2d(smem_w + stage * DG_W_BYTES, &tmap_w, &full_bar[stage], kb * DG_K, tile_m * DG_M);
                tma_load_2d(smem_x + stage * L.x_bytes, &tmap_x, &full_bar[stage], kb * DG_K, 0);
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = make_idesc_h16(DG_M, RB);
            int stage = 0; uint32_t phase = 0;
            for (int kb = kb0; kb < kb1; ++kb) {
                mbar_wait(&full_bar[stage], phase);
                tc_fence_after();
                const uint64_t da = make_desc_sw128(smem_u32(smem_w + stage * DG_W_BYTES), 1024, 0);
                const uint64_t db = make_desc_sw128(smem_u32(smem_x + stage * L.x_bytes), 1024, 0);
#pragma unroll
                for (int k = 0; k < DG_K / 16; ++k) umma_h16(tmem_base, da + 2 * k, db + 2 * k, idesc, (kb > kb0 || k) ? 1u : 0u);
                umma_commit(&empty_bar[stage]);
                if (++stage == STAGES) { stage = 0; phase ^= 1; }
            }
            umma_commit(tmem_full);
        }
    } else {
        mbar_wait(tmem_full, 0);          // every MMA of this CTA has retired: accumulator complete, operand ring free
        tc_fence_after();
        DG_STAMP(2);
    }

    const int q = warp & 3;                                   // TMEM lane quadrant of an epilogue warp (warps 2..5 -> 2,3,0,1)
    const int nl = q * 32 + lane;                             // weight row inside the tile = TMEM lane of this thread
    const int n0 = tile_m * DG_M;
    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);

    if (KS == 1) {
        // ---- transpose through shared memory (the operand ring is free): tile[r][128 n] fp32, then whole rows go out coalesced
        if (warp >= 2) {
            float* tile = reinterpret_cast<float*>(smem);
#pragma unroll 1
            for (int c0 = 0; c0 < p.R; c0 += 32) {
                uint32_t r[32];
                tmem_ld32(taddr + c0, r);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 32; ++j) tile[(c0 + j) * 128 + nl] = __uint_as_float(r[j]);      // rows >= R: zero columns, never read
            }
            epi_bar_sync();
            const int we = warp - 2, n = n0 + 4 * lane;
            float bias[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) bias[i] = (p.bias && n + i < p.N) ? __ldg(p.bias + n + i) : 0.0f;
            if (n < p.N) {
                for (int row = we; row < p.R; row += 4) {
                    const float4 t = *reinterpret_cast<const float4*>(tile + row * 128 + 4 * lane);
                    const float acc[4] = {t.x, t.y, t.z, t.w};
                    dg_store4(p, row, n, acc, bias);
                }
            }
        }
    } else {
        // ---- reduce-scatter of the KS partial accumulators through distributed shared memory: destination CTA j finishes
        // activation rows [j*cpd, (j+1)*cpd)
        const int cpd = (((p.R + KS - 1) / KS) + 7) & ~7;
        if (L.alias) {
            tc_fence_before();
            __syncthreads();              // all warps: this CTA's MMAs are done (the epilogue warps saw tmem_full)
            cluster_arrive();
        }
        cluster_wait();                   // ALIAS: every peer is past its MMAs (rings reusable); else: every peer is running
        DG_STAMP(3);
        const uint32_t my_rank = cluster_ctarank();
        // buffer: [src][cpd/4 column groups][128 weight rows] of float4 - a warp's 32 lanes always touch 512 contiguous bytes,
        // which is what distributed shared memory wants (lane-strided 16-byte stores were 3x slower) and is conflict-free to read
        const int src_stride = (cpd / 4) * 128 * 4;             // floats per source CTA
        if (warp >= 2) {
            tc_fence_after();
            const uint32_t local = smem_u32(red) + (uint32_t)((int)my_rank * src_stride + nl * 4) * 4u;
            for (int j = 0; j < KS; ++j) {
                const int c_begin = j * cpd;
                if (c_begin >= p.R) break;
                const uint32_t remote = mapa_shared(local, (uint32_t)j);
                for (int c = 0; c < cpd && c_begin + c < p.R; c += 16) {
                    uint32_t a[8], b[8];
                    const bool two = c + 8 < cpd && c_begin + c + 8 < p.R;
                    tmem_ld8(taddr + c_begin + c, a);
                    if (two) tmem_ld8(taddr + c_begin + c + 8, b);
                    tmem_ld_wait();
                    st_cluster_v4(remote + (uint32_t)((c / 4) * 128 * 16), a[0], a[1], a[2], a[3]);
                    st_cluster_v4(remote + (uint32_t)((c / 4 + 1) * 128 * 16), a[4], a[5], a[6], a[7]);
                    if (two) {
                        st_cluster_v4(remote + (uint32_t)((c / 4 + 2) * 128 * 16), b[0], b[1], b[2], b[3]);
                        st_cluster_v4(remote + (uint32_t)((c / 4 + 3) * 128 * 16), b[4], b[5], b[6], b[7]);
                    }
                }
            }
        }
        DG_STAMP(4);
        cluster_arrive();
        cluster_wait();                   // all partials have landed
        DG_STAMP(5);
        if (warp >= 2) {
            const int c_begin = (int)my_rank * cpd, n = n0 + nl;
            const float bias = (p.bias && n < p.N) ? __ldg(p.bias + n) : 0.0f;
            const float4* mine = reinterpret_cast<const float4*>(red) + nl;
            if (n < p.N) {
                for (int c = 0; c < cpd && c_begin + c < p.R; c += 4) {
                    float4 part[KS];
#pragma unroll
                    for (int s = 0; s < KS; ++s) part[s] = mine[(s * src_stride) / 4 + (c / 4) * 128];
                    float4 acc = part[0];
#pragma unroll
                    for (int s = 1; s < KS; ++s) { acc.x += part[s].x; acc.y += part[s].y; acc.z += part[s].z; acc.w += part[s].w; }  // fixed order
                    const float v[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i)
                        if (c_begin + c + i < p.R) dg_store(p, c_begin + c + i, n, v[i], bias);
                }
            }
        }
    }
    DG_STAMP(6);
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
    DG_STAMP(7);
}

template <int KS>
mw_status dg_launch(const CUtensorMap& tw, const CUtensorMap& tx, const DgParams& p, int tiles_m, cudaStream_t st) {
    static PerDeviceOnce attr_once;
    auto kern = decode_gemm_tcgen05_kernel<KS>;
    MW_CUDA_CHECK(attr_once.run([&] { return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, dg_layout(256).total); }));
    const DgLayout L = dg_layout(p.R);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(tiles_m, KS, 1);
    cfg.blockDim = dim3(DG_THREADS, 1, 1);
    cfg.dynamicSmemBytes = L.total;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 1;
    attr[0].val.clusterDim.y = KS;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    MW_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, tw, tx, p));
    count_launch();
    return MW_OK;
}

}  // namespace

bool decode_gemm_supported(int ldx, int ldw, int R, int N, int K) {
    return R >= 1 && R <= 256 && N >= 1 && K >= 64 && K % 64 == 0 && ldx % 8 == 0 && ldw % 8 == 0;
}

// split-K factor: enough CTAs to spread a small weight matrix over the machine, at least two 64-wide k-blocks per CTA
static int dg_pick_ks(int tiles_m, int nkb) {
    int ks = 1;
    for (int c : {2, 4, 8}) {
        if (tiles_m * c <= 160 && nkb / c >= 2) ks = c;
    }
    return ks;
}

static unsigned long long* g_dg_dbg = nullptr;
void decode_gemm_set_debug(unsigned long long* d_stamps) { g_dg_dbg = d_stamps; }

mw_status decode_gemm_launch(const void* X, int ldx, const void* W, int ldw, const float* bias, const float* resid, void* out,
                             int ldo, int R, int N, int K, int flags, cudaStream_t st) {
    MW_REQUIRE(decode_gemm_supported(ldx, ldw, R, N, K), "decode gemm: unsupported shape R=%d N=%d K=%d", R, N, K);
    MW_REQUIRE(((uintptr_t)X % 16 == 0) && ((uintptr_t)W % 16 == 0), "decode gemm: operands must be 16-byte aligned");
    const DgLayout L = dg_layout(R);
    static_assert(dg_layout(256).total <= 227 * 1024 && dg_layout(128).total <= 227 * 1024, "shared memory budget");
    const int tiles_m = ceil_div(N, DG_M), nkb = K / DG_K;
    CUtensorMap tw, tx;
    {
        uint64_t dims[2] = {(uint64_t)K, (uint64_t)N};
        uint64_t str[1] = {(uint64_t)ldw * 2};
        uint32_t box[2] = {DG_K, DG_M};
        mw_status s = encode_tensor_map(&tw, W, 2, dims, str, box, true);
        if (s != MW_OK) return s;
    }
    {
        uint64_t dims[2] = {(uint64_t)K, (uint64_t)R};
        uint64_t str[1] = {(uint64_t)ldx * 2};
        uint32_t box[2] = {DG_K, (uint32_t)L.rb};
        mw_status s = encode_tensor_map(&tx, X, 2, dims, str, box, true);
        if (s != MW_OK) return s;
    }
    DgParams p;
    p.R = R; p.N = N; p.nkb = nkb; p.ks = dg_pick_ks(tiles_m, nkb);
    p.bias = bias; p.resid = resid; p.out = out; p.ldo = ldo; p.flags = flags; p.dbg = g_dg_dbg;
    switch (p.ks) {
        case 1: return dg_launch<1>(tw, tx, p, tiles_m, st);
        case 2: return dg_launch<2>(tw, tx, p, tiles_m, st);
        case 4: return dg_launch<4>(tw, tx, p, tiles_m, st);
        default: return dg_launch<8>(tw, tx, p, tiles_m, st);
    }
}

}  // namespace mw

// D[R, N] = X[R, K] . W[N, K]^T (+bias) (gelu) (+residual) for R <= 256 rows: the decode-step projection, exposed for
// tests/test_gpu_kernels.py (flags: 1 = GELU, 2 = fp32 output; residual fp32 [R, N] with ld = N).
extern "C" mw_status mw_decode_gemm_h16(const void* d_x, const void* d_w, const float* d_bias, const float* d_residual,
                                        void* d_out, int R, int N, int K, int flags, void* stream) {
    return mw::decode_gemm_launch(d_x, K, d_w, K, d_bias, d_residual, d_out, N, R, N, K, flags, (cudaStream_t)stream);
}

// measurement hook: d_stamps (8 x u64, device) receives %globaltimer at the phase boundaries of CTA (0,0) of the following
// mw_decode_gemm_h16 calls (null switches it off): start, setup done, MMAs done, cluster barrier 1, scatter done,
// cluster barrier 2, stores done, end.
extern "C" void mw_decode_gemm_debug(unsigned long long* d_stamps) { mw::decode_gemm_set_debug(d_stamps); }
