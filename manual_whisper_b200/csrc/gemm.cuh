// Host-side interface of the tcgen05 GEMM (gemm.cu), shared by the encoder/decoder drivers.
#pragma once
#include "mw_common.cuh"
#include <cuda.h>

namespace mw {

// D[b, m, n] = sum_k A[b, m, k] * W[n, k]  (+ bias[n]) (gelu) (+ residual)
// A is addressed through a 3-D view (k, m, b) with arbitrary element strides, which is how the conv stem's
// im2col rows (overlapping windows of a time-major buffer) are fed without materialising them.
struct GemmArgs {
    const void* a = nullptr;        // bf16
    int64_t a_row_stride = 0;       // elements between consecutive m
    int64_t a_batch_stride = 0;     // elements between batches
    const void* w = nullptr;        // bf16 [N, K] row-major (ld = w_row_stride)
    int64_t w_row_stride = 0;
    const float* bias = nullptr;    // [N] or null
    const float* residual = nullptr;// f32, row r = b*res_batch_rows + m, ld = ld_res; null = none
    int64_t res_batch_rows = 0;
    int64_t ld_res = 0;
    void* out = nullptr;            // bf16 or f32; row r = b*out_batch_rows + out_row_off + m, ld = ld_out
    int64_t out_batch_rows = 0;
    int64_t out_row_off = 0;
    int64_t ld_out = 0;
    int batch = 1;
    int M = 0;                      // rows per batch
    int N = 0;
    int K = 0;
    bool gelu = false;
    bool out_f32 = false;
};

mw_status gemm_launch(const GemmArgs& args, cudaStream_t stream);

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time libcuda dependency)
mw_status encode_tensor_map(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                            const uint64_t* strides_bytes /* rank-1 */, const uint32_t* box, bool swizzle128);

int device_sm_count();

// decode_gemm.cu: out[R, N] = X[R, K] . W[N, K]^T (+bias) (gelu: flags & 1) (+resid f32, ld = ldo) -> h16 or f32 (flags & 2),
// R <= 256 rows, every weight byte streamed once (swap-AB tcgen05 tiles, split-K over a thread-block cluster)
bool decode_gemm_supported(int ldx, int ldw, int R, int N, int K);
mw_status decode_gemm_launch(const void* X, int ldx, const void* W, int ldw, const float* bias, const float* resid, void* out,
                             int ldo, int R, int N, int K, int flags, cudaStream_t st);

}  // namespace mw
