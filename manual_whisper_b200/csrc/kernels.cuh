// Launchers shared between the engine's translation units.
#pragma once
#include "mw_common.cuh"

namespace mw {

mw_status layernorm_launch(const float* x, const float* gamma, const float* beta, void* out_bf16, int rows, int d,
                           cudaStream_t st);
mw_status features_to_time_major_launch(const float* in, void* out_bf16, int B, int C, int F, cudaStream_t st);
// d_lens (may be null): per-window valid length for ragged self-attention - keys t >= d_lens[b] are masked, query tiles
// beyond it skipped (their output rows are left untouched).  The ragged contract (tests/test_gpu_tensor_core_paths.py):
//  * padded keys and values must be finite: a masked key gets P = 0, but 0 x NaN in P V is NaN;
//  * padded query rows of the tile that holds the window's last row are written (their attention over the valid keys);
//    rows of wholly padded 128-row tiles are not;
//  * a window's rows are those of its solo run (B = 1, T = its length) unless a padded query row of the boundary warp
//    moves the warp's exponent reference (the lazy rescale is decided per warp of 32 rows) where the solo run's zero rows do not
mw_status attention_launch(const void* d_qkv, void* d_out, int B, int T, int n_heads, cudaStream_t st, const int* d_lens = nullptr);
// LayerNorm variants of the wav2vec2 feature extractor: mode 1 = GELU(LN(x)) -> bf16, mode 2 = GELU(LN(x)) -> f32
mw_status layernorm_act_launch(const float* x, const float* gamma, const float* beta, void* out, int rows, int d, int mode,
                               cudaStream_t st);
// LN(x) -> h16 copy AND written back over x in fp32 (post-LayerNorm encoders)
mw_status layernorm_dual_launch(float* x_inout, const float* gamma, const float* beta, void* out_h16, int rows, int d,
                                cudaStream_t st);
mw_status attention_launch_general(const void* d_q, int64_t ldq, int colq0, const void* d_kv, int64_t ldkv, int colk0, int colv0,
                                   void* d_out, int out_ld, int B, int Tq, int Tk, int n_heads, cudaStream_t st,
                                   const int* d_kv_lens = nullptr);

}  // namespace mw
