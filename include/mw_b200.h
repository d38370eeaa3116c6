/*
 * mw_b200.h — C ABI of the B200-native Whisper hot path (libmw_b200.so).
 *
 * This is the drop-in boundary of SURVEY.md §8(b).  The reference has no native code of its own;
 * its hot path is entered from Python at
 *     /root/reference/transcribe.py:107-113   whisperx.load_model(...)
 *     /root/reference/transcribe.py:123       model.transcribe(audio, batch_size=..., language="zh")
 * and the arithmetic lives in three third-party seams beneath that call, which are what these
 * entry points replace one for one:
 *     S1  whisperx.audio.log_mel_spectrogram(audio, n_mels, padding, device)      -> mw_logmel / mw_logmel_long
 *     S2  ctranslate2.models.Whisper.encode(StorageView[B,n_mels,3000])            -> mw_encode
 *     S3  ctranslate2.models.Whisper.generate(enc, prompts, beam_size, patience,   -> mw_generate
 *             length_penalty, max_length, suppress_blank, suppress_tokens)
 *     (+) ctranslate2.models.Whisper.detect_language(enc)  [SURVEY §8(f) rank 2]   -> mw_detect_language
 *
 * Conventions
 *   - "h16" below = the 16-bit storage type mw_storage_dtype() reports (fp16 unless built otherwise).
 *   - plain C types only; every pointer named d_* is DEVICE memory owned by the caller, h_* is host.
 *   - every call returns mw_status (0 = ok); the message is in mw_last_error() (thread-local).
 *   - `stream` is a cudaStream_t passed as void*; work is enqueued there, no hidden sync unless stated.
 *   - one mw_model per GPU; calls on one model must be serialised by the caller; the library
 *     selects the model's device itself.
 *   - no allocation on the hot path: the model owns a workspace sized at create for max_batch.
 */
#ifndef MW_B200_H
#define MW_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MW_ABI_VERSION 2

typedef int32_t mw_status;
enum {
    MW_OK = 0,
    MW_ERR_INVALID = 1,   /* bad argument */
    MW_ERR_CUDA = 2,      /* CUDA runtime/driver error */
    MW_ERR_UNSUPPORTED = 3,
    MW_ERR_STATE = 4
};

int mw_abi_version(void);
/* 16-bit storage type of every "h16" buffer below (activations, K/V caches, weight matrices): 0 = IEEE fp16 (default:
 * the reference's GPU compute_type "float16", /root/reference/transcribe_colab.ipynb:119), 1 = bf16 (library built with
 * -DMW_STORAGE_BF16 for A/B runs).  Accumulation, residual stream, softmax statistics and logits are fp32 either way. */
int mw_storage_dtype(void);
const char* mw_last_error(void);
/* number of kernels this library has launched since load (process-wide); bench.py's gpu_launches */
uint64_t mw_launch_count(void);

/* ------------------------------------------------------------------ S1: log-mel ---------------- */
typedef struct mw_logmel_plan mw_logmel_plan;

/* h_filters: host float32 [n_mels, 201] mel filterbank (whisperx assets/mel_filters.npz layout).
 * max_chunks bounds n_chunks of later calls. */
mw_status mw_logmel_plan_create(int n_mels, const float* h_filters, int max_chunks, int device,
                                mw_logmel_plan** out_plan);
void mw_logmel_plan_destroy(mw_logmel_plan* plan);

/* The pipeline's per-chunk call: chunk c = d_audio[d_offsets[c] .. +d_lengths[c]) zero-padded to
 * 480000 samples, own global max.  d_out: float32 [n_chunks, n_mels, 3000].
 * d_out_t (may be NULL): additionally emits the h16 time-major copy [n_chunks, 3002, n_mels]
 * (rows 0 and 3001 zero) that mw_encode's conv stem reads. */
mw_status mw_logmel(mw_logmel_plan* plan, const float* d_audio, int64_t n_audio,
                    const int64_t* d_offsets, const int32_t* d_lengths, int n_chunks,
                    float* d_out, void* d_out_t, void* stream);

/* Un-chunked log_mel_spectrogram(audio[0:n], n_mels, padding): one global max over the whole
 * clip.  d_out: float32 [n_mels, (n+padding)/160]. */
mw_status mw_logmel_long(mw_logmel_plan* plan, const float* d_audio, int64_t n, int64_t padding,
                         float* d_out, void* stream);

/* ------------------------------------------------------------------ model ---------------------- */
typedef struct mw_model mw_model;

typedef struct mw_model_config {
    int32_t n_mels, d_model, n_heads, enc_layers, dec_layers, ffn, vocab;
    int32_t n_audio_ctx;   /* 1500 */
    int32_t n_text_ctx;    /* 448  */
    int32_t max_batch;     /* chunks per mw_encode / mw_generate call */
    int32_t max_beam;      /* 1 = greedy only */
    int32_t device;
} mw_model_config;

/* Weight table: device pointers in the order of enum mw_weight_id, then per-layer blocks.
 * Matrices are h16 row-major [out, in] (torch Linear layout); vectors are fp32.  Pointers are
 * BORROWED and must outlive the model.  Layouts the engine needs that differ from the checkpoint
 * (conv taps folded into K, q|k|v concatenated, zero k-bias) are prepared by the host shim
 * (manual_whisper_b200/engine.py: pack_weights). */
enum mw_weight_id {
    MW_W_CONV1 = 0,       /* h16 [d, 3*n_mels]  k-major: [co][tap][ci] */
    MW_B_CONV1,           /* f32  [d] */
    MW_W_CONV2,           /* h16 [d, 3*d]       [co][tap][ci] */
    MW_B_CONV2,           /* f32  [d] */
    MW_ENC_POS,           /* f32  [n_audio_ctx, d] */
    MW_ENC_LN_G, MW_ENC_LN_B,   /* f32 [d] final encoder LayerNorm */
    MW_DEC_EMB,           /* h16 [vocab, d] token embedding (tied output projection) */
    MW_DEC_POS,           /* f32  [n_text_ctx, d] */
    MW_DEC_LN_G, MW_DEC_LN_B,   /* f32 [d] final decoder LayerNorm */
    MW_GLOBAL_COUNT
};
enum mw_enc_layer_weight_id {
    MW_EL_LN1_G = 0, MW_EL_LN1_B,
    MW_EL_WQKV,           /* h16 [3d, d]   q|k|v rows */
    MW_EL_BQKV,           /* f32  [3d]      k part zero */
    MW_EL_WO, MW_EL_BO,   /* h16 [d, d], f32 [d] */
    MW_EL_LN2_G, MW_EL_LN2_B,
    MW_EL_W1, MW_EL_B1,   /* h16 [ffn, d], f32 [ffn] */
    MW_EL_W2, MW_EL_B2,   /* h16 [d, ffn], f32 [d] */
    MW_EL_COUNT
};
enum mw_dec_layer_weight_id {
    MW_DL_LN1_G = 0, MW_DL_LN1_B,
    MW_DL_WQKV, MW_DL_BQKV,
    MW_DL_WO, MW_DL_BO,
    MW_DL_LNX_G, MW_DL_LNX_B,   /* encoder_attn_layer_norm */
    MW_DL_WXQ, MW_DL_BXQ,       /* cross q: h16 [d,d], f32 [d] */
    MW_DL_WXKV, MW_DL_BXKV,     /* cross k|v: h16 [2d,d], f32 [2d] (k part zero) */
    MW_DL_WXO, MW_DL_BXO,
    MW_DL_LN2_G, MW_DL_LN2_B,
    MW_DL_W1, MW_DL_B1,
    MW_DL_W2, MW_DL_B2,
    MW_DL_COUNT
};
typedef struct mw_weight_table {
    int32_t n;               /* MW_GLOBAL_COUNT + enc_layers*MW_EL_COUNT + dec_layers*MW_DL_COUNT */
    const void* const* ptrs; /* host array of device pointers */
} mw_weight_table;

mw_status mw_model_create(const mw_model_config* cfg, const mw_weight_table* weights, mw_model** out_model);
void mw_model_destroy(mw_model* model);
/* bytes of device workspace the model allocated at create */
int64_t mw_model_workspace_bytes(const mw_model* model);

/* S2. d_mel: float32 [B, n_mels, 3000]; d_enc_out: h16 [B, n_audio_ctx, d_model]. */
mw_status mw_encode(mw_model* model, const float* d_mel, int B, void* d_enc_out, void* stream);
/* Same, reading the h16 time-major features mw_logmel emitted ([B, 3002, n_mels]). */
mw_status mw_encode_t(mw_model* model, const void* d_mel_t, int B, void* d_enc_out, void* stream);

typedef struct mw_gen_options {
    int32_t beam_size;            /* 1 = greedy */
    float   patience;
    float   length_penalty;
    int32_t max_length;           /* 448 */
    int32_t n_suppress;           /* ids masked at every step (already expanded, no -1) */
    const int32_t* h_suppress;    /* host */
    int32_t n_suppress_begin;     /* ids masked at the first generated step */
    const int32_t* h_suppress_begin;
    int32_t eot;
    int32_t timestamp_begin;
    int32_t no_timestamps;
    int32_t with_timestamps;      /* 1 = apply the timestamp rules */
    int32_t max_initial_timestamp_index;
    int32_t num_hypotheses;       /* <= beam_size */
    int32_t forced_eot_len;       /* bench-only knob: >0 forces <eot> after this many tokens; 0 = off */
} mw_gen_options;

/* S3.  d_enc: h16 [B, n_audio_ctx, d_model].  One shared prompt (whisperx passes [prompt]*B).
 * h_out_ids: host int32 [B, num_hypotheses, max_new] (max_new = min(max_length/2, max_length-prompt_len)),
 * h_out_len: host int32 [B, num_hypotheses], h_out_scores: host float [B, num_hypotheses].
 * Synchronises `stream` before returning (ids are returned to the host, like CT2). */
mw_status mw_generate(mw_model* model, const void* d_enc, int B, const int32_t* h_prompt, int prompt_len,
                      const mw_gen_options* opt, int32_t* h_out_ids, int32_t* h_out_len, float* h_out_scores,
                      void* stream);

/* Teacher-forced decoder logits for parity tests: tokens host int32 [B, n]; d_logits float32 [B, n, vocab]. */
mw_status mw_decoder_logits(mw_model* model, const void* d_enc, int B, const int32_t* h_tokens, int n,
                            float* d_logits, void* stream);

/* softmax over the language ids at the <sot> position: h_probs float [B, n_langs]. */
mw_status mw_detect_language(mw_model* model, const void* d_enc, int B, int32_t sot, int32_t first_lang,
                             int32_t n_langs, float* h_probs, void* stream);

/* ------------------------------------------------------------------ building blocks ------------
 * Exposed so tests can pin each kernel against torch on its own (tests/test_gpu_kernels.py). */
/* D[M,N] = A[M,K] . W[N,K]^T (+bias[N]) (gelu) (+residual f32[M,N]); A,W h16; out h16 or f32. */
mw_status mw_gemm_h16(const void* d_a, const void* d_w, const float* d_bias, const float* d_residual,
                       void* d_out, int M, int N, int K, int gelu, int out_f32, void* stream);
/* encoder self-attention on packed qkv h16 [B*T, 3*d]; out h16 [B*T, d] */
mw_status mw_attention_h16(const void* d_qkv, void* d_out, int B, int T, int n_heads, void* stream);
/* The decode-step projection (csrc/decode_gemm.cu): D[R,N] = X[R,K] . W[N,K]^T (+bias) (flags&1: GELU) (+residual f32 [R,N]);
 * X,W h16; out h16, or f32 when flags&2; R <= 256, K % 64 == 0.  W is streamed once for all R rows. */
mw_status mw_decode_gemm_h16(const void* d_x, const void* d_w, const float* d_bias, const float* d_residual,
                             void* d_out, int R, int N, int K, int flags, void* stream);
/* Scheduling hint for mw_generate: solo != 0 says this model (replica) is the only one decoding on its GPU, so the step is
 * built for latency (LayerNorm folded into the projections that consume it: 96 fewer launches per large-v3 step, -4 % per step);
 * solo == 0 (default) is the form that is faster when several replicas decode concurrently.  Same ids either way.  The host
 * mirror sets it per job (asr.py run_device_batches: one batch in flight -> solo), e.g. one recording sharded over 8 GPUs
 * (/root/reference/transcribe.py:123 with device_index=[0..7]). */
mw_status mw_set_solo(mw_model* model, int solo);
/* Measurement hook (bench.py "in_step"): keep only the kernel classes in `parts` (the mask of mw_bench_step, plus 64 = token
 * selection) in decode-step graphs captured from now on, process-wide; 127 restores the real step.  Ids are meaningless while a
 * class is missing; the change in step time is that class's cost inside the real, concurrent step. */
void mw_debug_step_parts(int parts);
/* Measurement hook: d_stamps (device, 8 x uint64) receives %globaltimer at the phase boundaries of CTA (0,0) of the
 * following mw_decode_gemm_h16 calls; NULL switches it off (scripts/gpu_dg_phases.py). */
void mw_decode_gemm_debug(unsigned long long* d_stamps);
mw_status mw_layernorm(const float* d_x, const float* d_gamma, const float* d_beta, void* d_out_h16,
                       int rows, int d, void* stream);
/* The tcgen05 GEMM in the full geometry of struct GemmArgs (csrc/gemm.cuh), for tests/test_gpu_tensor_core_paths.py:
 * out[b*out_batch_rows + out_row_off + m, n] (ld_out) = sum_k A[b*a_batch_stride + m*a_row_stride + k] W[n*w_row_stride + k]
 *     (+bias[n]) (gelu) (+resid[(b*res_batch_rows + m)*ld_res + n]).
 * A rows may overlap (a_row_stride < K); resid may equal out.  Shapes and strides are checked before any pointer. */
mw_status mw_gemm_general_h16(const void* d_a, int64_t a_row_stride, int64_t a_batch_stride, const void* d_w, int64_t w_row_stride,
                              const float* d_bias, const float* d_resid, int64_t res_batch_rows, int64_t ld_res,
                              void* d_out, int64_t out_batch_rows, int64_t out_row_off, int64_t ld_out,
                              int batch, int M, int N, int K, int gelu, int out_f32, void* stream);
/* attention_launch_general: q [B, Tq, ldq] head h at column colq0 + 64h; k|v [B, Tk, ldkv] at colk0 / colv0 + 64h;
 * out [B*Tq, out_ld] head h at column 64h; d_kv_lens (may be NULL, only with Tq == Tk): keys >= len masked, wholly padded
 * query tiles untouched (the ragged contract of attention_launch, csrc/kernels.cuh).  Column ranges are checked before any
 * pointer. */
mw_status mw_attention_general_h16(const void* d_q, int64_t ldq, int colq0, const void* d_kv, int64_t ldkv, int colk0, int colv0,
                                   void* d_out, int out_ld, int B, int Tq, int Tk, int n_heads, const int32_t* d_kv_lens,
                                   void* stream);
/* LayerNorm variants: mode 1 = GELU(LN) -> h16, 2 = GELU(LN) -> f32 (d <= 512); 3 = LN -> h16 AND written back over x in f32.
 * Mode 0 is mw_layernorm.  Shape and mode are checked before any pointer. */
mw_status mw_layernorm_mode(float* d_x, const float* d_gamma, const float* d_beta, void* d_out, int rows, int d, int mode,
                            void* stream);

/* The decode step's own kernels (csrc/decoder.cu) on caller buffers, for tests/test_gpu_decode_step.py.  The launch path is
 * named by an argument.  They may allocate a few bytes and synchronise. */
enum mw_step_path {
    MW_STEP_PATH_GREEDY = 0,        /* the step's routing in greedy search: tcgen05 decode GEMM from 96 rows, else mma.sync */
    MW_STEP_PATH_BEAM = 1,          /* the step's routing of the layer projections in beam search: mma.sync kernels only */
    MW_STEP_PATH_GREEDY_SOLO = 2,   /* the same two with mw_set_solo on (fused LayerNorm, one-tile K-halved fc2) */
    MW_STEP_PATH_BEAM_SOLO = 3,
    MW_STEP_PATH_ROWS16_WT1 = 4,    /* forced kernels: rows16 with one / two 16-row weight tiles per CTA, */
    MW_STEP_PATH_ROWS16_WT2 = 5,
    MW_STEP_PATH_KHALF_WT1 = 6,     /* the K-halved kernel (K = 2048 .. 5120) with one / two tiles, */
    MW_STEP_PATH_KHALF_WT2 = 7,
    MW_STEP_PATH_GENERIC = 8,       /* the generic kernel (any K % 32 == 0), */
    MW_STEP_PATH_LN_FUSED = 9,      /* LayerNorm folded into the projection (16-bit output), */
    MW_STEP_PATH_LN_SEPARATE = 10   /* LayerNorm, then the projection (beam routing), as two launches */
};
/* out[R,N] = X[R,K] . W[N,K]^T (+bias[N]) (flags&1: GELU) (+resid f32 [R,N]); out h16, or f32 when flags&2.  With gamma and
 * beta, X = LayerNorm(x_f32 [R,K]) and x_h16 is the scratch the stand-alone LayerNorm writes; otherwise X = x_h16.  A forced
 * kernel that does not exist for K returns MW_ERR_UNSUPPORTED. */
mw_status mw_step_projection_h16(const void* d_x_h16, const float* d_x_f32, const float* d_gamma, const float* d_beta,
                                 const void* d_w, const float* d_bias, const float* d_resid, void* d_out, int R, int N, int K,
                                 int flags, int path, void* stream);
/* Self-attention of one step: appends k, v of qkv h16 [R, 3d] at position pos of the caches h16 [R, ctx, d], then attends over
 * pos + 1 keys; key j < pos of row r is read from cache row d_idx[r*ctx + j] (int32 [R, ctx]; NULL = row r).  out h16 [R, d]. */
mw_status mw_step_self_attention_h16(const void* d_qkv, void* d_k_cache, void* d_v_cache, const int32_t* d_idx, int R,
                                     int n_heads, int ctx, int pos, void* d_out, void* stream);
/* Causal self-attention of the batched prompt prefill: qkv h16 [B*P, 3d], row b*P + p sees keys 0..p of its sequence. */
mw_status mw_step_prefill_attention_h16(const void* d_qkv, int B, int P, int n_heads, void* d_out, void* stream);
/* Cross-attention: G queries per sequence q h16 [B*G, d] over the sequence's keys/values kv h16 [B*T, 2d] (k | v);
 * out h16 [B*G, d].  G = 1: the streaming kernel with unr = 4 or 8 loads in flight per lane; G = 2..8: the grouped kernel of
 * beam search (G*T*4 bytes of scores must fit 96 KB). */
mw_status mw_step_cross_attention_h16(const void* d_q, const void* d_kv, int B, int G, int T, int n_heads, int unr,
                                      void* d_out, void* stream);

/* VAD front end (SURVEY.md §8f rank 1): RMS of consecutive frames of `frame` samples, d_out float32 [n / frame].
 * Feeds the energy VAD so the waveform is uploaded once and never revisited by the host. */
mw_status mw_frame_rms(const float* d_audio, int64_t n, int frame, float* d_out, void* stream);

/* The rest of that front end on the device: frame RMS (as written by mw_frame_rms, frame_s seconds per frame) -> energy
 * speech score (dB mapped between the 10 % and 95 % points of a 2048-bin histogram) -> Binarize hysteresis (onset / offset,
 * turns cut at max_duration_s) -> gaps shorter than min_off_s filled, turns shorter than min_on_s dropped ->
 * Vad.merge_chunks(chunk_size_s).  d_scratch: >= 8192 + 16 * max_turns bytes.  d_windows: double [max_windows][2] =
 * (start_s, end_s); d_counts: int32 [3] = {turns kept, windows written, overflow flag}.  Replaces the host pass of
 * whisperx's Binarize + merge_chunks (/root/reference/transcribe.py:43-46,112); manual_whisper_b200/vad.py: EnergyVad is
 * the host twin with the same float64 arithmetic. */
mw_status mw_vad_windows(const float* d_rms, int64_t n_frames, double frame_s, double onset, double offset,
                         double max_duration_s, double min_on_s, double min_off_s, double chunk_size_s,
                         void* d_scratch, int max_turns, double* d_windows, int max_windows, int32_t* d_counts,
                         void* stream);

/* Measurement hook for bench.py's roofline: average duration (ms, CUDA events on `stream`) of one hot decode
 * kernel launched `iters` times back to back over different layers' data (inputs larger than L2).
 * which: 0 = cross-attention decode, 1 = skinny GEMM (fc1 weights), 2 = skinny GEMM (out-proj weights). */
mw_status mw_bench_kernel(mw_model* model, int which, int B, int iters, float* h_ms_avg, void* stream);
/* Average ms of one decode step (CUDA-graph replay, B rows, position 0) restricted to the kernel classes in `parts`:
 * 1 embed, 2 LayerNorm, 4 skinny GEMMs, 8 self-attention, 16 cross-attention, 32 final LN + logits GEMM. */
mw_status mw_bench_step(mw_model* model, int B, int parts, int iters, float* h_ms_avg, void* stream);

/* ------------------------------------------------------------------ forced alignment (SURVEY.md §8f row 3) ------
 * Replaces what whisperx.align runs per segment (/root/reference/transcribe.py:127-135): the wav2vec2-CTC acoustic
 * model (Hugging Face Wav2Vec2ForCTC, feat_extract_norm="layer", do_stable_layer_norm=True - the XLSR-53 family
 * whisperx loads for "zh") -> log_softmax emissions, and the CTC trellis + backtrack of whisperx/alignment.py.
 * Windows of different lengths are batched: every per-frame op is row-wise, the positional conv sees zeros beyond a
 * window's last frame and self-attention masks keys beyond it, so each window's emissions equal a solo run. */
typedef struct mw_w2v mw_w2v;

typedef struct mw_w2v_config {
    int32_t n_layers, d_model, n_heads, ffn;
    int32_t vocab;           /* real CTC vocabulary; lm_head rows are padded to a multiple of 32 by the host */
    int32_t conv_dim;        /* 512: channels of the 7 feature-extractor convs (kernels 10,3,3,3,3,2,2; strides 5,2,2,2,2,2,2) */
    int32_t pos_kernel;      /* 128 */
    int32_t pos_groups;      /* 16; d_model / pos_groups must be 64 */
    int32_t max_batch;       /* windows per mw_w2v_emissions call */
    int32_t max_samples;     /* longest window in samples (480000 = 30 s) */
    int32_t device;
    int32_t variant;         /* 0: feat_extract_norm="layer", do_stable_layer_norm=True (XLSR-53 family: the reference's zh model);
                              * 1: wav2vec2-base (what whisperx loads for en/fr/de/es/it): GroupNorm after conv0 only, no conv
                              *    biases, post-LayerNorm encoder; d_model / pos_groups may then be 48 (pos-conv weight rows padded
                              *    to 64 per group by the host) */
} mw_w2v_config;

/* Weight table: MW_A_* globals, then n_layers blocks in the order of enum mw_enc_layer_weight_id (q|k|v rows
 * concatenated, all three biases real).  Matrices h16 row-major [out, in]; vectors fp32; pointers borrowed. */
enum mw_w2v_weight_id {
    MW_A_CONV0_W = 0,     /* f32 [conv_dim, 10] */
    MW_A_CONV0_B, MW_A_CONV0_LN_G, MW_A_CONV0_LN_B,
    MW_A_CONV1_W,         /* conv layer i = 1..6 at MW_A_CONV0_W + 4 i: h16 [conv_dim, k_i * conv_dim] as [co][tap][ci], */
    MW_A_CONV1_B, MW_A_CONV1_LN_G, MW_A_CONV1_LN_B,   /* then bias, LayerNorm gamma, beta */
    MW_A_FP_LN_G = 28, MW_A_FP_LN_B,   /* feature_projection.layer_norm */
    MW_A_FP_W, MW_A_FP_B,              /* feature_projection.projection: h16 [d, conv_dim], f32 [d] */
    MW_A_POS_W,           /* h16 [groups][64 out][pos_kernel taps][64 in]: effective (weight-normalised) pos-conv weight */
    MW_A_POS_B,           /* f32 [d] */
    MW_A_ENC_LN_G, MW_A_ENC_LN_B,      /* encoder.layer_norm (after the last layer) */
    MW_A_LM_W, MW_A_LM_B,              /* lm_head: h16 [ceil32(vocab), d], f32 [ceil32(vocab)] */
    MW_A_GLOBAL_COUNT
};

mw_status mw_w2v_create(const mw_w2v_config* cfg, const mw_weight_table* weights, mw_w2v** out_model);
void mw_w2v_destroy(mw_w2v* model);
int64_t mw_w2v_workspace_bytes(const mw_w2v* model);
/* frames the conv stack yields for n_samples (0 below 400 samples) */
int32_t mw_w2v_frames(int64_t n_samples);

/* Emissions of n windows: window c = d_audio[d_offsets[c] .. + d_lengths[c]), shorter than 400 samples is zero-padded to
 * 400 as whisperx does.  h_lengths: host copy of the lengths (sizes the launch).  d_out: f32, window c at
 * d_out + c * out_window_stride, [frames_c, vocab] log-probabilities (rows beyond frames_c are not written);
 * out_window_stride >= mw_w2v_frames(max length) * vocab. */
mw_status mw_w2v_emissions(mw_w2v* model, const float* d_audio, int64_t n_audio, const int64_t* d_offsets,
                           const int32_t* d_lengths, const int32_t* h_lengths, int n, float* d_out,
                           int64_t out_window_stride, void* stream);

/* Test hook: copies one internal buffer of the last mw_w2v_emissions call to d_dst (device): 0 = conv stack output f32
 * [n*T, conv_dim], 1 = residual stream f32 [n*T, d_model], 2 = GroupNorm statistics f32 [n, conv_dim, 2] (variant 1),
 * 3 = conv0 output h16 [n, T_0, conv_dim]. */
mw_status mw_w2v_debug_copy(mw_w2v* model, int which, void* d_dst, int64_t nbytes, void* stream);

/* CTC forced alignment of n windows (whisperx get_trellis + backtrack).  Emissions as written by mw_w2v_emissions;
 * d_frames[c] = valid frames; d_tokens [n, max_tokens] dictionary ids (-1 = wildcard: best non-blank symbol),
 * d_n_tokens[c] of them used.  Outputs per frame: d_frame_token [n, max_frames] = index into the window's token list,
 * d_frame_score [n, max_frames] = probability of the symbol the path emitted there; d_ok[c] = 0 when the window is not
 * alignable (more tokens than frames, or no tokens).  d_workspace: f32 [n * max_frames * (max_tokens + 1)] scratch. */
mw_status mw_ctc_align(const float* d_emissions, int64_t window_stride, int vocab, const int32_t* d_frames,
                       const int32_t* d_tokens, int max_tokens, const int32_t* d_n_tokens, int n, int blank,
                       int32_t* d_frame_token, float* d_frame_score, int max_frames, int32_t* d_ok,
                       float* d_workspace, void* stream);

/* ------------------------------------------------------------------ audio decode (SURVEY.md §8f row 4) -----------
 * The PCM leg of whisperx.load_audio (/root/reference/transcribe.py:117; `ffmpeg -ac 1 -ar 16000 -f s16le` then /32768):
 * interleaved PCM (sample_format 0 = int16, 1 = float32) [n_frames, channels] at rate orig*g -> mono float32 at new_rate*g
 * (orig:new_rate the reduced ratio).  d_kernels: f32 [new_rate, taps] polyphase windowed-sinc taps, taps = 2*width + orig
 * (torchaudio.functional.resample's filter, built by manual_whisper_b200/audio.py); d_lo_hi: int32 [new_rate, 2] non-zero
 * tap range of each phase.  d_out: f32 [n_out], n_out <= ceil(n_frames * new_rate / orig).  quantize_s16 != 0 rounds to
 * the int16 grid like the s16le pipe. */
mw_status mw_pcm_resample(const void* d_pcm, int64_t n_frames, int channels, int sample_format, int orig, int new_rate,
                          const float* d_kernels, const int32_t* d_lo_hi, int taps, int width, float* d_out,
                          int64_t n_out, int quantize_s16, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MW_B200_H */
