/*
 * d3pm_b200.h — C ABI of the B200-native D3PM / VQ-Diffusion reverse-diffusion token update.
 *
 * The reference (Developer-Zer0/GIF-synthesis-with-Discrete-Diffusion) is 100 % Python: the
 * "FFI" of this path is the method surface of
 *     src/models/motionencoder/diffusion_transformer.py  class DiffusionTransformer
 * Each entry point below names the reference method(s) (file:line) it replaces.  All pointers are
 * DEVICE pointers owned by the caller (PyTorch); the library allocates nothing persistent, keeps no
 * pointer past return, launches asynchronously on the given CUDA stream and never synchronises
 * (the one exception is the explicit d3pm_host_step handle near the end, for HOST input buffers).
 * Return value: 0 (D3PM_OK) or a negative error code; d3pm_last_error() gives the text.
 *
 * Memory layout ("token-major rows"): a logical [B, C, N] tensor of the reference (class dim = 1)
 * is stored as B*N rows of `pitch` floats, class index contiguous, pitch % 4 == 0, base 16-byte
 * aligned.  The denoiser's logits are already physically [B, N, K] (transformer_utils.py:442-443
 * returns a permuted view), so they are consumed in place with pitch = K.  Tensors that carry the
 * [MASK] class (K+1 entries) use pitch >= K+1 (K+4 for K = 4096): entry K of a row is the [MASK]
 * class, the padding is never read.
 */
#ifndef D3PM_B200_H
#define D3PM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define D3PM_VERSION 300 /* major*10000 + minor*100 + patch; 0.3.0: 16-bit logits (d3pm_step_desc.logits_dtype), video decoder */

#define D3PM_OK 0
#define D3PM_ERR_INVALID (-1)     /* null pointer, non-positive size, t/K/T inconsistent */
#define D3PM_ERR_ALIGN (-2)       /* pointer not 16-byte aligned or pitch % 4 != 0 */
#define D3PM_ERR_UNSUPPORTED (-3) /* shape outside what the kernels cover (K % 4 != 0, K > 8192) */
#define D3PM_ERR_CUDA (-4)        /* a CUDA runtime call failed (text holds cudaGetErrorString) */

/* bits OR-ed into the optional device status word by the kernels (the reference asserts these on
 * the host with .item() syncs, diffusion_transformer.py:45-46, :253) */
#define D3PM_STATUS_BAD_T 1u     /* some t[b] outside [0, T) */
#define D3PM_STATUS_BAD_TOKEN 2u /* some x_t outside [0, K] */
#define D3PM_STATUS_FALLBACK 4u  /* informational: a row needed the exhaustive sampling pass */

typedef void* d3pm_stream_t; /* cudaStream_t */

int d3pm_version(void);
const char* d3pm_last_error(void);

/* ---------------------------------------------------------------- schedule
 * Replaces: the eight registered buffers built in DiffusionTransformer.__init__
 * (diffusion_transformer.py:120-149) and every `extract(...)` gather on them (:36-39,
 * :186-189, :204-207, :263, :271).
 * `sched` = [8][T+1] floats in the order log_at, log_bt, log_ct, log_1_min_ct, log_cumprod_at,
 * log_cumprod_bt, log_cumprod_ct, log_1_min_cumprod_ct (per-step rows padded to T+1).
 * Writes table[T][D3PM_COEF_STRIDE]: per-timestep linear-domain coefficients (computed in
 * float64 on the device) that the step kernels index with t[b].                                  */
#define D3PM_COEF_STRIDE 32
int d3pm_build_coef_table(const float* sched, int T, int K, float* table, d3pm_stream_t stream);

/* ---------------------------------------------------------------- fused reverse step
 * Replaces, in ONE pass over the logits: predict_start's log-softmax/clamp (:231-236),
 * cf_predict_start (:240-249), q_posterior (:251-283) incl. q_pred / q_pred_one_timestep
 * (:185-218), log_sample_categorical (:354-359) and the index<->log-one-hot round trips
 * (:44-54) — i.e. p_pred (:285-296) + the prior_rule==0 branch of p_sample (:304-352).        */
#define D3PM_SAMPLE_NONE 0         /* outputs only (p_pred) */
#define D3PM_SAMPLE_GUMBEL 1       /* argmax(gumbel + posterior), noise injected by the caller */
#define D3PM_SAMPLE_PHILOX 2       /* in-kernel Philox4x32-7 noise (23-bit uniforms), thinned exponential race (production) */
#define D3PM_SAMPLE_PHILOX_EXACT 3 /* same noise, every class scored in log space (verification) */

#define D3PM_FROM_POSTERIOR 0 /* sample x_{t-1} from q_posterior's result (prior_rule 0, :347-350) */
#define D3PM_FROM_RECON 1     /* sample from log_x_recon = p(x0 | x_t) (prior_rule 1 / 2, :327-329) */

#define D3PM_KERNEL_AUTO 0
#define D3PM_KERNEL_ROWS 1   /* one CTA per token row, every shape and mode */
#define D3PM_KERNEL_STREAM 2 /* persistent TMA-pipelined kernel: PHILOX / PHILOX_EXACT, no outputs, K in {1024,2048,4096} */

#define D3PM_LOGITS_F32 0  /* logits_c / logits_u point at float rows */
#define D3PM_LOGITS_F16 1  /* ... at IEEE half rows (a denoiser run under torch.autocast, transformer_utils.py via :228-230) */
#define D3PM_LOGITS_BF16 2 /* ... at bfloat16 rows */

typedef struct d3pm_step_desc {
  /* inputs */
  const float* logits_c;   /* [B*N][pitch_logits] conditional denoiser logits (first K valid); element type = logits_dtype */
  const float* logits_u;   /* same shape, unconditional; NULL = guidance off (predict_start only) */
  const int64_t* x_t;      /* [B*N] current tokens in [0, K]; K = [MASK] */
  const int64_t* t;        /* [B] timestep per video, in [0, T) */
  const float* coef_table; /* from d3pm_build_coef_table */
  const float* gumbel;     /* [B*N][pitch_gumbel] Gumbel noise, entry K = [MASK]; D3PM_SAMPLE_GUMBEL only */
  /* outputs (each nullable) */
  int64_t* x_prev;     /* [B*N] sampled x_{t-1} */
  float* post;         /* [B*N][pitch_out] posterior log-probs, K+1 valid (q_posterior's return, clamp(-70,0)) */
  float* recon;        /* [B*N][pitch_out] log p(x0|x_t), K+1 valid (cf_predict_start's return) */
  float* gap;          /* [B*N] top-1 minus top-2 sampling score (near-tie log); GUMBEL / PHILOX_EXACT only */
  uint32_t* status;    /* one word, OR of D3PM_STATUS_* */
  /* sizes */
  int32_t B, N, K, T;
  int64_t pitch_logits, pitch_gumbel, pitch_out; /* in elements (pitch_logits: of logits_dtype) */
  /* parameters */
  float guidance_scale;
  int32_t sample_mode;   /* D3PM_SAMPLE_* */
  int32_t gumbel_is_uniform; /* 1: `gumbel` holds uniforms u (torch.rand_like's tensor); g = -log(-log(u+1e-30)+1e-30) in-kernel */
  uint64_t seed, offset; /* Philox key / per-call stream offset */
  int64_t row_offset;    /* global index of local row 0 (b_global*N + n): shards reproduce the 1-GPU stream */
  float thin_factor;     /* PHILOX thinning constant c (0 = default); smaller values make more rows take the second
                            attempt (stream kernel: c = 16), values < 0.01 force the exhaustive fallback */
  int32_t kernel;        /* D3PM_KERNEL_*: which implementation runs (AUTO picks by shape and mode) */
  d3pm_stream_t stream;
  /* purity-prior sampling (p_sample with prior_rule 1 / 2, :309-346); all optional.  D3PM_FROM_RECON + score with PHILOX
   * sampling runs on the stream kernel (its RECON instantiation); `sharpen` and the other modes on the rows kernel */
  int32_t sample_from;   /* D3PM_FROM_POSTERIOR (default) or D3PM_FROM_RECON: draw x from p(x0 | x_t) (:327-329) */
  int32_t logits_dtype;  /* D3PM_LOGITS_*.  16-bit rows are read as they lie in HBM and widened in registers - bit-identical to
                            running the fp32 path on logits.float() (the reference up-casts too: log_softmax(out.double()), :231) at
                            half the traffic.  Stream kernel only (PHILOX / PHILOX_EXACT sampling, no row outputs, D3PM_FROM_POSTERIOR,
                            K in {1024,2048,4096}, pitch_logits % 8 == 0); other requests return D3PM_ERR_UNSUPPORTED and the caller
                            casts */
  float* score;          /* [B*N] out: max_k p(x0 = k | x_t), the purity of :318 before its per-video normalisation */
  const float* sharpen;  /* [B*N] in: f = 1 + score * prior_weight; the draw is from softmax(f * log p(x0 | x_t)) (:323-325);
                            D3PM_FROM_RECON with GUMBEL / PHILOX_EXACT sampling only */
  float* winner_post;    /* [B*N] out, optional, stream kernel only (forces it): the posterior log-prob (clamp(log P, -70, 0),
                            :283; log p(x0 | x_t) with D3PM_FROM_RECON) of the class x_prev holds, exactly as the production
                            kernel computed it.  Verification hook: lets a test measure the 1e-4 posterior tolerance on the
                            kernel that is benchmarked, which otherwise outputs tokens only */
} d3pm_step_desc;

int d3pm_fused_step(const d3pm_step_desc* desc);

/* The uniforms D3PM_SAMPLE_PHILOX* draw, written as fp32 rows [rows][pitch] (K+1 valid) so a test can
 * inject the very same noise into the reference through torch.rand_like (:355).                     */
int d3pm_philox_uniform(float* u, int64_t rows, int K, int64_t pitch, uint64_t seed, uint64_t offset,
                        int64_t row_offset, d3pm_stream_t stream);

/* ---------------------------------------------------------------- fine-grained operators
 * q_posterior (:251-283) on an arbitrary log p(x0) (e.g. the one-hot truth of _train_loss :420).
 * log_x_start: [B*N][pitch_in], first K entries used (entry K is ignored, like the reference :278). */
int d3pm_q_posterior(const float* log_x_start, int64_t pitch_in, const int64_t* x_t, const int64_t* t,
                     const float* coef_table, float* post, int64_t pitch_out, int B, int N, int K, int T,
                     uint32_t* status, d3pm_stream_t stream);

/* log_sample_categorical (:354-359): x[row] = argmax_k(noise_k + logits[row][k]) over C classes.
 * noise_kind 0: `noise` holds Gumbel values; 1: `noise` holds uniforms u, g = -log(-log(u+1e-30)+1e-30);
 * 2: noise == NULL, Philox stream (seed, offset, row_offset) as in d3pm_fused_step.               */
int d3pm_gumbel_argmax(const float* logits, int64_t pitch_logits, const float* noise, int64_t pitch_noise,
                       int noise_kind, int64_t* x, float* gap, int64_t rows, int C, uint64_t seed,
                       uint64_t offset, int64_t row_offset, d3pm_stream_t stream);

/* index_to_log_onehot (:44-51): rows of C entries, 0 at x[row], log(1e-30) elsewhere. */
int d3pm_tokens_to_log_onehot(const int64_t* x, float* out, int64_t pitch, int64_t rows, int C,
                              uint32_t* status, d3pm_stream_t stream);

/* log_onehot_to_index (:53-54): first maximal class per token.
 * class_stride / token_stride / batch_stride in floats describe ANY [B, C, N] view:
 * token-major rows (class_stride 1) or the reference's contiguous layout (token_stride 1).        */
int d3pm_argmax_classes(const float* x, int64_t batch_stride, int64_t class_stride, int64_t token_stride,
                        int64_t* idx, int B, int C, int N, d3pm_stream_t stream);

/* Purity-prior reveal (the per-video loop of p_sample, :331-343).  Per video b: weights w_n = score[b][n] /
 * (max_n score[b][n] + 1e-10) where x_t[b][n] is [MASK], 0 elsewhere (:318-319, :334-337; score == NULL means
 * prior_rule 1, all ones); the n_reveal[b] positions with the largest w_n / q_n are revealed, x_out = x_t except
 * x_out[sel] = x_cand[sel] (:340-341).  q ~ Exp(1) is what torch.multinomial draws internally: `expo` injects it
 * ([B*N], parity tests), expo == NULL draws it from the Philox stream (seed, offset, row_offset).
 * revealed[b] = (#non-[MASK] in x_out) - (#non-[MASK] in x_t), the increment of `sampled[b]` (:342-343).
 * Ties (only the zero-weight positions, reached when a video holds fewer [MASK] tokens than n_reveal[b]) resolve
 * to the lowest position.  N <= 8192.                                                                          */
int d3pm_purity_select(const int64_t* x_t, const int64_t* x_cand, const float* score, const float* expo,
                       const int32_t* n_reveal, int64_t* x_out, int32_t* revealed, int B, int N, int K,
                       uint64_t seed, uint64_t offset, int64_t row_offset, d3pm_stream_t stream);

/* ---------------------------------------------------------------- training side (SURVEY.md §8 f1)
 * q_pred (:201-218, cumulative = 1, t wrapped modulo T+1) and q_pred_one_timestep (:185-199, cumulative = 0) on
 * rows of K+1 log-probabilities.  `sched` = the [8][T+1] schedule matrix of d3pm_build_coef_table.            */
int d3pm_q_pred(const float* in, int64_t pitch_in, const int64_t* t, const float* sched, int cumulative,
                float* out, int64_t pitch_out, int B, int N, int K, int T, d3pm_stream_t stream);

/* q_sample (:361-366) on integer tokens with the library's Philox noise: x_t[b][n] ~ q(x_t | x_0 = x0[b][n]) at the
 * per-video timestep t[b], i.e. index_to_log_onehot -> q_pred -> log_sample_categorical of the reference without any
 * of the three [B, K+1, N] tensors.  Bit-identical to d3pm_tokens_to_log_onehot + d3pm_q_pred + d3pm_gumbel_argmax
 * (Philox noise) with the same seed / offset / row_offset.  x0 in [0, K] (K = [MASK]); K % 4 == 0, K <= 8192.    */
int d3pm_q_sample_tokens(const int64_t* x0, const int64_t* t, const float* sched, int B, int N, int K, int T,
                         uint64_t seed, uint64_t offset, int64_t row_offset, int64_t* x_t, uint32_t* status,
                         d3pm_stream_t stream);

/* The variational-bound loss of _train_loss (:391-457) given the denoiser logits, the clean tokens x0, the noised
 * tokens x_t (from q_sample, :361-366) and t; and its gradient with respect to the logits.
 *   backward == 0: writes per-token tok_main / tok_aux (the caller sums them per video: kl_loss = sum tok_main,
 *                  vb_loss = kl_loss / pt + aux_weight * sum tok_aux / pt) and, optionally, x0_recon / xtm1_recon.
 *   backward == 1: recomputes the row and writes grad[row][k] = d( sum_b w_main[b] main_b + w_aux[b] auxc_b ) / d logits.
 *   backward == 2: both in ONE pass over the logits (forward outputs and the gradient for the given weights): the
 *                  training step's minimum of 16 KiB read + 16 KiB written per token.  A caller that learns the true
 *                  upstream gradient later rescales per video with d3pm_scale_rows (free when the factor is 1).
 * K in {1024, 2048, 4096} with >= 2048 rows runs the persistent TMA-pipelined kernel, other shapes one CTA per row.  */
typedef struct d3pm_train_desc {
  const float* logits;   /* [B*N][pitch] denoiser logits (first K valid); element type = logits_dtype */
  const int64_t* x0;     /* [B*N] in [0, K) */
  const int64_t* x_t;    /* [B*N] in [0, K] */
  const int64_t* t;      /* [B] */
  const float* coef_table;
  const float* w_main;   /* [B], backward only */
  const float* w_aux;    /* [B], backward only */
  float* tok_main;       /* [B*N], forward only */
  float* tok_aux;        /* [B*N], forward only */
  int64_t* x0_recon;     /* [B*N] arg-max of p(x0 | x_t), nullable (forward) */
  int64_t* xtm1_recon;   /* [B*N] arg-max of the model posterior, nullable (forward) */
  float* grad;           /* [B*N][pitch_grad], backward only; element type = logits_dtype */
  uint32_t* status;
  int32_t B, N, K, T;
  int64_t pitch, pitch_grad; /* in elements of logits_dtype */
  float mask_weight_masked, mask_weight_unmasked; /* mask_weight[0], mask_weight[1] (:423) */
  int32_t backward;
  d3pm_stream_t stream;
  int32_t logits_dtype;  /* D3PM_LOGITS_* of the logits AND grad rows (0 = F32).  16-bit logits are read as they lie in HBM and
                            widened in registers; the gradient is computed in fp32 and written in the same 16-bit type, rounded
                            to nearest even - bit-identical to running the fp32 path on logits.float() and casting grad with
                            tensor.to(dtype), at half the traffic each way.  Stream kernel only (K in {1024,2048,4096}, >= 2048
                            rows, both or neither of x0_recon / xtm1_recon; pitch and pitch_grad % 8 == 0, else
                            D3PM_ERR_ALIGN); other shapes return D3PM_ERR_UNSUPPORTED and the caller casts */
} d3pm_train_desc;

int d3pm_train_rows(const d3pm_train_desc* desc);

/* rows[b*N + n][0..K) *= factor[b]; videos whose factor is exactly 1.0f are skipped without touching memory. */
int d3pm_scale_rows(float* rows, int64_t pitch, const float* factor, int B, int N, int K, d3pm_stream_t stream);

/* ---------------------------------------------------------------- fused denoiser head + reverse step (SURVEY.md §8 f3)
 * Replaces the reference's prediction head `to_logits = LayerNorm(n_embd) + Linear(n_embd -> K)`
 * (transformer_utils.py:352-356, applied at :441) of BOTH denoiser passes of a step together with everything
 * d3pm_fused_step replaces: the [B, N, K] logits are produced tile by tile on the tensor cores (tcgen05, 3xTF32) and
 * consumed on chip; HBM sees the hidden states [B*N][D] and the tokens only.  n_embd D = 64 (the shipped config),
 * K in {1024, 2048, 4096}.
 *
 * d3pm_head_prepare: weight [K][D] / bias [K] (nullable) of the Linear -> `w_image` (d3pm_head_image_floats(K, D)
 * floats: per 128 classes the tf32 hi and lo parts of W * log2(e) in the 128-byte-swizzled K-major layout the tensor
 * core reads), `bias2` [K] = b * log2(e), and `stats` (2 floats, device): max_k ||W_k||_2 and max_k |b_k|, from which
 * the caller bounds |logit| <= stats[0] * (sqrt(D) * max|gamma| + ||beta||_2) + stats[1].  The fused kernel is valid
 * when that bound is <= (70 - ln K) / 2 (no -70 clamp of diffusion_transformer.py:236 can fire, so classifier-free
 * guidance commutes with the Linear); otherwise the caller must use the unfused path.                               */
int64_t d3pm_head_image_floats(int K, int D);
int d3pm_head_prepare(const float* weight, const float* bias, int K, int D, float* w_image, float* bias2, float* stats,
                      d3pm_stream_t stream);

#define D3PM_HEAD_STEP 0      /* sample x_{t-1} (production: Philox noise, thinned race, same stream as d3pm_fused_step) */
#define D3PM_HEAD_LOGITS 1    /* write the guidance-combined logits W (s a_c + (1-s) a_u) + b to logits_out (verification) */
#define D3PM_HEAD_REFERENCE 2 /* the same step on CUDA cores in plain fp32, exhaustive scoring (verification, slow) */

typedef struct d3pm_head_desc {
  const float* hidden_c;   /* [B*N][D] input of to_logits for the conditional pass (transformer_utils.py:441) */
  const float* hidden_u;   /* same for the unconditional pass; NULL = guidance off */
  const float* ln_weight;  /* [D] LayerNorm gamma, beta (to_logits[0]) */
  const float* ln_bias;
  const float* w_image;    /* from d3pm_head_prepare */
  const float* bias2;
  const int64_t* x_t;      /* [B*N] */
  const int64_t* t;        /* [B] */
  const float* coef_table;
  int64_t* x_prev;         /* [B*N] out (STEP, REFERENCE) */
  float* logits_out;       /* [B*N][K] out (LOGITS) */
  uint32_t* status;
  int32_t* redo_rows;      /* [B*N] scratch: rows the thinned race could not decide, rescored exhaustively */
  uint32_t* redo_count;    /* one word of scratch */
  int32_t B, N, K, T, D;
  int32_t mode;            /* D3PM_HEAD_* */
  float ln_eps, guidance_scale, thin_factor;
  float stat_slack;        /* > 0: the statistics pass (row maximum and sum of exponentials) runs in 1xTF32; the value bounds
                              |logit_1xTF32 - logit| in log2 units: 2^-9 * max_k ||W_k|| * ||a|| * log2(e) with ||a|| the largest
                              norm the combined LayerNorm output can have (d3pm_b200.head computes it).  Results do not change:
                              the thinning thresholds are widened by 2^slack and every score comes from exact 3xTF32 logits.
                              0 = statistics in 3xTF32 as well */
  uint64_t seed, offset;
  int64_t row_offset;
  d3pm_stream_t stream;
} d3pm_head_desc;

int d3pm_head_step(const d3pm_head_desc* desc);

/* ---------------------------------------------------------------- token -> video, first stage (SURVEY.md §8 f4)
 * VQVAE.decode (videogpt_vq_vae.py:53-56): h = post_vq_conv(shift_dim(F.embedding(tokens, codebook.embeddings), -1, 1)).
 * d3pm_decode_lut folds the codebook [K][E] and the 1x1x1 convolution (weight [C][E], bias [C] nullable) into
 * lut[K][C] once per weight version; d3pm_tokens_to_features then produces h as [B][C][N] (channels first, N = T*H*W, the
 * layout the decoder's Conv3d layers take) from the int64 [B][N] tokens this path samples.  Tokens outside [0, K) -- the
 * [MASK] class included -- set D3PM_STATUS_BAD_TOKEN and give zeros.                                                   */
int d3pm_decode_lut(const float* codebook, const float* conv_weight, const float* conv_bias, int K, int E, int C, float* lut,
                    d3pm_stream_t stream);
int d3pm_tokens_to_features(const int64_t* tokens, const float* lut, float* out, int B, int N, int K, int C,
                            uint32_t* status, d3pm_stream_t stream);

/* ---------------------------------------------------------------- token -> video, second stage (SURVEY.md §8 f4)
 * The reference's VQ-VAE `Decoder` (videogpt_vq_vae.py:258-287) in eval mode, layer by layer on channels-last activations
 * [B*T*H*W][C] (C % 32 == 0).  Every convolution / Linear is one call of d3pm_dec_conv, an implicit GEMM on the tensor cores
 * (tcgen05, 3xTF32 = fp32-grade, or terms = 1 for plain TF32 as cuDNN's default on the reference's GPU path);
 * d3pm_b200.decode.NativeDecoder holds the layer plan (which BatchNorm folds where, the parity classes of the transposed
 * convolutions).
 *
 * d3pm_dec_weight_image: w [nclass][N][Ktot] (row n = output channel, k = tap * Cin + input channel, contiguous) -> the
 * tf32 hi / lo parts in the swizzled K-major layout the kernel streams with bulk TMA; n_tile in {128, 256} is the tile
 * width d3pm_dec_conv will be called with, Ktot % 32 == 0.  d3pm_dec_image_floats gives the size of `image`.            */
#define D3PM_DEC_MAX_TAPS 32
#define D3PM_DEC_MAX_CLASSES 8
int64_t d3pm_dec_image_floats(int nclass, int N, int Ktot, int n_tile);
int d3pm_dec_weight_image(const float* w, int nclass, int N, int Ktot, int n_tile, float* image, d3pm_stream_t stream);

/* out[o(pos, class)][n] = act( bias[n] + residual[o][n] + sum_{tap, c} a(pos + tap_offset)[c] * w[class][n][tap * Cin + c] )
 * with a(q) = relu(x[q] * in_scale + in_shift) (or x[q] when in_scale == NULL) inside the input grid and 0 outside (the
 * reference's F.pad comes after the BatchNorm + ReLU: SamePadConv3d :302-310, SamePadConvTranspose3d :324-334), and
 * o(pos, class) = (b, t * stride_t + cls[class][0], h * stride_h + cls[class][1], w * stride_w + cls[class][2]) in the output
 * grid (T * stride_t, H * stride_h, W * stride_w): an ordinary convolution is one class with unit strides; a stride-2
 * transposed convolution is one class per output parity.  Replaces SamePadConv3d (:289-310), SamePadConvTranspose3d
 * (:312-334), the BatchNorm3d / ReLU pairs of AttentionResidualBlock (:120-136) and the four Linears of MultiHeadAttention
 * (model_utils.py:224-236).                                                                                          */
typedef struct d3pm_dec_conv_desc {
  const float* x;         /* [B*T*H*W][Cin] */
  const float* in_scale;  /* [Cin] or NULL */
  const float* in_shift;  /* [Cin], required with in_scale */
  const float* w_image;   /* from d3pm_dec_weight_image (same nclass, N = Nout, Ktot = ntaps * Cin, n_tile) */
  const float* bias;      /* [Nout rounded up to n_tile] or NULL */
  const float* residual;  /* rows like `out` (same ldo) or NULL */
  float* out;             /* [B*To*Ho*Wo][ldo], columns [0, Nout) written */
  int32_t B, T, H, W, Cin;
  int32_t ntaps, nclass;
  int32_t cta_pair;       /* 1: pairs of CTAs (tcgen05 cta_group::2, M = 256 per instruction) share a weight tile, each staging half of its
                             rows: half the L2 weight stream and half the shared-memory operand reads per CTA; same results */
  int32_t Nout;           /* Nout % 4 == 0 */
  int32_t out_transposed; /* 1: out[(row / ldo) * Nout * ldo + n * ldo + row % ldo] - planes of ldo consecutive output rows, channel-major
                             inside a plane (with ldo = H * W: the layout d3pm_dec_col2im reads); no residual */
  int64_t ldo;            /* row pitch of out in floats, % 4 == 0 (transposed: rows per plane, must divide the number of output rows) */
  int32_t stride_t, stride_h, stride_w;
  int32_t relu_out;
  int32_t terms;          /* 3: 3xTF32 (fp32-grade), 1: TF32 */
  int32_t n_tile;         /* 128 or 256 */
  int8_t tap[D3PM_DEC_MAX_CLASSES][D3PM_DEC_MAX_TAPS][4]; /* (dt, dh, dw, 0) per class and tap */
  int8_t cls[D3PM_DEC_MAX_CLASSES][4];                    /* (pt, ph, pw, 0) per class */
  d3pm_stream_t stream;
} d3pm_dec_conv_desc;
int d3pm_dec_conv(const d3pm_dec_conv_desc* desc);

/* h[row] = lut[tokens[row]] (lut from d3pm_decode_lut): the channels-last input of the decoder. */
int d3pm_dec_embed_rows(const int64_t* tokens, const float* lut, float* out, int64_t rows, int K, int C, uint32_t* status,
                        d3pm_stream_t stream);

/* AxialBlock's three attentions (videogpt_vq_vae.py:100-118; AxialAttention / scaled_dot_product_attention,
 * model_utils.py:318-336, :586-600) on qkv [M][3 axes (W, H, T)][q, k, v][heads][head_dim] -> att [M][3 axes][heads][head_dim];
 * softmax(softmax_scale * q k^T) v along one grid axis, fp32; softmax_scale <= 0 means 1 / sqrt(head_dim) (a caller whose
 * heads are zero-padded up to head_dim passes 1 / sqrt(true width)).  head_dim in {32, 64, 128}, T, H, W <= 32.        */
int d3pm_dec_axial_attention(const float* qkv, float* att, int B, int T, int H, int W, int heads, int head_dim,
                             float softmax_scale, d3pm_stream_t stream);

/* Last SamePadConvTranspose3d (kernel 4, stride (st, sh, sw) in {1, 2}, Cout <= 4): y_t [B*T][64 * Cout][H*W] holds the per-tap
 * contributions (row ((kt*4 + kh)*4 + kw) * Cout + c of plane (b, t), column = (h, w); from d3pm_dec_conv with one tap,
 * N = 64 * Cout, out_transposed = 1 and ldo = H*W); out [B][Cout][T*st][H*sh][W*sw] = bias + the contributions landing on
 * each voxel: the reference's video layout.                                                                             */
int d3pm_dec_col2im(const float* y_t, const float* bias, float* out, int B, int T, int H, int W, int Cout, int st, int sh, int sw,
                    d3pm_stream_t stream);

/* ---------------------------------------------------------------- denoiser self-attention (SURVEY.md §8 f3)
 * The self-attention of the denoiser's blocks, FullAttention (transformer_utils.py:24-62), after its q / k / v Linears and
 * before `proj`, forward only, fp32:
 *     y[b*N + n][h*hd + c] = sum_j softmax_j(scale * q_{b,n,h} . k_{b,j,h}) v_{b,j,h}[c]
 * with x_{b,n,h} = x[b*N + n][h*hd .. h*hd + hd).  q, k and v are rows of pitch_qkv floats as the three Linear outputs lie
 * ([B*T][C] each, pitch_qkv = C); y is written as [B*N][pitch_y], the layout of the reference's
 * `y.transpose(1, 2).contiguous().view(B, T, C)`.  The [N, N] scores never leave registers (no workspace), the softmax is
 * exact (running maximum per block of 32 keys, ex2.approx on pre-scaled scores).  The head-averaged attention map the
 * reference also returns is not produced.  head_dim = 4 (n_embd 64 / 16 heads, the shipped model) only: other values
 * return D3PM_ERR_UNSUPPORTED.  Any N >= 1 and B >= 1, heads <= 65535; pointers 16-byte aligned, pitches % 4 == 0.       */
typedef struct d3pm_attn_desc {
  const float* q;      /* [B*N][pitch_qkv] */
  const float* k;      /* [B*N][pitch_qkv] */
  const float* v;      /* [B*N][pitch_qkv] */
  float* y;            /* [B*N][pitch_y] out, columns [0, heads * head_dim) written */
  int32_t B, N, heads, head_dim;
  int64_t pitch_qkv, pitch_y; /* in floats, >= heads * head_dim */
  float scale;         /* softmax scale, 1 / sqrt(head_dim) in the reference */
  d3pm_stream_t stream;
} d3pm_attn_desc;

int d3pm_self_attention(const d3pm_attn_desc* desc);

/* ---------------------------------------------------------------- denoiser cross-attention (SURVEY.md §8 f3)
 * The cross-attention of the denoiser's blocks, CrossAttention (the blocks' attn2 over the M condition tokens), after its
 * q / k / v Linears and before `proj`, forward only, fp32:
 *     y[b*N + n][h*hd + c] = sum_{j < M} softmax_j(scale * q_{b,n,h} . k_{b,j,h}) v_{b,j,h}[c]
 * with q_{b,n,h} = q[b*N + n][h*hd .. h*hd + hd) and k_{b,j,h} = k[b*M + j][h*hd .. h*hd + hd) (v alike).  q is the output of
 * `query(x)` ([B*N][pitch_q]); k and v are the outputs of `key(encoder_output)` and `value(encoder_output)` ([B*M][pitch_kv]
 * each), read in place; y is written as [B*N][pitch_y], the layout `proj` takes.  The numerics of d3pm_self_attention: the
 * [N, M] scores never leave registers (no workspace), exact running maximum per block of keys, ex2.approx on pre-scaled
 * scores, Kahan-compensated block sums.  The head-averaged attention map the reference also returns is not produced.
 * head_dim = 4 only (other values return D3PM_ERR_UNSUPPORTED).  Any N, M >= 1 and B >= 1, heads <= 65535; pointers
 * 16-byte aligned, pitches % 4 == 0 and >= heads * head_dim.  Launches on `stream` only (CUDA-graph capturable).        */
typedef struct d3pm_cross_attn_desc {
  const float* q;      /* [B*N][pitch_q] */
  const float* k;      /* [B*M][pitch_kv] */
  const float* v;      /* [B*M][pitch_kv] */
  float* y;            /* [B*N][pitch_y] out, columns [0, heads * head_dim) written */
  int32_t B, N, M, heads, head_dim;
  int64_t pitch_q, pitch_kv, pitch_y; /* in floats, >= heads * head_dim */
  float scale;         /* softmax scale, 1 / sqrt(head_dim) in the reference */
  d3pm_stream_t stream;
} d3pm_cross_attn_desc;

int d3pm_cross_attention(const d3pm_cross_attn_desc* desc);

/* ---------------------------------------------------------------- host-buffer entry points
 * For a caller whose denoiser output lives in HOST memory (the reference's CPU tensors; bench.py's `e2e`): a handle owns
 * the device staging buffers for one batch shape, a copy stream and a compute stream.  `run` copies the inputs up in
 * chunks of whole videos, runs d3pm_fused_step (production Philox sampling) on each chunk while the next one is on the
 * bus, copies the int64 tokens down into x_prev and RETURNS WHEN THEY ARE THERE (the one synchronous entry point of the
 * library).  Host buffers should be page-locked (cudaHostRegister / torch pin_memory) for the copies to overlap.
 * coef_table (and the head weights of the second form) stay DEVICE pointers on `device`: they are per-model constants.
 * status_out (nullable) receives the OR of D3PM_STATUS_* of this call.
 *   D = 0: the handle stages logits [B*N][K] (+ the unconditional tensor when guidance != 0)   -> d3pm_host_step_run
 *   D = 64: it stages the hidden states [B*N][D] that enter to_logits                           -> d3pm_host_head_step_run
 * chunks <= 0 picks the default (4 when B % 4 == 0 and a chunk holds >= 1024 rows, else 1).                          */
typedef struct d3pm_host_step d3pm_host_step;
int d3pm_host_step_create(d3pm_host_step** out, int device, int B, int N, int K, int T, int D, int guidance, int chunks);
int d3pm_host_step_destroy(d3pm_host_step* h);
int64_t d3pm_host_step_h2d_bytes(const d3pm_host_step* h); /* bytes one run moves host -> device */
int64_t d3pm_host_step_d2h_bytes(const d3pm_host_step* h); /* and device -> host */
/* Element type of the HOST logits of a D = 0 handle (D3PM_LOGITS_*; default F32): float16 / bfloat16 rows cross the bus at half
 * the bytes and are stepped in place (d3pm_step_desc.logits_dtype); logits_c / logits_u of d3pm_host_step_run then point at
 * 16-bit rows.  K % 8 == 0.                                                                                              */
int d3pm_host_step_set_logits_dtype(d3pm_host_step* h, int logits_dtype);
int d3pm_host_step_run(d3pm_host_step* h, const float* logits_c, const float* logits_u, const int64_t* x_t, const int64_t* t,
                       const float* coef_table, float guidance_scale, uint64_t seed, uint64_t offset, int64_t row_offset,
                       int64_t* x_prev, uint32_t* status_out);
int d3pm_host_head_step_run(d3pm_host_step* h, const float* hidden_c, const float* hidden_u, const int64_t* x_t,
                            const int64_t* t, const float* ln_weight, const float* ln_bias, float ln_eps,
                            const float* w_image, const float* bias2, const float* coef_table, float guidance_scale,
                            float stat_slack, uint64_t seed, uint64_t offset, int64_t row_offset, int64_t* x_prev,
                            uint32_t* status_out);

/* [B, C, N] contiguous (reference layout) -> token-major rows [B*N][pitch]. */
int d3pm_to_token_major(const float* src, float* dst, int64_t pitch, int B, int C, int N,
                        d3pm_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* D3PM_B200_H */
