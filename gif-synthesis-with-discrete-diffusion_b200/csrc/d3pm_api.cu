// C ABI of libd3pm_b200.so (see include/d3pm_b200.h).  Host side only validates, picks a kernel
// instantiation and launches on the caller's stream; nothing here allocates, synchronises or keeps
// state beyond a thread-local error string -- except the explicit d3pm_host_step handle at the end of
// the file, which owns device staging buffers and two streams for callers whose inputs are HOST buffers.
#include <cstdarg>
#include <cstdio>
#include <type_traits>

#include "d3pm_host.h"
#include "d3pm_ops.cuh"
#include "d3pm_step_rows.cuh"
#include "d3pm_step_stream.cuh"
#include "d3pm_train_rows.cuh"
#include "d3pm_train_stream.cuh"
#include "d3pm_head_step.cuh"

namespace {
thread_local char g_err[512] = "";
}  // namespace

namespace d3pm {
namespace host {

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int check_launch(const char* what) {
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(D3PM_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
  return D3PM_OK;
}

}  // namespace host
}  // namespace d3pm

namespace {

using d3pm::host::check_launch;
using d3pm::host::DeviceGuard;
using d3pm::host::fail;

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

constexpr int64_t kMaxGrid = 2147483647LL;

template <int V, bool HAS_U>
void launch_rows(const d3pm::StepParams& p, cudaStream_t s) {
  const dim3 grid(static_cast<unsigned>(p.rows)), block(d3pm::kRowThreads);
  if (p.sample_mode == D3PM_SAMPLE_PHILOX && p.post == nullptr && p.recon == nullptr && p.sharpen == nullptr)
    d3pm::step_rows_kernel<V, HAS_U, true><<<grid, block, 0, s>>>(p);
  else
    d3pm::step_rows_kernel<V, HAS_U, false><<<grid, block, 0, s>>>(p);
}

template <int V>
void launch_train(const d3pm::TrainParams& p, bool backward, cudaStream_t s) {
  const dim3 grid(static_cast<unsigned>(p.rows)), block(d3pm::kRowThreads);
  if (backward) d3pm::train_rows_kernel<V, true><<<grid, block, 0, s>>>(p);
  else d3pm::train_rows_kernel<V, false><<<grid, block, 0, s>>>(p);
}

// launch(std::integral_constant<int, V>) with V = float4 chunks per thread of a one-CTA-per-row kernel: the fewest of
// 1, 2, 4, 8 that cover K classes
template <typename Launch>
void with_row_chunks(int K, Launch launch) {
  const int chunks = (K / 4 + d3pm::kRowThreads - 1) / d3pm::kRowThreads;
  if (chunks <= 1) launch(std::integral_constant<int, 1>{});
  else if (chunks <= 2) launch(std::integral_constant<int, 2>{});
  else if (chunks <= 4) launch(std::integral_constant<int, 4>{});
  else launch(std::integral_constant<int, 8>{});
}

}  // namespace

extern "C" {

int d3pm_version(void) { return D3PM_VERSION; }

const char* d3pm_last_error(void) { return g_err; }

int d3pm_build_coef_table(const float* sched, int T, int K, float* table, d3pm_stream_t stream) {
  if (sched == nullptr || table == nullptr) return fail(D3PM_ERR_INVALID, "coef_table: null pointer");
  const DeviceGuard on_device(table);
  if (T <= 0 || K <= 0) return fail(D3PM_ERR_INVALID, "coef_table: T=%d K=%d must be positive", T, K);
  if (!aligned16(table)) return fail(D3PM_ERR_ALIGN, "coef_table: table must be 16-byte aligned");
  d3pm::coef_table_kernel<<<(T + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(sched, T, K, table);
  return check_launch("coef_table");
}

int d3pm_fused_step(const d3pm_step_desc* d) {
  if (d == nullptr) return fail(D3PM_ERR_INVALID, "fused_step: null descriptor");
  const DeviceGuard on_device(d->logits_c);
  if (d->logits_c == nullptr || d->x_t == nullptr || d->t == nullptr || d->coef_table == nullptr)
    return fail(D3PM_ERR_INVALID, "fused_step: logits_c, x_t, t and coef_table are required");
  if (d->B <= 0 || d->N <= 0 || d->K <= 0 || d->T <= 0)
    return fail(D3PM_ERR_INVALID, "fused_step: B=%d N=%d K=%d T=%d must be positive", d->B, d->N, d->K, d->T);
  if (d->K % 4 != 0 || d->K > 8192)
    return fail(D3PM_ERR_UNSUPPORTED, "fused_step: K=%d must be a multiple of 4 and <= 8192", d->K);
  const int64_t rows = static_cast<int64_t>(d->B) * d->N;
  if (rows > kMaxGrid) return fail(D3PM_ERR_UNSUPPORTED, "fused_step: B*N=%lld exceeds the grid limit", (long long)rows);
  if (d->logits_dtype < D3PM_LOGITS_F32 || d->logits_dtype > D3PM_LOGITS_BF16)
    return fail(D3PM_ERR_INVALID, "fused_step: unknown logits_dtype %d", d->logits_dtype);
  const int pitch_mult = d->logits_dtype == D3PM_LOGITS_F32 ? 4 : 8;  // rows start on 16-byte boundaries
  if (d->pitch_logits < d->K || d->pitch_logits % pitch_mult != 0)
    return fail(D3PM_ERR_ALIGN, "fused_step: pitch_logits=%lld must be >= K and a multiple of %d", (long long)d->pitch_logits, pitch_mult);
  if (!aligned16(d->logits_c) || !aligned16(d->logits_u) || !aligned16(d->coef_table))
    return fail(D3PM_ERR_ALIGN, "fused_step: logits and coef_table must be 16-byte aligned");
  const int mode = d->sample_mode;
  if (mode < D3PM_SAMPLE_NONE || mode > D3PM_SAMPLE_PHILOX_EXACT)
    return fail(D3PM_ERR_INVALID, "fused_step: unknown sample_mode %d", mode);
  if (mode == D3PM_SAMPLE_NONE && d->post == nullptr && d->recon == nullptr && d->score == nullptr)
    return fail(D3PM_ERR_INVALID, "fused_step: nothing to do (no sampling and no output requested)");
  if (d->sample_from != D3PM_FROM_POSTERIOR && d->sample_from != D3PM_FROM_RECON)
    return fail(D3PM_ERR_INVALID, "fused_step: unknown sample_from %d", d->sample_from);
  if (d->sharpen != nullptr && (d->sample_from != D3PM_FROM_RECON || mode == D3PM_SAMPLE_PHILOX || mode == D3PM_SAMPLE_NONE))
    return fail(D3PM_ERR_INVALID, "fused_step: sharpen needs D3PM_FROM_RECON with GUMBEL or PHILOX_EXACT sampling");
  if (d->sample_from == D3PM_FROM_RECON && d->post != nullptr)
    return fail(D3PM_ERR_INVALID, "fused_step: post is the q_posterior output; it cannot be combined with D3PM_FROM_RECON");
  if (mode != D3PM_SAMPLE_NONE && d->x_prev == nullptr)
    return fail(D3PM_ERR_INVALID, "fused_step: x_prev is required when sampling");
  if (mode == D3PM_SAMPLE_GUMBEL) {
    if (d->gumbel == nullptr) return fail(D3PM_ERR_INVALID, "fused_step: D3PM_SAMPLE_GUMBEL needs the gumbel tensor");
    if (d->pitch_gumbel < d->K + 1 || d->pitch_gumbel % 4 != 0 || !aligned16(d->gumbel))
      return fail(D3PM_ERR_ALIGN, "fused_step: gumbel rows need pitch >= K+1, pitch %% 4 == 0, 16-byte base");
  }
  if (d->post != nullptr || d->recon != nullptr) {
    if (d->pitch_out < d->K + 1 || d->pitch_out % 4 != 0 || !aligned16(d->post) || !aligned16(d->recon))
      return fail(D3PM_ERR_ALIGN, "fused_step: output rows need pitch >= K+1, pitch %% 4 == 0, 16-byte base");
  }
  if (d->gap != nullptr && (mode == D3PM_SAMPLE_NONE || mode == D3PM_SAMPLE_PHILOX))
    return fail(D3PM_ERR_INVALID, "fused_step: gap is produced only by the GUMBEL and PHILOX_EXACT modes");
  if (d->thin_factor < 0.f) return fail(D3PM_ERR_INVALID, "fused_step: thin_factor must be >= 0");

  d3pm::StepParams p;
  p.logits_c = d->logits_c, p.logits_u = d->logits_u, p.x_t = d->x_t, p.t = d->t, p.coef_table = d->coef_table;
  p.gumbel = d->gumbel, p.x_prev = d->x_prev, p.post = d->post, p.recon = d->recon, p.gap = d->gap;
  p.status = d->status;
  p.B = d->B, p.N = d->N, p.K = d->K, p.T = d->T;
  p.pitch_logits = d->pitch_logits, p.pitch_gumbel = d->pitch_gumbel, p.pitch_out = d->pitch_out;
  p.guidance_scale = d->guidance_scale, p.sample_mode = mode, p.gumbel_is_uniform = d->gumbel_is_uniform;
  p.seed = d->seed, p.offset = d->offset, p.row_offset = d->row_offset, p.thin_factor = d->thin_factor;
  p.rows = rows;
  p.sample_from = d->sample_from, p.score = d->score, p.sharpen = d->sharpen;
  p.winner_post = d->winner_post;
  p.logits_dtype = d->logits_dtype;
  d3pm::expand_round_keys(p.seed, p.keys);
  const cudaStream_t s = static_cast<cudaStream_t>(d->stream);

  if (d->kernel < D3PM_KERNEL_AUTO || d->kernel > D3PM_KERNEL_STREAM)
    return fail(D3PM_ERR_INVALID, "fused_step: unknown kernel selector %d", d->kernel);
  const bool can_stream = d3pm::stream_kernel_supports(p) && rows <= d3pm::stream_kernel_max_rows();
  if (d->winner_post != nullptr && !(can_stream && d->kernel != D3PM_KERNEL_ROWS))
    return fail(D3PM_ERR_UNSUPPORTED, "fused_step: winner_post is an output of the stream kernel (PHILOX sampling, K in {1024,2048,4096}); "
                                      "the rows kernel offers the whole posterior row (post) instead");
  if (d->logits_dtype != D3PM_LOGITS_F32 && !(can_stream && d->kernel != D3PM_KERNEL_ROWS))
    return fail(D3PM_ERR_UNSUPPORTED, "fused_step: 16-bit logits are read by the stream kernel only (PHILOX sampling of the posterior, no row "
                                      "outputs, K in {1024,2048,4096}); cast to float for the other modes");
  if (d->kernel == D3PM_KERNEL_STREAM && !can_stream)
    return fail(D3PM_ERR_UNSUPPORTED, "fused_step: the stream kernel needs PHILOX sampling, no outputs and K in {1024,2048,4096}");
  if (d->kernel == D3PM_KERNEL_STREAM || (d->kernel == D3PM_KERNEL_AUTO && can_stream &&
                                            (rows >= d3pm::kStreamMinRows || d->winner_post != nullptr || d->logits_dtype != D3PM_LOGITS_F32))) {
    const int rc = d3pm::launch_step_stream(p, s);
    if (rc != D3PM_OK) return fail(rc, "fused_step: stream kernel launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    return check_launch("fused_step(stream)");
  }
  with_row_chunks(d->K, [&](auto v) {
    if (p.logits_u != nullptr) launch_rows<decltype(v)::value, true>(p, s);
    else launch_rows<decltype(v)::value, false>(p, s);
  });
  return check_launch("fused_step");
}

int d3pm_philox_uniform(float* u, int64_t rows, int K, int64_t pitch, uint64_t seed, uint64_t offset,
                        int64_t row_offset, d3pm_stream_t stream) {
  if (u == nullptr || rows <= 0 || K <= 0 || pitch < K + 1 || rows > kMaxGrid)
    return fail(D3PM_ERR_INVALID, "philox_uniform: bad arguments (rows=%lld K=%d pitch=%lld)", (long long)rows, K, (long long)pitch);
  const DeviceGuard on_device(u);
  d3pm::philox_uniform_kernel<<<static_cast<unsigned>(rows), d3pm::kOpThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      u, K, pitch, seed, offset, row_offset);
  return check_launch("philox_uniform");
}

int d3pm_q_posterior(const float* log_x_start, int64_t pitch_in, const int64_t* x_t, const int64_t* t,
                     const float* coef_table, float* post, int64_t pitch_out, int B, int N, int K, int T,
                     uint32_t* status, d3pm_stream_t stream) {
  if (log_x_start == nullptr || x_t == nullptr || t == nullptr || coef_table == nullptr || post == nullptr)
    return fail(D3PM_ERR_INVALID, "q_posterior: null pointer");
  const DeviceGuard on_device(post);
  if (B <= 0 || N <= 0 || K <= 0 || T <= 0) return fail(D3PM_ERR_INVALID, "q_posterior: sizes must be positive");
  const int64_t rows = static_cast<int64_t>(B) * N;
  if (rows > kMaxGrid) return fail(D3PM_ERR_UNSUPPORTED, "q_posterior: B*N too large");
  if (pitch_in < K || pitch_out < K + 1) return fail(D3PM_ERR_INVALID, "q_posterior: pitch_in >= K and pitch_out >= K+1 required");
  if (!aligned16(coef_table)) return fail(D3PM_ERR_ALIGN, "q_posterior: coef_table must be 16-byte aligned");
  d3pm::q_posterior_rows_kernel<<<static_cast<unsigned>(rows), d3pm::kOpThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      log_x_start, pitch_in, x_t, t, coef_table, post, pitch_out, N, K, T, status);
  return check_launch("q_posterior");
}

int d3pm_gumbel_argmax(const float* logits, int64_t pitch_logits, const float* noise, int64_t pitch_noise,
                       int noise_kind, int64_t* x, float* gap, int64_t rows, int C, uint64_t seed,
                       uint64_t offset, int64_t row_offset, d3pm_stream_t stream) {
  if (logits == nullptr || x == nullptr || rows <= 0 || C <= 0 || pitch_logits < C || rows > kMaxGrid)
    return fail(D3PM_ERR_INVALID, "gumbel_argmax: bad arguments");
  const DeviceGuard on_device(x);
  if (noise_kind < 0 || noise_kind > 2) return fail(D3PM_ERR_INVALID, "gumbel_argmax: noise_kind %d", noise_kind);
  if (noise_kind != 2 && (noise == nullptr || pitch_noise < C))
    return fail(D3PM_ERR_INVALID, "gumbel_argmax: noise tensor required for noise_kind %d", noise_kind);
  const dim3 grid(static_cast<unsigned>(rows)), block(d3pm::kOpThreads);
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (noise_kind == 0)
    d3pm::gumbel_argmax_rows_kernel<0><<<grid, block, 0, s>>>(logits, pitch_logits, noise, pitch_noise, x, gap, C, seed, offset, row_offset);
  else if (noise_kind == 1)
    d3pm::gumbel_argmax_rows_kernel<1><<<grid, block, 0, s>>>(logits, pitch_logits, noise, pitch_noise, x, gap, C, seed, offset, row_offset);
  else if (gap == nullptr && C <= 8193)
    d3pm::gumbel_argmax_thin_rows_kernel<<<grid, block, 0, s>>>(logits, pitch_logits, x, C, seed, offset, row_offset);
  else
    d3pm::gumbel_argmax_rows_kernel<2><<<grid, block, 0, s>>>(logits, pitch_logits, nullptr, 0, x, gap, C, seed, offset, row_offset);
  return check_launch("gumbel_argmax");
}

int d3pm_tokens_to_log_onehot(const int64_t* x, float* out, int64_t pitch, int64_t rows, int C, uint32_t* status,
                              d3pm_stream_t stream) {
  if (x == nullptr || out == nullptr || rows <= 0 || C <= 0 || pitch < C || rows > kMaxGrid)
    return fail(D3PM_ERR_INVALID, "tokens_to_log_onehot: bad arguments");
  const DeviceGuard on_device(out);
  d3pm::tokens_to_log_onehot_kernel<<<static_cast<unsigned>(rows), d3pm::kOpThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      x, out, pitch, C, status);
  return check_launch("tokens_to_log_onehot");
}

int d3pm_argmax_classes(const float* x, int64_t batch_stride, int64_t class_stride, int64_t token_stride,
                        int64_t* idx, int B, int C, int N, d3pm_stream_t stream) {
  if (x == nullptr || idx == nullptr || B <= 0 || C <= 0 || N <= 0)
    return fail(D3PM_ERR_INVALID, "argmax_classes: bad arguments");
  const DeviceGuard on_device(idx);
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t rows = static_cast<int64_t>(B) * N;
  if (class_stride == 1) {
    if (rows > kMaxGrid) return fail(D3PM_ERR_UNSUPPORTED, "argmax_classes: B*N too large");
    d3pm::argmax_rows_kernel<<<static_cast<unsigned>(rows), d3pm::kOpThreads, 0, s>>>(x, batch_stride, token_stride, idx, C, N);
  } else {
    if (B > 65535) return fail(D3PM_ERR_UNSUPPORTED, "argmax_classes: B > 65535 in the strided layout");
    const dim3 grid((N + d3pm::kOpThreads - 1) / d3pm::kOpThreads, B);
    d3pm::argmax_strided_kernel<<<grid, d3pm::kOpThreads, 0, s>>>(x, batch_stride, class_stride, token_stride, idx, C, N);
  }
  return check_launch("argmax_classes");
}

int d3pm_purity_select(const int64_t* x_t, const int64_t* x_cand, const float* score, const float* expo,
                       const int32_t* n_reveal, int64_t* x_out, int32_t* revealed, int B, int N, int K, uint64_t seed,
                       uint64_t offset, int64_t row_offset, d3pm_stream_t stream) {
  if (x_t == nullptr || x_cand == nullptr || n_reveal == nullptr || x_out == nullptr)
    return fail(D3PM_ERR_INVALID, "purity_select: x_t, x_cand, n_reveal and x_out are required");
  const DeviceGuard on_device(x_out);
  if (B <= 0 || N <= 0 || K <= 0) return fail(D3PM_ERR_INVALID, "purity_select: sizes must be positive");
  if (N > d3pm::kPurityMaxN) return fail(D3PM_ERR_UNSUPPORTED, "purity_select: N=%d exceeds %d", N, d3pm::kPurityMaxN);
  int n2 = 1;
  while (n2 < N) n2 <<= 1;
  const size_t smem = static_cast<size_t>(n2) * sizeof(unsigned long long);
  if (cudaFuncSetAttribute(d3pm::purity_select_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) != cudaSuccess)
    return fail(D3PM_ERR_CUDA, "purity_select: %s", cudaGetErrorString(cudaGetLastError()));
  d3pm::purity_select_kernel<<<static_cast<unsigned>(B), d3pm::kPurityThreads, smem, static_cast<cudaStream_t>(stream)>>>(
      x_t, x_cand, score, expo, n_reveal, x_out, revealed, N, n2, K, seed, offset, row_offset);
  return check_launch("purity_select");
}

int d3pm_q_pred(const float* in, int64_t pitch_in, const int64_t* t, const float* sched, int cumulative, float* out,
                int64_t pitch_out, int B, int N, int K, int T, d3pm_stream_t stream) {
  if (in == nullptr || t == nullptr || sched == nullptr || out == nullptr) return fail(D3PM_ERR_INVALID, "q_pred: null pointer");
  const DeviceGuard on_device(out);
  if (B <= 0 || N <= 0 || K <= 0 || T <= 0 || pitch_in < K + 1 || pitch_out < K + 1)
    return fail(D3PM_ERR_INVALID, "q_pred: bad sizes (rows need K+1 entries)");
  const int64_t rows = static_cast<int64_t>(B) * N;
  if (rows > kMaxGrid) return fail(D3PM_ERR_UNSUPPORTED, "q_pred: B*N too large");
  d3pm::q_pred_rows_kernel<<<static_cast<unsigned>(rows), d3pm::kRowThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      in, pitch_in, t, 0, sched, T, K, N, cumulative ? 1 : 0, out, pitch_out);
  return check_launch("q_pred");
}

int d3pm_q_sample_tokens(const int64_t* x0, const int64_t* t, const float* sched, int B, int N, int K, int T, uint64_t seed,
                         uint64_t offset, int64_t row_offset, int64_t* x_t, uint32_t* status, d3pm_stream_t stream) {
  if (x0 == nullptr || t == nullptr || sched == nullptr || x_t == nullptr) return fail(D3PM_ERR_INVALID, "q_sample_tokens: null pointer");
  const DeviceGuard on_device(x_t);
  if (B <= 0 || N <= 0 || K <= 0 || T <= 0) return fail(D3PM_ERR_INVALID, "q_sample_tokens: sizes must be positive");
  if (K % 4 != 0 || K > 8192) return fail(D3PM_ERR_UNSUPPORTED, "q_sample_tokens: K=%d must be a multiple of 4 and <= 8192", K);
  const int64_t rows = static_cast<int64_t>(B) * N;
  const int64_t grid = (rows + d3pm::kQSampleWarps - 1) / d3pm::kQSampleWarps;
  if (grid > kMaxGrid) return fail(D3PM_ERR_UNSUPPORTED, "q_sample_tokens: B*N too large");
  d3pm::q_sample_tokens_kernel<<<static_cast<unsigned>(grid), 32 * d3pm::kQSampleWarps, 0, static_cast<cudaStream_t>(stream)>>>(
      x0, t, sched, T, K, N, rows, seed, offset, row_offset, x_t, status);
  return check_launch("q_sample_tokens");
}

int d3pm_train_rows(const d3pm_train_desc* d) {
  if (d == nullptr) return fail(D3PM_ERR_INVALID, "train_rows: null descriptor");
  const DeviceGuard on_device(d->logits);
  if (d->logits == nullptr || d->x0 == nullptr || d->x_t == nullptr || d->t == nullptr || d->coef_table == nullptr)
    return fail(D3PM_ERR_INVALID, "train_rows: logits, x0, x_t, t and coef_table are required");
  if (d->B <= 0 || d->N <= 0 || d->K <= 0 || d->T <= 0) return fail(D3PM_ERR_INVALID, "train_rows: sizes must be positive");
  if (d->K % 4 != 0 || d->K > 8192) return fail(D3PM_ERR_UNSUPPORTED, "train_rows: K=%d must be a multiple of 4 and <= 8192", d->K);
  if (d->logits_dtype < D3PM_LOGITS_F32 || d->logits_dtype > D3PM_LOGITS_BF16)
    return fail(D3PM_ERR_INVALID, "train_rows: unknown logits_dtype %d", d->logits_dtype);
  const int pitch_mult = d->logits_dtype == D3PM_LOGITS_F32 ? 4 : 8;  // rows start on 16-byte boundaries
  if (d->pitch < d->K || d->pitch % pitch_mult != 0 || !aligned16(d->logits) || !aligned16(d->coef_table))
    return fail(D3PM_ERR_ALIGN, "train_rows: logits rows need pitch >= K, pitch %% %d == 0, 16-byte base", pitch_mult);
  const int64_t rows = static_cast<int64_t>(d->B) * d->N;
  if (rows > kMaxGrid) return fail(D3PM_ERR_UNSUPPORTED, "train_rows: B*N too large");
  if (d->backward < 0 || d->backward > 2) return fail(D3PM_ERR_INVALID, "train_rows: backward must be 0, 1 or 2");
  if (d->backward != 0) {
    if (d->grad == nullptr || d->w_main == nullptr || d->w_aux == nullptr)
      return fail(D3PM_ERR_INVALID, "train_rows: the gradient needs grad, w_main and w_aux");
    if (d->pitch_grad < d->K || d->pitch_grad % pitch_mult != 0 || !aligned16(d->grad))
      return fail(D3PM_ERR_ALIGN, "train_rows: grad rows need pitch >= K, pitch %% %d == 0, 16-byte base", pitch_mult);
  }
  if (d->backward != 1 && (d->tok_main == nullptr || d->tok_aux == nullptr))
    return fail(D3PM_ERR_INVALID, "train_rows: the forward outputs need tok_main and tok_aux");
  d3pm::TrainParams p;
  p.logits = d->logits, p.x0 = d->x0, p.x_t = d->x_t, p.t = d->t, p.coef_table = d->coef_table;
  p.w_main = d->w_main, p.w_aux = d->w_aux, p.tok_main = d->tok_main, p.tok_aux = d->tok_aux;
  p.x0_recon = d->x0_recon, p.xtm1_recon = d->xtm1_recon, p.grad = d->grad, p.status = d->status;
  p.B = d->B, p.N = d->N, p.K = d->K, p.T = d->T, p.pitch = d->pitch, p.pitch_grad = d->pitch_grad;
  p.mask_weight_masked = d->mask_weight_masked, p.mask_weight_unmasked = d->mask_weight_unmasked;
  p.rows = rows;
  p.logits_dtype = d->logits_dtype;
  if (d->backward == 0) p.grad = nullptr;  // a forward pass writes no gradient: its pitch does not matter
  const cudaStream_t s = static_cast<cudaStream_t>(d->stream);
  const bool can_stream = d3pm::train_stream_supports(p) && (d->x0_recon == nullptr) == (d->xtm1_recon == nullptr);
  if (d->logits_dtype != D3PM_LOGITS_F32 && !can_stream)
    return fail(D3PM_ERR_UNSUPPORTED, "train_rows: 16-bit logits are read by the stream kernel only (K in {1024,2048,4096}, "
                                      ">= 2048 rows, both or neither of x0_recon / xtm1_recon); cast to float for other shapes");
  if (can_stream) {
    if (d->backward == 1) p.tok_main = nullptr, p.tok_aux = nullptr, p.x0_recon = nullptr, p.xtm1_recon = nullptr;
    const int rc = d3pm::launch_train_stream(p, d->backward != 0, s);
    if (rc != D3PM_OK) return fail(rc, "train_rows: stream kernel launch failed: %s", cudaGetErrorString(cudaGetLastError()));
    return check_launch("train_rows(stream)");
  }
  for (int pass = 0; pass < 2; ++pass) {  // one CTA per row: forward and gradient are separate launches
    const bool bwd = pass == 1;
    if ((bwd && d->backward == 0) || (!bwd && d->backward == 1)) continue;
    with_row_chunks(d->K, [&](auto v) { launch_train<decltype(v)::value>(p, bwd, s); });
  }
  return check_launch("train_rows");
}

int d3pm_scale_rows(float* rows, int64_t pitch, const float* factor, int B, int N, int K, d3pm_stream_t stream) {
  if (rows == nullptr || factor == nullptr || B <= 0 || N <= 0 || K <= 0 || K % 4 != 0 || pitch < K || pitch % 4 != 0 || !aligned16(rows))
    return fail(D3PM_ERR_INVALID, "scale_rows: bad arguments");
  const DeviceGuard on_device(rows);
  const int64_t n = static_cast<int64_t>(B) * N;
  if (n > kMaxGrid) return fail(D3PM_ERR_UNSUPPORTED, "scale_rows: B*N too large");
  d3pm::scale_rows_kernel<<<static_cast<unsigned>(n), 256, 0, static_cast<cudaStream_t>(stream)>>>(rows, pitch, factor, N, K);
  return check_launch("scale_rows");
}

int64_t d3pm_head_image_floats(int K, int D) {
  if (D != 64 || K <= 0 || K % 1024 != 0) return 0;
  return static_cast<int64_t>(K / d3pm::head::kChunk) * d3pm::head::Geo<64>::kChunkFloats;
}

int d3pm_head_prepare(const float* weight, const float* bias, int K, int D, float* w_image, float* bias2, float* stats,
                      d3pm_stream_t stream) {
  if (weight == nullptr || w_image == nullptr || bias2 == nullptr || stats == nullptr)
    return fail(D3PM_ERR_INVALID, "head_prepare: null pointer");
  const DeviceGuard on_device(w_image);
  if (D != 64) return fail(D3PM_ERR_UNSUPPORTED, "head_prepare: n_embd D=%d (the fused head is built for D = 64)", D);
  if (K != 1024 && K != 2048 && K != 4096) return fail(D3PM_ERR_UNSUPPORTED, "head_prepare: K=%d must be 1024, 2048 or 4096", K);
  if (!aligned16(weight) || !aligned16(w_image) || !aligned16(bias2))
    return fail(D3PM_ERR_ALIGN, "head_prepare: weight, w_image and bias2 must be 16-byte aligned");
  const cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (cudaMemsetAsync(stats, 0, 2 * sizeof(float), s) != cudaSuccess) return fail(D3PM_ERR_CUDA, "head_prepare: memset failed");
  const int threads = K * (D / 4);
  d3pm::head::head_prepare_kernel<64><<<(threads + 255) / 256, 256, 0, s>>>(weight, bias, K, w_image, bias2,
                                                                            reinterpret_cast<uint32_t*>(stats));
  return check_launch("head_prepare");
}

int d3pm_head_step(const d3pm_head_desc* d) {
  namespace H = d3pm::head;
  if (d == nullptr) return fail(D3PM_ERR_INVALID, "head_step: null descriptor");
  const DeviceGuard on_device(d->hidden_c);
  if (d->hidden_c == nullptr || d->ln_weight == nullptr || d->ln_bias == nullptr || d->w_image == nullptr || d->bias2 == nullptr)
    return fail(D3PM_ERR_INVALID, "head_step: hidden_c, ln_weight, ln_bias, w_image and bias2 are required");
  if (d->D != 64) return fail(D3PM_ERR_UNSUPPORTED, "head_step: n_embd D=%d (built for D = 64)", d->D);
  if (d->K != 1024 && d->K != 2048 && d->K != 4096) return fail(D3PM_ERR_UNSUPPORTED, "head_step: K=%d must be 1024, 2048 or 4096", d->K);
  if (d->B <= 0 || d->N <= 0) return fail(D3PM_ERR_INVALID, "head_step: B and N must be positive");
  if (d->mode < D3PM_HEAD_STEP || d->mode > D3PM_HEAD_REFERENCE) return fail(D3PM_ERR_INVALID, "head_step: unknown mode %d", d->mode);
  if (!aligned16(d->hidden_c) || !aligned16(d->hidden_u) || !aligned16(d->w_image) || !aligned16(d->bias2) || !aligned16(d->logits_out))
    return fail(D3PM_ERR_ALIGN, "head_step: hidden, w_image, bias2 and logits_out must be 16-byte aligned");
  const int64_t rows = static_cast<int64_t>(d->B) * d->N;
  if (rows > kMaxGrid) return fail(D3PM_ERR_UNSUPPORTED, "head_step: B*N too large");
  if (d->mode == D3PM_HEAD_LOGITS) {
    if (d->logits_out == nullptr) return fail(D3PM_ERR_INVALID, "head_step: LOGITS mode needs logits_out");
  } else {
    if (d->x_t == nullptr || d->t == nullptr || d->coef_table == nullptr || d->x_prev == nullptr || d->T <= 0)
      return fail(D3PM_ERR_INVALID, "head_step: x_t, t, coef_table and x_prev are required");
    if (d->mode == D3PM_HEAD_STEP && (d->redo_rows == nullptr || d->redo_count == nullptr))
      return fail(D3PM_ERR_INVALID, "head_step: redo_rows [B*N] and redo_count scratch are required");
    if (!aligned16(d->coef_table)) return fail(D3PM_ERR_ALIGN, "head_step: coef_table must be 16-byte aligned");
  }
  H::HeadParams p;
  p.hidden_c = d->hidden_c, p.hidden_u = d->hidden_u, p.ln_weight = d->ln_weight, p.ln_bias = d->ln_bias;
  p.w_image = d->w_image, p.bias2 = d->bias2, p.x_t = d->x_t, p.t = d->t, p.coef_table = d->coef_table;
  p.x_prev = d->x_prev, p.logits_out = d->logits_out, p.status = d->status;
  p.redo_rows = d->redo_rows, p.redo_count = d->redo_count;
  p.N = d->N, p.K = d->K, p.T = d->T, p.rows = rows;
  p.ln_eps = d->ln_eps, p.guidance_scale = d->guidance_scale, p.thin_factor = d->thin_factor;
  p.stat_slack = d->stat_slack > 0.f ? d->stat_slack : 0.f;
  p.seed = d->seed, p.offset = d->offset, p.row_offset = d->row_offset;
  const cudaStream_t s = static_cast<cudaStream_t>(d->stream);
  const bool has_u = d->hidden_u != nullptr;
  const int sms = d3pm::host::sm_count();
  if (sms == 0) return fail(D3PM_ERR_CUDA, "head_step: cannot query the device");
  if (d->mode == D3PM_HEAD_REFERENCE) {
    const unsigned grid = static_cast<unsigned>(rows < 8LL * sms ? rows : 8LL * sms);
    if (has_u) H::head_redo_kernel<64, true><<<grid, H::kRedoThreads, 0, s>>>(p, 1);
    else H::head_redo_kernel<64, false><<<grid, H::kRedoThreads, 0, s>>>(p, 1);
    return check_launch("head_step(reference)");
  }
  const size_t smem = H::smem_bytes<64>();
  const long long tiles = (rows + H::kTileM - 1) / H::kTileM;
  const unsigned grid = static_cast<unsigned>(tiles < sms ? tiles : sms);
  auto launch = [&](auto kern) -> int {
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) != cudaSuccess)
      return fail(D3PM_ERR_CUDA, "head_step: %s", cudaGetErrorString(cudaGetLastError()));
    kern<<<grid, H::kThreads, smem, s>>>(p);
    return D3PM_OK;
  };
  int rc;
  if (d->mode == D3PM_HEAD_LOGITS) {
    rc = has_u ? launch(H::head_step_kernel<64, true, true>) : launch(H::head_step_kernel<64, false, true>);
    if (rc != D3PM_OK) return rc;
    return check_launch("head_step(logits)");
  }
  if (cudaMemsetAsync(d->redo_count, 0, sizeof(uint32_t), s) != cudaSuccess) return fail(D3PM_ERR_CUDA, "head_step: memset failed");
  rc = has_u ? launch(H::head_step_kernel<64, true, false>) : launch(H::head_step_kernel<64, false, false>);
  if (rc != D3PM_OK) return rc;
  rc = check_launch("head_step");
  if (rc != D3PM_OK) return rc;
  if (has_u) H::head_redo_kernel<64, true><<<sms, H::kRedoThreads, 0, s>>>(p, 0);
  else H::head_redo_kernel<64, false><<<sms, H::kRedoThreads, 0, s>>>(p, 0);
  return check_launch("head_step(redo)");
}

int d3pm_decode_lut(const float* codebook, const float* conv_weight, const float* conv_bias, int K, int E, int C, float* lut,
                    d3pm_stream_t stream) {
  if (codebook == nullptr || conv_weight == nullptr || lut == nullptr || K <= 0 || E <= 0 || C <= 0 || E > 8192)
    return fail(D3PM_ERR_INVALID, "decode_lut: bad arguments (K=%d E=%d C=%d)", K, E, C);
  const DeviceGuard on_device(lut);
  d3pm::decode_lut_kernel<<<static_cast<unsigned>(K), 256, static_cast<size_t>(E) * sizeof(float), static_cast<cudaStream_t>(stream)>>>(
      codebook, conv_weight, conv_bias, E, C, lut);
  return check_launch("decode_lut");
}

int d3pm_tokens_to_features(const int64_t* tokens, const float* lut, float* out, int B, int N, int K, int C, uint32_t* status,
                            d3pm_stream_t stream) {
  if (tokens == nullptr || lut == nullptr || out == nullptr || B <= 0 || N <= 0 || K <= 0 || C <= 0 || B > 65535)
    return fail(D3PM_ERR_INVALID, "tokens_to_features: bad arguments");
  const DeviceGuard on_device(out);
  const dim3 grid((N + 31) / 32, B);
  d3pm::tokens_to_features_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(tokens, lut, out, N, K, C, status);
  return check_launch("tokens_to_features");
}

int d3pm_to_token_major(const float* src, float* dst, int64_t pitch, int B, int C, int N, d3pm_stream_t stream) {
  if (src == nullptr || dst == nullptr || B <= 0 || C <= 0 || N <= 0 || pitch < C || B > 65535)
    return fail(D3PM_ERR_INVALID, "to_token_major: bad arguments");
  const DeviceGuard on_device(dst);
  const dim3 grid((N + 31) / 32, (C + 31) / 32, B);
  d3pm::to_token_major_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(src, dst, pitch, C, N);
  return check_launch("to_token_major");
}

}  // extern "C"

// ---------------------------------------------------------------- host-buffer entry points
// The reference's tensors live wherever its caller put them; a caller whose logits (or hidden states) are HOST
// buffers goes through a handle that owns the device staging memory, a copy stream and a compute stream.  The inputs
// travel in chunks of whole videos on the copy stream and the fused step of a chunk runs while the next chunk is on
// the bus (the noise is keyed by the global row, so the chunks reproduce the one-launch result bit for bit).
struct d3pm_host_step {
  int device = 0;
  int B = 0, N = 0, K = 0, T = 0, D = 0, chunks = 1;
  int logits_dtype = D3PM_LOGITS_F32;  // element type of the HOST logits handed to d3pm_host_step_run
  bool guidance = false;
  float *logits_c = nullptr, *logits_u = nullptr, *hidden_c = nullptr, *hidden_u = nullptr;
  int64_t *x_t = nullptr, *t = nullptr, *x_prev = nullptr;
  int32_t* redo_rows = nullptr;
  uint32_t *redo_count = nullptr, *status = nullptr;
  cudaStream_t copy = nullptr, compute = nullptr;
  cudaEvent_t landed[16] = {};
  cudaEvent_t idle = nullptr;
};

namespace {
#define D3PM_CUDA_OK(call, what)                                                                   \
  do {                                                                                             \
    const cudaError_t e_ = (call);                                                                 \
    if (e_ != cudaSuccess) return fail(D3PM_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e_));     \
  } while (0)
}  // namespace

extern "C" int d3pm_host_step_destroy(d3pm_host_step* h) {
  if (h == nullptr) return D3PM_OK;
  const DeviceGuard on_device(h->device);
  if (h->compute != nullptr) cudaStreamSynchronize(h->compute);
  if (h->copy != nullptr) cudaStreamSynchronize(h->copy);
  for (void* ptr : {static_cast<void*>(h->logits_c), static_cast<void*>(h->logits_u), static_cast<void*>(h->hidden_c),
                    static_cast<void*>(h->hidden_u), static_cast<void*>(h->x_t), static_cast<void*>(h->t),
                    static_cast<void*>(h->x_prev), static_cast<void*>(h->redo_rows), static_cast<void*>(h->redo_count),
                    static_cast<void*>(h->status)})
    if (ptr != nullptr) cudaFree(ptr);
  for (cudaEvent_t ev : h->landed)
    if (ev != nullptr) cudaEventDestroy(ev);
  if (h->idle != nullptr) cudaEventDestroy(h->idle);
  if (h->copy != nullptr) cudaStreamDestroy(h->copy);
  if (h->compute != nullptr) cudaStreamDestroy(h->compute);
  delete h;
  cudaGetLastError();
  return D3PM_OK;
}

extern "C" int d3pm_host_step_create(d3pm_host_step** out, int device, int B, int N, int K, int T, int D, int guidance, int chunks) {
  if (out == nullptr) return fail(D3PM_ERR_INVALID, "host_step_create: null handle pointer");
  *out = nullptr;
  if (B <= 0 || N <= 0 || T <= 0 || (K != 1024 && K != 2048 && K != 4096) || (D != 0 && D != 64))
    return fail(D3PM_ERR_UNSUPPORTED, "host_step_create: B=%d N=%d T=%d must be positive, K=%d in {1024,2048,4096}, D=%d in {0,64}", B, N, T, K, D);
  if (chunks <= 0) chunks = (B % 4 == 0 && static_cast<int64_t>(B) * N / 4 >= 1024) ? 4 : 1;
  if (chunks > 16 || B % chunks != 0) return fail(D3PM_ERR_INVALID, "host_step_create: chunks=%d must divide B=%d and be <= 16", chunks, B);
  const DeviceGuard on_device(device);
  d3pm_host_step* h = new d3pm_host_step;
  h->device = device, h->B = B, h->N = N, h->K = K, h->T = T, h->D = D, h->chunks = chunks, h->guidance = guidance != 0;
  const size_t rows = static_cast<size_t>(B) * N;
  auto alloc = [&](auto** ptr, size_t bytes) { return cudaMalloc(reinterpret_cast<void**>(ptr), bytes) == cudaSuccess; };
  bool ok = true;
  if (D == 0) {
    ok = ok && alloc(&h->logits_c, rows * K * sizeof(float));
    if (h->guidance) ok = ok && alloc(&h->logits_u, rows * K * sizeof(float));
  } else {
    ok = ok && alloc(&h->hidden_c, rows * D * sizeof(float));
    if (h->guidance) ok = ok && alloc(&h->hidden_u, rows * D * sizeof(float));
    ok = ok && alloc(&h->redo_rows, rows * sizeof(int32_t)) && alloc(&h->redo_count, sizeof(uint32_t));
  }
  ok = ok && alloc(&h->x_t, rows * 8) && alloc(&h->t, static_cast<size_t>(B) * 8) && alloc(&h->x_prev, rows * 8) && alloc(&h->status, 4);
  ok = ok && cudaMemset(h->status, 0, 4) == cudaSuccess;
  ok = ok && cudaStreamCreateWithFlags(&h->copy, cudaStreamNonBlocking) == cudaSuccess;
  ok = ok && cudaStreamCreateWithFlags(&h->compute, cudaStreamNonBlocking) == cudaSuccess;
  for (int c = 0; c < chunks && ok; ++c) ok = cudaEventCreateWithFlags(&h->landed[c], cudaEventDisableTiming) == cudaSuccess;
  ok = ok && cudaEventCreateWithFlags(&h->idle, cudaEventDisableTiming) == cudaSuccess;
  if (!ok) {
    const cudaError_t e = cudaGetLastError();
    d3pm_host_step_destroy(h);
    return fail(D3PM_ERR_CUDA, "host_step_create: %s", cudaGetErrorString(e));
  }
  *out = h;
  return D3PM_OK;
}

extern "C" int64_t d3pm_host_step_h2d_bytes(const d3pm_host_step* h) {
  if (h == nullptr) return 0;
  const int64_t rows = static_cast<int64_t>(h->B) * h->N;
  const int64_t width = h->D == 0 ? h->K : h->D;
  const int64_t elem = (h->D == 0 && h->logits_dtype != D3PM_LOGITS_F32) ? 2 : 4;
  return rows * width * elem * (h->guidance ? 2 : 1) + rows * 8 + static_cast<int64_t>(h->B) * 8;
}

extern "C" int d3pm_host_step_set_logits_dtype(d3pm_host_step* h, int logits_dtype) {
  if (h == nullptr || h->D != 0) return d3pm::host::fail(D3PM_ERR_INVALID, "host_step_set_logits_dtype: needs a handle created for logits (D = 0)");
  if (logits_dtype < D3PM_LOGITS_F32 || logits_dtype > D3PM_LOGITS_BF16)
    return d3pm::host::fail(D3PM_ERR_INVALID, "host_step_set_logits_dtype: unknown dtype %d", logits_dtype);
  if (logits_dtype != D3PM_LOGITS_F32 && h->K % 8 != 0) return d3pm::host::fail(D3PM_ERR_ALIGN, "host_step_set_logits_dtype: 16-bit rows need K %% 8 == 0");
  h->logits_dtype = logits_dtype;
  return D3PM_OK;
}
extern "C" int64_t d3pm_host_step_d2h_bytes(const d3pm_host_step* h) { return h == nullptr ? 0 : static_cast<int64_t>(h->B) * h->N * 8; }

// shared driver of the two run calls: `launch(b0, nb)` enqueues the step of videos [b0, b0 + nb) on h->compute
template <typename Launch>
static int host_step_run(d3pm_host_step* h, const float* in_c, const float* in_u, float* dev_c, float* dev_u, int64_t width,
                         const int64_t* x_t, const int64_t* t, int64_t* x_prev, uint32_t* status_out, Launch launch, size_t elem = 4) {
  const DeviceGuard on_device(h->device);
  const size_t rows = static_cast<size_t>(h->B) * h->N;
  D3PM_CUDA_OK(cudaMemcpyAsync(h->x_t, x_t, rows * 8, cudaMemcpyHostToDevice, h->compute), "host_step: x_t copy");
  D3PM_CUDA_OK(cudaMemcpyAsync(h->t, t, static_cast<size_t>(h->B) * 8, cudaMemcpyHostToDevice, h->compute), "host_step: t copy");
  const int per = h->B / h->chunks;
  const size_t chunk_bytes = static_cast<size_t>(per) * h->N * width * elem;  // (16-bit logits use the front half of the staging buffers)
  auto at = [&](const float* base, int c) { return reinterpret_cast<const unsigned char*>(base) + c * chunk_bytes; };
  auto at_dev = [&](float* base, int c) { return reinterpret_cast<unsigned char*>(base) + c * chunk_bytes; };
  for (int c = 0; c < h->chunks; ++c) {
    D3PM_CUDA_OK(cudaMemcpyAsync(at_dev(dev_c, c), at(in_c, c), chunk_bytes, cudaMemcpyHostToDevice, h->copy), "host_step: input copy");
    if (h->guidance)
      D3PM_CUDA_OK(cudaMemcpyAsync(at_dev(dev_u, c), at(in_u, c), chunk_bytes, cudaMemcpyHostToDevice, h->copy), "host_step: input copy");
    D3PM_CUDA_OK(cudaEventRecord(h->landed[c], h->copy), "host_step: event");
    D3PM_CUDA_OK(cudaStreamWaitEvent(h->compute, h->landed[c], 0), "host_step: wait");
    const int rc = launch(c * per, per);
    if (rc != D3PM_OK) return rc;
  }
  D3PM_CUDA_OK(cudaMemcpyAsync(x_prev, h->x_prev, rows * 8, cudaMemcpyDeviceToHost, h->compute), "host_step: token copy");
  uint32_t st = 0;
  D3PM_CUDA_OK(cudaMemcpyAsync(&st, h->status, 4, cudaMemcpyDeviceToHost, h->compute), "host_step: status copy");
  D3PM_CUDA_OK(cudaMemsetAsync(h->status, 0, 4, h->compute), "host_step: status reset");
  // the next call's copies must not overwrite staging buffers a kernel of this call still reads
  D3PM_CUDA_OK(cudaEventRecord(h->idle, h->compute), "host_step: event");
  D3PM_CUDA_OK(cudaStreamWaitEvent(h->copy, h->idle, 0), "host_step: wait");
  D3PM_CUDA_OK(cudaStreamSynchronize(h->compute), "host_step: synchronize");
  if (status_out != nullptr) *status_out = st;
  return D3PM_OK;
}

extern "C" int d3pm_host_step_run(d3pm_host_step* h, const float* logits_c, const float* logits_u, const int64_t* x_t, const int64_t* t,
                       const float* coef_table, float guidance_scale, uint64_t seed, uint64_t offset, int64_t row_offset,
                       int64_t* x_prev, uint32_t* status_out) {
  if (h == nullptr || logits_c == nullptr || x_t == nullptr || t == nullptr || coef_table == nullptr || x_prev == nullptr)
    return fail(D3PM_ERR_INVALID, "host_step_run: handle, logits_c, x_t, t, coef_table and x_prev are required");
  if (h->D != 0) return fail(D3PM_ERR_INVALID, "host_step_run: the handle was created for hidden states (D = %d)", h->D);
  if (h->guidance != (logits_u != nullptr)) return fail(D3PM_ERR_INVALID, "host_step_run: logits_u must be given exactly when the handle has guidance");
  auto launch = [&](int b0, int nb) {
    d3pm_step_desc d = {};
    const size_t at = static_cast<size_t>(b0) * h->N;
    const size_t esz = h->logits_dtype == D3PM_LOGITS_F32 ? 4 : 2;
    auto row_ptr = [&](float* base) { return reinterpret_cast<const float*>(reinterpret_cast<unsigned char*>(base) + at * h->K * esz); };
    d.logits_c = row_ptr(h->logits_c), d.logits_u = h->guidance ? row_ptr(h->logits_u) : nullptr;
    d.logits_dtype = h->logits_dtype;
    d.x_t = h->x_t + at, d.t = h->t + b0, d.coef_table = coef_table, d.x_prev = h->x_prev + at, d.status = h->status;
    d.B = nb, d.N = h->N, d.K = h->K, d.T = h->T, d.pitch_logits = h->K;
    d.guidance_scale = guidance_scale, d.sample_mode = D3PM_SAMPLE_PHILOX;
    d.seed = seed, d.offset = offset, d.row_offset = row_offset + static_cast<int64_t>(at);
    d.kernel = D3PM_KERNEL_AUTO, d.stream = h->compute;
    return d3pm_fused_step(&d);
  };
  return host_step_run(h, logits_c, logits_u, h->logits_c, h->logits_u, h->K, x_t, t, x_prev, status_out, launch,
                       h->logits_dtype == D3PM_LOGITS_F32 ? 4 : 2);
}

extern "C" int d3pm_host_head_step_run(d3pm_host_step* h, const float* hidden_c, const float* hidden_u, const int64_t* x_t, const int64_t* t,
                            const float* ln_weight, const float* ln_bias, float ln_eps, const float* w_image, const float* bias2,
                            const float* coef_table, float guidance_scale, float stat_slack, uint64_t seed, uint64_t offset,
                            int64_t row_offset, int64_t* x_prev, uint32_t* status_out) {
  if (h == nullptr || hidden_c == nullptr || x_t == nullptr || t == nullptr || coef_table == nullptr || x_prev == nullptr)
    return fail(D3PM_ERR_INVALID, "host_head_step_run: handle, hidden_c, x_t, t, coef_table and x_prev are required");
  if (h->D == 0) return fail(D3PM_ERR_INVALID, "host_head_step_run: the handle was created for logits (D = 0)");
  if (h->guidance != (hidden_u != nullptr)) return fail(D3PM_ERR_INVALID, "host_head_step_run: hidden_u must be given exactly when the handle has guidance");
  auto launch = [&](int b0, int nb) {
    d3pm_head_desc d = {};
    const size_t at = static_cast<size_t>(b0) * h->N;
    d.hidden_c = h->hidden_c + at * h->D, d.hidden_u = h->guidance ? h->hidden_u + at * h->D : nullptr;
    d.ln_weight = ln_weight, d.ln_bias = ln_bias, d.w_image = w_image, d.bias2 = bias2;
    d.x_t = h->x_t + at, d.t = h->t + b0, d.coef_table = coef_table, d.x_prev = h->x_prev + at, d.status = h->status;
    d.redo_rows = h->redo_rows + at, d.redo_count = h->redo_count;
    d.B = nb, d.N = h->N, d.K = h->K, d.T = h->T, d.D = h->D, d.mode = D3PM_HEAD_STEP;
    d.ln_eps = ln_eps, d.guidance_scale = guidance_scale, d.stat_slack = stat_slack;
    d.seed = seed, d.offset = offset, d.row_offset = row_offset + static_cast<int64_t>(at), d.stream = h->compute;
    return d3pm_head_step(&d);
  };
  return host_step_run(h, hidden_c, hidden_u, h->hidden_c, h->hidden_u, h->D, x_t, t, x_prev, status_out, launch);
}
