// C ABI of the denoiser's fused self-attention (include/d3pm_b200.h, d3pm_self_attention).
#include <cmath>

#include "d3pm_attention.cuh"
#include "d3pm_host.h"

namespace {
using d3pm::host::fail;
using d3pm::host::check_launch;
using d3pm::host::DeviceGuard;

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
}  // namespace

extern "C" {

int d3pm_self_attention(const d3pm_attn_desc* d) {
  namespace A = d3pm::attn;
  if (d == nullptr) return fail(D3PM_ERR_INVALID, "self_attention: null descriptor");
  if (d->q == nullptr || d->k == nullptr || d->v == nullptr || d->y == nullptr)
    return fail(D3PM_ERR_INVALID, "self_attention: q, k, v and y are required");
  if (d->B <= 0 || d->N <= 0 || d->heads <= 0)
    return fail(D3PM_ERR_INVALID, "self_attention: B=%d N=%d heads=%d must be positive", d->B, d->N, d->heads);
  if (d->head_dim != A::kHeadDim)
    return fail(D3PM_ERR_UNSUPPORTED, "self_attention: head_dim=%d (only %d is implemented)", d->head_dim, A::kHeadDim);
  if (d->heads > 65535) return fail(D3PM_ERR_UNSUPPORTED, "self_attention: heads=%d must be <= 65535 (grid y)", d->heads);
  if (d->pitch_qkv % 4 != 0 || d->pitch_y % 4 != 0)
    return fail(D3PM_ERR_ALIGN, "self_attention: pitch_qkv=%lld and pitch_y=%lld must be multiples of 4", (long long)d->pitch_qkv,
                (long long)d->pitch_y);
  const long long width = static_cast<long long>(d->heads) * d->head_dim;
  if (d->pitch_qkv < width || d->pitch_y < width)
    return fail(D3PM_ERR_INVALID, "self_attention: pitches %lld / %lld shorter than heads * head_dim = %lld", (long long)d->pitch_qkv,
                (long long)d->pitch_y, width);
  if (!aligned16(d->q) || !aligned16(d->k) || !aligned16(d->v) || !aligned16(d->y))
    return fail(D3PM_ERR_ALIGN, "self_attention: q, k, v and y must be 16-byte aligned");
  if (!std::isfinite(d->scale)) return fail(D3PM_ERR_INVALID, "self_attention: scale is not finite");
  const DeviceGuard on_device(d->q);
  const int sms = d3pm::host::sm_count();
  if (sms == 0) return fail(D3PM_ERR_CUDA, "self_attention: cannot query the device");
  // 2 queries per thread.  Halve the CTA while the grid would not give every SM two CTAs (config 1, B = 1 and N = 1024, has
  // only 16 (video, head) pairs): small shapes then spread over the whole GPU.
  int threads = A::kMaxThreads;
  auto ctas = [&](int t) { return static_cast<long long>((d->N + 2 * t - 1) / (2 * t)) * d->heads * d->B; };
  while (threads > 32 && ctas(threads) < 2LL * sms) threads /= 2;
  A::Params p;
  p.N = d->N, p.pitch_qkv = d->pitch_qkv, p.pitch_y = d->pitch_y;
  p.scale_log2 = static_cast<float>(static_cast<double>(d->scale) * 1.4426950408889634);
  const cudaStream_t s = static_cast<cudaStream_t>(d->stream);
  // videos are grid z (at most 65535 per launch): a larger batch runs as several launches on the same stream
  constexpr int kMaxGridZ = 65535;
  for (int b0 = 0; b0 < d->B; b0 += kMaxGridZ) {
    const long long rows = static_cast<long long>(b0) * d->N;
    p.q = d->q + rows * d->pitch_qkv, p.k = d->k + rows * d->pitch_qkv, p.v = d->v + rows * d->pitch_qkv;
    p.y = d->y + rows * d->pitch_y;
    const int videos = d->B - b0 < kMaxGridZ ? d->B - b0 : kMaxGridZ;
    const dim3 grid(static_cast<unsigned>((d->N + 2 * threads - 1) / (2 * threads)), static_cast<unsigned>(d->heads),
                    static_cast<unsigned>(videos));
    A::self_attention_kernel<<<grid, threads, 0, s>>>(p);
    const int rc = check_launch("self_attention");
    if (rc != D3PM_OK) return rc;
  }
  return D3PM_OK;
}

}  // extern "C"
