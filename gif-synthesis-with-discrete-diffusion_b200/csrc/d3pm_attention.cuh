// Fused self-attention of the denoiser blocks (include/d3pm_b200.h, d3pm_self_attention): the reference's
// FullAttention (transformer_utils.py:24-62) at head dimension 4, forward, fp32, without the [B, heads, N, N] score
// matrix.
//
// At head dimension 4 a (query, key) pair costs ~8 FMAs and one exponential, so the kernel is bound by the MUFU
// exponential unit (16 ex2 per clock per SM), not by memory.  Layout of the work:
//   * grid (query tiles, heads, videos); a CTA of `blockDim.x` threads owns 2 * blockDim.x queries of one (video, head),
//     each thread two of them (n and n + blockDim.x), held as float2 pairs so every FMA, add and multiply of the inner
//     loop is one packed FFMA2 / FADD2 / FMUL2 for both queries;
//   * the head's K and V (16 B each per key) are staged in shared memory kTileKeys keys at a time and read back as
//     broadcast LDS.128 (every thread reads the same key);
//   * online softmax with an exact stabiliser: per block of 32 keys the scores stay in registers, their maximum raises the
//     running maximum, accumulator and denominator are rescaled once, then the 32 exponentials are taken.  Scores are
//     pre-scaled by scale * log2(e) (folded into q) so each exponential is one ex2.approx.  The exponent is never above
//     0 and the largest term of the row is exactly 1, so the row can neither overflow nor underflow to an empty sum.
#pragma once

#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

namespace d3pm {
namespace attn {

constexpr int kHeadDim = 4;
constexpr int kKeyBlock = 32;     // keys per maximum / rescale
constexpr int kTileKeys = 1024;   // keys of K and V staged per pass: 32 KiB of shared memory
constexpr int kMaxThreads = 128;  // 3 CTAs per SM leave 170 registers a thread (2 x 256 capped it at 128 and spilled)

struct Params {
  const float* q;
  const float* k;
  const float* v;
  float* y;
  int N;
  long long pitch_qkv, pitch_y;
  float scale_log2;  // softmax scale * log2(e)
};

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ float2 splat(float a) { return make_float2(a, a); }

// Running softmax state of a thread's two queries: maximum m (log2 units), denominator l and numerator acc[c], each sum
// with its Kahan compensation.  The sums are compensated because one key can outweigh all others by many orders (a
// dominant key, or scores spread over hundreds): added one by one, every later term below half an ulp of the running sum
// would be lost, an error that grows with N (1e-4 of max|v| at N = 8200 in a plain fp32 sum).  Each block of 32 keys is
// therefore summed from zero and its partial sums are added to the running sums once, compensated.
struct RowState {
  float2 m, l, cl;
  float2 acc[kHeadDim], cacc[kHeadDim];
};

__device__ __forceinline__ void kahan_add(float2& sum, float2& comp, float2 x) {
  const float2 y = __fadd2_rn(x, make_float2(-comp.x, -comp.y));
  const float2 t = __fadd2_rn(sum, y);
  comp = __fadd2_rn(__fadd2_rn(t, make_float2(-sum.x, -sum.y)), make_float2(-y.x, -y.y));
  sum = t;
}

// One block of keys for the thread's two queries.  kTail: fewer than kKeyBlock valid keys (the last block of the row);
// the others score -inf and weigh exactly 0, and their (stale) shared-memory values are not read.
template <bool kTail>
__device__ __forceinline__ void key_block(const float4* __restrict__ ks, const float4* __restrict__ vs, int valid,
                                          const float2 (&q)[kHeadDim], RowState& st) {
  float2 s[kKeyBlock];
#pragma unroll
  for (int j = 0; j < kKeyBlock; ++j) {
    const float4 kk = ks[j];
    float2 d = __fmul2_rn(q[0], splat(kk.x));
    d = __ffma2_rn(q[1], splat(kk.y), d);
    d = __ffma2_rn(q[2], splat(kk.z), d);
    d = __ffma2_rn(q[3], splat(kk.w), d);
    if (kTail && j >= valid) d = splat(-CUDART_INF_F);
    s[j] = d;
  }
  float2 mx = st.m;
#pragma unroll
  for (int j = 0; j < kKeyBlock; j += 2) {
    mx.x = fmaxf(fmaxf(mx.x, s[j].x), s[j + 1].x);
    mx.y = fmaxf(fmaxf(mx.y, s[j].y), s[j + 1].y);
  }
  // the first block turns m = -inf into a finite maximum: ex2(-inf) = 0 clears the (zero) sums
  const float2 alpha = make_float2(ex2(st.m.x - mx.x), ex2(st.m.y - mx.y));
  st.m = mx;
  const float2 neg = make_float2(-mx.x, -mx.y);
  float2 lb = splat(0.f), ab[kHeadDim] = {splat(0.f), splat(0.f), splat(0.f), splat(0.f)};
#pragma unroll
  for (int j = 0; j < kKeyBlock; ++j) {
    if (kTail && j >= valid) break;
    const float2 e = __fadd2_rn(s[j], neg);
    const float2 p = make_float2(ex2(e.x), ex2(e.y));
    lb = __fadd2_rn(lb, p);
    const float4 vv = vs[j];
    ab[0] = __ffma2_rn(p, splat(vv.x), ab[0]);
    ab[1] = __ffma2_rn(p, splat(vv.y), ab[1]);
    ab[2] = __ffma2_rn(p, splat(vv.z), ab[2]);
    ab[3] = __ffma2_rn(p, splat(vv.w), ab[3]);
  }
  st.l = __fmul2_rn(st.l, alpha), st.cl = __fmul2_rn(st.cl, alpha);
  kahan_add(st.l, st.cl, lb);
#pragma unroll
  for (int c = 0; c < kHeadDim; ++c) {
    st.acc[c] = __fmul2_rn(st.acc[c], alpha), st.cacc[c] = __fmul2_rn(st.cacc[c], alpha);
    kahan_add(st.acc[c], st.cacc[c], ab[c]);
  }
}

// y[b, n, 4h .. 4h+3] = sum_j softmax_j(scale q_{b,n,h} . k_{b,j,h}) v_{b,j,h}; blockIdx = (query tile, h, b).
__global__ void __launch_bounds__(kMaxThreads, 3) self_attention_kernel(const Params p) {
  __shared__ float4 sk[kTileKeys];
  __shared__ float4 sv[kTileKeys];
  const int h = blockIdx.y;
  const long long row0 = static_cast<long long>(blockIdx.z) * p.N;  // first token row of video b
  const int na = blockIdx.x * 2 * blockDim.x + threadIdx.x, nb = na + blockDim.x;
  // queries past the end compute on the last token and store nothing (they still take part in the barriers)
  const float4 qa = __ldg(reinterpret_cast<const float4*>(p.q + (row0 + min(na, p.N - 1)) * p.pitch_qkv + kHeadDim * h));
  const float4 qb = __ldg(reinterpret_cast<const float4*>(p.q + (row0 + min(nb, p.N - 1)) * p.pitch_qkv + kHeadDim * h));
  const float2 q[kHeadDim] = {make_float2(qa.x * p.scale_log2, qb.x * p.scale_log2), make_float2(qa.y * p.scale_log2, qb.y * p.scale_log2),
                              make_float2(qa.z * p.scale_log2, qb.z * p.scale_log2), make_float2(qa.w * p.scale_log2, qb.w * p.scale_log2)};
  RowState st;
  st.m = splat(-CUDART_INF_F), st.l = st.cl = splat(0.f);
#pragma unroll
  for (int c = 0; c < kHeadDim; ++c) st.acc[c] = st.cacc[c] = splat(0.f);
  const float* kbase = p.k + row0 * p.pitch_qkv + kHeadDim * h;
  const float* vbase = p.v + row0 * p.pitch_qkv + kHeadDim * h;
  for (int t0 = 0; t0 < p.N; t0 += kTileKeys) {
    const int nk = min(kTileKeys, p.N - t0);
    __syncthreads();  // the previous tile is consumed
    for (int j = threadIdx.x; j < nk; j += blockDim.x) {
      sk[j] = __ldg(reinterpret_cast<const float4*>(kbase + (t0 + j) * p.pitch_qkv));
      sv[j] = __ldg(reinterpret_cast<const float4*>(vbase + (t0 + j) * p.pitch_qkv));
    }
    __syncthreads();
    const int full = nk / kKeyBlock * kKeyBlock;
    for (int j = 0; j < full; j += kKeyBlock) key_block<false>(sk + j, sv + j, kKeyBlock, q, st);
    if (full < nk) key_block<true>(sk + full, sv + full, nk - full, q, st);
  }
  const float2 inv = make_float2(1.f / st.l.x, 1.f / st.l.y);
  const float2(&acc)[kHeadDim] = st.acc;
  if (na < p.N)
    *reinterpret_cast<float4*>(p.y + (row0 + na) * p.pitch_y + kHeadDim * h) =
        make_float4(acc[0].x * inv.x, acc[1].x * inv.x, acc[2].x * inv.x, acc[3].x * inv.x);
  if (nb < p.N)
    *reinterpret_cast<float4*>(p.y + (row0 + nb) * p.pitch_y + kHeadDim * h) =
        make_float4(acc[0].y * inv.y, acc[1].y * inv.y, acc[2].y * inv.y, acc[3].y * inv.y);
}

}  // namespace attn
}  // namespace d3pm
