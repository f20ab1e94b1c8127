// Training-side use of the path (SURVEY.md §8 f1): the variational-bound loss of `_train_loss`
// (diffusion_transformer.py:391-457) and its gradient with respect to the denoiser logits, one CTA per token row.
//
// Per token, with c = logits row, x0 the clean token, j = x_t the noised token, t the video's timestep:
//   recon_k = clamp(log_softmax(c)_k, -70, 0), p = exp(recon)                       (predict_start, :231-236)
//   M_k     = clamp(log P_k, -70, 0),  P_k = p_k A_k + BO_k e^L,  e^L = sum p_k W_k + 1e-30   (q_posterior, :251-283)
//   T_k     = the same posterior for the one-hot x0 (takes four distinct values)              (:420)
//   kl      = sum_{k<=K} T_k (log T_k - M_k)                                                 (:421, :181-183)
//   nll     = -M_{x0},   aux = -recon_{x0}      (log_categorical :427 and the auxiliary KL :445; the 1e-30-weighted
//                                                tails of both sums are below fp32 resolution and dropped)
//   main = t == 0 ? nll : w kl,  auxc = t == 0 ? nll : w aux   (w = mask_weight of the token, :422-424, :430-431, :448)
// and, for the backward pass with per-video weights am (on main) and aa (on auxc):
//   gM_k = d/dM_k = -am w T_k (t > 0) or -(am + aa) [k = x0] (t = 0);   gP_k = gM_k / P_k where -70 <= log P_k <= 0
//   G    = sum_k gP_k BO_k;   h_k = p_k (gP_k A_k + W_k G) - aa w [k = x0, t > 0], zeroed where recon_k was clamped
//   dL/dc_k = h_k - softmax(c)_k sum_m h_m
// The forward pass writes per-token `main` / `auxc` (summed per video by the caller, deterministically), the backward
// pass recomputes the row and writes the gradient row: the logits are read once per pass, nothing else is stored.
#pragma once

#include "d3pm_common.cuh"

namespace d3pm {

struct TrainParams {
  const float* logits;     // [rows][pitch]
  const int64_t* x0;       // [rows] clean tokens in [0, K)
  const int64_t* x_t;      // [rows] noised tokens in [0, K]
  const int64_t* t;        // [B]
  const float* coef_table;
  const float* w_main;     // [B] weight of `main` in the gradient (backward only)
  const float* w_aux;      // [B] weight of `auxc` in the gradient (backward only)
  float* tok_main;         // [rows] out (forward)
  float* tok_aux;          // [rows] out (forward)
  int64_t* x0_recon;       // [rows] out, argmax of recon (nullable)
  int64_t* xtm1_recon;     // [rows] out, argmax of the model posterior (nullable)
  float* grad;             // [rows][pitch_grad] out (backward)
  uint32_t* status;
  int32_t B, N, K, T;
  int64_t pitch, pitch_grad;
  float mask_weight_masked, mask_weight_unmasked;
  int64_t rows;
  int32_t logits_dtype;    // D3PM_LOGITS_*: element type of the logits and grad rows (16-bit: stream kernel only)
};

template <int NW>
__device__ __forceinline__ float block_sum_f(float x, float* scratch) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  x = warp_sum(x);
  __syncthreads();  // scratch may still be read from the previous use
  if (lane == 0) scratch[warp] = x;
  __syncthreads();
  float s = 0.f;
#pragma unroll
  for (int w = 0; w < NW; ++w) s += scratch[w];
  return s;
}

template <int V, bool WRITE_GRAD>
__global__ void __launch_bounds__(kRowThreads) train_rows_kernel(const TrainParams p) {
  constexpr int NW = kRowThreads / 32;
  __shared__ float sf[NW];
  __shared__ unsigned long long sk[NW];
  const int tid = threadIdx.x;
  const int64_t row = blockIdx.x;
  const int b = static_cast<int>(row / p.N);
  const int K = p.K, nq = K >> 2;

  long long tt = p.t[b], jj = p.x_t[row], x0l = p.x0[row];
  uint32_t st = 0;
  if (tt < 0 || tt >= p.T) st |= D3PM_STATUS_BAD_T, tt = tt < 0 ? 0 : p.T - 1;
  if (jj < 0 || jj > K) st |= D3PM_STATUS_BAD_TOKEN, jj = K;
  if (x0l < 0 || x0l >= K) st |= D3PM_STATUS_BAD_TOKEN, x0l = 0;
  if (st != 0 && tid == 0 && p.status != nullptr) atomicOr(p.status, st);
  const bool masked = (jj == K), t0 = (tt == 0);
  const uint32_t j = static_cast<uint32_t>(jj), x0 = static_cast<uint32_t>(x0l);
  const RowCoef cf = load_row_coef(p.coef_table, static_cast<int>(tt), masked);
  const float* __restrict__ rc = p.logits + row * p.pitch;

  // ---- the row, its maximum (and arg-max = x0_recon), its softmax ----
  float x[V][4], e[V][4];
  int nvalid = 0;
  float mloc = -CUDART_INF_F;
  unsigned long long kbest = 0ull;
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const int q = tid + i * kRowThreads;
    if (q < nq) {
      nvalid = i + 1;
      const float4 a = ld_stream4(rc + 4 * q);
      x[i][0] = a.x, x[i][1] = a.y, x[i][2] = a.z, x[i][3] = a.w;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        mloc = fmaxf(mloc, x[i][c]);
        const unsigned long long key = pack_key(x[i][c], 4 * q + c);
        kbest = key > kbest ? key : kbest;
      }
    } else {
#pragma unroll
      for (int c = 0; c < 4; ++c) x[i][c] = -CUDART_INF_F;
    }
  }
  kbest = group_max_u64<NW>(kbest, sk, CtaSync());
  const float M = fmaxf(key_score(kbest), -3.0e38f);
  if (!WRITE_GRAD && tid == 0 && p.x0_recon != nullptr) p.x0_recon[row] = key_class(kbest);
  const float M2 = to_log2_units(M);
  float sloc = 0.f;
#pragma unroll
  for (int i = 0; i < V; ++i)
#pragma unroll
    for (int c = 0; c < 4; ++c)
      if (i < nvalid) {
        e[i][c] = ex2(fmaf(x[i][c], kLog2e, -M2));
        sloc += e[i][c];
      }
  const float S = block_sum_f<NW>(sloc, sf);
  const float lnS = ln_rel_sum(M, S), rS = 1.0f / S;

  // ---- scalars of the two special classes and of the one-hot ("true") posterior ----
  const float c_x0 = __ldg(rc + x0), c_j = masked ? 0.f : __ldg(rc + j);
  const float recon_x0 = fmaxf((c_x0 - M) - lnS, kClampLo);
  const float p_x0 = fminf(fmaxf(ex2(fmaf(c_x0, kLog2e, -M2)) * rS, kPFloor), 1.0f);
  const float p_j = masked ? 0.f : fminf(fmaxf(ex2(fmaf(c_j, kLog2e, -M2)) * rS, kPFloor), 1.0f);
  const float eL = masked ? cf.W + kTiny : fmaf(cf.W, 1.0f - p_j, fmaf(cf.WS, p_j, kTiny));
  const float Bc = cf.BO * eL;
  const bool j_is_x0 = (!masked && j == x0);
  // model posterior at the specials
  const float P_j = masked ? 1.0f : fmaf(p_j, cf.AS, cf.BOS * eL);
  const float P_x0 = j_is_x0 ? P_j : fmaf(p_x0, cf.A, Bc);
  const float P_K = fmaf(cf.PK1, eL, cf.PK0);
  // true posterior: p' = 1 at x0, 1e-30 elsewhere
  const float sumpt = 1.0f;  // 1 + (K-1) 1e-30
  const float ptj = j_is_x0 ? 1.0f : kTiny;
  const float eLt = masked ? fmaf(cf.W, sumpt, kTiny) : fmaf(cf.W, sumpt - ptj, fmaf(cf.WS, ptj, kTiny));
  const float Tg_lin = fmaf(kTiny, cf.A, cf.BO * eLt);
  const float Tj_lin = masked ? 1.0f : fmaf(ptj, cf.AS, cf.BOS * eLt);
  const float Tx0_lin = j_is_x0 ? Tj_lin : fmaf(1.0f, cf.A, cf.BO * eLt);
  const float TK_lin = fmaf(cf.PK1, eLt, cf.PK0);
  const float Tg_log = log_prob_clamped(Tg_lin), Tj_log = log_prob_clamped(Tj_lin);
  const float Tx0_log = log_prob_clamped(Tx0_lin), TK_log = log_prob_clamped(TK_lin);
  const float Tg = expf(Tg_log), Tj = expf(Tj_log), Tx0 = expf(Tx0_log), TK = expf(TK_log);
  const float M_x0 = log_prob_clamped(P_x0), M_j = log_prob_clamped(P_j), M_K = log_prob_clamped(P_K);
  const float wtok = masked ? p.mask_weight_masked : p.mask_weight_unmasked;

  // ---- generic classes: sum of model log-probs (KL tail), sum of 1/P (gradient tail), arg-max of the posterior ----
  float sumM = 0.f, sumInvP = 0.f;
  unsigned long long kpost = 0ull;
  const bool want_arg = (!WRITE_GRAD && p.xtm1_recon != nullptr);
#pragma unroll
  for (int i = 0; i < V; ++i)
    if (i < nvalid) {
      const int q = tid + i * kRowThreads;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const uint32_t k = 4 * q + c;
        const float pk = fminf(fmaxf(e[i][c] * rS, kPFloor), 1.0f);
        const float Pk = fmaf(pk, cf.A, Bc);
        const float lp = lg2(Pk) * kLn2;
        const float Mk = fminf(fmaxf(lp, kClampLo), 0.0f);
        const bool generic = (k != x0) && (k != j);
        if (generic) {
          sumM += Mk;
          if (WRITE_GRAD && lp >= kClampLo && lp <= 0.0f) sumInvP += __frcp_rn(Pk);
        }
        if (want_arg) {
          const float Mreal = (k == j) ? M_j : Mk;  // x0 != j uses the generic coefficients already
          const unsigned long long key = pack_key(Mreal, k);
          kpost = key > kpost ? key : kpost;
        }
      }
    }
  sumM = block_sum_f<NW>(sumM, sf);
  const int n_generic = K - 1 - ((!masked && !j_is_x0) ? 1 : 0);

  if (!WRITE_GRAD) {
    if (want_arg) {
      if (tid == 0) {
        const unsigned long long key = pack_key(M_K, K);
        kpost = key > kpost ? key : kpost;
      }
      kpost = group_max_u64<NW>(kpost, sk, CtaSync());
      if (tid == 0) p.xtm1_recon[row] = key_class(kpost);
    }
    if (tid == 0) {
      float kl = Tg * fmaf(static_cast<float>(n_generic), Tg_log, -sumM);
      kl += Tx0 * (Tx0_log - M_x0) + TK * (TK_log - M_K);
      if (!masked && !j_is_x0) kl += Tj * (Tj_log - M_j);
      const float nll = -M_x0;
      const float aux = -recon_x0;
      p.tok_main[row] = t0 ? nll : wtok * kl;
      p.tok_aux[row] = t0 ? nll : wtok * aux;
    }
    return;
  }

  // ---- backward ----
  sumInvP = block_sum_f<NW>(sumInvP, sf);
  const float am = p.w_main[b], aa = p.w_aux[b];
  auto inside = [](float Pv) {
    const float lp = lg2(Pv) * kLn2;
    return lp >= kClampLo && lp <= 0.0f;
  };
  // gP at the specials and the generic multiplier
  const float g_gen = t0 ? 0.f : -am * wtok * Tg;                    // gM of a generic class
  const float gP_x0 = inside(P_x0) ? (t0 ? -(am + aa) : -am * wtok * Tx0) / P_x0 : 0.f;
  const float gP_j = (!masked && !j_is_x0 && !t0 && inside(P_j)) ? (-am * wtok * Tj) / P_j : 0.f;
  const float gP_K = (!t0 && inside(P_K)) ? (-am * wtok * TK) / P_K : 0.f;
  float G = g_gen * cf.BO * sumInvP + gP_K * cf.PK1;
  if (j_is_x0) G += gP_x0 * cf.BOS;
  else G += gP_x0 * cf.BO + gP_j * cf.BOS;
  float hsum = 0.f;
#pragma unroll
  for (int i = 0; i < V; ++i)
    if (i < nvalid) {
      const int q = tid + i * kRowThreads;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const uint32_t k = 4 * q + c;
        const float sm = e[i][c] * rS;                       // softmax(c)_k
        const float pk = fminf(fmaxf(sm, kPFloor), 1.0f);
        const bool unclamped = ((x[i][c] - M) - lnS) >= kClampLo;
        float gP, Ak, Wk;
        if (k == x0) {
          gP = gP_x0, Ak = j_is_x0 ? cf.AS : cf.A, Wk = j_is_x0 ? cf.WS : cf.W;
        } else if (k == j) {
          gP = gP_j, Ak = cf.AS, Wk = cf.WS;
        } else {
          const float Pk = fmaf(pk, cf.A, Bc);
          gP = inside(Pk) ? g_gen * __frcp_rn(Pk) : 0.f;
          Ak = cf.A, Wk = cf.W;
        }
        float h = pk * fmaf(gP, Ak, Wk * G);
        if (k == x0 && !t0) h -= aa * wtok;
        h = unclamped ? h : 0.f;
        hsum += h;
        x[i][c] = h;   // logits no longer needed
        e[i][c] = sm;
      }
    }
  hsum = block_sum_f<NW>(hsum, sf);
  float* __restrict__ rg = p.grad + row * p.pitch_grad;
#pragma unroll
  for (int i = 0; i < V; ++i)
    if (i < nvalid) {
      const int q = tid + i * kRowThreads;
      st_stream4(rg + 4 * q, make_float4(fmaf(-e[i][0], hsum, x[i][0]), fmaf(-e[i][1], hsum, x[i][1]),
                                         fmaf(-e[i][2], hsum, x[i][2]), fmaf(-e[i][3], hsum, x[i][3])));
    }
}

// ---------------------------------------------------------------- q_pred / q_pred_one_timestep on rows
// out_k = log_add_exp(x_k + la, lb) for k < K, out_K = log_add_exp(x_K + l1c, lc) with the per-video schedule
// scalars of :186-189 (one step) or :203-207 (cumulative, t wrapped modulo T+1).  sched = [8][T+1].
__device__ __forceinline__ float lae32(float a, float b) {  // the reference's fp32 log_add_exp (:32-34)
  const float m = fmaxf(a, b);
  if (m == -CUDART_INF_F) return m;
  return m + logf(expf(a - m) + expf(b - m));
}
__global__ void __launch_bounds__(kRowThreads) q_pred_rows_kernel(const float* __restrict__ in, int64_t pitch_in,
                                                                  const int64_t* __restrict__ t, int t_shift,
                                                                  const float* __restrict__ sched, int T, int K, int N,
                                                                  int cumulative, float* __restrict__ out,
                                                                  int64_t pitch_out) {
  const int64_t row = blockIdx.x;
  const int P = T + 1;
  long long tt = t[row / N] + t_shift;
  float la, lb, lc, l1c;
  if (cumulative) {
    tt = ((tt % P) + P) % P;
    la = sched[4 * P + tt], lb = sched[5 * P + tt], lc = sched[6 * P + tt], l1c = sched[7 * P + tt];
  } else {
    tt = tt < 0 ? 0 : (tt >= T ? T - 1 : tt);
    la = sched[0 * P + tt], lb = sched[1 * P + tt], lc = sched[2 * P + tt], l1c = sched[3 * P + tt];
  }
  const float* __restrict__ r = in + row * pitch_in;
  float* __restrict__ o = out + row * pitch_out;
  for (int k = threadIdx.x; k < K; k += kRowThreads) o[k] = lae32(r[k] + la, lb);
  if (threadIdx.x == 0) o[K] = lae32(r[K] + l1c, lc);
}


// ---------------------------------------------------------------- q_sample on integer tokens (:361-366), Philox noise
// x_t ~ q(x_t | x_0) for a one-hot x_0.  The reference materialises the log one-hot, q_pred and the Gumbel tensor; the
// row q_pred would produce takes three values only (x_0 itself, any other code, [MASK]), so this kernel forms them
// with the SAME expressions as q_pred_rows_kernel on a log one-hot and runs the SAME race as gumbel_argmax_rows_kernel
// in its Philox mode (score = q_k + Gumbel(u_k), u_k from NoiseStream::draw) - but thinned: a code other than x_0 can
// only win if its 16 coarse noise bits are below c P_other / P_tot, one integer compare per class and no memory
// traffic at all.  One warp per token; tokens identical to the three-kernel route (tested).
constexpr int kQSampleWarps = 8;
// exact score of one class (rare: ~6 codes + 2 special classes per token); a real call keeps the sweep below small
__device__ __noinline__ unsigned long long q_sample_score(uint32_t k, uint64_t grow, uint64_t seed, uint64_t offset, float q) {
  const NoiseStream rng(seed, offset);
  return pack_key(gumbel_from_uniform(uniform_from_draw(rng.draw(k, grow))) + q, k);
}
__global__ void __launch_bounds__(32 * kQSampleWarps) q_sample_tokens_kernel(
    const int64_t* __restrict__ x0, const int64_t* __restrict__ t, const float* __restrict__ sched, int T, int K, int N,
    int64_t rows, uint64_t seed, uint64_t offset, int64_t row_offset, int64_t* __restrict__ x_t, uint32_t* status) {
  const int lane = threadIdx.x & 31;
  const int64_t row = static_cast<int64_t>(blockIdx.x) * kQSampleWarps + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int P = T + 1;
  long long tt = t[row / N];
  tt = ((tt % P) + P) % P;
  const float la = sched[4 * P + tt], lb = sched[5 * P + tt], lc = sched[6 * P + tt], l1c = sched[7 * P + tt];
  long long j64 = x0[row];
  if (j64 < 0 || j64 > K) {  // the log one-hot of such a token has no 0 entry at all
    if (lane == 0 && status != nullptr) atomicOr(status, D3PM_STATUS_BAD_TOKEN);
    j64 = -1;
  }
  const uint32_t j = static_cast<uint32_t>(j64);  // 0xffffffff: no class is "self"
  const float q_self = lae32(0.0f + la, lb), q_other = lae32(kLogTiny + la, lb);
  const float q_mask = lae32((j64 == K ? 0.0f : kLogTiny) + l1c, lc);
  const NoiseStream rng(seed, offset);
  const uint64_t grow = static_cast<uint64_t>(row_offset + row);
  auto score_of = [&](uint32_t k) {
    const float q = (k == static_cast<uint32_t>(K)) ? q_mask : (k == j ? q_self : q_other);
    return q_sample_score(k, grow, seed, offset, q);
  };
  // thinning: E_k >= h_k / 2^16, a code other than x_0 can only reach ln(P_tot / c) if E_k <= c P_other / P_tot
  const float p_other = expf(q_other);
  const float p_tot = fmaf(static_cast<float>(K - 1), p_other, expf(q_self) + expf(q_mask));
  const float c = 12.0f;  // other codes carry almost no mass (b_t is tiny), so a wide bound costs nothing and the
                          // score-everything fallback below (e^-c of the tokens) stays out of the launch's tail
  const float hf = (c * p_other / p_tot) * 65536.0f * 1.001f + 2.0f;
  const uint32_t hmax = hf >= 65535.0f ? 0xffffu : static_cast<uint32_t>(hf);
  const float accept = logf(p_tot / c) + 0.02f;
  unsigned long long best = 0ull;
  const int nq = K >> 2;                               // float4 chunks of the codes
  const int ncalls = ((nq + 255) >> 8) << 7;           // coarse calls that cover them
  for (int call = lane; call < ncalls; call += 32) {
    const uint4 cw = rng.coarse(static_cast<uint32_t>(call), grow);
    const uint32_t w4[4] = {cw.x, cw.y, cw.z, cw.w};
    const int chunk_lo = ((call >> 7) << 8) | (call & 127);
    // smallest of the eight halves first: almost every call ends here
    const uint32_t m01 = min(min(w4[0] & 0xffffu, w4[0] >> 16), min(w4[1] & 0xffffu, w4[1] >> 16));
    const uint32_t m23 = min(min(w4[2] & 0xffffu, w4[2] >> 16), min(w4[3] & 0xffffu, w4[3] >> 16));
    if (min(m01, m23) > hmax) continue;
    uint32_t hits = 0;
#pragma unroll
    for (int h = 0; h < 8; ++h) {
      const uint32_t half = (h & 1) ? (w4[h >> 1] >> 16) : (w4[h >> 1] & 0xffffu);
      hits |= (half <= hmax ? 1u : 0u) << h;
    }
    while (hits != 0) {
      const int h = __ffs(hits) - 1;
      hits &= hits - 1;
      const uint32_t k = 4u * static_cast<uint32_t>(chunk_lo + 128 * (h >> 2)) + (h & 3);
      if (k < static_cast<uint32_t>(K) && k != j) {
        const unsigned long long key = score_of(k);
        best = key > best ? key : best;
      }
    }
  }
  if (lane == 0) {
    const unsigned long long key = score_of(static_cast<uint32_t>(K));
    best = key > best ? key : best;
  }
  if (lane == 1 && j < static_cast<uint32_t>(K)) {
    const unsigned long long key = score_of(j);
    best = key > best ? key : best;
  }
  best = warp_max_u64(best);
  if (!(key_score(best) >= accept)) {  // probability ~e^-c: score every class
    best = 0ull;
    for (uint32_t k = lane; k <= static_cast<uint32_t>(K); k += 32) {
      const unsigned long long key = score_of(k);
      best = key > best ? key : best;
    }
    best = warp_max_u64(best);
  }
  if (lane == 0) x_t[row] = key_class(best);
}

}  // namespace d3pm
