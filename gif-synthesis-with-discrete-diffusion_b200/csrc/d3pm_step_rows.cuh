// Fused reverse step, general kernel: one CTA of 256 threads per token row, the row held in registers.
//
// This is the shape-general implementation (any K % 4 == 0 up to 8192, every output / sampling
// mode).  d3pm_step_stream.cuh holds the persistent TMA-pipelined kernel used for the production
// mode on large batches; both share the per-row mathematics below (RowMath), so they agree bit for
// bit on the quantities they both compute.
#pragma once

#include "d3pm_common.cuh"

namespace d3pm {

struct StepParams {
  const float* logits_c;
  const float* logits_u;
  const int64_t* x_t;
  const int64_t* t;
  const float* coef_table;
  const float* gumbel;
  int64_t* x_prev;
  float* post;
  float* recon;
  float* gap;
  uint32_t* status;
  int32_t B, N, K, T;
  int64_t pitch_logits, pitch_gumbel, pitch_out;
  float guidance_scale;
  int32_t sample_mode;
  int32_t gumbel_is_uniform;
  uint64_t seed, offset;
  int64_t row_offset;
  float thin_factor;
  int64_t rows;
  int32_t sample_from;   // D3PM_FROM_POSTERIOR / D3PM_FROM_RECON
  float* score;          // [rows] out: max_k p(x0 = k | x_t)
  const float* sharpen;  // [rows] in: draw from softmax(f * recon)
  float* winner_post;    // [rows] out (stream kernel): log-posterior of the sampled class as the kernel computed it
  int32_t logits_dtype;  // D3PM_LOGITS_*: storage type behind logits_c / logits_u (16-bit: stream kernel only)
  PhiloxRoundKeys keys;  // the round keys of `seed`, expanded on the host (stream kernel: constant-bank operands)
};

// Everything a row needs once the softmax statistics are known.  Identical in every kernel.
struct RowMath {
  float A, Bc;      // P_k = p_k*A + Bc           (k != x_t)
  float Pj;         // P at k == x_t (unmasked rows)
  float PK;         // P at the [MASK] class
  float Ptot;       // sum of all K+1 P's (for the thinning threshold)
  uint32_t j;       // x_t (== K when masked)

  // p_j = exp(recon_j) as a probability in [exp(-70), 1]; ignored for masked rows.  qj = sum_{k != j} p_k: the kernels that
  // write posterior ROWS (p_pred) accumulate it class by class, because 1 - p_j loses everything when the denoiser is sure
  // of x_t (p_j within 1e-7 of 1) while W = 1 / b_t is ~1e8 at small t; the token-only kernels pass 1 - p_j, whose error
  // there is ~1e-7 of absolute probability mass
  __device__ __forceinline__ void init(const RowCoef& cf, bool masked, float pj, uint32_t jj, int K) {
    init(cf, masked, pj, 1.0f - pj, jj, K);
  }
  __device__ __forceinline__ void init(const RowCoef& cf, bool masked, float pj, float qj, uint32_t jj, int K) {
    j = jj;
    const float eL = masked ? cf.W + kTiny : fmaf(cf.W, qj, fmaf(cf.WS, pj, kTiny));
    A = cf.A;
    Bc = cf.BO * eL;
    Pj = masked ? 0.0f : fmaf(pj, cf.AS, cf.BOS * eL);
    PK = fmaf(cf.PK1, eL, cf.PK0);
    Ptot = masked ? fmaf(static_cast<float>(K), Bc, A) + PK
                  : fmaf(static_cast<float>(K - 1), Bc, A * qj) + Pj + PK;
  }
  // the distribution the purity-prior branch samples (:327-329): log_x_recon itself, i.e. P_k = p_k for the codes
  // and exp(-70) for [MASK]; every sampling path below then works unchanged
  __device__ __forceinline__ void init_recon(float pj, uint32_t jj) {
    j = jj;
    A = 1.0f, Bc = 0.0f, Pj = pj, PK = kPFloor, Ptot = 1.0f + kPFloor;
  }
  // posterior log-prob of class k (< K) given its softmax numerator e and the thread's scale r
  __device__ __forceinline__ float post_of(uint32_t k, float e, float r) const {
    const float p = fminf(fmaxf(e * r, kPFloor), 1.0f);
    const float P = (k == j) ? Pj : fmaf(p, A, Bc);
    return log_prob_clamped(P);
  }
  __device__ __forceinline__ float post_self() const { return log_prob_clamped(Pj); }
  __device__ __forceinline__ float post_mask() const { return log_prob_clamped(PK); }
};

// Thinning rule of the production sampler (shared by every kernel so they take identical decisions).
// A class is kept when its 16 coarse noise bits h satisfy 1 + h*2^-23 <= e_k*(r*scaleA) + thrB, i.e.
// h/2^16 <= c*P_k/Ptot up to rounding slack that can only admit more classes; the best survivor is
// accepted when its exact score reaches `accept` = ln(Ptot/c) + slack, which no discarded class can.
constexpr float kDefaultThin = 8.0f;
struct ThinRule {
  float scaleA, thrB, accept;
  __device__ __forceinline__ ThinRule(const RowMath& rm, float thin_factor) {
    const float c = thin_factor > 0.f ? thin_factor : kDefaultThin;
    const float inv = __fdividef(c, rm.Ptot);  // approximate is fine: the filter and the bound use the same value
    scaleA = rm.A * inv * 0.0078125f;                                  // * 2^-7: h sits in the low mantissa bits
    thrB = fmaf(rm.Bc * inv, 0.0078125f, 1.0f) + 2.384185791015625e-7f;  // + 2 ulps of slack
    accept = -lg2(inv) * kLn2 + 0.02f;
  }
};

template <int NV, int NW, typename Sync>
__device__ __forceinline__ void group_max_sum_n(float (&m)[NV], float (&s)[NV], float* scratch, Sync sync) {
  const int lane = threadIdx.x & 31, warp = (threadIdx.x >> 5) % NW;
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const float mw = warp_max(m[v]);
    const float sw =
        warp_sum(m[v] == -CUDART_INF_F ? 0.0f : s[v] * ex2(to_log2_units(m[v]) - to_log2_units(mw)));
    if (lane == 0) {
      scratch[(2 * v) * NW + warp] = mw;
      scratch[(2 * v + 1) * NW + warp] = sw;
    }
  }
  sync();
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    float M = scratch[(2 * v) * NW];
#pragma unroll
    for (int w = 1; w < NW; ++w) M = fmaxf(M, scratch[(2 * v) * NW + w]);
    const float M2 = to_log2_units(M);
    float S = 0.0f;
#pragma unroll
    for (int w = 0; w < NW; ++w) {
      const float mwv = scratch[(2 * v) * NW + w];
      S += (mwv == -CUDART_INF_F) ? 0.0f : scratch[(2 * v + 1) * NW + w] * ex2(to_log2_units(mwv) - M2);
    }
    m[v] = M;
    s[v] = S;
  }
}

// V = float4 chunks per thread; THIN = production Philox mode (thinned exponential race, token only)
template <int V, bool HAS_U, bool THIN>
__global__ void __launch_bounds__(kRowThreads) step_rows_kernel(const StepParams p) {
  constexpr int NW = kRowThreads / 32;
  __shared__ float sred[3][4 * NW];
  __shared__ unsigned long long skey[2][NW];
  __shared__ float sgap[NW];
  const CtaSync sync;

  const int tid = threadIdx.x;
  const int64_t row = blockIdx.x;
  const int b = static_cast<int>(row / p.N);
  const int K = p.K, nq = K >> 2;

  // ---- row scalars --------------------------------------------------------------------------
  long long tt = p.t[b];
  long long jj = p.x_t[row];
  uint32_t st = 0;
  if (tt < 0 || tt >= p.T) {
    st |= D3PM_STATUS_BAD_T;
    tt = tt < 0 ? 0 : p.T - 1;
  }
  if (jj < 0 || jj > K) {
    st |= D3PM_STATUS_BAD_TOKEN;
    jj = K;
  }
  if (st != 0 && tid == 0 && p.status != nullptr) atomicOr(p.status, st);
  const bool masked = (jj == K);
  const uint32_t j = static_cast<uint32_t>(jj);
  const RowCoef cf = load_row_coef(p.coef_table, static_cast<int>(tt), masked);

  const float* __restrict__ rc = p.logits_c + row * p.pitch_logits;
  const float* __restrict__ ru = HAS_U ? p.logits_u + row * p.pitch_logits : nullptr;

  // ---- load the row: x = conditional logits, z = unconditional ---------------------------------
  float x[V][4], z[V][4];
  int nvalid = 0;
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const int q = tid + i * kRowThreads;
    if (q < nq) {
      nvalid = i + 1;
      const float4 a = ld_stream4(rc + 4 * q);
      x[i][0] = a.x, x[i][1] = a.y, x[i][2] = a.z, x[i][3] = a.w;
      if (HAS_U) {
        const float4 c = ld_stream4(ru + 4 * q);
        z[i][0] = c.x, z[i][1] = c.y, z[i][2] = c.z, z[i][3] = c.w;
      }
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e) x[i][e] = -CUDART_INF_F, z[i][e] = -CUDART_INF_F;
    }
  }
  float xj = 0.f, zj = 0.f;  // the logits of class x_t (unmasked rows), same for every thread
  if (!masked) {
    xj = __ldg(rc + j);
    if (HAS_U) zj = __ldg(ru + j);
  }

  // ---- softmax statistics of the raw logits (:231) -------------------------------------------
  float m[2] = {-CUDART_INF_F, -CUDART_INF_F}, s[2] = {0.f, 0.f};
#pragma unroll
  for (int i = 0; i < V; ++i)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      m[0] = fmaxf(m[0], x[i][e]);
      if (HAS_U) m[1] = fmaxf(m[1], z[i][e]);
    }
  {
    const float m0 = to_log2_units(m[0]), m1 = to_log2_units(m[1]);
#pragma unroll
    for (int i = 0; i < V; ++i)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (i < nvalid) {
          const float ec = ex2(fmaf(x[i][e], kLog2e, -m0));
          s[0] += ec;
          if (HAS_U) s[1] += ex2(fmaf(z[i][e], kLog2e, -m1));
          else z[i][e] = ec;  // guidance off: these are already the softmax numerators
        }
      }
  }
  const float m_local = m[0], m_local_c2 = to_log2_units(m[0]);
  if (HAS_U) {
    group_max_sum_n<2, NW>(m, s, sred[0], sync);
  } else {
    float m1[1] = {m[0]}, s1[1] = {s[0]};
    group_max_sum_n<1, NW>(m1, s1, sred[0], sync);
    m[0] = m1[0], s[0] = s1[0];
  }

  // ---- guidance combine + renormalisation (:245-247), or pass-through when guidance is off ------
  float My, Sy, Sother, lnSy, r, yj;
  if (HAS_U) {
    const float lnSc = ln_rel_sum(m[0], s[0]), lnSu = ln_rel_sum(m[1], s[1]);
    const float gs = p.guidance_scale;
    float my = -CUDART_INF_F;
#pragma unroll
    for (int i = 0; i < V; ++i)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (i < nvalid) {
          const float lc = fmaxf((x[i][e] - m[0]) - lnSc, kClampLo);  // clamp of :236 (upper bound is automatic)
          const float lu = fmaxf((z[i][e] - m[1]) - lnSu, kClampLo);
          const float y = fmaf(gs, lc - lu, lu);
          x[i][e] = y;
          my = fmaxf(my, y);
        }
      }
    {
      const float lc = fmaxf((xj - m[0]) - lnSc, kClampLo), lu = fmaxf((zj - m[1]) - lnSu, kClampLo);
      yj = fmaf(gs, lc - lu, lu);
    }
    const float my2 = to_log2_units(my);
    float sy = 0.f, so = 0.f;  // so: the classes other than x_t, summed on their own (see RowMath::init)
#pragma unroll
    for (int i = 0; i < V; ++i)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (i < nvalid) {
          const float ey = ex2(fmaf(x[i][e], kLog2e, -my2));
          z[i][e] = ey;
          sy += ey;
          so += (static_cast<uint32_t>(4 * (tid + i * kRowThreads) + e) == j) ? 0.f : ey;
        }
      }
    float mm[2] = {my, my}, ss[2] = {sy, so};
    group_max_sum_n<2, NW>(mm, ss, sred[1], sync);
    My = mm[0], Sy = ss[0], Sother = ss[1];
    r = (nvalid > 0) ? ex2(my2 - to_log2_units(My)) / Sy : 0.f;
  } else {
    // guidance off: z holds the numerators relative to the thread-local maximum of the first pass
    float so = 0.f;
#pragma unroll
    for (int i = 0; i < V; ++i)
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if (i < nvalid) so += (static_cast<uint32_t>(4 * (tid + i * kRowThreads) + e) == j) ? 0.f : z[i][e];
    float mm[1] = {m_local}, ss[1] = {so};
    group_max_sum_n<1, NW>(mm, ss, sred[1], sync);
    My = m[0], Sy = s[0], Sother = ss[0];
    yj = xj;
    r = (nvalid > 0) ? ex2(m_local_c2 - to_log2_units(My)) / Sy : 0.f;
  }
  lnSy = ln_rel_sum(My, Sy);

  // ---- per-row posterior coefficients (:251-283 collapsed, see d3pm_common.cuh) ------------------
  const float pj = masked ? 0.f : fminf(fmaxf(ex2(fmaf(yj, kLog2e, -to_log2_units(My))) / Sy, kPFloor), 1.0f);
  RowMath rm;
  const bool from_recon = (p.sample_from == D3PM_FROM_RECON);
  if (from_recon) rm.init_recon(masked ? 0.f : pj, masked ? static_cast<uint32_t>(K) + 1u : j);
  else rm.init(cf, masked, pj, masked ? 1.0f : fminf(Sother / Sy, 1.0f), j, K);
  // purity (:318): max_k exp(log_x_recon_k).clamp(0, 1); the largest recon entry is clamp(-lnSy, -70, 0)
  if (p.score != nullptr && tid == 0) p.score[row] = expf(fminf(fmaxf(-lnSy, kClampLo), 0.0f));

  const uint64_t grow = static_cast<uint64_t>(p.row_offset + row);
  const NoiseStream rng(p.seed, p.offset);
  unsigned long long best = 0ull;

  // exact Gumbel score of class k from its softmax numerator e and its 23-bit draw m (:356-357)
  auto score_exact = [&](uint32_t k, float e, uint32_t m) {
    return rm.post_of(k, e, r) + gumbel_from_uniform(uniform_from_draw(m));
  };
  // the noise of the four classes of chunk q: 16 coarse bits each, plus (exact paths) the 7 fine bits
  auto chunk_draws = [&](int q, uint32_t (&m)[4]) {
    const uint4 cw = rng.coarse(NoiseStream::coarse_call_of_chunk(q), grow);
    const uint4 fw = rng.fine(q >> 2, grow);
#pragma unroll
    for (int e = 0; e < 4; ++e)
      m[e] = (NoiseStream::half_of(cw, (((q >> 7) & 1) << 2) | e) << 7) | NoiseStream::low7_of(fw, ((q & 3) << 2) | e);
  };

  if (!THIN) {
    // ================= log-domain pass: optional outputs + exact Gumbel-max =====================
    const int mode = p.sample_mode;
    float* __restrict__ rpost = p.post ? p.post + row * p.pitch_out : nullptr;
    float* __restrict__ rrec = p.recon ? p.recon + row * p.pitch_out : nullptr;
    const float* __restrict__ rg = (mode == D3PM_SAMPLE_GUMBEL) ? p.gumbel + row * p.pitch_gumbel : nullptr;
    // sharpened draw (:323-325): prob = log_softmax(f * log_x_recon) over all K+1 classes, clamp(-70, 0).
    // f >= 1 and recon <= 0, so the largest entry is f * max(recon) = f * clamp(-lnSy, -70, 0).
    const bool sharp = from_recon && p.sharpen != nullptr;
    float fsh = 1.0f, sh_off = 0.0f;  // prob_k = f * recon_k - sh_off
    if (sharp) {
      fsh = __ldg(p.sharpen + row);
      const float top = fsh * fminf(fmaxf(-lnSy, kClampLo), 0.0f);
      float acc = 0.f;
#pragma unroll
      for (int i = 0; i < V; ++i)
        if (i < nvalid)
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float rcv = fminf(fmaxf((x[i][e] - My) - lnSy, kClampLo), 0.0f);
            acc += expf(fmaf(fsh, rcv, -top));
          }
      if (tid == 0) acc += expf(fmaf(fsh, kClampLo, -top));  // the [MASK] row of log_x_recon (-70)
      float mm[1] = {0.f}, ss[1] = {acc};
      group_max_sum_n<1, NW>(mm, ss, sred[2], sync);
      sh_off = top + logf(ss[0]);
    }
#pragma unroll
    for (int i = 0; i < V; ++i) {
      if (i < nvalid) {
        const int q = tid + i * kRowThreads;
        float o[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          if (sharp) {
            const float rcv = fminf(fmaxf((x[i][e] - My) - lnSy, kClampLo), 0.0f);
            o[e] = fminf(fmaxf(fmaf(fsh, rcv, -sh_off), kClampLo), 0.0f);
          } else {
            o[e] = rm.post_of(4 * q + e, z[i][e], r);
          }
        }
        if (rpost) st_stream4(rpost + 4 * q, make_float4(o[0], o[1], o[2], o[3]));
        if (rrec) {
          float rc4[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) rc4[e] = fminf(fmaxf((x[i][e] - My) - lnSy, kClampLo), 0.0f);
          st_stream4(rrec + 4 * q, make_float4(rc4[0], rc4[1], rc4[2], rc4[3]));
        }
        if (mode != D3PM_SAMPLE_NONE) {
          float g[4];
          if (mode == D3PM_SAMPLE_GUMBEL) {
            const float4 gv = ld_stream4(rg + 4 * q);
            g[0] = gv.x, g[1] = gv.y, g[2] = gv.z, g[3] = gv.w;
            if (p.gumbel_is_uniform) {
#pragma unroll
              for (int e = 0; e < 4; ++e) g[e] = gumbel_from_uniform(g[e]);
            }
          } else {
            uint32_t m[4];
            chunk_draws(q, m);
#pragma unroll
            for (int e = 0; e < 4; ++e) g[e] = gumbel_from_uniform(uniform_from_draw(m[e]));
          }
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float sc = g[e] + o[e];
            z[i][e] = sc;  // kept for the near-tie gap
            const unsigned long long key = pack_key(sc, 4 * q + e);
            best = key > best ? key : best;
          }
        }
      }
    }
    float scoreK = 0.f;
    if (tid == 0) {  // the [MASK] class
      const float oK = sharp ? fminf(fmaxf(fmaf(fsh, kClampLo, -sh_off), kClampLo), 0.0f) : rm.post_mask();
      if (rpost) rpost[K] = oK;
      if (rrec) rrec[K] = kClampLo;  // constant -70 row of :235, :248
      if (mode != D3PM_SAMPLE_NONE) {
        float gK;
        if (mode == D3PM_SAMPLE_GUMBEL) gK = p.gumbel_is_uniform ? gumbel_from_uniform(__ldg(rg + K)) : __ldg(rg + K);
        else gK = gumbel_from_uniform(uniform_from_draw(rng.draw(K, grow)));
        scoreK = gK + oK;
        const unsigned long long key = pack_key(scoreK, K);
        best = key > best ? key : best;
      }
    }
    if (mode == D3PM_SAMPLE_NONE) return;
    best = group_max_u64<NW>(best, skey[0], sync);
    if (tid == 0 && p.x_prev) p.x_prev[row] = key_class(best);
    if (p.gap != nullptr) {  // runner-up score, for the near-tie log
      const uint32_t win = key_class(best);
      float second = -CUDART_INF_F;
#pragma unroll
      for (int i = 0; i < V; ++i)
        if (i < nvalid) {
          const int q = tid + i * kRowThreads;
#pragma unroll
          for (int e = 0; e < 4; ++e)
            if (static_cast<uint32_t>(4 * q + e) != win) second = fmaxf(second, z[i][e]);
        }
      if (tid == 0 && win != static_cast<uint32_t>(K)) second = fmaxf(second, scoreK);
      second = group_max_f32<NW>(second, sgap, sync);
      if (tid == 0) p.gap[row] = key_score(best) - second;
    }
    return;
  }

  // ================= production sampling: thinned exponential race ===============================
  // argmax_k (post_k + g_k) = argmax_k P_k / E_k with E_k = -log u_k.  A class can only win if
  // E_k < c * P_k / Ptot for a modest c (the winner's ratio is distributed as Ptot / Exp(1)); since
  // E_k >= v_k = 1 - u_k >= h_k / 2^16, testing the 16 coarse noise bits against that bound discards all but
  // ~c of the K classes before any logarithm is taken.  Survivors are scored exactly as in the log-domain
  // pass, so the result is the same argmax; if the best survivor does not clear the bound (probability
  // e^-c per row) the row is rescored exhaustively.
  const ThinRule thin(rm, p.thin_factor);
  const float thrA = r * thin.scaleA;

#pragma unroll
  for (int i = 0; i < V; ++i) {
    if (i < nvalid) {
      const int q = tid + i * kRowThreads;
      const uint4 cw = rng.coarse(NoiseStream::coarse_call_of_chunk(q), grow);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const uint32_t h = NoiseStream::half_of(cw, (((q >> 7) & 1) << 2) | e);
        if (__uint_as_float(0x3f800000u | h) <= fmaf(z[i][e], thrA, thin.thrB)) {
          const uint32_t k = 4 * q + e;
          const uint32_t m = (h << 7) | NoiseStream::low7_of(rng.fine(k >> 4, grow), k & 15u);
          const unsigned long long key = pack_key(score_exact(k, z[i][e], m), k);
          best = key > best ? key : best;
        }
      }
    }
  }
  if (tid == 0) {  // the two classes with their own coefficients are always scored
    const unsigned long long kK = pack_key(rm.post_mask() + gumbel_from_uniform(uniform_from_draw(rng.draw(K, grow))), K);
    best = kK > best ? kK : best;
    if (!masked) {
      const unsigned long long kj =
          pack_key(rm.post_self() + gumbel_from_uniform(uniform_from_draw(rng.draw(j, grow))), j);
      best = kj > best ? kj : best;
    }
  }
  best = group_max_u64<NW>(best, skey[0], sync);
  if (!(key_score(best) >= thin.accept)) {  // exhaustive rescoring (row-uniform branch)
    best = 0ull;
#pragma unroll
    for (int i = 0; i < V; ++i) {
      if (i < nvalid) {
        const int q = tid + i * kRowThreads;
        uint32_t m[4];
        chunk_draws(q, m);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const unsigned long long key = pack_key(score_exact(4 * q + e, z[i][e], m[e]), 4 * q + e);
          best = key > best ? key : best;
        }
      }
    }
    if (tid == 0) {
      const unsigned long long kK =
          pack_key(rm.post_mask() + gumbel_from_uniform(uniform_from_draw(rng.draw(K, grow))), K);
      best = kK > best ? kK : best;
      if (p.status != nullptr) atomicOr(p.status, D3PM_STATUS_FALLBACK);
    }
    best = group_max_u64<NW>(best, skey[1], sync);
  }
  if (tid == 0 && p.x_prev) p.x_prev[row] = key_class(best);
}

}  // namespace d3pm
