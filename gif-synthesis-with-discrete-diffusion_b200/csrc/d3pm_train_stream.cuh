// Training-side loss (SURVEY.md §8 f1), production kernel: persistent CTAs, TMA-staged logit rows, loss AND gradient in
// one pass.  Same mathematics as train_rows_kernel (d3pm_train_rows.cuh, `_train_loss` diffusion_transformer.py:391-457);
// what changes is the schedule:
//   * one CTA of 512 threads per SM, split into independent groups of K / 32 threads (see TrainShape); a group owns every
//     G-th token row;
//   * a two-stage shared-memory ring per group, filled with 1-D bulk TMA (16 KiB per row for K = 4096): two rows per
//     group are in flight while a third is processed from registers (128 KiB per SM);
//   * the row lives in registers: first the logits, from the first sweep on their softmax numerators IN PLACE; every class
//     is treated by the GENERIC formula and the (at most two) special classes x_0 and x_t are corrected on scalars
//     afterwards, so the inner loops carry no per-class compares;
//   * the sum over classes of the gradient's softmax term is obtained in closed form from sums accumulated in the
//     forward sweep, so a row needs two group exchanges (none across warps for the one-warp groups), not four;
//   * the gradient row is written with streaming 128-bit stores straight from registers;
//   * float16 / bfloat16 logits (LD, a denoiser run under autocast) are copied as they lie in HBM and widened in registers
//     (LogitType, as in the reverse step); the gradient row then has the logits' type, each fp32 value rounded to nearest
//     even - bit-identical to the fp32 kernel on logits.float() followed by grad.to(dtype), at half the bytes each way;
//   * a row's scalars (x_0, x_t, t of its video, the per-video gradient weights) are loaded one row ahead and the
//     coefficient table is staged in shared memory.
// HBM traffic is the algorithmic minimum of a fused forward + backward: 16 KiB read and 16 KiB written per token.
#pragma once

#include "d3pm_ptx.cuh"
#include "d3pm_stream.cuh"
#include "d3pm_train_rows.cuh"

namespace d3pm {

__device__ __forceinline__ float rcp_fast(float x) {  // MUFU.RCP, 1 ulp: plenty for a gradient checked to 5e-5
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Shape of one instantiation.  NP = K / 1024.  A thread holds 32 classes of the row (numerators + reciprocals: 64 registers),
// so a group is K / 32 threads wide - 4 groups of 128 threads at K = 4096 (as in round 1), 8 groups of 64 at K = 2048, 16
// one-warp groups at K = 1024 - and the per-row scalar work, 59 % of a warp's instructions at K = 4096, costs the same per
// class for every codebook (round 1 ran 128-thread groups for every K: 0.231 ms instead of 0.100 ms at K = 1024, 64 videos).
// Measured and NOT kept for K = 4096: 64 classes per thread in groups of 64 threads - with 512 threads per CTA the 128
// registers spill, with 256 threads (255 registers) the 8 warps left per SM cannot hide the latency of the scalar sections
// (0.139 instead of 0.104 ms either way).
template <int NP>
struct TrainShape {
  static constexpr int K = 1024 * NP;
  static constexpr int CPT = 8;                   // float4 chunks per thread
  static constexpr int THREADS = kStreamThreads;
  static constexpr int GT = 256 * NP / CPT;       // threads per group: 128 / 64 / 32
  static constexpr int NW = GT / 32;
  static constexpr int NG = THREADS / GT;         // groups per CTA: 4 / 8 / 16
};

template <int NP, int LD = D3PM_LOGITS_F32>
struct __align__(128) TrainGroupSmem {
  // two rows per group in flight while a third is processed from registers (16-bit rows: half the bytes)
  float stage[2][1024 * NP * LogitType<LD>::kBytes / sizeof(float)];
  alignas(16) float red[2][4 * 4];     // reduction scratch: [value][warp], padded to four warps
  unsigned long long keys[2][4];
  unsigned long long full[2];
};

// WRITE_GRAD false: forward only (per-token losses, arg-maxes); true: forward + gradient rows in the same pass.
// LD: D3PM_LOGITS_* of the logits and gradient rows.
template <int NP, bool WRITE_GRAD, int LD = D3PM_LOGITS_F32>
__global__ void __launch_bounds__(TrainShape<NP>::THREADS, 1) train_stream_kernel(const TrainParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  using Sh = TrainShape<NP>;
  using LT = LogitType<LD>;
  constexpr int K = Sh::K, NC = Sh::CPT, GT = Sh::GT, NW = Sh::NW, NG = Sh::NG;
  constexpr uint32_t kRowBytes = K * LT::kBytes;
  uint32_t tid;
  asm volatile("mov.u32 %0, %%tid.x;" : "=r"(tid));
  const int g = tid / GT, tg = tid % GT;
  const int lane = tid & 31, warp = (tid >> 5) & (NW - 1);
  TrainGroupSmem<NP, LD>& S = reinterpret_cast<TrainGroupSmem<NP, LD>*>(smem_raw)[g];
  const StreamSync<NW> sync{g + 1};
  // row indices are 32-bit (the launcher refuses more than 2^31 - 1 rows)
  const int G = static_cast<int>(gridDim.x) * NG;
  const int first_row = g * static_cast<int>(gridDim.x) + static_cast<int>(blockIdx.x);
  const int rows = static_cast<int>(p.rows);
  auto issue_row = [&](int row, int st) {
    fence_proxy_async();
    mbar_expect_tx(&S.full[st], kRowBytes);
    tma_load(S.stage[st], LT::row(p.logits, static_cast<unsigned long long>(row) * p.pitch), kRowBytes, &S.full[st]);
  };
  if (tg == 0) {
    // A fence after each init, as the kernel was tuned.  One fence after both changes the machine code only in this
    // set-up (and the addresses of everything behind it), yet measured 0.2 - 0.9 % slower (B200 at 1000 W).
    mbar_init(&S.full[0], 1);
    fence_mbarrier_init();
    mbar_init(&S.full[1], 1);
    fence_mbarrier_init();
  }
  // CTA-wide copy of the coefficient table (16 floats per timestep) when it fits
  float* coef_s = reinterpret_cast<float*>(smem_raw + sizeof(TrainGroupSmem<NP, LD>) * NG);
  const bool coef_in_smem = p.T <= kCoefSmemRows;
  if (coef_in_smem) {
    for (int i = tid; i < p.T * 16; i += Sh::THREADS)
      coef_s[i] = __ldg(p.coef_table + static_cast<size_t>(i >> 4) * D3PM_COEF_STRIDE + (i & 15));
  }
  __syncthreads();
  if (tg == 0) {
    if (first_row < rows) issue_row(first_row, 0);
    if (first_row + G < rows) issue_row(first_row + G, 1);
  }
  uint32_t phase[2] = {0, 0};
  uint32_t status_bits = 0;
  const bool want_arg = (p.x0_recon != nullptr);

  // scalars of a row, loaded one row ahead
  long long tt_n = 0, jj_n = 0, x0_n = 0;
  float am_n = 0.f, aa_n = 0.f;
  auto load_scalars = [&](int r_) {
    const int b_ = static_cast<int>(static_cast<uint32_t>(r_) / static_cast<uint32_t>(p.N));  // rows < 2^31 (launcher)
    tt_n = p.t[b_], jj_n = p.x_t[r_], x0_n = p.x0[r_];
    if (WRITE_GRAD) am_n = __ldg(p.w_main + b_), aa_n = __ldg(p.w_aux + b_);
  };
  if (first_row < rows) load_scalars(first_row);
  int it = 0;
  for (int row = first_row; row < rows; row += G, ++it) {
    const int st = it & 1;
    long long tt = tt_n, jj = jj_n, x0l = x0_n;
    const float am = am_n, aa = aa_n;
    asm volatile("" : "+l"(tt), "+l"(jj), "+l"(x0l) : : "memory");  // consume before the next loads are issued
    if (row + G < rows) load_scalars(row + G);
    if (static_cast<unsigned long long>(tt) >= static_cast<unsigned long long>(p.T)) status_bits |= D3PM_STATUS_BAD_T, tt = tt < 0 ? 0 : p.T - 1;
    if (static_cast<unsigned long long>(jj) > static_cast<unsigned long long>(K)) status_bits |= D3PM_STATUS_BAD_TOKEN, jj = K;
    if (static_cast<unsigned long long>(x0l) >= static_cast<unsigned long long>(K)) status_bits |= D3PM_STATUS_BAD_TOKEN, x0l = 0;
    const bool masked = (jj == K), t0 = (tt == 0);
    const uint32_t j = static_cast<uint32_t>(jj), x0 = static_cast<uint32_t>(x0l);
    RowCoef cf;
    if (coef_in_smem) {
      const float* crow = coef_s + static_cast<int>(tt) * 16 + (masked ? 0 : 8);
      cf = row_coef_from(lds4(crow), lds4(crow + 4), masked);
    } else {
      cf = load_row_coef(p.coef_table, static_cast<int>(tt), masked);
    }

    mbar_wait_spin(&S.full[st], phase[st]);
    phase[st] ^= 1u;
    const float* __restrict__ rowbuf = S.stage[st];
    // class pairs (0,1) and (2,3) of chunk i (float4 number GT i + tg), packed for the f32x2 pipe; first the logits, from
    // the first sweep on their softmax numerators (in place)
    float2 e[NC][2];
#pragma unroll
    for (int i = 0; i < NC; ++i) LT::chunk(rowbuf, GT * i + tg, e[i][0], e[i][1]);
    const float c_x0 = LT::one(rowbuf, x0), c_j = masked ? 0.f : LT::one(rowbuf, j);

    // ---- exchange 1: (max, sum of exponentials relative to the thread-local max) and the arg-max of the logits ----
    float m = fmaxf(fmaxf(e[0][0].x, e[0][0].y), fmaxf(e[0][1].x, e[0][1].y));
    float lo = fminf(fminf(e[0][0].x, e[0][0].y), fminf(e[0][1].x, e[0][1].y));
#pragma unroll
    for (int i = 1; i < NC; ++i) {  // 3-input min / max: two instructions per four classes each
      m = fmaxf(fmaxf(m, e[i][0].x), fmaxf(e[i][0].y, fmaxf(e[i][1].x, e[i][1].y)));
      lo = fminf(fminf(lo, e[i][0].x), fminf(e[i][0].y, fminf(e[i][1].x, e[i][1].y)));
    }
    unsigned long long kbest = 0ull;
    uint32_t idx = 0;
    if (want_arg) {  // first class (lowest index) that attains the thread-local maximum
#pragma unroll
      for (int i = NC - 1; i >= 0; --i)
#pragma unroll
        for (int c = 3; c >= 0; --c) {
          const float xv = (c & 1) ? e[i][c >> 1].y : e[i][c >> 1].x;
          idx = (xv == m) ? 4u * (static_cast<uint32_t>(GT) * i + tg) + c : idx;
        }
    }
    const float e_top = ex2(fmaf(m, kLog2e, -to_log2_units(fmaxf(m, -3.0e38f))));  // numerator of the thread's best class
    m = fmaxf(m, -3.0e38f);
    const float m2 = to_log2_units(m);
    float sloc;
    {
      const float2 l2e = make_float2(kLog2e, kLog2e), nm2 = make_float2(-m2, -m2);
      float2 s2[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
#pragma unroll
      for (int i = 0; i < NC; ++i)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const float2 a = __ffma2_rn(e[i][h], l2e, nm2);
          e[i][h] = make_float2(ex2(a.x), ex2(a.y));
          s2[h] = __fadd2_rn(s2[h], e[i][h]);
        }
      sloc = (s2[0].x + s2[0].y) + (s2[1].x + s2[1].y);
    }
    float M, Ssum, xmin;
    {
      const float mw = warp_max(m);
      const float mw2 = to_log2_units(mw);
      const float sw = warp_sum(sloc * ex2(m2 - mw2));
      const float lw = warp_min(lo);
      if (want_arg) kbest = warp_argmax_key(m, idx);
      if (NW > 1 && lane == 0) {
        S.red[0][warp] = mw, S.red[0][4 + warp] = sw, S.red[0][8 + warp] = lw;
        if (want_arg) S.keys[0][warp] = kbest;
      }
      sync();  // everyone has drained the stage (and published its partials)
      if (tg == 0 && row + 2 * G < rows) issue_row(row + 2 * G, st);
      if (NW > 1) {
        const float4 mw_ = lds_warps<NW>(S.red[0], -CUDART_INF_F), sw_ = lds_warps<NW>(S.red[0] + 4, 0.f);
        const float4 lw_ = lds_warps<NW>(S.red[0] + 8, CUDART_INF_F);
        xmin = fminf(fminf(lw_.x, lw_.y), fminf(lw_.z, lw_.w));
        M = fmaxf(fmaxf(mw_.x, mw_.y), fmaxf(mw_.z, mw_.w));
        const float M2g = to_log2_units(M);
        Ssum = fmaf(sw_.x, ex2(to_log2_units(mw_.x) - M2g), sw_.y * ex2(to_log2_units(mw_.y) - M2g));
        if (NW == 4) Ssum += fmaf(sw_.z, ex2(to_log2_units(mw_.z) - M2g), sw_.w * ex2(to_log2_units(mw_.w) - M2g));
      } else {
        xmin = lw, M = mw, Ssum = sw;
      }
      if (want_arg && tg == 0) {  // the thread that writes the arg-max combines the warps' keys
        if (NW > 1) {
          kbest = S.keys[0][0];
#pragma unroll
          for (int w = 1; w < NW; ++w) kbest = S.keys[0][w] > kbest ? S.keys[0][w] : kbest;
        }
        p.x0_recon[row] = key_class(kbest);
      }
    }
    const float M2 = to_log2_units(M);
    const float lnS = ln_rel_sum(M, Ssum), rS = rcp_fast(Ssum);
    const float r = ex2(m2 - M2) * rS;  // thread-local numerators -> softmax

    // ---- scalars of the special classes and of the one-hot ("true") posterior (as train_rows_kernel) ----
    const float recon_x0 = fmaxf((c_x0 - M) - lnS, kClampLo);
    const float sm_x0 = ex2(fmaf(c_x0, kLog2e, -M2)) * rS, sm_j = masked ? 0.f : ex2(fmaf(c_j, kLog2e, -M2)) * rS;
    const float p_x0 = fminf(fmaxf(sm_x0, kPFloor), 1.0f);
    const float p_j = masked ? 0.f : fminf(fmaxf(sm_j, kPFloor), 1.0f);
    const float eL = masked ? cf.W + kTiny : fmaf(cf.W, 1.0f - p_j, fmaf(cf.WS, p_j, kTiny));
    const float Bc = cf.BO * eL;
    const bool j_is_x0 = (!masked && j == x0);
    const bool j_other = (!masked && !j_is_x0);
    const float P_j = masked ? 1.0f : fmaf(p_j, cf.AS, cf.BOS * eL);
    const float P_x0 = j_is_x0 ? P_j : fmaf(p_x0, cf.A, Bc);
    const float P_K = fmaf(cf.PK1, eL, cf.PK0);
    const float ptj = j_is_x0 ? 1.0f : kTiny;
    const float eLt = masked ? fmaf(cf.W, 1.0f, kTiny) : fmaf(cf.W, 1.0f - ptj, fmaf(cf.WS, ptj, kTiny));
    // the "true" posterior of the one-hot x_0 takes four values per row; clamp(log T, -70, 0) is a clamp of T itself to
    // [exp(-70), 1], so the linear values every thread needs for the gradient cost no logarithm (the logs are taken by
    // the one thread that forms the loss)
    const float Tg = fminf(fmaxf(fmaf(kTiny, cf.A, cf.BO * eLt), kPFloor), 1.0f);
    const float Tj = masked ? 1.0f : fminf(fmaxf(fmaf(ptj, cf.AS, cf.BOS * eLt), kPFloor), 1.0f);
    const float Tx0 = j_is_x0 ? Tj : fminf(fmaxf(fmaf(1.0f, cf.A, cf.BO * eLt), kPFloor), 1.0f);
    const float TK = fminf(fmaxf(fmaf(cf.PK1, eLt, cf.PK0), kPFloor), 1.0f);
    const float wtok = masked ? p.mask_weight_masked : p.mask_weight_unmasked;

    // ---- forward sweep over the classes, all by the generic formula ----
    // sumM = sum M_k; with "inside" = the posterior clamp did not fire and "open" = the recon clamp did not fire:
    // sInv = sum_{inside} 1/P_k,  sPP = sum_{inside & open} p_k / P_k,  sP = sum_{open} p_k
    float sumM = 0.f, sInv = 0.f, sPP = 0.f, sP = 0.f;
    float2 inv[WRITE_GRAD ? NC : 1][2];  // 1 / P_k (0 where the posterior clamp fired), kept for the gradient
    unsigned long long kpost = 0ull;
    float post_best = -CUDART_INF_F;
    uint32_t post_idx = 0;
    // Clamp-free fast path (row-uniform): when no log-softmax entry can reach -70 (smallest logit of the row) and every
    // generic P_k = p_k A + Bc lies in [exp(-70), 1] (Bc and A + Bc say so), none of the clamps of :236 / :283 can fire for
    // a generic class: the sweep needs no predicates, and the posterior arg-max is the logits' arg-max.
    const bool fast = ((xmin - M) - lnS >= kClampLo + 1.0e-3f) && (Bc >= 1.01f * kPFloor) && (cf.A + Bc <= 0.9999f) &&
                      (cf.A >= 0.f);
    if (fast) {
      const float2 r2 = make_float2(r, r), A2 = make_float2(cf.A, cf.A), Bc2 = make_float2(Bc, Bc);
      float2 sL[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)}, sI[2] = {sL[0], sL[0]}, sQ[2] = {sL[0], sL[0]};
#pragma unroll
      for (int i = 0; i < NC; ++i)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const float2 sm = __fmul2_rn(e[i][h], r2);
          const float2 Pk = __ffma2_rn(sm, A2, Bc2);
          sL[h] = __fadd2_rn(sL[h], make_float2(lg2(Pk.x), lg2(Pk.y)));
          if (WRITE_GRAD) {
            const float2 iv = make_float2(rcp_fast(Pk.x), rcp_fast(Pk.y));
            inv[i][h] = iv;
            sI[h] = __fadd2_rn(sI[h], iv);
            sQ[h] = __ffma2_rn(sm, iv, sQ[h]);
          }
        }
      sumM = kLn2 * ((sL[0].x + sL[0].y) + (sL[1].x + sL[1].y));
      if (WRITE_GRAD) {
        sInv = (sI[0].x + sI[0].y) + (sI[1].x + sI[1].y);
        sPP = (sQ[0].x + sQ[0].y) + (sQ[1].x + sQ[1].y);
        sP = sloc * r;  // every class is "open" here
      }
      post_best = log_prob_clamped(fmaf(fminf(e_top * r, 1.0f), cf.A, Bc));
      post_idx = idx;
    } else {
#pragma unroll
      for (int i = 0; i < NC; ++i)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float sm = ((c & 1) ? e[i][c >> 1].y : e[i][c >> 1].x) * r;
          const float pk = fminf(fmaxf(sm, kPFloor), 1.0f);
          const float Pk = fmaf(pk, cf.A, Bc);
          const float lp = lg2(Pk) * kLn2;
          const float Mk = fminf(fmaxf(lp, kClampLo), 0.0f);
          sumM += Mk;
          if (WRITE_GRAD) {
            const bool inside = (Pk >= kPFloor) && (Pk <= 1.0f), open = sm >= kPFloor;
            const float iv = inside ? rcp_fast(Pk) : 0.f;
            if (c & 1) inv[i][c >> 1].y = iv;
            else inv[i][c >> 1].x = iv;
            sInv += iv;
            sPP += open ? pk * iv : 0.f;
            sP += open ? pk : 0.f;
          }
          if (want_arg) {  // strict ">" keeps the lowest class of a tie inside the thread (classes ascend with i, c)
            const bool better = Mk > post_best;
            post_best = better ? Mk : post_best;
            post_idx = better ? 4u * (static_cast<uint32_t>(GT) * i + tg) + c : post_idx;
          }
        }
    }
    // The sweep scored x_t with the generic coefficients; its true term M_j joins at the end (first thread, with
    // [MASK]), so the thread that owns class x_t must offer its best class OTHER than x_t.  Nothing to do unless
    // x_t is that thread's best; then (fast rows) the runner-up among its softmax numerators, or (rows with clamps)
    // a rescoring of its classes.
    if (want_arg && !masked && tg == static_cast<int>((j >> 2) & static_cast<uint32_t>(GT - 1)) && post_idx == j) {
      if (fast) {
        float e2nd = -1.0f;
        uint32_t i2nd = 0;
#pragma unroll
        for (int i = 0; i < NC; ++i)
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const uint32_t k = 4u * (static_cast<uint32_t>(GT) * i + tg) + c;
            const float ev = (c & 1) ? e[i][c >> 1].y : e[i][c >> 1].x;
            const bool better = (ev > e2nd) && (k != j);
            e2nd = better ? ev : e2nd;
            i2nd = better ? k : i2nd;
          }
        post_best = log_prob_clamped(fmaf(fminf(e2nd * r, 1.0f), cf.A, Bc));
        post_idx = i2nd;
      } else {
        post_best = -CUDART_INF_F;
#pragma unroll
        for (int i = 0; i < NC; ++i)
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const uint32_t k = 4u * (static_cast<uint32_t>(GT) * i + tg) + c;
            const float pk = fminf(fmaxf(((c & 1) ? e[i][c >> 1].y : e[i][c >> 1].x) * r, kPFloor), 1.0f);
            const float Mk = log_prob_clamped(fmaf(pk, cf.A, Bc));
            const bool better = (Mk > post_best) && (k != j);
            post_best = better ? Mk : post_best;
            post_idx = better ? k : post_idx;
          }
      }
    }
    // ---- exchange 2 ----
    {
      float tot = 0.f;
      if (WRITE_GRAD) {
        // four warp sums in one butterfly: after the xor-16 step a lane carries two of the four values, after the xor-8
        // step one; lanes 0 / 8 / 16 / 24 end with the totals of sumM / sInv / sPP / sP (18 instructions instead of 40)
        const bool up16 = (lane & 16) != 0, up8 = (lane & 8) != 0;
        const float k0 = (up16 ? sPP : sumM) + __shfl_xor_sync(0xffffffffu, up16 ? sumM : sPP, 16);
        const float k1 = (up16 ? sP : sInv) + __shfl_xor_sync(0xffffffffu, up16 ? sInv : sP, 16);
        tot = (up8 ? k1 : k0) + __shfl_xor_sync(0xffffffffu, up8 ? k0 : k1, 8);
        tot += __shfl_xor_sync(0xffffffffu, tot, 4);
        tot += __shfl_xor_sync(0xffffffffu, tot, 2);
        tot += __shfl_xor_sync(0xffffffffu, tot, 1);
      } else {
        tot = warp_sum(sumM);
      }
      if (want_arg) kpost = warp_argmax_key(post_best, post_idx);
      if (NW > 1) {
        if (WRITE_GRAD) {
          if ((lane & 7) == 0) S.red[1][(lane >> 3) * 4 + warp] = tot;
        } else if (lane == 0) {
          S.red[1][warp] = tot;
        }
        if (lane == 0 && want_arg) S.keys[1][warp] = kpost;
        sync();
        const float4 a0 = lds_warps<NW>(S.red[1], 0.f), a1 = lds_warps<NW>(S.red[1] + 4, 0.f);
        const float4 a2 = lds_warps<NW>(S.red[1] + 8, 0.f), a3 = lds_warps<NW>(S.red[1] + 12, 0.f);
        sumM = (a0.x + a0.y) + (a0.z + a0.w), sInv = (a1.x + a1.y) + (a1.z + a1.w);
        sPP = (a2.x + a2.y) + (a2.z + a2.w), sP = (a3.x + a3.y) + (a3.z + a3.w);
      } else {
        if (WRITE_GRAD) {  // the four totals sit in lanes 0 / 8 / 16 / 24
          sumM = __shfl_sync(0xffffffffu, tot, 0), sInv = __shfl_sync(0xffffffffu, tot, 8);
          sPP = __shfl_sync(0xffffffffu, tot, 16), sP = __shfl_sync(0xffffffffu, tot, 24);
        } else {
          sumM = tot;
        }
      }
    }
    // remove what the generic formula contributed for the special classes (they are re-added with their own terms)
    auto generic_terms = [&](float sm_k, float pk, float& Pk, float& iv, float& pp, float& po) {
      Pk = fmaf(pk, cf.A, Bc);
      const bool inside = (Pk >= kPFloor) && (Pk <= 1.0f), open = sm_k >= kPFloor;  // the clamp of :283 did not fire
      iv = inside ? rcp_fast(Pk) : 0.f;
      pp = open ? pk * iv : 0.f;
      po = open ? pk : 0.f;
    };
    float gP_gen_x0, gi_x0, gpp_x0, gpo_x0, gP_gen_j = 1.0f, gi_j = 0.f, gpp_j = 0.f, gpo_j = 0.f;
    generic_terms(sm_x0, p_x0, gP_gen_x0, gi_x0, gpp_x0, gpo_x0);
    if (j_other) generic_terms(sm_j, p_j, gP_gen_j, gi_j, gpp_j, gpo_j);
    const int n_generic = K - 1 - (j_other ? 1 : 0);

    if (tg == 0) {
      const float M_x0 = log_prob_clamped(P_x0), M_j = log_prob_clamped(P_j), M_K = log_prob_clamped(P_K);
      const float sumM_gen = sumM - log_prob_clamped(gP_gen_x0) - (j_other ? log_prob_clamped(gP_gen_j) : 0.f);
      const float Tg_log = lg2(Tg) * kLn2, Tj_log = lg2(Tj) * kLn2, Tx0_log = lg2(Tx0) * kLn2, TK_log = lg2(TK) * kLn2;
      float kl = Tg * fmaf(static_cast<float>(n_generic), Tg_log, -sumM_gen);
      kl += Tx0 * (Tx0_log - M_x0) + TK * (TK_log - M_K);
      if (j_other) kl += Tj * (Tj_log - M_j);
      const float nll = -M_x0, aux = -recon_x0;
      if (p.tok_main != nullptr) p.tok_main[row] = t0 ? nll : wtok * kl;
      if (p.tok_aux != nullptr) p.tok_aux[row] = t0 ? nll : wtok * aux;
      if (want_arg && p.xtm1_recon != nullptr) {
        unsigned long long kb = kpost;
        if (NW > 1) {
          kb = S.keys[1][0];
#pragma unroll
          for (int w = 1; w < NW; ++w) kb = S.keys[1][w] > kb ? S.keys[1][w] : kb;
        }
        const unsigned long long kK = pack_key(M_K, K), kJ = masked ? 0ull : pack_key(M_j, j);
        kb = kK > kb ? kK : kb;
        kb = kJ > kb ? kJ : kb;
        p.xtm1_recon[row] = key_class(kb);
      }
    }
    if (!WRITE_GRAD) continue;

    // ---- gradient (same formulas as train_rows_kernel) ----
    auto inside_of = [](float Pv) { return Pv >= kPFloor && Pv <= 1.0f; };
    const float g_gen = t0 ? 0.f : -am * wtok * Tg;
    const float gP_x0 = inside_of(P_x0) ? (t0 ? -(am + aa) : -am * wtok * Tx0) * rcp_fast(P_x0) : 0.f;
    const float gP_j = (j_other && !t0 && inside_of(P_j)) ? (-am * wtok * Tj) * rcp_fast(P_j) : 0.f;
    const float gP_K = (!t0 && inside_of(P_K)) ? (-am * wtok * TK) * rcp_fast(P_K) : 0.f;
    const float sInv_gen = sInv - gi_x0 - gi_j;
    float Gs = g_gen * cf.BO * sInv_gen + gP_K * cf.PK1;
    if (j_is_x0) Gs += gP_x0 * cf.BOS;
    else Gs += gP_x0 * cf.BO + gP_j * cf.BOS;
    // h_k = p_k (gP_k A_k + W_k G) - aa w [k = x0, t > 0], zero where the recon clamp fired
    const bool open_x0 = sm_x0 >= kPFloor, open_j = j_other && (sm_j >= kPFloor);
    float h_x0 = p_x0 * fmaf(gP_x0, j_is_x0 ? cf.AS : cf.A, (j_is_x0 ? cf.WS : cf.W) * Gs);
    if (!t0) h_x0 -= aa * wtok;
    h_x0 = open_x0 ? h_x0 : 0.f;
    const float h_j = open_j ? p_j * fmaf(gP_j, cf.AS, cf.WS * Gs) : 0.f;
    const float gA = g_gen * cf.A, WG = cf.W * Gs;
    const float hsum = fmaf(gA, sPP - gpp_x0 - gpp_j, WG * (sP - gpo_x0 - gpo_j)) + h_x0 + h_j;
    typename LT::Elem* __restrict__ rg = reinterpret_cast<typename LT::Elem*>(p.grad) + static_cast<long long>(row) * p.pitch_grad;
    const uint32_t q_x0 = x0 >> 2, q_j = j_other ? (j >> 2) : 0xffffffffu;
#pragma unroll
    for (int i = 0; i < NC; ++i) {
      const uint32_t q = static_cast<uint32_t>(GT) * i + tg;
      float o[4];
      if (fast) {
        const float2 r2 = make_float2(r, r), gA2 = make_float2(gA, gA), wh2 = make_float2(WG - hsum, WG - hsum);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const float2 v = __fmul2_rn(__fmul2_rn(e[i][h], r2), __ffma2_rn(gA2, inv[i][h], wh2));
          o[2 * h] = v.x, o[2 * h + 1] = v.y;
        }
      } else {
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float sm = ((c & 1) ? e[i][c >> 1].y : e[i][c >> 1].x) * r;
          const float iv = (c & 1) ? inv[i][c >> 1].y : inv[i][c >> 1].x;
          const float hk = (sm >= kPFloor) ? fmaf(gA, iv, WG) : 0.f;  // h_k / p_k, 0 where the recon clamp fired
          o[c] = fminf(sm, 1.0f) * hk - sm * hsum;
        }
      }
      LT::store4(rg, q, o);
    }
    // the two special classes: their owners overwrite the generic value (same thread, same address: program order)
    if (tg == static_cast<int>(q_x0 & static_cast<uint32_t>(GT - 1))) rg[x0] = LT::narrow1(fmaf(-sm_x0, hsum, h_x0));
    if (j_other && tg == static_cast<int>(q_j & static_cast<uint32_t>(GT - 1))) rg[j] = LT::narrow1(fmaf(-sm_j, hsum, h_j));
  }
  if (status_bits != 0 && tg == 0 && p.status != nullptr) atomicOr(p.status, status_bits);
}

// grad[row][:] *= factor[video of row]; rows whose factor is exactly 1 are left untouched (no memory traffic), which is
// the common case: the gradient was written with the scale the caller announced (see d3pm_train_rows, backward == 2)
__global__ void __launch_bounds__(256) scale_rows_kernel(float* __restrict__ rows, int64_t pitch, const float* __restrict__ factor,
                                                         int N, int K) {
  const int64_t row = blockIdx.x;
  const float f = __ldg(factor + row / N);
  if (f == 1.0f) return;
  float* __restrict__ r = rows + row * pitch;
  for (int q = threadIdx.x; q < (K >> 2); q += 256) {
    float4 v = *reinterpret_cast<float4*>(r + 4 * q);
    v.x *= f, v.y *= f, v.z *= f, v.w *= f;
    *reinterpret_cast<float4*>(r + 4 * q) = v;
  }
}

// 16-bit rows start on 16-byte boundaries too: both pitches a multiple of 8 elements
inline bool train_stream_supports(const TrainParams& p) {
  return (p.K == 1024 || p.K == 2048 || p.K == 4096) && p.rows >= 2048 && p.pitch % 4 == 0 &&
         (p.logits_dtype == D3PM_LOGITS_F32 || (p.pitch % 8 == 0 && (p.grad == nullptr || p.pitch_grad % 8 == 0)));
}

template <int NP, int LD>
int launch_train_stream_np(const TrainParams& p, bool write_grad, cudaStream_t s) {
  const size_t smem = sizeof(TrainGroupSmem<NP, LD>) * TrainShape<NP>::NG + kCoefSmemRows * 16 * sizeof(float);
  return launch_persistent(write_grad ? train_stream_kernel<NP, true, LD> : train_stream_kernel<NP, false, LD>,
                           TrainShape<NP>::THREADS, smem, p, s);
}

template <int LD>
int launch_train_stream_ld(const TrainParams& p, bool write_grad, cudaStream_t s) {
  switch (p.K) {
    case 1024: return launch_train_stream_np<1, LD>(p, write_grad, s);
    case 2048: return launch_train_stream_np<2, LD>(p, write_grad, s);
    case 4096: return launch_train_stream_np<4, LD>(p, write_grad, s);
    default: return D3PM_ERR_UNSUPPORTED;
  }
}

inline int launch_train_stream(const TrainParams& p, bool write_grad, cudaStream_t s) {
  switch (p.logits_dtype) {
    case D3PM_LOGITS_F32: return launch_train_stream_ld<D3PM_LOGITS_F32>(p, write_grad, s);
    case D3PM_LOGITS_F16: return launch_train_stream_ld<D3PM_LOGITS_F16>(p, write_grad, s);
    case D3PM_LOGITS_BF16: return launch_train_stream_ld<D3PM_LOGITS_BF16>(p, write_grad, s);
    default: return D3PM_ERR_INVALID;
  }
}

}  // namespace d3pm
