// Fused reverse step, production kernel: persistent CTAs, TMA-staged rows, register-resident math.
//
// One CTA of 512 threads per SM, split into independent GROUPS; a group owns every G-th token row (G = number of
// groups in the grid).  A thread always holds 32 classes of the row (64 without guidance, where the softmax numerators
// overwrite the logits in place), so the group is K/32 (K/64) threads wide:
//
//     K = 4096, guidance on : 4 groups of 128 threads      K = 4096, guidance off : 8 groups of 64 threads
//     K = 2048, guidance on : 8 groups of  64 threads      K = 2048, guidance off : 16 groups of one warp
//     K = 1024              : 16 groups of one warp
//
// The per-row work that does not depend on the class (reductions, row coefficients, thinning thresholds, loop
// bookkeeping: ~250 of the ~690 instructions a warp spends on a row at K = 4096) is executed by every warp of a group, so
// its cost per class is the same for every codebook size instead of doubling each time K halves (round 1: 79 % / 51 % of
// the copy peak at K = 2048 / 1024, 72 % without guidance).  One-warp groups need no barrier at all.  Per row:
//   * one elected thread issues the bulk-TMA copies (cp.async.bulk) of the conditional / unconditional logit rows into
//     the group's shared-memory stage, completion signalled on an mbarrier; the copy of row r+1 flies while row r is
//     being computed from registers;
//   * the threads pull the row into registers (class pairs packed for the f32x2 pipe) and run the softmax statistics,
//     the guidance combine and the posterior entirely in registers with thread-local maxima, so that only two group
//     barriers per row are needed;
//   * sampling is the thinned exponential race (see ThinRule): 16 Philox bits per class decide whether the
//     class can still win; the ~8 survivors per row are appended to a per-row list in shared memory;
//   * every kScoreBatch rows the group scores the survivors of the whole batch exactly (Gumbel score in
//     accurate fp32, argmax with first-index ties), two rows per warp pass, and writes the tokens;
//   * rows whose best survivor does not clear the acceptance bound (probability e^-8, ~25 of 65 536 rows)
//     are queued and redone by the same group after its main loop: the same race thinned at c = 16 with the
//     survivors scored on the spot, and exhaustively only if that fails too (e^-16).
// HBM traffic is the algorithmic minimum: each logit is read once, 8 bytes of token go out per row.
#pragma once

#include <type_traits>

#include "d3pm_host.h"
#include "d3pm_ptx.cuh"
#include "d3pm_step_rows.cuh"
#include "d3pm_stream.cuh"

namespace d3pm {

constexpr int kCandPerRow = 30;   // survivors kept per row (a row with more is redone); the scoring pass takes one or two
                                  // rounds of 16 lanes per row: up to 14 survivors + [MASK] + x_t in the first
constexpr float kStreamThin = 8.0f;  // ~8 survivors per row; a row's best survivor misses the bound with probability e^-8
constexpr float kRedoThin = 16.0f;  // bound of the second attempt at a row whose best survivor did not clear the first
struct RowInfo {  // what the scoring pass needs to finish a row
  float A, Bc, Pj, PK, accept;
  uint32_t j;      // x_t, == K when masked
  int32_t rel;     // row index relative to the group's first row, in units of G
  int32_t pad;
};

// Shape of one instantiation.  NP = K / 1024; CPT = float4 chunks a thread holds per tensor (8, or 16 without guidance).
template <int NP, int CPT, bool HAS_U>
struct StreamShape {
  static_assert(CPT == 8 || (CPT == 16 && !HAS_U), "64 classes per thread only fit in registers without the second tensor");
  static constexpr int K = 1024 * NP;
  static constexpr int GT = 256 * NP / CPT;        // threads per group
  static constexpr int NW = GT / 32;               // warps per group
  static constexpr int NG = kStreamThreads / GT;   // groups per CTA
  static constexpr int SB = 128 / NG;              // rows whose survivors are scored together
  static constexpr int RC = 8192 / NG;             // rows a group can queue for rescoring (= max rows per group)
  static constexpr int PS = 128 / GT;              // a coarse Philox call serves chunks q and q + 128: slots i and i + PS
  static constexpr int NCALL = CPT / 2;            // coarse calls per thread and row
  static_assert(GT >= 32 && GT <= 128 && NG <= 16, "unsupported group shape");
};

template <int NP, int CPT, bool HAS_U>
struct __align__(128) GroupSmem {
  using Sh = StreamShape<NP, CPT, HAS_U>;
  float c[1024 * NP];                   // conditional logits of the row in flight
  float u[HAS_U ? 1024 * NP : 4];       // unconditional logits
  alignas(16) float red[3][6 * 4];      // reduction scratch, read back with 128-bit loads
  unsigned long long full;              // mbarrier: TMA bytes landed
  unsigned long long keys[4];
  uint32_t redo_cnt;
  uint32_t pad;
  RowInfo info[Sh::SB];
  uint32_t cand_cnt[Sh::SB];
  uint32_t cand_k[Sh::SB][kCandPerRow];
  float cand_p[Sh::SB][kCandPerRow];
  int32_t redo[Sh::RC];
};

// Group-wide (max, sum) of per-thread softmax partials, one barrier.  m: thread-local max (natural units),
// s: sum of 2^(x*log2e - fl(m*log2e)).  Returns the group max and the sum relative to it.
template <int NW, int NV, typename Sync>
__device__ __forceinline__ void stream_max_sum(float (&m)[NV], float (&s)[NV], float* scratch, Sync sync) {
  const int lane = threadIdx.x & 31, warp = (threadIdx.x >> 5) & (NW - 1);
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const float mw = warp_max(m[v]);
    const float mw2 = to_log2_units(mw);
    const float sw = warp_sum(s[v] * ex2(to_log2_units(m[v]) - mw2));
    if (NW == 1) {
      m[v] = mw, s[v] = sw;
    } else if (lane == 0) {
      scratch[(3 * v) * 4 + warp] = mw;
      scratch[(3 * v + 1) * 4 + warp] = mw2;
      scratch[(3 * v + 2) * 4 + warp] = sw;
    }
  }
  sync();
  if constexpr (NW > 1) {
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const float4 mw = lds_warps<NW>(scratch + (3 * v) * 4, -CUDART_INF_F), mw2 = lds_warps<NW>(scratch + (3 * v + 1) * 4, 0.f);
    const float4 sw = lds_warps<NW>(scratch + (3 * v + 2) * 4, 0.f);
    if (NW == 4) {
      const float M = fmaxf(fmaxf(mw.x, mw.y), fmaxf(mw.z, mw.w));
      const float M2 = to_log2_units(M);
      m[v] = M;
      s[v] = fmaf(sw.x, ex2(mw2.x - M2), fmaf(sw.y, ex2(mw2.y - M2), fmaf(sw.z, ex2(mw2.z - M2), sw.w * ex2(mw2.w - M2))));
    } else {
      const float M = fmaxf(mw.x, mw.y);
      const float M2 = to_log2_units(M);
      m[v] = M;
      s[v] = fmaf(sw.x, ex2(mw2.x - M2), sw.y * ex2(mw2.y - M2));
    }
  }
  }
}

// Group-wide max of NV values (one CREDUX per value, one barrier).
template <int NW, int NV, typename Sync>
__device__ __forceinline__ void stream_max(float* mx, float* scratch, Sync sync) {
  const int lane = threadIdx.x & 31, warp = (threadIdx.x >> 5) & (NW - 1);
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const float a = warp_max(mx[v]);
    if (NW == 1) mx[v] = a;
    else if (lane == 0) scratch[v * 4 + warp] = a;
  }
  sync();
  if constexpr (NW > 1) {
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const float4 a = lds_warps<NW>(scratch + v * 4, -CUDART_INF_F);
    mx[v] = fmaxf(fmaxf(a.x, a.y), fmaxf(a.z, a.w));
  }
  }
}

// Group-wide sums (all relative to the same, already global, maximum).
template <int NW, int NV, typename Sync>
__device__ __forceinline__ void stream_sum(float (&s)[NV], float* scratch, Sync sync) {
  const int lane = threadIdx.x & 31, warp = (threadIdx.x >> 5) & (NW - 1);
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const float sw = warp_sum(s[v]);
    if (NW == 1) s[v] = sw;
    else if (lane == 0) scratch[v * 4 + warp] = sw;
  }
  sync();
  if constexpr (NW > 1) {
#pragma unroll
  for (int v = 0; v < NV; ++v) {
    const float4 a = lds_warps<NW>(scratch + v * 4, 0.f);
    s[v] = (a.x + a.y) + (a.z + a.w);
  }
  }
}

// group arg-max of 64-bit keys (rare paths only)
template <int NW, typename Sync>
__device__ __forceinline__ unsigned long long stream_max_u64(unsigned long long key, unsigned long long* scratch, Sync sync) {
  const int lane = threadIdx.x & 31, warp = (threadIdx.x >> 5) & (NW - 1);
  key = warp_max_u64(key);
  if (NW == 1) {
    sync();
    return key;
  }
  if (lane == 0) scratch[warp] = key;
  sync();
  unsigned long long best = scratch[0];
#pragma unroll
  for (int w = 1; w < NW; ++w) best = scratch[w] > best ? scratch[w] : best;
  return best;
}

// Exact finish of a batch of rows from their survivor lists: 16 lanes per row (14 survivors, the [MASK] class,
// the row's own class), every lane scores one class exactly as the log-domain kernel does, a 16-lane
// segmented argmax picks the winner, which is accepted if it clears the row's bound and queued otherwise.
template <int NP, int CPT, bool HAS_U>
__device__ __noinline__ void score_batch(GroupSmem<NP, CPT, HAS_U>& S, int nslots, const ParamNoiseStream& rng, const StepParams& p, int G,
                                         int first_row) {
  using Sh = StreamShape<NP, CPT, HAS_U>;
  constexpr uint32_t K = 1024u * NP;
  const int lane = threadIdx.x & 31, warp = (threadIdx.x >> 5) & (Sh::NW - 1);
  const int sub = lane & 15;
  for (int slot = 2 * warp + (lane >> 4); slot - (lane >> 4) < nslots; slot += 2 * Sh::NW) {
    unsigned long long key = 0ull;
    float lp = 0.f;  // log-posterior of this lane's class (kept for the optional winner_post output)
    const bool live = slot < nslots;
    RowInfo ri;
    ri.accept = 0.f, ri.rel = 0;
    uint32_t cnt = 0;
    if (live) {
      ri = S.info[slot];
      cnt = S.cand_cnt[slot];
      const uint32_t n = cnt < static_cast<uint32_t>(kCandPerRow) ? cnt : static_cast<uint32_t>(kCandPerRow);
      // items 0 .. n-1: the survivors, item n: [MASK], item n+1: the row's own class; one round of 16 lanes, a second one
      // for the rare row with more than 14 survivors
      const uint64_t grow = static_cast<uint64_t>(p.row_offset + (first_row + ri.rel * G));
      for (uint32_t item = static_cast<uint32_t>(sub); item < n + 2u; item += 16u) {
        uint32_t k = 0;
        float P = 0.f;
        bool have = false;
        if (item < n) {
          k = S.cand_k[slot][item];
          const float pe = fminf(fmaxf(S.cand_p[slot][item], kPFloor), 1.0f);
          P = fmaf(pe, ri.A, ri.Bc);
          have = (k != ri.j);  // the row's own class has its own coefficients and its own item
        } else if (item == n) {
          k = K, P = ri.PK, have = true;
        } else if (ri.j != K) {
          k = ri.j, P = ri.Pj, have = true;
        }
        if (have) {
          const float lpk = log_prob_clamped(P);
          const float sc = lpk + gumbel_from_uniform(uniform_from_draw(rng.draw(k, grow)));
          const unsigned long long kk = pack_key(sc, k);
          if (kk > key) key = kk, lp = lpk;
        }
      }
    }
    const unsigned long long mine = key;
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {  // argmax within each 16-lane half
      const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
      key = other > key ? other : key;
    }
    const bool accepted = live && cnt <= static_cast<uint32_t>(kCandPerRow) && key_score(key) >= ri.accept;
    if (live && sub == 0) {
      if (accepted) {
        p.x_prev[first_row + ri.rel * G] = key_class(key);
      } else {
        S.redo[atomicAdd(&S.redo_cnt, 1u)] = ri.rel;
      }
      S.cand_cnt[slot] = 0;
    }
    // verification output: what THIS kernel computed as the posterior log-prob of the class it sampled
    if (p.winner_post != nullptr && accepted && mine == key && mine != 0ull) p.winner_post[first_row + ri.rel * G] = lp;
  }
}

// RECON: the purity-prior variant (draw from p(x0 | x_t), write the purity score); its own instantiation so that the
// plain step's code is not perturbed
template <int NP, int CPT, bool HAS_U, bool RECON, int LD = D3PM_LOGITS_F32>
__global__ void __launch_bounds__(kStreamThreads, 1) step_stream_kernel(const __grid_constant__ StepParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  using Sh = StreamShape<NP, CPT, HAS_U>;
  using Smem = GroupSmem<NP, CPT, HAS_U>;
  constexpr int K = Sh::K, GT = Sh::GT, NW = Sh::NW, NG = Sh::NG, PS = Sh::PS, NCALL = Sh::NCALL;
  constexpr int NC = CPT;  // float4 chunks per thread per tensor
  using LT = LogitType<LD>;
  constexpr uint32_t kRowBytes = K * LT::kBytes;
  uint32_t tid;  // read once: a volatile read cannot be rematerialised as an S2R in every row
  asm volatile("mov.u32 %0, %%tid.x;" : "=r"(tid));
  const int g = tid / GT;
  const int tg = tid % GT;
  Smem& S = reinterpret_cast<Smem*>(smem_raw)[g];
  const StreamSync<NW> sync{g + 1};
  // row indices are 32-bit throughout (the launcher refuses more than 2^31 - 1 rows)
  const int G = static_cast<int>(gridDim.x) * NG;
  const int first_row = g * static_cast<int>(gridDim.x) + static_cast<int>(blockIdx.x);  // neighbouring rows -> different SMs
  const int rows = static_cast<int>(p.rows);
  const uint32_t pitch = static_cast<uint32_t>(p.pitch_logits);
  const bool exact_mode = (p.sample_mode == D3PM_SAMPLE_PHILOX_EXACT);
  // The very first thing a group does is to get its first row moving: the elected thread arms the group's mbarrier and
  // issues the copies, and the set-up below (coefficient table into shared memory, list counters) runs under that latency.
  if (tg == 0) {
    mbar_init(&S.full, 1);
    fence_mbarrier_init();
    S.redo_cnt = 0;
    if (!exact_mode && first_row < rows) {
      const unsigned long long at = static_cast<unsigned long long>(static_cast<uint32_t>(first_row)) * pitch;
      mbar_expect_tx(&S.full, HAS_U ? 2 * kRowBytes : kRowBytes);
      tma_load(S.c, LT::row(p.logits_c, at), kRowBytes, &S.full);
      if (HAS_U) tma_load(S.u, LT::row(p.logits_u, at), kRowBytes, &S.full);
    }
  }
  // CTA-wide copy of the coefficient table (16 floats per timestep) when it fits: per-row lookups become LDS
  float* coef_s = reinterpret_cast<float*>(smem_raw + sizeof(Smem) * NG);
  const bool coef_in_smem = p.T <= kCoefSmemRows;
  if (coef_in_smem) {
    for (int i = tid; i < p.T * 16; i += kStreamThreads)
      coef_s[i] = __ldg(p.coef_table + static_cast<size_t>(i >> 4) * D3PM_COEF_STRIDE + (i & 15));
  }
  const ParamNoiseStream rng(NoiseKeysParam(p.keys), p.offset);  // round keys straight from the parameter block
  const float thin_c = p.thin_factor > 0.f ? p.thin_factor : kStreamThin;
  for (int i = tg; i < Sh::SB; i += GT) S.cand_cnt[i] = 0;
  __syncthreads();  // the table, the counters and every group's barrier are set up

  auto issue_row = [&](int row) {  // elected thread: arm the barrier and launch both row copies
    const unsigned long long at = static_cast<unsigned long long>(static_cast<uint32_t>(row)) * pitch;
    fence_proxy_async();
    mbar_expect_tx(&S.full, HAS_U ? 2 * kRowBytes : kRowBytes);
    tma_load(S.c, LT::row(p.logits_c, at), kRowBytes, &S.full);
    if (HAS_U) tma_load(S.u, LT::row(p.logits_u, at), kRowBytes, &S.full);
  };
  // slot (register chunk index) of the low chunk of coarse call c: chunks q and q + 128 share a call, i.e. slots
  // i and i + PS of the same thread
  auto slot_lo = [](int c) { return (c / PS) * 2 * PS + (c % PS); };

  uint32_t phase = 0;
  uint32_t status_bits = 0;
#ifdef D3PM_STREAM_TIMING  // debug build: p.status is a [groups][8] uint32 trace buffer (word 0 of the grid = origin)
  auto now_ns = [] { unsigned long long v; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(v)); return v; };
  const unsigned long long tm_start = now_ns();
  unsigned long long tm_main = 0;
  uint32_t tm_rows = 0, tm_redo = 0;
#endif

  // ------------------------------------------------------------------------------------------------
  // one row.  `exact` (compile time): rows outside the batched path (PHILOX_EXACT mode and redone rows); otherwise the
  // row's survivors are left in slot `slot` for the next score_batch.
  // ------------------------------------------------------------------------------------------------
  auto process_row = [&](auto exact_c, int row, int next_row, uint32_t j, int tt, int slot, int rel) {
    constexpr bool exact = decltype(exact_c)::value;
    const bool masked = (j == static_cast<uint32_t>(K));
    mbar_wait_spin(&S.full, phase);
    phase ^= 1u;

    // ---- shared -> registers: chunk i of this thread is float4 number GT*i + tg (conflict-free 128-bit
    //      reads); x[i][0] = classes (0,1) of the chunk, x[i][1] = classes (2,3), packed for the f32x2 pipe.
    //      Without guidance the softmax numerators later overwrite x in place (e_of below) ----
    float2 x[NC][2], z[HAS_U ? NC : 1][2];
#pragma unroll
    for (int i = 0; i < NC; ++i) {
      const int q = GT * i + tg;
      LT::chunk(S.c, q, x[i][0], x[i][1]);
      if (HAS_U) LT::chunk(S.u, q, z[i][0], z[i][1]);
    }
    auto e_of = [&](int i, int h) -> float2& {  // the softmax numerators of the row (relative to the thread-local max)
      if constexpr (HAS_U) return z[i][h];
      else return x[i][h];
    };
    const float xj = masked ? 0.f : LT::one(S.c, j);
    const float zj = (HAS_U && !masked) ? LT::one(S.u, j) : 0.f;

    // ---- largest |logit| of each tensor: thread-local, then one cheap group reduction ----
    float am[2] = {0.f, 0.f};
    if (HAS_U) {
      am[0] = fmaxf(fmaxf(fabsf(x[0][0].x), fabsf(x[0][0].y)), fmaxf(fabsf(x[0][1].x), fabsf(x[0][1].y)));
      am[1] = fmaxf(fmaxf(fabsf(z[0][0].x), fabsf(z[0][0].y)), fmaxf(fabsf(z[0][1].x), fabsf(z[0][1].y)));
    }
#pragma unroll
    for (int i = 1; i < NC; ++i) {
      if (HAS_U)
        am[0] = fmaxf(fmaxf(am[0], fabsf(x[i][0].x)), fmaxf(fabsf(x[i][0].y), fmaxf(fabsf(x[i][1].x), fabsf(x[i][1].y))));
      if (HAS_U)
        am[1] = fmaxf(fmaxf(am[1], fabsf(z[i][0].x)), fmaxf(fabsf(z[i][0].y), fmaxf(fabsf(z[i][1].x), fabsf(z[i][1].y))));
    }
    if (HAS_U) stream_max<NW, 2>(am, S.red[0], sync);  // barrier 1: every thread is done with the stage
    else sync();                                        // (without guidance nothing depends on the range of the logits)
    // the stage is free: prefetch the next row now (exhaustive rows park their numerators in it first)
    if (!exact && tg == 0 && next_row >= 0) issue_row(next_row);  // (`exact` is a constant here)

    const uint64_t grow = static_cast<uint64_t>(p.row_offset + row);

    float My2, rSy, r, yj;
    const float2 l2e = make_float2(kLog2e, kLog2e);
    if (HAS_U) {
      // ---- guidance combine (:245) ----
      const float gs = p.guidance_scale, og = 1.0f - gs;
      const float2 gs2 = make_float2(gs, gs), og2 = make_float2(og, og);
      float my = -CUDART_INF_F;
      // log-softmax can only reach the -70 clamp of :236 if some logit lies more than 70 - ln K below the row
      // maximum (lse <= max + ln K).  When |logit| <= (70 - ln K) / 2 throughout neither tensor can, both
      // normalisers are constants that cancel in the renormalisation of :246, so  y = s c + (1 - s) u  up to a
      // constant: no exponential of the raw logits is needed.  (|y| stays below ~100, two fused roundings.)
      constexpr float kLnK = NP == 4 ? 8.3178f : (NP == 2 ? 7.6247f : 6.9315f);
      constexpr float kSafeAbs = 0.5f * (69.99f - kLnK);
      const bool no_clamp = (am[0] <= kSafeAbs) && (am[1] <= kSafeAbs) && (fabsf(gs) * am[0] + fabsf(og) * am[1] <= 160.0f);
      if (no_clamp) {
#pragma unroll
        for (int i = 0; i < NC; ++i)
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const float2 y = __ffma2_rn(gs2, x[i][h], __fmul2_rn(og2, z[i][h]));
            x[i][h] = y;
            my = fmaxf(my, fmaxf(y.x, y.y));
          }
        yj = fmaf(gs, xj, og * zj);
      } else {
        // general path: softmax normalisers of both tensors (:231), clamps of :236 applied as thresholds.
        // With a = x - max, log-softmax clamped at -70 is max(a, -70 + lnS) - lnS, so
        //   y = lu + s (lc - lu) = s a' + (1 - s) b' + C,  C = -s lnSc - (1 - s) lnSu
        float mx[2], s[2];
        mx[0] = fmaxf(fmaxf(x[0][0].x, x[0][0].y), fmaxf(x[0][1].x, x[0][1].y));
        mx[1] = fmaxf(fmaxf(z[0][0].x, z[0][0].y), fmaxf(z[0][1].x, z[0][1].y));
#pragma unroll
        for (int i = 1; i < NC; ++i) {
          mx[0] = fmaxf(fmaxf(mx[0], x[i][0].x), fmaxf(x[i][0].y, fmaxf(x[i][1].x, x[i][1].y)));
          mx[1] = fmaxf(fmaxf(mx[1], z[i][0].x), fmaxf(z[i][0].y, fmaxf(z[i][1].x, z[i][1].y)));
        }
        stream_max<NW, 2>(mx, S.red[2], sync);  // extra barriers, general path only
        mx[0] = fmaxf(mx[0], -3.0e38f), mx[1] = fmaxf(mx[1], -3.0e38f);  // an all--inf row stays finite
        {
          const float mc2 = to_log2_units(mx[0]), mu2 = to_log2_units(mx[1]);
          const float2 nmc = make_float2(-mc2, -mc2), nmu = make_float2(-mu2, -mu2);
          float2 sc[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)}, su[2] = {sc[0], sc[0]};
#pragma unroll
          for (int i = 0; i < NC; ++i)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const float2 ac = __ffma2_rn(x[i][h], l2e, nmc), au = __ffma2_rn(z[i][h], l2e, nmu);
              sc[h] = __fadd2_rn(sc[h], make_float2(ex2(ac.x), ex2(ac.y)));
              su[h] = __fadd2_rn(su[h], make_float2(ex2(au.x), ex2(au.y)));
            }
          s[0] = (sc[0].x + sc[0].y) + (sc[1].x + sc[1].y);
          s[1] = (su[0].x + su[0].y) + (su[1].x + su[1].y);
        }
        stream_sum<NW, 2>(s, S.red[2] + 2 * 4, sync);
        const float lnSc = ln_rel_sum(mx[0], s[0]), lnSu = ln_rel_sum(mx[1], s[1]);
        const float ta = kClampLo + lnSc, tb = kClampLo + lnSu;
        const float C = fmaf(-gs, lnSc, -og * lnSu);
        const float2 nMc = make_float2(-mx[0], -mx[0]), nMu = make_float2(-mx[1], -mx[1]), C2 = make_float2(C, C);
#pragma unroll
        for (int i = 0; i < NC; ++i)
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            float2 a = __fadd2_rn(x[i][h], nMc), b = __fadd2_rn(z[i][h], nMu);
            a.x = fmaxf(a.x, ta), a.y = fmaxf(a.y, ta);
            b.x = fmaxf(b.x, tb), b.y = fmaxf(b.y, tb);
            const float2 y = __ffma2_rn(gs2, a, __ffma2_rn(og2, b, C2));
            x[i][h] = y;
            my = fmaxf(my, fmaxf(y.x, y.y));
          }
        yj = fmaf(gs, fmaxf(xj - mx[0], ta), fmaf(og, fmaxf(zj - mx[1], tb), C));
      }
      // ---- renormalisation (:246): numerators relative to the thread-local max, one reduction ----
      const float my2 = to_log2_units(my);
      {
        const float2 nmy = make_float2(-my2, -my2);
        float2 sy[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
#pragma unroll
        for (int i = 0; i < NC; ++i)
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const float2 ay = __ffma2_rn(x[i][h], l2e, nmy);
            const float2 ey = make_float2(ex2(ay.x), ex2(ay.y));
            e_of(i, h) = ey;
            sy[h] = __fadd2_rn(sy[h], ey);
          }
        float mm[1] = {my}, ss[1] = {(sy[0].x + sy[0].y) + (sy[1].x + sy[1].y)};
        stream_max_sum<NW, 1>(mm, ss, S.red[1], sync);  // barrier 2
        My2 = to_log2_units(mm[0]);
        rSy = __fdividef(1.0f, ss[0]);
      }
      r = ex2(my2 - My2) * rSy;
    } else {
      // ---- guidance off: p(x0) is the softmax of the conditional logits alone (predict_start, :231-236) ----
      float mx[1];
      mx[0] = fmaxf(fmaxf(x[0][0].x, x[0][0].y), fmaxf(x[0][1].x, x[0][1].y));
#pragma unroll
      for (int i = 1; i < NC; ++i) mx[0] = fmaxf(fmaxf(mx[0], x[i][0].x), fmaxf(x[i][0].y, fmaxf(x[i][1].x, x[i][1].y)));
      mx[0] = fmaxf(mx[0], -3.0e38f);
      const float mc2 = to_log2_units(mx[0]);  // thread-local max: one reduction yields both max and sum
      const float2 nmc = make_float2(-mc2, -mc2);
      float2 sc[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
#pragma unroll
      for (int i = 0; i < NC; ++i)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const float2 ac = __ffma2_rn(x[i][h], l2e, nmc);
          const float2 ec = make_float2(ex2(ac.x), ex2(ac.y));
          e_of(i, h) = ec;  // in place: the logits themselves are not needed any more
          sc[h] = __fadd2_rn(sc[h], ec);
        }
      float ss[1] = {(sc[0].x + sc[0].y) + (sc[1].x + sc[1].y)};
      stream_max_sum<NW, 1>(mx, ss, S.red[1], sync);  // barrier 2
      My2 = to_log2_units(mx[0]);
      rSy = __fdividef(1.0f, ss[0]);
      r = ex2(mc2 - My2) * rSy;
      yj = xj;
    }
    const float pj = masked ? 0.f : fminf(fmaxf(ex2(fmaf(yj, kLog2e, -My2)) * rSy, kPFloor), 1.0f);
    RowCoef cf;
    if (coef_in_smem) {
      const float* crow = coef_s + tt * 16 + (masked ? 0 : 8);
      cf = row_coef_from(lds4(crow), lds4(crow + 4), masked);
    } else {
      cf = load_row_coef(p.coef_table, tt, masked);
    }
    RowMath rm;
    if (RECON) {
      // purity-prior sampling (:309-346) draws the candidate from p(x0 | x_t) itself and scores the token by its
      // largest probability, 1 / (sum of the softmax numerators relative to the row maximum)
      rm.init_recon(masked ? 0.f : pj, masked ? static_cast<uint32_t>(K) + 1u : j);
      if (tg == 0 && p.score != nullptr) p.score[row] = fminf(fmaxf(rSy, kPFloor), 1.0f);
    } else {
      rm.init(cf, masked, pj, j, K);
    }

    if constexpr (!exact) {
      // ---- thinned race: 16 noise bits per class, survivors go to this row's slot.  One Philox call = 8 x 16 bits:
      //      word w of call c serves classes (2w, 2w+1) of chunk slot_lo(c) (w < 2) / slot_lo(c) + PS (w >= 2);
      //      four calls are drawn together (four independent Philox chains to interleave) ----
      const ThinRule thin(rm, thin_c);
      const float thrA = r * thin.scaleA, nthrB = -thin.thrB;
      const float2 tA2 = make_float2(thrA, thrA);
      if (tg == 0) {
        RowInfo ri;
        ri.A = rm.A, ri.Bc = rm.Bc, ri.Pj = rm.Pj, ri.PK = rm.PK, ri.accept = thin.accept;
        ri.j = j, ri.rel = rel, ri.pad = 0;
        S.info[slot] = ri;
      }
#pragma unroll
      for (int c0 = 0; c0 < NCALL; c0 += 4) {
        uint4 cws[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) cws[c] = rng.coarse(ParamNoiseStream::coarse_call_of_chunk(GT * slot_lo(c0 + c) + tg), grow);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const int lo = slot_lo(c0 + c);
          // the halves are spliced under the exponent of -1.0f so that nf = -(1 + h 2^-23) comes out of one PRMT; a class
          // survives when e thrA + nf >= -thrB (one packed FMA per two classes, the comparison once per call)
          const uint32_t w4[4] = {cws[c].x, cws[c].y, cws[c].z, cws[c].w};
          float slack = -4.0f;  // max over the 8 classes of e thrA + nf
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            const float2 nf = make_float2(__uint_as_float(__byte_perm(w4[w], 0xbf80u, 0x5410)),
                                          __uint_as_float(__byte_perm(w4[w], 0xbf80u, 0x5432)));
            const float2 d = __ffma2_rn(e_of(lo + (w >> 1) * PS, w & 1), tA2, nf);
            slack = fmaxf(slack, fmaxf(d.x, d.y));
          }
          if (slack >= nthrB) {
#pragma unroll
            for (int w = 0; w < 4; ++w)
#pragma unroll
              for (int hl = 0; hl < 2; ++hl) {
                const float2 ee = e_of(lo + (w >> 1) * PS, w & 1);
                const float e = hl ? ee.y : ee.x;
                const uint32_t h16 = hl ? (w4[w] >> 16) : (w4[w] & 0xffffu);
                const float nf = __uint_as_float(0xbf800000u | h16);
                if (fmaf(e, thrA, nf) >= nthrB) {
                  const uint32_t pos = atomicAdd(&S.cand_cnt[slot], 1u);
                  if (pos < static_cast<uint32_t>(kCandPerRow)) {
                    S.cand_k[slot][pos] = 4u * (GT * (lo + (w >> 1) * PS) + tg) + 2u * (w & 1) + hl;
                    S.cand_p[slot][pos] = e * r;
                  }
                }
              }
          }
        }
      }
      return;
    } else {
    // ---- rows outside the batched path ----
    unsigned long long best = 0ull;
    float best_lp = 0.f;  // log-posterior of this thread's best class (winner_post output)
    bool settled = false;
    if (!exact_mode) {
      // a row whose best survivor missed the acceptance bound: the same thinned race at a bound that fails with
      // probability e^-16, survivors scored on the spot (exactly as score_batch scores them)
      // (a test knob: thin_factor < 0.01 is used for this attempt too, which then fails and reaches the code below)
      const ThinRule thin2(rm, (p.thin_factor > 0.f && p.thin_factor < 0.01f) ? p.thin_factor : kRedoThin);
      const float thrA = r * thin2.scaleA;
      const float2 tA2 = make_float2(thrA, thrA), tB2 = make_float2(thin2.thrB, thin2.thrB);
#pragma unroll
      for (int c = 0; c < NCALL; ++c) {
        const int lo = slot_lo(c);
        const uint4 cw = rng.coarse(ParamNoiseStream::coarse_call_of_chunk(GT * lo + tg), grow);
        const uint32_t w4[4] = {cw.x, cw.y, cw.z, cw.w};
        uint32_t hits = 0;  // bit 2 w + h: class h of word w passed the coarse test
        float ev[8];
#pragma unroll
        for (int w = 0; w < 4; ++w) {
          const float2 ee = e_of(lo + (w >> 1) * PS, w & 1);
          ev[2 * w] = ee.x, ev[2 * w + 1] = ee.y;
          const float2 nf = make_float2(__uint_as_float(__byte_perm(w4[w], 0xbf80u, 0x5410)),
                                        __uint_as_float(__byte_perm(w4[w], 0xbf80u, 0x5432)));
          const float2 d = __ffma2_rn(ee, tA2, __fadd2_rn(tB2, nf));
          hits |= (d.x >= 0.0f ? 1u : 0u) << (2 * w);
          hits |= (d.y >= 0.0f ? 1u : 0u) << (2 * w + 1);
        }
        while (hits != 0) {  // ~16 classes per row in all
          const int b = __ffs(hits) - 1;
          hits &= hits - 1;
          float e = 0.f;
#pragma unroll
          for (int q = 0; q < 8; ++q) e = (b == q) ? ev[q] : e;  // picked with selects, never through memory
          const uint32_t k = 4u * (GT * (lo + (b >> 2) * PS) + tg) + static_cast<uint32_t>(b & 3);
          if (k != j) {
            const float lpk = rm.post_of(k, e, r);
            const unsigned long long key = pack_key(lpk + gumbel_from_uniform(uniform_from_draw(rng.draw(k, grow))), k);
            if (key > best) best = key, best_lp = lpk;
          }
        }
      }
      if (tg == 0) {
        const float lpk = rm.post_mask();
        const unsigned long long key = pack_key(lpk + gumbel_from_uniform(uniform_from_draw(rng.draw(K, grow))), K);
        if (key > best) best = key, best_lp = lpk;
      }
      if (tg == GT - 1 && !masked) {  // the row's own class has its own coefficients
        const float lpk = rm.post_self();
        const unsigned long long key = pack_key(lpk + gumbel_from_uniform(uniform_from_draw(rng.draw(j, grow))), j);
        if (key > best) best = key, best_lp = lpk;
      }
      const unsigned long long mine = best;
      best = stream_max_u64<NW>(best, S.keys, sync);  // barrier 3
      settled = key_score(best) >= thin2.accept;
      if (settled) {
        if (p.winner_post != nullptr && mine == best) p.winner_post[row] = best_lp;
      } else {
        best = 0ull;
        sync();  // S.keys is about to be reused
      }
    }
    if (!settled) {
      // ---- exhaustive scoring (PHILOX_EXACT mode, or the second attempt failed too): kept small rather than
      //      fast.  The softmax numerators are parked in the idle conditional stage (the prefetch of the next row is
      //      deferred to the end of an exhaustive row) and scored in a rolled loop.
#pragma unroll
      for (int i = 0; i < NC; ++i) {
        const float2 a = e_of(i, 0), b = e_of(i, 1);
        *reinterpret_cast<float4*>(S.c + 4 * (GT * i + tg)) = make_float4(a.x, a.y, b.x, b.y);
      }
#pragma unroll 1
      for (int i = 0; i < NC; ++i) {
        const uint32_t q = static_cast<uint32_t>(GT) * i + tg;
        const float4 e4 = lds4(S.c + 4 * q);
        const float ev[4] = {e4.x, e4.y, e4.z, e4.w};
        const uint4 cw = rng.coarse(ParamNoiseStream::coarse_call_of_chunk(q), grow);
        const uint4 fw = rng.fine(q >> 2, grow);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const uint32_t k = 4u * q + e;
          const uint32_t mdraw =
              (ParamNoiseStream::half_of(cw, (((q >> 7) & 1u) << 2) | e) << 7) | ParamNoiseStream::low7_of(fw, ((q & 3u) << 2) | e);
          const float lpk = rm.post_of(k, ev[e], r);
          const unsigned long long key = pack_key(lpk + gumbel_from_uniform(uniform_from_draw(mdraw)), k);
          if (key > best) best = key, best_lp = lpk;
        }
      }
      if (tg == 0) {
        const float lpk = rm.post_mask();
        const unsigned long long key = pack_key(lpk + gumbel_from_uniform(uniform_from_draw(rng.draw(K, grow))), K);
        if (key > best) best = key, best_lp = lpk;
      }
      const unsigned long long mine = best;
      best = stream_max_u64<NW>(best, S.keys, sync);  // barrier 3 (also: every thread has read its parked numerators)
      if (p.winner_post != nullptr && mine == best) p.winner_post[row] = best_lp;
    }
    if (tg == 0) {
      p.x_prev[row] = key_class(best);
      if (next_row >= 0) issue_row(next_row);
    }
    }
  };

  // ---- the group's rows (main pass, batched scoring), then the rows it queued - or, in PHILOX_EXACT mode, all of them ----
  const int N = p.N;
  auto token_of = [&](int r_) { return static_cast<long long>(p.x_t[r_]); };
  auto time_of = [&](int b_) { return static_cast<long long>(p.t[b_]); };
  // range checks of a row's scalars (the reference asserts them on the host, :45-46, :253)
  auto checked = [&](long long tt, long long jj, int& t_cur, uint32_t& j_cur) {
    if (static_cast<unsigned long long>(tt) >= static_cast<unsigned long long>(p.T)) {
      status_bits |= D3PM_STATUS_BAD_T;
      tt = tt < 0 ? 0 : p.T - 1;
    }
    if (static_cast<unsigned long long>(jj) > static_cast<unsigned long long>(K)) {
      status_bits |= D3PM_STATUS_BAD_TOKEN;
      jj = K;
    }
    t_cur = static_cast<int>(tt), j_cur = static_cast<uint32_t>(jj);
    // consume the scalars (loaded one row ahead) BEFORE the next prefetch is issued: the consumer waits on the scoreboard
    // slot the loads share, so the other order would stall on the loads just issued
    asm volatile("" : "+r"(t_cur), "+r"(j_cur) : : "memory");
  };
  if (!exact_mode) {
    const int stepB = G / N, stepR = G % N;  // video index b = row / N is tracked incrementally (row advances by G)
    int vb = first_row / N, vr = first_row % N;
    int row = first_row < rows ? first_row : -1;
    long long jj = 0, tt = 0;
    if (row >= 0) {  // (its copies were issued at the top of the kernel)
      jj = token_of(row);
      tt = time_of(vb);
    }
    int it = 0, in_batch = 0;
    while (row >= 0) {
      int t_cur;
      uint32_t j_cur;
      checked(tt, jj, t_cur, j_cur);
      const int next = row + G < rows ? row + G : -1;
      vb += stepB, vr += stepR;
      if (vr >= N) vr -= N, ++vb;
      if (next >= 0) {  // software prefetch of the next row's scalars
        jj = token_of(next);
        tt = time_of(vb);
      }
      process_row(std::false_type{}, row, next, j_cur, t_cur, in_batch, it);
#ifdef D3PM_STREAM_TIMING
      ++tm_rows;
#endif
      row = next;
      ++it;
      if (++in_batch == Sh::SB || row < 0) {  // finish the rows accumulated so far
        sync();  // every thread has finished appending survivors
        score_batch<NP, CPT, HAS_U>(S, in_batch, rng, p, G, first_row);
        sync();  // slots may be reused, redo_cnt is final for this batch
        in_batch = 0;
      }
    }
  }
#ifdef D3PM_STREAM_TIMING
  tm_main = now_ns();
#endif
  {
    const uint32_t n2 = exact_mode ? (first_row < rows ? static_cast<uint32_t>((rows - first_row + G - 1) / G) : 0u) : S.redo_cnt;
    auto row_at = [&](uint32_t i) { return first_row + (exact_mode ? static_cast<int>(i) : S.redo[i]) * G; };
    if (n2 > 0) {
      if (!exact_mode) status_bits |= D3PM_STATUS_FALLBACK;
      int row = row_at(0);
      if (tg == 0) issue_row(row);
      long long jj = token_of(row), tt = time_of(row / N);
      for (uint32_t i = 0; i < n2; ++i) {
        int t_cur;
        uint32_t j_cur;
        checked(tt, jj, t_cur, j_cur);
        const int next = (i + 1 < n2) ? row_at(i + 1) : -1;
        if (next >= 0) {
          jj = token_of(next);
          tt = time_of(next / N);
        }
        process_row(std::true_type{}, row, next, j_cur, t_cur, 0, 0);
#ifdef D3PM_STREAM_TIMING
        ++tm_redo;
#endif
        row = next;
      }
    }
  }
#ifdef D3PM_STREAM_TIMING
  if (tg == 0 && p.status != nullptr) {
    const unsigned long long tm_end = now_ns();
    uint32_t* o = p.status + 8 * (blockIdx.x * NG + g);
    uint32_t smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    o[0] = static_cast<uint32_t>(tm_start), o[1] = static_cast<uint32_t>(tm_start >> 32);
    o[2] = static_cast<uint32_t>(tm_main - tm_start), o[3] = static_cast<uint32_t>(tm_end - tm_start);
    o[4] = tm_rows, o[5] = tm_redo, o[6] = smid, o[7] = 0;
  }
#else
  if (status_bits != 0 && tg == 0 && p.status != nullptr) atomicOr(p.status, status_bits);
#endif
}

constexpr long long kStreamMinRows = 1024;  // below this the one-CTA-per-row kernel has less latency (config 1, 1024
                                            // rows: 14.6 us here, 20.6 us there)

inline bool stream_kernel_supports(const StepParams& p) {
  if (p.sample_mode != D3PM_SAMPLE_PHILOX && p.sample_mode != D3PM_SAMPLE_PHILOX_EXACT) return false;
  if (p.post != nullptr || p.recon != nullptr || p.gap != nullptr || p.x_prev == nullptr) return false;
  if (p.sharpen != nullptr || (p.score != nullptr && p.sample_from != D3PM_FROM_RECON)) return false;
  if (p.K != 1024 && p.K != 2048 && p.K != 4096) return false;
  if (p.pitch_logits >= (1LL << 32)) return false;  // row offsets are formed as 32 x 32 -> 64 bit products
  if (p.logits_dtype != D3PM_LOGITS_F32 && (p.sample_from == D3PM_FROM_RECON || p.pitch_logits % 8 != 0)) return false;
  return true;
}

// every group must be able to queue all of its rows for rescoring (RC * NG = 8192 rows per CTA in every shape)
inline long long stream_kernel_max_rows() { return 8192LL * host::sm_count(); }

template <int NP, int CPT, bool HAS_U>
int launch_step_stream_t(const StepParams& p, cudaStream_t s) {
  const size_t smem = sizeof(GroupSmem<NP, CPT, HAS_U>) * StreamShape<NP, CPT, HAS_U>::NG + kCoefSmemRows * 16 * sizeof(float);
  const bool recon = p.sample_from == D3PM_FROM_RECON;
  // 16-bit logits: the plain step only (the purity-prior draw of an autocast caller goes through a cast)
  if (p.logits_dtype == D3PM_LOGITS_F16)
    return recon ? D3PM_ERR_UNSUPPORTED : launch_persistent(step_stream_kernel<NP, CPT, HAS_U, false, D3PM_LOGITS_F16>, kStreamThreads, smem, p, s);
  if (p.logits_dtype == D3PM_LOGITS_BF16)
    return recon ? D3PM_ERR_UNSUPPORTED : launch_persistent(step_stream_kernel<NP, CPT, HAS_U, false, D3PM_LOGITS_BF16>, kStreamThreads, smem, p, s);
  return launch_persistent(recon ? step_stream_kernel<NP, CPT, HAS_U, true> : step_stream_kernel<NP, CPT, HAS_U, false>,
                           kStreamThreads, smem, p, s);
}

inline int launch_step_stream(const StepParams& p, cudaStream_t s) {
  const bool has_u = p.logits_u != nullptr;
  switch (p.K) {
    case 1024: return has_u ? launch_step_stream_t<1, 8, true>(p, s) : launch_step_stream_t<1, 8, false>(p, s);
    case 2048: return has_u ? launch_step_stream_t<2, 8, true>(p, s) : launch_step_stream_t<2, 16, false>(p, s);
    case 4096: return has_u ? launch_step_stream_t<4, 8, true>(p, s) : launch_step_stream_t<4, 16, false>(p, s);
    default: return D3PM_ERR_UNSUPPORTED;
  }
}

}  // namespace d3pm
