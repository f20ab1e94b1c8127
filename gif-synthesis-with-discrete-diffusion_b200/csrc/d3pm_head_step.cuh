// Fused denoiser head + reverse step (SURVEY.md §8 f3): the [B, N, K] logits never touch HBM.
//
// Replaces, in one kernel, the reference's prediction head `to_logits = LayerNorm(D) + Linear(D -> K)`
// (transformer_utils.py:352-356, applied at :441) for BOTH denoiser passes of a step, plus everything
// d3pm_fused_step replaces (predict_start / cf_predict_start / q_posterior / log_sample_categorical,
// diffusion_transformer.py:220-283, :354-359).  Inputs are the hidden states that feed the head.
//
// Mathematics.  Rows whose logits cannot reach the -70 clamps of :236 (|logit| <= (70 - ln K) / 2, guaranteed for ALL
// rows by a bound on the weights that the host checks once, see d3pm_head_prepare) satisfy
//     y = s * log_softmax(c) + (1 - s) * log_softmax(u) = W (s a_c + (1 - s) a_u) + b + const,
// a_* = LayerNorm(h_*): the guidance combine moves in front of the GEMM, so ONE [128 x D] x [D x K] product per token
// tile yields the combined logits.  The product runs on the 5th-gen tensor cores (tcgen05.mma, kind::tf32, M = 128,
// N = 128, accumulators in TMEM) as a 3xTF32 split (a_hi w_hi + a_lo w_hi + a_hi w_lo, fp32-grade accuracy).
// A 128 x K fp32 tile of logits (2 MB) does not fit on chip, so the kernel makes two passes over the classes, recomputing
// the product: pass 1 accumulates the softmax statistics (max, sum) of every row, pass 2 regenerates the logits and runs
// the thinned exponential race of the stream kernel (same Philox stream, same ThinRule, same exact scoring of the
// survivors), so a token differs from the unfused path only where the logits' last bits decide a near-tie.
//
// Roles (576 threads, one CTA per SM, persistent over 128-token tiles):
//   warp 0      one lane issues tcgen05.mma and the tcgen05.commit's that drive the mbarrier pipeline
//   warps 1-16  (a) produce the A operand of the tile: LayerNorm, guidance combine, hi/lo split, 128B-swizzled K-major
//               canonical layout in shared memory; (b) epilogue: tcgen05.ld a TMEM lane (= token row) per thread, so all
//               row reductions are thread-local (four threads per row, one per quarter of the columns)
//   warp 17     one lane streams the pre-swizzled weight image (hi and lo, 64 KiB per 128 classes) through a two-stage
//               shared-memory ring with 1-D bulk TMA
// TMEM: 4 accumulators of 128 columns (all 512 columns); the epilogue consumes them in pairs 512 classes apart because one
// Philox call serves classes (4c..4c+3) and (4c+512..4c+515).
#pragma once

#include "d3pm_ptx.cuh"
#include "d3pm_step_rows.cuh"

namespace d3pm {
namespace head {

constexpr int kTileM = 128;      // token rows per tile = TMEM lanes
constexpr int kChunk = 128;      // classes per accumulator and per weight stage
constexpr int kAccStages = 4;
constexpr int kBStages = 2;
constexpr int kEpiWarps = 16;    // 4 per TMEM lane quarter: each thread owns one row and a quarter of the columns
constexpr int kColSplit = kEpiWarps / 4;
constexpr int kCols = kChunk / kColSplit;  // columns of a chunk per thread (32)
constexpr int kEpiThreads = 32 * kEpiWarps;
constexpr int kThreads = 32 * (kEpiWarps + 2);
constexpr int kRowThreads4 = kEpiThreads / kTileM;  // threads that build one row of the A operand (4)
static_assert(kCols == 32 && kRowThreads4 == 4, "the epilogue below is written for 16 epilogue warps");
// Survivor lists of 28 classes per row and a thinning constant of 8 (the unfused kernels: 14 and 6): a row the race
// cannot decide costs a whole CTA of head_redo_kernel (2 MiB of weight image through L2, ~25 us), so they are made
// rare - e^-8 of the rows, ~20 per 65 536 - at the price of 8 instead of 6 survivors per row to score.
constexpr int kCand = 28;
constexpr float kThin = 8.0f;
constexpr int kBlockBytes = kTileM * 128;  // one 128-byte k-block of a 128-row operand
constexpr uint32_t kIdesc = idesc_tf32(kTileM, kChunk);

struct HeadParams {
  const float* hidden_c;  // [rows][D]
  const float* hidden_u;  // nullable (guidance off)
  const float* ln_weight;
  const float* ln_bias;
  const float* w_image;   // [K/128][2 terms][D/32][128 rows x 128 B, swizzled], scaled by log2(e)
  const float* bias2;     // [K], scaled by log2(e)
  const int64_t* x_t;
  const int64_t* t;
  const float* coef_table;
  int64_t* x_prev;
  float* logits_out;      // dump mode: [rows][K] combined logits (natural units)
  uint32_t* status;
  int32_t* redo_rows;
  uint32_t* redo_count;
  int32_t N, K, T;
  int64_t rows;
  float ln_eps, guidance_scale, thin_factor;
  float stat_slack;       // > 0: the statistics pass runs in 1xTF32 and its logits are within this many log2 units of the exact ones
  uint64_t seed, offset;
  int64_t row_offset;
};

template <int D>
struct Geo {
  static_assert(D == 64, "the fused head is built for n_embd = 64 (configs/model/motionencoder/transformer_utils.yaml)");
  static constexpr int KB = D / 32;
  static constexpr int kTermBytes = KB * kBlockBytes;  // hi (or lo) part of a 128-row operand
  static constexpr int kABytes = 2 * kTermBytes;
  static constexpr int kBStageBytes = 2 * kTermBytes;
  static constexpr int kOperandBytes = kABytes + kBStages * kBStageBytes;
  static constexpr int kChunkFloats = kBStageBytes / 4;  // floats of the weight image per 128 classes
};

struct HeadRowInfo {  // what score_tile needs to finish a row exactly
  uint32_t j;      // x_t, == K when masked
  int32_t tt;      // timestep of the row's video
  float yj_rel;    // log2-unit logit of class x_t minus the row's stabiliser
  float pad;
};

struct Ctl {
  unsigned long long b_full[kBStages], b_empty[kBStages], acc_full[kAccStages], acc_empty[kAccStages], a_ready, a_free;
  uint32_t tmem_base, pad;
  float stat_m[kColSplit][kTileM], stat_s[kColSplit][kTileM];
  float yj2[kTileM];
  float sum2[kColSplit][kTileM];   // pass 2: the exact sum of the row's numerators, per column quarter
  HeadRowInfo info[kTileM];
  uint32_t cand_cnt[kTileM];
  float cand_p[kTileM][kCand];     // softmax NUMERATORS of the survivors (relative to the row's stabiliser)
  uint16_t cand_k[kTileM][kCand];  // K <= 8192
};

template <int D>
constexpr size_t smem_bytes() {
  return 1024 + Geo<D>::kOperandBytes + sizeof(Ctl);
}

__device__ __forceinline__ void epi_bar() { asm volatile("bar.sync 1, %0;" ::"n"(kEpiThreads) : "memory"); }

// class chunk processed at position `ci` of a pass: pairs (p, p + 4) inside every block of 8 chunks (1024 classes)
__device__ __forceinline__ int chunk_of(int ci) { return (ci & ~7) + ((ci & 7) >> 1) + ((ci & 1) << 2); }

// float offset, inside the weight image, of the 16-byte piece `piece` (4 floats of hidden dims 32 kb + 4 piece ..) of
// class k: image[k / 128][term][kb][k % 128][(piece ^ (k % 8)) * 4 ..]
template <int D>
__device__ __host__ __forceinline__ size_t image_offset(int k, int term, int kb, int piece) {
  const int r = k & 127;
  return static_cast<size_t>(k >> 7) * Geo<D>::kChunkFloats + static_cast<size_t>(term * Geo<D>::KB + kb) * (kBlockBytes / 4) +
         r * 32 + ((piece ^ (r & 7)) << 2);
}

// ---- weight preparation --------------------------------------------------------------------------------------
// One thread per (class, 4 hidden dims).  w' = w * log2(e); hi = w' with the 13 low mantissa bits cleared (exactly a
// tf32 number), lo = w' - hi (exact in fp32).  stats[0] = max_k ||w_k||_2, stats[1] = max_k |b_k| (as float bits).
template <int D>
__global__ void head_prepare_kernel(const float* __restrict__ weight, const float* __restrict__ bias, int K,
                                    float* __restrict__ image, float* __restrict__ bias2, uint32_t* __restrict__ stats) {
  constexpr int PPR = D / 4;  // 16-byte pieces per class
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int k = idx / PPR, pp = idx % PPR;
  float ss = 0.f;
  if (k < K) {
    const float4 w = *reinterpret_cast<const float4*>(weight + static_cast<size_t>(k) * D + 4 * pp);
    const float v[4] = {w.x, w.y, w.z, w.w};
    float hi[4], lo[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float s = v[e] * kLog2e;
      hi[e] = __uint_as_float(__float_as_uint(s) & 0xffffe000u);
      lo[e] = s - hi[e];
      ss = fmaf(v[e], v[e], ss);
    }
    const int kb = pp >> 3, piece = pp & 7;
    *reinterpret_cast<float4*>(image + image_offset<D>(k, 0, kb, piece)) = make_float4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<float4*>(image + image_offset<D>(k, 1, kb, piece)) = make_float4(lo[0], lo[1], lo[2], lo[3]);
    if (pp == 0) {
      const float b = bias != nullptr ? bias[k] : 0.f;
      bias2[k] = b * kLog2e;
      atomicMax(stats + 1, __float_as_uint(fabsf(b)));
    }
  }
  // the PPR threads of a class are adjacent lanes (PPR = 16 divides 32)
#pragma unroll
  for (int o = PPR / 2; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  if (k < K && pp == 0) atomicMax(stats, __float_as_uint(sqrtf(ss)));
}

// LayerNorm of 16 of the 64 hidden values of a row held by this thread (4 adjacent lanes hold a row; part = which 16).
__device__ __forceinline__ void layer_norm_part(float (&x)[16], const float* __restrict__ gamma, const float* __restrict__ beta,
                                                int part, float eps) {
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) sum += x[i];
  sum += __shfl_xor_sync(0xffffffffu, sum, 1);
  sum += __shfl_xor_sync(0xffffffffu, sum, 2);
  const float mean = sum * (1.0f / 64.0f);
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const float d = x[i] - mean;
    sq = fmaf(d, d, sq);
  }
  sq += __shfl_xor_sync(0xffffffffu, sq, 1);
  sq += __shfl_xor_sync(0xffffffffu, sq, 2);
  const float rstd = 1.0f / sqrtf(sq * (1.0f / 64.0f) + eps);
#pragma unroll
  for (int i = 0; i < 16; ++i) x[i] = fmaf((x[i] - mean) * rstd, __ldg(gamma + 16 * part + i), __ldg(beta + 16 * part + i));
}

// ---- the kernel ----------------------------------------------------------------------------------------------
template <int D, bool HAS_U, bool DUMP>
__global__ void __launch_bounds__(kThreads, 1) head_step_kernel(const HeadParams p) {
  using G = Geo<D>;
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
  unsigned char* sA = smem;
  unsigned char* sB = smem + G::kABytes;
  Ctl& C = *reinterpret_cast<Ctl*>(smem + G::kOperandBytes);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int NCH = p.K / kChunk;                // chunks per pass
  const int NIT = DUMP ? NCH : 2 * NCH;        // accumulator iterations per tile
  const bool stat1x = !DUMP && p.stat_slack > 0.f;
  const long long ntiles = (p.rows + kTileM - 1) / kTileM;

  if (tid == 0) {
    // A fence after every init, as the kernel was tuned.  One fence after all of them changes the machine code only in
    // this set-up (and the addresses of everything behind it), yet measured 0.15 % slower (B200 at 1000 W).
    auto init = [](unsigned long long* bar, uint32_t count) { mbar_init(bar, count), fence_mbarrier_init(); };
    for (int i = 0; i < kBStages; ++i) init(&C.b_full[i], 1), init(&C.b_empty[i], 1);
    for (int i = 0; i < kAccStages; ++i) init(&C.acc_full[i], 1), init(&C.acc_empty[i], kEpiWarps);
    init(&C.a_ready, kEpiThreads);
    init(&C.a_free, 1);
  }
  if (tid < kTileM) C.cand_cnt[tid] = 0;
  if (warp == 0) {  // the whole tensor memory: 4 accumulators x 128 columns
    tmem_alloc<1, 512>(&C.tmem_base);
    tmem_relinquish<1>();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = C.tmem_base;

  if (warp == kEpiWarps + 1) {
    // =========================== weight stream (bulk TMA) ===========================
    if (lane == 0) {
      long long g = 0;
      for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
        for (int it = 0; it < NIT; ++it, ++g) {
          const int st = static_cast<int>(g & 1);
          mbar_wait(&C.b_empty[st], static_cast<uint32_t>(((g >> 1) & 1) ^ 1));
          const bool hi_only = stat1x && it < NCH;  // the statistics pass multiplies the hi parts only
          mbar_expect_tx(&C.b_full[st], hi_only ? G::kTermBytes : G::kBStageBytes);
          const float* src = p.w_image + static_cast<size_t>(chunk_of(it % NCH)) * G::kChunkFloats;
          unsigned char* dst = sB + st * G::kBStageBytes;
          const int nblk = (hi_only ? G::kTermBytes : G::kBStageBytes) / kBlockBytes;
          for (int q = 0; q < nblk; ++q)
            tma_load(dst + q * kBlockBytes, src + q * (kBlockBytes / 4), kBlockBytes, &C.b_full[st]);
        }
    }
  } else if (warp == 0) {
    // =========================== MMA issue ===========================
    if (lane == 0) {
      long long g = 0;
      uint32_t tcount = 0;
      const uint32_t a_addr = smem_u32(sA);
      for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tcount) {
        mbar_wait(&C.a_ready, tcount & 1);
        for (int it = 0; it < NIT; ++it, ++g) {
          const int st = static_cast<int>(g & 1), acc = it & 3;
          mbar_wait(&C.b_full[st], static_cast<uint32_t>((g >> 1) & 1));
          mbar_wait(&C.acc_empty[acc], static_cast<uint32_t>(((g >> 2) & 1) ^ 1));
          tc_fence_after();
          const uint32_t b_addr = smem_u32(sB + st * G::kBStageBytes);
          const uint32_t d_tmem = tmem + acc * kChunk;
          uint32_t accum = 0;
          // small terms first: a_lo w_hi, a_hi w_lo, then a_hi w_hi (the statistics pass in 1xTF32: a_hi w_hi only)
          const int term0 = (stat1x && it < NCH) ? 2 : 0;
#pragma unroll
          for (int term = 0; term < 3; ++term) {
            if (term < term0) continue;
            const uint32_t a_off = (term == 0) ? G::kTermBytes : 0;  // 0 = hi, 1 = lo
            const uint32_t b_off = (term == 1) ? G::kTermBytes : 0;
#pragma unroll
            for (int kb = 0; kb < G::KB; ++kb)
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {  // 4 MMAs of K = 8 per 128-byte k-block
                const uint32_t off = kb * kBlockBytes + ks * 32;
                tc_mma_tf32(d_tmem, smem_desc(a_addr + a_off + off), smem_desc(b_addr + b_off + off), kIdesc, accum);
                accum = 1;
              }
          }
          tc_commit(&C.b_empty[st]);
          tc_commit(&C.acc_full[acc]);
        }
        tc_commit(&C.a_free);
      }
    }
  } else {
    // =========================== A producer + epilogue (warps 1..16) ===========================
    const int et = tid - 32;            // 0..511
    const int q = warp & 3;             // TMEM lane quarter this warp may access
    const int cs = (warp - 1) >> 2;     // which 32 of the 128 columns of a chunk
    const int erow = 32 * q + lane;     // row (TMEM lane) of this thread in the epilogue
    const uint32_t t_lane = tmem + (static_cast<uint32_t>(32 * q) << 16) + kCols * cs;
    const NoiseStream rng(p.seed, p.offset);
    const float thin_c = p.thin_factor > 0.f ? p.thin_factor : kThin;
    uint32_t status_bits = 0;
    uint32_t tcount = 0;
    long long prev_tile = -1;

    // exact finish of the previous tile's rows from their survivor lists (16 lanes per row, as score_batch).  Everything
    // that enters a score is formed HERE from exact quantities - the row's sum of numerators accumulated in pass 2 (3xTF32
    // logits), the fp32 logit of class x_t - so the approximate statistics of a 1xTF32 first pass never reach a result.
    auto score_tile = [&](long long tile) {
      const int sub = lane & 15;
      for (int slot = 2 * (warp - 1) + (lane >> 4); slot < kTileM; slot += 2 * kEpiWarps) {
        const long long lrow = tile * kTileM + slot;
        const bool live = lrow < p.rows;
        unsigned long long key = 0ull;
        float accept = 0.f;
        uint32_t cnt = 0;
        if (live) {
          const HeadRowInfo hi = C.info[slot];
          const float S = (C.sum2[0][slot] + C.sum2[1][slot]) + (C.sum2[2][slot] + C.sum2[3][slot]);
          const float rS = __frcp_rn(S);
          const bool masked = (hi.j == static_cast<uint32_t>(p.K));
          const float pj = masked ? 0.f : fminf(fmaxf(ex2(hi.yj_rel) * rS, kPFloor), 1.0f);
          RowMath rm;
          rm.init(load_row_coef(p.coef_table, hi.tt, masked), masked, pj, hi.j, p.K);
          accept = ThinRule(rm, thin_c).accept;
          cnt = C.cand_cnt[slot];
          const uint32_t n = cnt < static_cast<uint32_t>(kCand) ? cnt : static_cast<uint32_t>(kCand);
          // items 0 .. n-1: the survivors, item n: [MASK], item n+1: the row's own class; one or two rounds of 16 lanes
          for (uint32_t item = static_cast<uint32_t>(sub); item < n + 2u; item += 16u) {
            uint32_t k = 0;
            float P = 0.f;
            bool have = false;
            if (item < n) {
              k = C.cand_k[slot][item];
              const float pe = fminf(fmaxf(C.cand_p[slot][item] * rS, kPFloor), 1.0f);
              P = fmaf(pe, rm.A, rm.Bc);
              have = (k != hi.j);
            } else if (item == n) {
              k = static_cast<uint32_t>(p.K), P = rm.PK, have = true;
            } else if (!masked) {
              k = hi.j, P = rm.Pj, have = true;
            }
            if (have) {
              const float sc = log_prob_clamped(P) +
                               gumbel_from_uniform(uniform_from_draw(rng.draw(k, static_cast<uint64_t>(p.row_offset + lrow))));
              const unsigned long long kk = pack_key(sc, k);
              key = kk > key ? kk : key;
            }
          }
        }
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) {
          const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, o);
          key = other > key ? other : key;
        }
        if (live && sub == 0) {
          if (cnt <= static_cast<uint32_t>(kCand) && key_score(key) >= accept) {
            p.x_prev[lrow] = key_class(key);
          } else {
            p.redo_rows[atomicAdd(p.redo_count, 1u)] = static_cast<int32_t>(lrow);
          }
          C.cand_cnt[slot] = 0;
        }
      }
    };

    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++tcount) {
      // ---------------- A operand: LayerNorm, guidance combine, hi/lo split, swizzled store ----------------
      {
        const int arow = et >> 2, part = et & 3;  // 4 adjacent lanes per row, 16 hidden values each
        const long long lrow = tile * kTileM + arow;
        const bool valid = lrow < p.rows;
        float a[16];
        if (valid) {
          const float4* src = reinterpret_cast<const float4*>(p.hidden_c + lrow * D + 16 * part);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float4 v = __ldg(src + i);
            a[4 * i] = v.x, a[4 * i + 1] = v.y, a[4 * i + 2] = v.z, a[4 * i + 3] = v.w;
          }
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) a[i] = 0.f;
        }
        layer_norm_part(a, p.ln_weight, p.ln_bias, part, p.ln_eps);
        if (HAS_U) {
          float u[16];
          if (valid) {
            const float4* src = reinterpret_cast<const float4*>(p.hidden_u + lrow * D + 16 * part);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float4 v = __ldg(src + i);
              u[4 * i] = v.x, u[4 * i + 1] = v.y, u[4 * i + 2] = v.z, u[4 * i + 3] = v.w;
            }
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) u[i] = 0.f;
          }
          layer_norm_part(u, p.ln_weight, p.ln_bias, part, p.ln_eps);
          const float gs = p.guidance_scale, og = 1.0f - gs;
#pragma unroll
          for (int i = 0; i < 16; ++i) a[i] = fmaf(gs, a[i], og * u[i]);
        }
        if (!valid) {
#pragma unroll
          for (int i = 0; i < 16; ++i) a[i] = 0.f;
        }
        const int kb = part >> 1, piece0 = 4 * (part & 1);  // k-block and first 16-byte piece of this thread's values
        // logit (log2 units) of the row's current token, needed by the posterior of unmasked rows
        if (!DUMP) {
          long long jj = valid ? p.x_t[lrow] : p.K;
          if (jj < 0 || jj > p.K) status_bits |= D3PM_STATUS_BAD_TOKEN, jj = p.K;
          float dot = 0.f;
          if (jj < p.K) {
            const int j = static_cast<int>(jj);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float4 hi = __ldg(reinterpret_cast<const float4*>(p.w_image + image_offset<D>(j, 0, kb, piece0 + i)));
              const float4 lo = __ldg(reinterpret_cast<const float4*>(p.w_image + image_offset<D>(j, 1, kb, piece0 + i)));
              dot = fmaf(a[4 * i], hi.x + lo.x, dot);
              dot = fmaf(a[4 * i + 1], hi.y + lo.y, dot);
              dot = fmaf(a[4 * i + 2], hi.z + lo.z, dot);
              dot = fmaf(a[4 * i + 3], hi.w + lo.w, dot);
            }
          }
          dot += __shfl_xor_sync(0xffffffffu, dot, 1);
          dot += __shfl_xor_sync(0xffffffffu, dot, 2);
          if (part == 0) C.yj2[arow] = (jj < p.K) ? dot + __ldg(p.bias2 + jj) : 0.f;
        }
        if (tcount > 0) mbar_wait(&C.a_free, (tcount - 1) & 1);  // the previous tile's MMAs no longer read A
        unsigned char* rowp = sA + kb * kBlockBytes + arow * 128;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float hi[4], lo[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            hi[e] = __uint_as_float(__float_as_uint(a[4 * i + e]) & 0xffffe000u);
            lo[e] = a[4 * i + e] - hi[e];
          }
          const int sw = ((piece0 + i) ^ (arow & 7)) * 16;
          *reinterpret_cast<float4*>(rowp + sw) = make_float4(hi[0], hi[1], hi[2], hi[3]);
          *reinterpret_cast<float4*>(rowp + G::kTermBytes + sw) = make_float4(lo[0], lo[1], lo[2], lo[3]);
        }
        fence_proxy_async();
        mbar_arrive(&C.a_ready);
      }
      // the tensor pipe is busy with this tile now: finish the previous one
      if (!DUMP && prev_tile >= 0) score_tile(prev_tile);

      const long long lrow = tile * kTileM + erow;
      const bool live = lrow < p.rows;

      if (DUMP) {
        for (int it = 0; it < NIT; ++it) {
          const int acc = it & 3;
          mbar_wait(&C.acc_full[acc], static_cast<uint32_t>((it >> 2) & 1));
          tc_fence_after();
          const int k0 = chunk_of(it) * kChunk + kCols * cs;
          uint32_t v[32];
          tmem_ld32(t_lane + acc * kChunk, v);
          tmem_ld_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&C.acc_empty[acc]);
          if (live) {
            float* dst = p.logits_out + lrow * p.K + k0;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias2 + k0) + i);
              *reinterpret_cast<float4*>(dst + 4 * i) =
                  make_float4((__uint_as_float(v[4 * i]) + b.x) * kLn2, (__uint_as_float(v[4 * i + 1]) + b.y) * kLn2,
                              (__uint_as_float(v[4 * i + 2]) + b.z) * kLn2, (__uint_as_float(v[4 * i + 3]) + b.w) * kLn2);
            }
          }
        }
        continue;
      }

      // ---------------- pass 1: softmax statistics of the row (log2 units) ----------------
      float m = -CUDART_INF_F, s = 0.f;
      for (int it = 0; it < NCH; ++it) {
        const int acc = it & 3;
        mbar_wait(&C.acc_full[acc], static_cast<uint32_t>((it >> 2) & 1));
        tc_fence_after();
        const int k0 = chunk_of(it) * kChunk + kCols * cs;
        uint32_t v[32];
        tmem_ld32(t_lane + acc * kChunk, v);
        // the bias of these 32 classes while the TMEM load is in flight
        float4 b[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) b[i] = __ldg(reinterpret_cast<const float4*>(p.bias2 + k0) + i);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&C.acc_empty[acc]);
        float2 y[16];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          y[2 * i] = __fadd2_rn(make_float2(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1])), make_float2(b[i].x, b[i].y));
          y[2 * i + 1] = __fadd2_rn(make_float2(__uint_as_float(v[4 * i + 2]), __uint_as_float(v[4 * i + 3])), make_float2(b[i].z, b[i].w));
        }
        float cm = fmaxf(y[0].x, y[0].y);
#pragma unroll
        for (int i = 1; i < 16; ++i) cm = fmaxf(cm, fmaxf(y[i].x, y[i].y));
        const float mn = fmaxf(m, cm);
        s *= ex2(m - mn);
        m = mn;
        const float2 nm = make_float2(-m, -m);
        float2 part[2] = {make_float2(0.f, 0.f), make_float2(0.f, 0.f)};
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float2 d = __fadd2_rn(y[i], nm);
          part[i & 1] = __fadd2_rn(part[i & 1], make_float2(ex2(d.x), ex2(d.y)));
        }
        s += (part[0].x + part[0].y) + (part[1].x + part[1].y);
      }
      C.stat_m[cs][erow] = m;
      C.stat_s[cs][erow] = s;
      epi_bar();  // all parts of every row are in; the previous tile's lists have been scored and reset
      float M2 = C.stat_m[0][erow];
#pragma unroll
      for (int c = 1; c < kColSplit; ++c) M2 = fmaxf(M2, C.stat_m[c][erow]);
      float S = 0.f;
#pragma unroll
      for (int c = 0; c < kColSplit; ++c) S = fmaf(C.stat_s[c][erow], ex2(C.stat_m[c][erow] - M2), S);
      const float rS = __frcp_rn(S);

      // ---------------- per-row posterior coefficients and thinning thresholds ----------------
      long long jj = live ? p.x_t[lrow] : p.K;
      if (jj < 0 || jj > p.K) jj = p.K;  // flagged by the A producer
      long long tt = live ? p.t[lrow / p.N] : 0;
      if (tt < 0 || tt >= p.T) status_bits |= D3PM_STATUS_BAD_T, tt = tt < 0 ? 0 : p.T - 1;
      const bool masked = (jj == p.K);
      const uint32_t j = static_cast<uint32_t>(jj);
      const RowCoef cf = load_row_coef(p.coef_table, static_cast<int>(tt), masked);
      const float yj_rel = masked ? 0.f : C.yj2[erow] - M2;
      // Thinning thresholds.  With exact statistics (3xTF32 first pass) they are those of the unfused kernels.  With a
      // 1xTF32 first pass the stabiliser M2 is merely close to the row maximum (harmless: any stabiliser works) and S is
      // within a factor 2^slack of the exact sum, so the thresholds are made CONSERVATIVE: 1/S and p_j are taken at the
      // ends of their intervals and the larger threshold of the two ends is used (A c / Ptot and Bc c / Ptot are ratios
      // of functions linear in p_j, hence monotone) - the survivor lists can only grow, by ~2^(2 slack).  The acceptance
      // bound and every score are formed from exact quantities in score_tile.
      const float grow_f = stat1x ? ex2(p.stat_slack) : 1.0f;
      const float pj_mid = masked ? 0.f : ex2(yj_rel) * rS;
      RowMath rm;
      rm.init(cf, masked, masked ? 0.f : fminf(fmaxf(pj_mid * grow_f, kPFloor), 1.0f), j, p.K);
      ThinRule thin(rm, thin_c);
      if (stat1x && !masked) {
        RowMath rm_lo;
        rm_lo.init(cf, masked, fminf(fmaxf(pj_mid / grow_f, kPFloor), 1.0f), j, p.K);
        const ThinRule thin_lo(rm_lo, thin_c);
        thin.scaleA = fmaxf(thin.scaleA, thin_lo.scaleA), thin.thrB = fmaxf(thin.thrB, thin_lo.thrB);
      }
      const float thrA = rS * grow_f * thin.scaleA;
      if (cs == 0) {
        HeadRowInfo hi;
        hi.j = j, hi.tt = static_cast<int32_t>(tt), hi.yj_rel = yj_rel, hi.pad = 0.f;
        C.info[erow] = hi;
      }
      const uint64_t grow = static_cast<uint64_t>(p.row_offset + lrow);
      const float2 nM2 = make_float2(-M2, -M2), tA2 = make_float2(thrA, thrA);
      const float nthrB = -thin.thrB;
      float2 esum = make_float2(0.f, 0.f);  // exact sum of this thread's numerators

      // ---------------- pass 2: regenerate the logits, thinned race, survivors to the row's list ----------------
      // The noise (integer pipe) is generated one group of eight classes AHEAD of the exponentials (MUFU pipe) that
      // consume it, in the same basic block, so that the two pipes overlap inside every warp.
      auto coarse_of = [&](int pr_, int c8_) {
        const int kk = chunk_of(2 * pr_) * kChunk + kCols * cs;
        return rng.coarse(NoiseStream::coarse_call_of_chunk(static_cast<uint32_t>(kk >> 2) + c8_), grow);
      };
      uint4 cw_next = coarse_of(0, 0);
      for (int pr = 0; pr < NCH / 2; ++pr) {
        const int itA = NCH + 2 * pr, itB = itA + 1;
        const int accA = itA & 3, accB = itB & 3;
        // classes k0 .. k0+31 from the first chunk of the pair and the same + 512 from the second (chunk_of(2 pr + 1) =
        // chunk_of(2 pr) + 4): one Philox call serves four classes of each
        const int k0 = chunk_of(2 * pr) * kChunk + kCols * cs;
        mbar_wait(&C.acc_full[accA], static_cast<uint32_t>((itA >> 2) & 1));
        mbar_wait(&C.acc_full[accB], static_cast<uint32_t>((itB >> 2) & 1));
        tc_fence_after();
        // the accumulators are read 16 columns at a time (two halves of the thread's 32 columns): 32 live registers for
        // the logits instead of 64, which is what keeps this loop free of spills at 96 registers per thread
        uint32_t va[16], vb[16];
#pragma unroll
        for (int c8 = 0; c8 < 8; ++c8) {
          if ((c8 & 3) == 0) {
            tmem_ld16(t_lane + accA * kChunk + 4 * c8, va);
            tmem_ld16(t_lane + accB * kChunk + 4 * c8, vb);
            tmem_ld_wait();
            if (c8 == 4) {  // both halves are in registers: the tensor pipe may overwrite the two accumulators
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive(&C.acc_empty[accA]), mbar_arrive(&C.acc_empty[accB]);
            }
          }
          const int c4 = c8 & 3;
          const uint4 cw = cw_next;
          if (c8 < 7) cw_next = coarse_of(pr, c8 + 1);
          else if (pr + 1 < NCH / 2) cw_next = coarse_of(pr + 1, 0);
          const float4 ba = __ldg(reinterpret_cast<const float4*>(p.bias2 + k0) + c8);
          const float4 bb = __ldg(reinterpret_cast<const float4*>(p.bias2 + k0 + 512) + c8);
          float2 e[4], d[4];
          e[0] = __fadd2_rn(__fadd2_rn(make_float2(__uint_as_float(va[4 * c4]), __uint_as_float(va[4 * c4 + 1])), make_float2(ba.x, ba.y)), nM2);
          e[1] = __fadd2_rn(__fadd2_rn(make_float2(__uint_as_float(va[4 * c4 + 2]), __uint_as_float(va[4 * c4 + 3])), make_float2(ba.z, ba.w)), nM2);
          e[2] = __fadd2_rn(__fadd2_rn(make_float2(__uint_as_float(vb[4 * c4]), __uint_as_float(vb[4 * c4 + 1])), make_float2(bb.x, bb.y)), nM2);
          e[3] = __fadd2_rn(__fadd2_rn(make_float2(__uint_as_float(vb[4 * c4 + 2]), __uint_as_float(vb[4 * c4 + 3])), make_float2(bb.z, bb.w)), nM2);
          const uint32_t w4[4] = {cw.x, cw.y, cw.z, cw.w};
          float slack = -4.0f;  // max over the 8 classes of e thrA + nf, nf = -(1 + h 2^-23); a class survives when >= -thrB
#pragma unroll
          for (int w = 0; w < 4; ++w) {
            e[w] = make_float2(ex2(e[w].x), ex2(e[w].y));
            esum = __fadd2_rn(esum, e[w]);
            // the 16-bit halves spliced under the exponent of -1.0f: -(1 + h 2^-23)
            const float2 nf = make_float2(__uint_as_float(__byte_perm(w4[w], 0xbf80u, 0x5410)),
                                          __uint_as_float(__byte_perm(w4[w], 0xbf80u, 0x5432)));
            d[w] = __ffma2_rn(e[w], tA2, nf);
            slack = fmaxf(slack, fmaxf(d[w].x, d[w].y));
          }
          if (slack >= nthrB && live) {  // ~1 % of the lanes: some class of the eight survives
#pragma unroll
            for (int w = 0; w < 4; ++w)
#pragma unroll
              for (int hl = 0; hl < 2; ++hl)
                if ((hl ? d[w].y : d[w].x) >= nthrB) {
                  const uint32_t pos = atomicAdd(&C.cand_cnt[erow], 1u);
                  if (pos < static_cast<uint32_t>(kCand)) {
                    C.cand_k[erow][pos] = static_cast<uint16_t>(k0 + 4 * c8 + (w >> 1) * 512 + 2 * (w & 1) + hl);
                    C.cand_p[erow][pos] = hl ? e[w].y : e[w].x;
                  }
                }
          }
        }
      }
      C.sum2[cs][erow] = esum.x + esum.y;
      epi_bar();  // every survivor of the tile is listed, every row's exact sum is in
      prev_tile = tile;
    }
    if (!DUMP && prev_tile >= 0) score_tile(prev_tile);
    if (status_bits != 0 && p.status != nullptr) atomicOr(p.status, status_bits);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc<1, 512>(tmem);
  }
}

// ---- rescoring of the rows the race could not decide (probability ~e^-c per row) and reference CUDA-core path ----------
// One CTA per listed row: the combined logits of the row in plain fp32 FMAs, then exhaustive exact Gumbel scoring (the
// same arithmetic as the exhaustive path of step_rows_kernel).
// 1024 threads per row (at most 8 classes each, their weight loads all in flight at once): the launch lasts as long as
// ONE row when few rows are listed, and that latency follows every fused step.
constexpr int kRedoThreads = 1024;
template <int D, bool HAS_U>
__global__ void __launch_bounds__(kRedoThreads) head_redo_kernel(const HeadParams p, int all_rows) {
  constexpr int NW = kRedoThreads / 32;
  constexpr int kPer = 8;  // K <= 8192
  __shared__ float sa[D];
  __shared__ float sred[2][NW];
  __shared__ float ys[1024 * kPer];  // the row's logits (log2 units)
  __shared__ unsigned long long skey[NW];
  __shared__ float syj;
  const int tid = threadIdx.x;
  const long long count = all_rows ? p.rows : static_cast<long long>(*p.redo_count);
  const NoiseStream rng(p.seed, p.offset);
  for (long long e = blockIdx.x; e < count; e += gridDim.x) {
    const long long lrow = all_rows ? e : p.redo_rows[e];
    __syncthreads();
    if (tid < 32) {  // one warp: the combined, normalised hidden vector (2 values per lane)
      float x[2] = {p.hidden_c[lrow * D + tid], p.hidden_c[lrow * D + 32 + tid]};
      auto ln = [&](float (&v)[2]) {
        const float mean = warp_sum(v[0] + v[1]) * (1.0f / D);
        const float d0 = v[0] - mean, d1 = v[1] - mean;
        const float rstd = 1.0f / sqrtf(warp_sum(d0 * d0 + d1 * d1) * (1.0f / D) + p.ln_eps);
        v[0] = fmaf(d0 * rstd, p.ln_weight[tid], p.ln_bias[tid]);
        v[1] = fmaf(d1 * rstd, p.ln_weight[32 + tid], p.ln_bias[32 + tid]);
      };
      ln(x);
      if (HAS_U) {
        float u[2] = {p.hidden_u[lrow * D + tid], p.hidden_u[lrow * D + 32 + tid]};
        ln(u);
        const float gs = p.guidance_scale, og = 1.0f - gs;
        x[0] = fmaf(gs, x[0], og * u[0]), x[1] = fmaf(gs, x[1], og * u[1]);
      }
      sa[tid] = x[0], sa[32 + tid] = x[1];
    }
    __syncthreads();
    long long jj = p.x_t[lrow], tt = p.t[lrow / p.N];
    if (jj < 0 || jj > p.K) jj = p.K;
    if (tt < 0 || tt >= p.T) tt = tt < 0 ? 0 : p.T - 1;
    const bool masked = (jj == p.K);
    const uint32_t j = static_cast<uint32_t>(jj);
    // logits of the row: the eight lanes of a class read the eight 16-byte pieces of its 128-byte image rows (one
    // coalesced line per class, term and k-block; one class per thread touched 32 lines per load instruction and the
    // kernel spent its time in the load queue), four classes per warp pass, products summed across the eight lanes
    {
      const int piece = tid & 7, c4 = (tid >> 3) & 3, wrp = tid >> 5;
      float4 av[Geo<D>::KB];
#pragma unroll
      for (int kb = 0; kb < Geo<D>::KB; ++kb) av[kb] = *reinterpret_cast<const float4*>(sa + 32 * kb + 4 * piece);
#pragma unroll 4
      for (int k = 4 * wrp + c4; k < p.K; k += 4 * NW) {
        float dot = 0.f;
#pragma unroll
        for (int kb = 0; kb < Geo<D>::KB; ++kb) {
          const float4 hi = __ldg(reinterpret_cast<const float4*>(p.w_image + image_offset<D>(k, 0, kb, piece)));
          const float4 lo = __ldg(reinterpret_cast<const float4*>(p.w_image + image_offset<D>(k, 1, kb, piece)));
          dot = fmaf(av[kb].x, hi.x + lo.x, dot), dot = fmaf(av[kb].y, hi.y + lo.y, dot);
          dot = fmaf(av[kb].z, hi.z + lo.z, dot), dot = fmaf(av[kb].w, hi.w + lo.w, dot);
        }
        dot += __shfl_xor_sync(0xffffffffu, dot, 1);
        dot += __shfl_xor_sync(0xffffffffu, dot, 2);
        dot += __shfl_xor_sync(0xffffffffu, dot, 4);
        if (piece == 0) ys[k] = dot + __ldg(p.bias2 + k);
      }
    }
    __syncthreads();
    float y[kPer];  // classes tid + 1024 i
    float m = -CUDART_INF_F;
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
      const int k = tid + kRedoThreads * i;
      y[i] = k < p.K ? ys[k] : -CUDART_INF_F;
      m = fmaxf(m, y[i]);
    }
    if (tid == 0 && !masked) syj = ys[j];
    // softmax statistics in log2 units
    m = warp_max(m);
    if ((tid & 31) == 0) sred[0][tid >> 5] = m;
    __syncthreads();
    float M2 = sred[0][0];
    for (int w = 1; w < NW; ++w) M2 = fmaxf(M2, sred[0][w]);
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < kPer; ++i) {
      y[i] = ex2(y[i] - M2);  // 0 for the slots beyond K
      s += y[i];
    }
    s = warp_sum(s);
    if ((tid & 31) == 0) sred[1][tid >> 5] = s;
    __syncthreads();
    float S = 0.f;
    for (int w = 0; w < NW; ++w) S += sred[1][w];
    const float rS = __frcp_rn(S);
    const RowCoef cf = load_row_coef(p.coef_table, static_cast<int>(tt), masked);
    const float pj = masked ? 0.f : fminf(fmaxf(ex2(syj - M2) * rS, kPFloor), 1.0f);
    RowMath rm;
    rm.init(cf, masked, pj, j, p.K);
    const uint64_t grow = static_cast<uint64_t>(p.row_offset + lrow);
    unsigned long long best = 0ull;
#pragma unroll 2
    for (int i = 0; i < kPer; ++i) {
      const uint32_t k = tid + kRedoThreads * i;
      if (k >= static_cast<uint32_t>(p.K)) break;
      const float sc = rm.post_of(k, y[i], rS) + gumbel_from_uniform(uniform_from_draw(rng.draw(k, grow)));
      const unsigned long long key = pack_key(sc, k);
      best = key > best ? key : best;
    }
    if (tid == 0) {
      const unsigned long long key =
          pack_key(rm.post_mask() + gumbel_from_uniform(uniform_from_draw(rng.draw(p.K, grow))), p.K);
      best = key > best ? key : best;
    }
    best = warp_max_u64(best);
    if ((tid & 31) == 0) skey[tid >> 5] = best;
    __syncthreads();
    if (tid == 0) {
      for (int w = 0; w < NW; ++w) best = skey[w] > best ? skey[w] : best;
      p.x_prev[lrow] = key_class(best);
    }
  }
}

}  // namespace head
}  // namespace d3pm
