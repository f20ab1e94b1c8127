// Token -> video, second stage (SURVEY.md §8 f4): the reference's VQ-VAE `Decoder` (videogpt_vq_vae.py:258-287) in eval
// mode - attention residual blocks (:120-136: BatchNorm3d, ReLU, SamePadConv3d 3x3x3, 1x1x1, AxialBlock :100-118 with the
// MultiHeadAttention of utils/model_utils.py:214-297) followed by SamePadConvTranspose3d layers (:312-334).
//
// Every convolution and every Linear of the decoder is ONE kernel here, an implicit GEMM on the 5th-gen tensor cores:
//   * activations are channels-last rows [B*T*H*W][C] (one 128-byte line per 32 channels of a position);
//   * a tile is 128 positions x NT output channels, accumulated in tensor memory (tcgen05.mma kind::tf32, M = 128,
//     N = NT, K = 8 per instruction) as a 3xTF32 split (a_lo w_hi + a_hi w_lo + a_hi w_hi: fp32-grade results; `terms = 1`
//     multiplies the hi parts only, which is what cuDNN's default TF32 convolutions of the reference on a GPU do);
//   * the A operand is produced in the kernel, k-block by k-block (one filter tap x 32 input channels): eight warps
//     gather the shifted input rows (zero outside the grid: the SamePad padding), apply the BatchNorm + ReLU that
//     precedes the convolution in the reference as a per-channel affine, split hi / lo and store into the 128-byte
//     swizzled K-major layout the tensor core reads; the B operand (weights, BatchNorms that FOLLOW a convolution folded
//     in) is a pre-swizzled image streamed with 1-D bulk TMA through the same ring of shared-memory stages;
//   * the epilogue reads the accumulator row per thread (tcgen05.ld 32x32b), adds bias / residual, applies ReLU and stores
//     channels-last rows (128 contiguous bytes per thread and 32 channels).
// A transposed convolution with stride 2 is decomposed by output parity: every parity class is an ordinary convolution over
// the INPUT grid with 2 taps per strided dimension (4 per unit-stride dimension), its results scattered to the class's
// output positions, so no zero-stuffed input is ever formed.  The last layer (3 output channels) runs the other way round:
// a plain GEMM [positions x C] x [C x 64 taps * 3] followed by col2im_kernel, which sums the 16 contributions of each
// output voxel and writes the channels-first video the reference returns.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "d3pm_b200.h"
#include "d3pm_ptx.cuh"

namespace d3pm {
namespace dec {

constexpr int kTileM = 128;
constexpr int kProdWarps = 8;                     // A producers, then the epilogue
constexpr int kProdThreads = 32 * kProdWarps;
constexpr int kBlockBytes = kTileM * 128;         // one k-block (32 floats) of a 128-row operand
constexpr int kMaxTaps = D3PM_DEC_MAX_TAPS;
constexpr int kMaxClasses = D3PM_DEC_MAX_CLASSES;
constexpr int kMaxCin = 1024;

struct GemmParams {
  const float* x;         // [B*T*H*W][Cin]
  const float* in_scale;  // [Cin] or null
  const float* in_shift;
  const float* w_image;   // [class][N tile][k-block][term][NT rows x 128 B swizzled]
  const float* bias;      // [Npad] or null
  const float* residual;  // rows laid out like `out`, or null
  float* out;
  int B, T, H, W, Cin;
  int ntaps, nclass;
  int Npad, Nout;
  long long ldo;
  int To, Ho, Wo, st, sh, sw;
  int relu_out, terms;
  int out_transposed;     // 1: out[(row / ldo) * Nout * ldo + n * ldo + row % ldo]: planes of ldo rows, channel-major inside a plane
                          // (the col2im input; a plane = one (video, frame) keeps a tile's 64 * Cout rows within a few pages)
  signed char tap[kMaxClasses][kMaxTaps][4];  // (dt, dh, dw) of every tap of every class
  signed char cls[kMaxClasses][4];            // (pt, ph, pw): output position = input position * stride + this
};

// nearest tf32 number (10 mantissa bits, ties away from zero): the tensor core ignores the 13 low bits, so rounding here makes
// the single-product mode unbiased; in the 3xTF32 mode lo = x - hi stays exact either way
__device__ __forceinline__ float tf32_round(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u); }

// ---- weight image ---------------------------------------------------------------------------------------------
// floats of the image of one parity class: [Npad / NT][Ktot / 32][2 terms][NT][32]
__host__ __device__ inline int64_t image_floats(int Npad, int Ktot) { return static_cast<int64_t>(Npad) * Ktot * 2; }

// w: [nclass][N][Ktot] row-major fp32 (k contiguous: the K-major operand), rows n >= N are zero in the image.
// hi = w rounded to the nearest tf32 number, lo = w - hi (exact in fp32).
__global__ void weight_image_kernel(const float* __restrict__ w, int N, int Npad, int Ktot, int NT, float* __restrict__ image) {
  const int KB = Ktot / 32;
  const int64_t pieces = static_cast<int64_t>(Npad) * KB * 8;  // 16-byte pieces of one class
  const int64_t idx = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= pieces) return;
  const int cls = blockIdx.y;
  const int piece = static_cast<int>(idx & 7);
  const int kb = static_cast<int>((idx >> 3) % KB);
  const int n = static_cast<int>((idx >> 3) / KB);
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (n < N) v = *reinterpret_cast<const float4*>(w + (static_cast<size_t>(cls) * N + n) * Ktot + kb * 32 + piece * 4);
  const float s[4] = {v.x, v.y, v.z, v.w};
  float hi[4], lo[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    hi[e] = tf32_round(s[e]);
    lo[e] = s[e] - hi[e];
  }
  const int ntile = n / NT, r = n % NT;
  float* blk = image + static_cast<size_t>(cls) * image_floats(Npad, Ktot) +
               (static_cast<size_t>(ntile) * KB + kb) * (2 * NT * 32);
  const int at = r * 32 + ((piece ^ (r & 7)) << 2);
  *reinterpret_cast<float4*>(blk + at) = make_float4(hi[0], hi[1], hi[2], hi[3]);
  *reinterpret_cast<float4*>(blk + NT * 32 + at) = make_float4(lo[0], lo[1], lo[2], lo[3]);
}

// ---- the implicit-GEMM convolution ------------------------------------------------------------------------------
// TERMS = 3: 3xTF32, a stage holds the hi and lo halves of both operands; TERMS = 1: plain TF32, hi halves only, so twice
// as many stages fit (the single-product mode is bound by the producers' latency, which deeper staging hides)
// CTAS = 2: a pair of CTAs (cluster of two on one TPC) computes 256 positions x NT channels with M = 256 MMAs
// (tcgen05 cta_group::2): every CTA gathers the A rows of its own 128 positions and stages HALF of the weight rows, so its L2
// weight stream and the shared-memory reads of the B operand are halved - the two floors of the single-CTA kernel.
template <int NT, int TERMS, int CTAS>
struct GemmGeo {
  static constexpr int kHalves = TERMS == 1 ? 1 : 2;
  static constexpr int kBRows = NT / CTAS;                        // weight rows this CTA stages
  static constexpr int kBBytes = kBRows * 128;                    // one term of them
  static constexpr int kABytes = kHalves * kBlockBytes;           // A part of a stage
  static constexpr int kStageBytes = kABytes + kHalves * kBBytes;
  static constexpr int kStages = 196608 / kStageBytes < 6 ? 196608 / kStageBytes : 6;
  static constexpr uint32_t kIdesc = idesc_tf32(kTileM * CTAS, NT);  // M = 128 per CTA
};

struct GemmCtl {
  unsigned long long full_a[6], full_b[6], empty[6], peer_full[6], acc_full[2], acc_empty[2];
  uint32_t tmem_base, pad;
  signed char taps[kMaxClasses][kMaxTaps][4];
  int tap_shift[kMaxClasses][kMaxTaps];  // element offset of a tap's source row relative to the row itself
  alignas(16) float scale[kMaxCin];
  alignas(16) float shift[kMaxCin];
  alignas(16) float stage[4][32][36];    // epilogue: 32 rows x 32 columns per warp, rows padded to 144 B (conflict-free 128-bit access)
};

template <int NT, int TERMS, int CTAS>
constexpr size_t gemm_smem_bytes() {
  return 1024 + GemmGeo<NT, TERMS, CTAS>::kStages * GemmGeo<NT, TERMS, CTAS>::kStageBytes + sizeof(GemmCtl);
}

// Persistent: a CTA walks the tiles  t = blockIdx.x, blockIdx.x + gridDim.x, ...  of the launch, tile t = (parity class, M tile,
// N tile) with the N tile fastest (neighbouring CTAs gather the same input rows: L2).  Fourteen warps:
//   warp 0      one lane issues the MMAs of a tile into accumulator (tile & 1) and the commits that free stages / publish it
//   warp 1      one lane streams the weight image (bulk TMA)
//   warps 2-9   produce the A operand, k-block after k-block, running ahead across tile boundaries
//   warps 10-13 epilogue of tile i while the MMAs of tile i + 1 fill the other accumulator
constexpr int kEpiWarps = 4;
constexpr int kGemmThreads = 32 * (2 + kProdWarps + kEpiWarps);

template <int NT, int TERMS, int CTAS>
__global__ void __launch_bounds__(kGemmThreads, 1) conv_gemm_kernel(const __grid_constant__ GemmParams p) {
  using G = GemmGeo<NT, TERMS, CTAS>;
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_dyn) + 1023) & ~uintptr_t(1023));
  GemmCtl& C = *reinterpret_cast<GemmCtl*>(smem + G::kStages * G::kStageBytes);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = CTAS == 2 ? cluster_ctarank() : 0u;   // rank 0 of a pair is the leader: it issues the MMAs
  const long long unit0 = blockIdx.x / CTAS;                  // a "unit" = the CTA or the pair that walks tiles together
  const long long nunits = gridDim.x / CTAS;
  const int ntiles_n = p.Npad / NT;
  const int CB = p.Cin >> 5;            // k-blocks per tap
  const int KB = p.ntaps * CB;          // k-blocks of a tile
  const long long M = static_cast<long long>(p.B) * p.T * p.H * p.W;
  const long long mtiles = ((M + kTileM - 1) / kTileM + CTAS - 1) / CTAS;  // tiles of 128 * CTAS positions
  const long long per_class = mtiles * ntiles_n;
  const long long total = per_class * p.nclass;
  const int HW = p.H * p.W;

  if (tid == 0) {
    for (int i = 0; i < G::kStages; ++i)
      mbar_init(&C.full_a[i], kProdThreads), mbar_init(&C.full_b[i], 1), mbar_init(&C.empty[i], 1), mbar_init(&C.peer_full[i], 1);
    for (int i = 0; i < 2; ++i) mbar_init(&C.acc_full[i], 1), mbar_init(&C.acc_empty[i], kEpiWarps * CTAS);
    fence_mbarrier_init();
  }
  if (p.in_scale != nullptr)
    for (int i = tid; i < p.Cin; i += kGemmThreads) C.scale[i] = p.in_scale[i], C.shift[i] = p.in_shift[i];
  for (int i = tid; i < p.nclass * p.ntaps; i += kGemmThreads) {
    const int c = i / p.ntaps, t = i - c * p.ntaps;
    for (int e = 0; e < 4; ++e) C.taps[c][t][e] = p.tap[c][t][e];
    C.tap_shift[c][t] = ((p.tap[c][t][0] * p.H + p.tap[c][t][1]) * p.W + p.tap[c][t][2]) * p.Cin;
  }
  if (warp == 0) {  // two accumulators of NT columns (in both CTAs of a pair: the same warp of each allocates)
    tmem_alloc<CTAS, 2 * NT>(&C.tmem_base);
    tmem_relinquish<CTAS>();
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (CTAS == 2) cluster_sync();  // the partner's barriers exist before anything arrives on them
  tc_fence_after();
  const uint32_t tmem = C.tmem_base;

  if (warp == 1) {
    // =========================== weight stream (bulk TMA) ===========================
    if (lane == 0) {
      constexpr uint32_t bytes = G::kHalves * G::kBBytes;
      constexpr uint32_t piece = G::kBBytes < kBlockBytes ? G::kBBytes : kBlockBytes;
      int st = 0;
      uint32_t par = 1;
      for (long long tile = unit0; tile < total; tile += nunits) {
        const int cls = static_cast<int>(tile / per_class);
        const int ntile = static_cast<int>(tile % ntiles_n);
        // this CTA's rows of the N tile: [rank * kBRows, (rank + 1) * kBRows) of the hi block and of the lo block
        const float* src = p.w_image + static_cast<size_t>(cls) * image_floats(p.Npad, KB * 32) + static_cast<size_t>(ntile) * KB * (2 * NT * 32) +
                           static_cast<size_t>(rank) * (G::kBBytes / 4);
        for (int kb = 0; kb < KB; ++kb) {
          mbar_wait(&C.empty[st], par);
          mbar_expect_tx(&C.full_b[st], bytes);
          unsigned char* dst = smem + st * G::kStageBytes + G::kABytes;
          const float* s = src + static_cast<size_t>(kb) * (2 * NT * 32);
#pragma unroll
          for (int half = 0; half < G::kHalves; ++half)
            for (uint32_t q = 0; q < G::kBBytes; q += piece)
              tma_load(dst + half * G::kBBytes + q, s + half * (NT * 32) + q / 4, piece, &C.full_b[st]);
          if (++st == G::kStages) st = 0, par ^= 1u;
        }
      }
    }
  } else if (warp == 0) {
    if (rank != 0) {
      // =========================== partner CTA: tell the leader when this CTA's half of a stage is in place ===========================
      // one lane per stage, so that the remote arrivals of consecutive k-blocks do not queue behind each other
      // (polled without suspending: a lane that slept on its stage would hold up the lanes of the stages that complete first)
      const long long my_tiles = unit0 < total ? (total - unit0 + nunits - 1) / nunits : 0;
      const long long nkb = my_tiles * KB;
      long long g = lane;
      uint32_t par = 0;
      bool active = lane < G::kStages && g < nkb;
      const int st = lane < G::kStages ? lane : 0;
      while (__any_sync(0xffffffffu, active)) {
        if (active && mbar_test(&C.full_a[st], par) && mbar_test(&C.full_b[st], par)) {
          mbar_arrive_remote(&C.peer_full[st], 0);
          g += G::kStages, par ^= 1u;
          active = g < nkb;
        }
      }
    } else if (lane == 0) {
      // =========================== MMA issue ===========================
      int st = 0;
      uint32_t par = 0, tc = 0;
      for (long long tile = unit0; tile < total; tile += nunits, ++tc) {
        const uint32_t acc = tc & 1u;
        // the epilogue (of both CTAs) of tile tc - 2 has drained this accumulator
        if constexpr (CTAS == 2) mbar_wait_cluster(&C.acc_empty[acc], ((tc >> 1) & 1u) ^ 1u);
        else mbar_wait(&C.acc_empty[acc], ((tc >> 1) & 1u) ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem + acc * NT;
        uint32_t accum = 0;
        for (int kb = 0; kb < KB; ++kb) {
          mbar_wait(&C.full_a[st], par);
          mbar_wait(&C.full_b[st], par);
          if constexpr (CTAS == 2) mbar_wait_cluster(&C.peer_full[st], par);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + st * G::kStageBytes);
          const uint32_t b_addr = a_addr + G::kABytes;
          // small terms first: a_lo w_hi, a_hi w_lo, then a_hi w_hi (terms == 1: a_hi w_hi only)
#pragma unroll
          for (int term = (TERMS == 1 ? 2 : 0); term < 3; ++term) {
            const uint32_t a_off = (term == 0) ? kBlockBytes : 0;
            const uint32_t b_off = (term == 1) ? G::kBBytes : 0;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {  // 4 MMAs of K = 8 per 128-byte k-block
              if constexpr (CTAS == 2)
                tc_mma_tf32_pair(d_tmem, smem_desc(a_addr + a_off + ks * 32), smem_desc(b_addr + b_off + ks * 32), G::kIdesc, accum);
              else
                tc_mma_tf32(d_tmem, smem_desc(a_addr + a_off + ks * 32), smem_desc(b_addr + b_off + ks * 32), G::kIdesc, accum);
              accum = 1;
            }
          }
          if constexpr (CTAS == 2) tc_commit_pair(&C.empty[st]);
          else tc_commit(&C.empty[st]);
          if (++st == G::kStages) st = 0, par ^= 1u;
        }
        if constexpr (CTAS == 2) tc_commit_pair(&C.acc_full[acc]);
        else tc_commit(&C.acc_full[acc]);
      }
    }
  } else if (warp < 2 + kProdWarps) {
    // =========================== A producer (warps 2..9) ===========================
    // Everything that depends on the tile only is formed once per tile: per row a bit mask of the taps that stay inside the
    // grid and a 32-bit element offset.  A k-block then costs four 128-bit loads, the transform and four (eight) 128-bit
    // shared stores per thread.  The fetch side runs two k-blocks ahead of the store side, across tile boundaries.
    const int pt = tid - 64;        // 0..255
    const int piece = pt & 7;       // 16-byte piece of the 128-byte k-block row
    const int r0 = pt >> 3;         // rows r0 + 32 i
    uint32_t okmask[4];             // bit `tap`: the tap's source position of row i exists
    uint32_t base[4];               // element offset of the row's own position (+ this thread's piece)
    uint32_t soff[4];               // byte offset of (row, piece) inside a swizzled k-block
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = r0 + 32 * i;
      soff[i] = static_cast<uint32_t>(r * 128 + ((piece ^ (r & 7)) << 4));
    }
    long long f_tile = unit0;  // tile the fetch side is in
    int f_cls = 0, f_tap = 0, f_cb = 0;
    auto enter_tile = [&]() {
      if (f_tile >= total) return;
      f_cls = static_cast<int>(f_tile / per_class);
      const long long mtile = (f_tile % per_class) / ntiles_n * CTAS + rank;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const long long m = mtile * kTileM + r0 + 32 * i;
        const bool rowok = m < M;
        const long long mm = rowok ? m : 0;
        const int inb = static_cast<int>(mm % (static_cast<long long>(p.T) * HW));
        const int ct = inb / HW, ch = (inb % HW) / p.W, cw = inb % p.W;
        uint32_t mask = 0;
        for (int tap = 0; tap < p.ntaps; ++tap) {
          const bool ok = rowok && static_cast<unsigned>(ct + C.taps[f_cls][tap][0]) < static_cast<unsigned>(p.T) &&
                          static_cast<unsigned>(ch + C.taps[f_cls][tap][1]) < static_cast<unsigned>(p.H) &&
                          static_cast<unsigned>(cw + C.taps[f_cls][tap][2]) < static_cast<unsigned>(p.W);
          mask |= (ok ? 1u : 0u) << tap;
        }
        okmask[i] = mask;
        base[i] = static_cast<uint32_t>(mm * p.Cin + piece * 4);
      }
    };
    enter_tile();
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t scale_at = smem_u32(C.scale) + piece * 16, shift_at = smem_u32(C.shift) + piece * 16;
    auto fetch = [&](float4 (&v)[4], uint32_t& ok4) {
      const int shift = C.tap_shift[f_cls][f_tap] + f_cb * 32;  // may be negative: 32-bit wrap-around arithmetic on the offsets
      ok4 = 0;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const bool ok = (okmask[i] >> f_tap) & 1u;
        v[i] = ok ? __ldg(reinterpret_cast<const float4*>(p.x + static_cast<uint32_t>(base[i] + static_cast<uint32_t>(shift))))
                  : make_float4(0.f, 0.f, 0.f, 0.f);
        ok4 |= (ok ? 1u : 0u) << i;
      }
      if (++f_cb == CB) {
        f_cb = 0;
        if (++f_tap == p.ntaps) {
          f_tap = 0;
          f_tile += nunits;
          enter_tile();
        }
      }
    };
    const bool affine = p.in_scale != nullptr;
    constexpr bool want_lo = TERMS != 1;
    int e_st = 0, e_cb = 0;
    uint32_t e_par = 1;  // parity to wait for on the stage's `empty` barrier (first round: passes at once)
    // transform (BatchNorm + ReLU in front of the convolution; the zero padding comes AFTER it: F.pad of the activated
    // tensor), hi / lo split and swizzled store of one k-block
    auto emit = [&](const float4 (&cur)[4], uint32_t cur_ok) {
      mbar_wait(&C.empty[e_st], e_par);
      const uint32_t a_hi = smem_base + e_st * G::kStageBytes;
      float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
      if (affine) {
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(sc.x), "=f"(sc.y), "=f"(sc.z), "=f"(sc.w) : "r"(scale_at + e_cb * 128));
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(sh.x), "=f"(sh.y), "=f"(sh.z), "=f"(sh.w) : "r"(shift_at + e_cb * 128));
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float a[4] = {cur[i].x, cur[i].y, cur[i].z, cur[i].w};
        if (affine) {
          const bool ok = (cur_ok >> i) & 1u;
          a[0] = ok ? fmaxf(fmaf(a[0], sc.x, sh.x), 0.f) : 0.f;
          a[1] = ok ? fmaxf(fmaf(a[1], sc.y, sh.y), 0.f) : 0.f;
          a[2] = ok ? fmaxf(fmaf(a[2], sc.z, sh.z), 0.f) : 0.f;
          a[3] = ok ? fmaxf(fmaf(a[3], sc.w, sh.w), 0.f) : 0.f;
        }
        float hi[4], lo[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          hi[e] = tf32_round(a[e]);
          lo[e] = a[e] - hi[e];
        }
        asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a_hi + soff[i]), "f"(hi[0]), "f"(hi[1]), "f"(hi[2]), "f"(hi[3]) : "memory");
        if (want_lo)
          asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a_hi + kBlockBytes + soff[i]), "f"(lo[0]), "f"(lo[1]), "f"(lo[2]), "f"(lo[3])
                       : "memory");
      }
      fence_proxy_async();
      mbar_arrive(&C.full_a[e_st]);
      if (++e_st == G::kStages) e_st = 0, e_par ^= 1u;
      if (++e_cb == CB) e_cb = 0;
    };
    // k-blocks this CTA produces in all; two of them in flight per thread (32 KiB per SM): the gather is latency-bound at one
    const long long my_tiles = unit0 < total ? (total - unit0 + nunits - 1) / nunits : 0;
    const long long nkb = my_tiles * KB;
    float4 buf0[4], buf1[4];
    uint32_t ok0 = 0, ok1 = 0;
    if (nkb > 0) fetch(buf0, ok0);
    if (nkb > 1) fetch(buf1, ok1);
    for (long long g = 0; g < nkb; g += 2) {
      {
        float4 cur[4];
        const uint32_t cur_ok = ok0;
#pragma unroll
        for (int i = 0; i < 4; ++i) cur[i] = buf0[i];
        if (g + 2 < nkb) fetch(buf0, ok0);
        emit(cur, cur_ok);
      }
      if (g + 1 < nkb) {
        float4 cur[4];
        const uint32_t cur_ok = ok1;
#pragma unroll
        for (int i = 0; i < 4; ++i) cur[i] = buf1[i];
        if (g + 3 < nkb) fetch(buf1, ok1);
        emit(cur, cur_ok);
      }
    }
  } else {
    // =========================== epilogue (warps 10..13) ===========================
    const int q = warp & 3;                 // TMEM lane quarter this warp may access
    const int r = 32 * q + lane;
    // transposed output of a plain product (output row = input row) with 4-aligned planes: whole-column stores
    const bool tfast = p.out_transposed && p.st == 1 && p.sh == 1 && p.sw == 1 && p.nclass == 1 && (p.ldo & 3) == 0 && (M & 3) == 0;
    uint32_t tc = 0;
    for (long long tile = unit0; tile < total; tile += nunits, ++tc) {
      const int cls = static_cast<int>(tile / per_class);
      const long long mtile = (tile % per_class) / ntiles_n * CTAS + rank;
      const int ntile = static_cast<int>(tile % ntiles_n);
      const long long m = mtile * kTileM + r;
      const bool live = m < M;
      long long orow = 0;
      if (live) {
        const long long THW = static_cast<long long>(p.T) * HW;
        const long long b = m / THW;
        const int inb = static_cast<int>(m - b * THW);
        const int t = inb / HW, h = (inb % HW) / p.W, w = inb % p.W;
        orow = ((b * p.To + (t * p.st + p.cls[cls][0])) * p.Ho + (h * p.sh + p.cls[cls][1])) * p.Wo + (w * p.sw + p.cls[cls][2]);
      }
      const uint32_t acc = tc & 1u;
      mbar_wait(&C.acc_full[acc], (tc >> 1) & 1u);
      tc_fence_after();
      const uint32_t t_lane = tmem + acc * NT + (static_cast<uint32_t>(32 * q) << 16);
#pragma unroll 1
      for (int c0 = 0; c0 < NT; c0 += 32) {
        const int n0 = ntile * NT + c0;
        if (n0 >= p.Nout) break;  // (uniform) the padded columns of the last N tile
        uint32_t v[32];
        tmem_ld32(t_lane + c0, v);
        tmem_ld_wait();
        if (p.out_transposed && tfast) {
          // The four epilogue warps exchange their 32 x 32 blocks through shared memory ([column][128 rows]) so that a warp
          // writes whole columns: 512 contiguous bytes per store instruction instead of 128.
          float* stT = &C.stage[0][0][0];
          asm volatile("bar.sync 2, 128;" ::: "memory");  // the previous block has been read
#pragma unroll
          for (int i = 0; i < 32; ++i) stT[i * kTileM + r] = __uint_as_float(v[i]);
          asm volatile("bar.sync 2, 128;" ::: "memory");
          const long long m0 = mtile * kTileM + 4 * lane;  // rows 4 lane .. 4 lane + 3 of the tile (same plane: ldo % 4 == 0)
          if (m0 < M) {
            const long long plane = m0 / p.ldo;
            float* dst0 = p.out + (plane * p.Nout + n0) * p.ldo + (m0 - plane * p.ldo);
            const int cw = 8 * (warp - (2 + kProdWarps));
#pragma unroll
            for (int cc = 0; cc < 8; ++cc) {
              const int c = cw + cc;
              if (n0 + c < p.Nout) {
                float4 o = *reinterpret_cast<const float4*>(stT + c * kTileM + 4 * lane);
                if (p.bias != nullptr) {
                  const float bc = __ldg(p.bias + n0 + c);
                  o.x += bc, o.y += bc, o.z += bc, o.w += bc;
                }
                if (p.relu_out) o.x = fmaxf(o.x, 0.f), o.y = fmaxf(o.y, 0.f), o.z = fmaxf(o.z, 0.f), o.w = fmaxf(o.w, 0.f);
                *reinterpret_cast<float4*>(dst0 + static_cast<long long>(c) * p.ldo) = o;
              }
            }
          }
        } else if (live && p.out_transposed) {
          // lanes = consecutive rows: every column is one coalesced 128-byte store of the warp
          const long long plane = orow / p.ldo;
          float* dst = p.out + (plane * p.Nout + n0) * p.ldo + (orow - plane * p.ldo);
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            if (n0 + i < p.Nout) {
              float o = __uint_as_float(v[i]);
              if (p.bias != nullptr) o += __ldg(p.bias + n0 + i);
              if (p.relu_out) o = fmaxf(o, 0.f);
              dst[static_cast<long long>(i) * p.ldo] = o;
            }
          }
        } else if (!p.out_transposed) {
          // Through shared memory so that the global accesses are coalesced: a thread owns a ROW of the accumulator, but
          // eight lanes should write the 128 contiguous bytes of one output row.  Row r of this warp's 32 x 32 block goes to
          // stage[r][*]; then lane l handles piece (l & 7) of rows 4 j + (l >> 3), j = 0..7.
          float (*stg)[36] = C.stage[warp - (2 + kProdWarps)];
          __syncwarp();  // the previous chunk's readers are done with the block
#pragma unroll
          for (int i = 0; i < 8; ++i)
            *reinterpret_cast<float4*>(&stg[lane][4 * i]) = make_float4(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]),
                                                                        __uint_as_float(v[4 * i + 2]), __uint_as_float(v[4 * i + 3]));
          __syncwarp();
          const int pc = lane & 7, rsub = lane >> 3;
          const bool col_ok = n0 + 4 * pc < p.Nout;
          float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
          if (p.bias != nullptr && col_ok) b4 = __ldg(reinterpret_cast<const float4*>(p.bias + n0) + pc);
          float4 r4[8];
          const bool has_res = p.residual != nullptr;
          if (has_res) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {  // all eight residual loads in flight before the first one is used
              const int rr = 4 * j + rsub;
              const long long orr = __shfl_sync(0xffffffffu, orow, rr);
              const bool ok = __shfl_sync(0xffffffffu, live ? 1 : 0, rr) != 0 && col_ok;
              r4[j] = ok ? __ldg(reinterpret_cast<const float4*>(p.residual + orr * p.ldo + n0) + pc) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int rr = 4 * j + rsub;
            const long long orr = __shfl_sync(0xffffffffu, orow, rr);
            const bool ok = __shfl_sync(0xffffffffu, live ? 1 : 0, rr) != 0 && col_ok;
            float4 o = *reinterpret_cast<const float4*>(&stg[rr][4 * pc]);
            if (ok) {
              o.x += b4.x, o.y += b4.y, o.z += b4.z, o.w += b4.w;
              if (has_res) o.x += r4[j].x, o.y += r4[j].y, o.z += r4[j].z, o.w += r4[j].w;
              if (p.relu_out) o.x = fmaxf(o.x, 0.f), o.y = fmaxf(o.y, 0.f), o.z = fmaxf(o.z, 0.f), o.w = fmaxf(o.w, 0.f);
              reinterpret_cast<float4*>(p.out + orr * p.ldo + n0)[pc] = o;
            }
          }
        }
      }
      // this warp's tensor-memory reads of the accumulator are complete: hand it back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (CTAS == 2 && rank != 0) mbar_arrive_remote(&C.acc_empty[acc], 0);  // the leader's MMA warp waits for both CTAs
        else mbar_arrive(&C.acc_empty[acc]);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if constexpr (CTAS == 2) cluster_sync();  // both CTAs are done with the pair's tensor memory and barriers
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc<CTAS, 2 * NT>(tmem);
  }
}

// ---- codebook rows ----------------------------------------------------------------------------------------------
// h[row][0..C) = lut[tokens[row]][0..C): the channels-last form of post_vq_conv(embedding(tokens)) (videogpt_vq_vae.py:54-55)
__global__ void embed_rows_kernel(const int64_t* __restrict__ tokens, const float* __restrict__ lut, float* __restrict__ out,
                                  long long rows, int K, int C, uint32_t* status) {
  const int per_row = C >> 2;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= rows * per_row) return;
  const long long row = idx / per_row;
  const int c4 = static_cast<int>(idx - row * per_row);
  const long long tok = tokens[row];
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  if (tok >= 0 && tok < K) v = __ldg(reinterpret_cast<const float4*>(lut + tok * C) + c4);
  else if (c4 == 0 && status != nullptr) atomicOr(status, D3PM_STATUS_BAD_TOKEN);
  reinterpret_cast<float4*>(out + row * C)[c4] = v;
}

// ---- axial attention (AxialBlock, videogpt_vq_vae.py:100-118; scaled_dot_product_attention, model_utils.py:586-600) ----
// qkv: [M][3 axes][q, k, v][heads][dh]; att: [M][3 axes][heads][dh].  One launch per axis, one warp per (sequence along the
// axis, head): K and V of the sequence (L <= LMAX positions) staged in shared memory, a lane holds VPL = dh / 32 channels of
// every vector.  Per query the LMAX partial dot products of a lane are reduced over the warp by a transposing butterfly
// (at every level a lane keeps half of its values and hands the other half to its partner: LMAX - 1 shuffles instead of
// 5 LMAX), after which lane l holds the complete score of key l >> (5 - log2 LMAX); the softmax then runs across lanes.
// Several warps share a job (four queries each), so that a job's Q / K / V tile (24 KiB at 16 positions x 128 channels) serves
// four warps: 36 warps per SM instead of 8, and the load burst of one job overlaps the arithmetic of the others.
struct AttnShape {
  int wj, bw, jpb;  // warps per job, warps per block, jobs per block
};
__host__ __device__ constexpr AttnShape attn_shape(int lmax) {
  const int wj = lmax >= 8 ? lmax / 4 : 1;
  const int bw = wj > 4 ? wj : 4;
  return AttnShape{wj, bw, bw / wj};
}

template <int N>
__device__ __forceinline__ void transpose_reduce(float (&s)[N], int lane, int o) {
  // pairs (m, m + N/2): the lane whose bit `o` is clear keeps the lower half, its partner the upper half
  if constexpr (N >= 2) {
    const bool up = (lane & o) != 0;
#pragma unroll
    for (int m = 0; m < N / 2; ++m) {
      const float keep = up ? s[m + N / 2] : s[m];
      const float send = up ? s[m] : s[m + N / 2];
      s[m] = keep + __shfl_xor_sync(0xffffffffu, send, o);
    }
  }
}

template <int VPL, int LMAX>
__global__ void __launch_bounds__(32 * attn_shape(LMAX).bw) axial_attention_kernel(const float* __restrict__ qkv, float* __restrict__ att, int B,
                                                                                   int T, int H, int W, int heads, int axis, float softmax_scale) {
  constexpr int DH = 32 * VPL;
  constexpr AttnShape SH = attn_shape(LMAX);
  constexpr int QPW = LMAX / SH.wj;  // queries (and rows to load) per warp
  constexpr int LOG = LMAX == 32 ? 5 : (LMAX == 16 ? 4 : (LMAX == 8 ? 3 : 2));
  constexpr int REP = 32 / LMAX;  // lanes that end up holding the same key's score
  static_assert(LMAX == 4 || LMAX == 8 || LMAX == 16 || LMAX == 32, "LMAX must be 4, 8, 16 or 32");
  __shared__ __align__(16) float kv_smem[SH.jpb][3][LMAX][DH];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int jl = warp / SH.wj, wj = warp % SH.wj;  // job of this warp inside the block, and its part of the job
  // axis 0: along W (attn_w, axial_dim -2), 1: along H, 2: along T
  const int L = axis == 0 ? W : (axis == 1 ? H : T);
  const long long M = static_cast<long long>(B) * T * H * W;
  const long long nseq = M / L;
  const long long job = static_cast<long long>(blockIdx.x) * SH.jpb + jl;
  const bool have = job < nseq * heads;
  const long long seq = have ? job / heads : 0;
  const int head = have ? static_cast<int>(job - seq * heads) : 0;
  long long row0, rstride;
  const long long HW = static_cast<long long>(H) * W;
  if (axis == 0) row0 = seq * W, rstride = 1;
  else if (axis == 1) row0 = (seq / W) * HW + seq % W, rstride = W;
  else row0 = (seq / HW) * (T * HW) + seq % HW, rstride = HW;
  const int C = heads * DH;
  const int ldq = 9 * C;  // floats per row of qkv
  float (*ks)[DH] = kv_smem[jl][0];
  float (*vs)[DH] = kv_smem[jl][1];
  float (*qs)[DH] = kv_smem[jl][2];
  const float* qbase = qkv + static_cast<size_t>(axis) * 3 * C + head * DH + lane * VPL;
  auto load_vec = [](const float* src, float (&dst)[VPL]) {
    if constexpr (VPL == 4) {
      const float4 t = __ldg(reinterpret_cast<const float4*>(src));
      dst[0] = t.x, dst[1] = t.y, dst[2] = t.z, dst[3] = t.w;
    } else if constexpr (VPL == 2) {
      const float2 t = __ldg(reinterpret_cast<const float2*>(src));
      dst[0] = t.x, dst[1] = t.y;
    } else {
      dst[0] = __ldg(src);
    }
  };
  // this warp's rows of the job's Q / K / V tile (rows past the sequence are zero)
#pragma unroll
  for (int jj = 0; jj < QPW; ++jj) {
    const int j = wj * QPW + jj;
    float qq[VPL], kk[VPL], vv[VPL];
#pragma unroll
    for (int e = 0; e < VPL; ++e) qq[e] = 0.f, kk[e] = 0.f, vv[e] = 0.f;
    if (have && j < L) {
      const float* rowp = qbase + (row0 + j * rstride) * ldq;
      load_vec(rowp, qq);
      load_vec(rowp + C, kk);
      load_vec(rowp + 2 * C, vv);
    }
#pragma unroll
    for (int e = 0; e < VPL; ++e) qs[j][lane * VPL + e] = qq[e], ks[j][lane * VPL + e] = kk[e], vs[j][lane * VPL + e] = vv[e];
  }
  __syncthreads();
  if (!have) return;
  const float scale = (softmax_scale > 0.f ? softmax_scale : rsqrtf(static_cast<float>(DH))) * 1.4426950408889634f;  // scores in log2 units
  const int myj = lane >> (5 - LOG);  // the key whose score this lane holds after the reduction
  for (int i = wj * QPW; i < (wj + 1) * QPW && i < L; ++i) {
    float qv[VPL];
#pragma unroll
    for (int e = 0; e < VPL; ++e) qv[e] = qs[i][lane * VPL + e];
    float s[LMAX];
#pragma unroll
    for (int j = 0; j < LMAX; ++j) {
      float d = 0.f;
#pragma unroll
      for (int e = 0; e < VPL; ++e) d = fmaf(qv[e], ks[j][lane * VPL + e], d);
      s[j] = d;
    }
    // transposing butterfly: after the level with offset o a lane holds the values whose index has bit (o's rank) equal to
    // its own lane bit; log2(LMAX) levels leave one value per lane, the remaining levels are plain butterflies
    if constexpr (LOG >= 1) transpose_reduce<LMAX>(s, lane, 16);
    if constexpr (LOG >= 2) transpose_reduce<LMAX / 2>(reinterpret_cast<float (&)[LMAX / 2]>(s), lane, 8);
    if constexpr (LOG >= 3) transpose_reduce<LMAX / 4>(reinterpret_cast<float (&)[LMAX / 4]>(s), lane, 4);
    if constexpr (LOG >= 4) transpose_reduce<LMAX / 8>(reinterpret_cast<float (&)[LMAX / 8]>(s), lane, 2);
    if constexpr (LOG >= 5) transpose_reduce<LMAX / 16>(reinterpret_cast<float (&)[LMAX / 16]>(s), lane, 1);
    float sc = s[0];
#pragma unroll
    for (int o = 16 >> LOG; o > 0; o >>= 1) sc += __shfl_xor_sync(0xffffffffu, sc, o);
    // lane l: score of key myj (bits of the key index follow the lane bits from the top: level 16 decided the highest bit)
    sc = myj < L ? sc * scale : -3.0e38f;
    float mx = sc;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    const float e_ = myj < L ? exp2f(sc - mx) : 0.f;
    float sum = e_;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float pr = e_ * (static_cast<float>(REP) / sum);  // every key is counted REP times in `sum`
    float acc[VPL];
#pragma unroll
    for (int e = 0; e < VPL; ++e) acc[e] = 0.f;
#pragma unroll
    for (int j = 0; j < LMAX; ++j) {
      const float pj = __shfl_sync(0xffffffffu, pr, j << (5 - LOG));
#pragma unroll
      for (int e = 0; e < VPL; ++e) acc[e] = fmaf(pj, vs[j][lane * VPL + e], acc[e]);
    }
    float* o = att + (row0 + i * rstride) * (3 * C) + axis * C + head * DH + lane * VPL;
    if constexpr (VPL == 4) *reinterpret_cast<float4*>(o) = make_float4(acc[0], acc[1], acc[2], acc[3]);
    else if constexpr (VPL == 2) *reinterpret_cast<float2*>(o) = make_float2(acc[0], acc[1]);
    else o[0] = acc[0];
  }
}

// ---- col2im of the last transposed convolution ----------------------------------------------------------------------
// yT: [B * T][64 * Cout][H * W] (the plane-transposed rows of the last GEMM: row ((kt*4 + kh)*4 + kw)*Cout + c of plane (b, it),
// column = (ih, iw)) = contribution of an input position through filter tap (kt, kh, kw) to output channel c.
// out: [B][Cout][To][Ho][Wo] (the reference's layout) = bias + the contributions that land on each voxel: along a dimension
// of stride s, tap k of input i lands on y = (i + pf) * s + k - 3, pf = ceil((4 - s) / 2) (F.pad of SamePadConvTranspose3d
// :324-328, then ConvTranspose3d with padding 3 :330-332).  A thread owns the sw output voxels above one input column
// position, so the lanes of a warp read consecutive input positions of one (tap, channel) row: coalesced.
__global__ void col2im_kernel(const float* __restrict__ yT, const float* __restrict__ bias, float* __restrict__ out, int B, int T, int H,
                              int W, int Cout, int st, int sh, int sw) {
  const int To = T * st, Ho = H * sh;
  const long long Wo = static_cast<long long>(W) * sw;
  const long long total = static_cast<long long>(B) * To * Ho * W;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int mw = static_cast<int>(idx % W);
  const int yh = static_cast<int>((idx / W) % Ho);
  const int yt = static_cast<int>((idx / (static_cast<long long>(W) * Ho)) % To);
  const long long b = idx / (static_cast<long long>(W) * Ho * To);
  const int pft = (4 - st + 1) / 2, pfh = (4 - sh + 1) / 2, pfw = (4 - sw + 1) / 2;
  const long long P = static_cast<long long>(H) * W;
  float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
  for (int kt = 0; kt < 4; ++kt) {
    const int nt = yt + 3 - kt;
    if (nt % st != 0) continue;
    const int it = nt / st - pft;
    if (it < 0 || it >= T) continue;
    const float* plane = yT + (b * T + it) * (64LL * Cout) * P;
    for (int kh = 0; kh < 4; ++kh) {
      const int nh = yh + 3 - kh;
      if (nh % sh != 0) continue;
      const int ih = nh / sh - pfh;
      if (ih < 0 || ih >= H) continue;
#pragma unroll
      for (int pw = 0; pw < 2; ++pw) {
        if (pw >= sw) break;
        const int yw = mw * sw + pw;
#pragma unroll
        for (int kw = 0; kw < 4; ++kw) {
          const int nw = yw + 3 - kw;
          if (nw % sw != 0) continue;
          const int iw = nw / sw - pfw;
          if (iw < 0 || iw >= W) continue;
          const float* src = plane + static_cast<long long>(((kt * 4 + kh) * 4 + kw) * Cout) * P + ih * W + iw;
          for (int c = 0; c < Cout && c < 4; ++c) acc[pw][c] += __ldg(src + c * P);
        }
      }
    }
  }
  for (int c = 0; c < Cout && c < 4; ++c) {
    float* dst = out + (((b * Cout + c) * To + yt) * Ho + yh) * Wo + static_cast<long long>(mw) * sw;
    const float bc = bias != nullptr ? bias[c] : 0.f;
    if (sw == 2) *reinterpret_cast<float2*>(dst) = make_float2(acc[0][c] + bc, acc[1][c] + bc);
    else dst[0] = acc[0][c] + bc;
  }
}

// The same for the strides the decoder's last layer has in practice, (ST, 2, 2): the taps that land on a voxel are known up
// to the parities of yt / yh, so the 16 (ST = 1) or 8 (ST = 2) x 2 x 3 loads of a thread are straight-line code with range
// predicates only - they are all in flight together instead of one per loop iteration.
template <int ST>
__global__ void __launch_bounds__(256) col2im_s22_kernel(const float* __restrict__ yT, const float* __restrict__ bias, float* __restrict__ out,
                                                         int B, int T, int H, int W, int Cout) {
  const int To = T * ST, Ho = H * 2;
  const long long Wo = 2LL * W;
  const long long total = static_cast<long long>(B) * To * Ho * W;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int mw = static_cast<int>(idx % W);
  const int yh = static_cast<int>((idx / W) % Ho);
  const int yt = static_cast<int>((idx / (static_cast<long long>(W) * Ho)) % To);
  const long long b = idx / (static_cast<long long>(W) * Ho * To);
  const long long P = static_cast<long long>(H) * W;
  constexpr int NKT = 4 / ST;
  const int kt0 = ST == 1 ? 0 : ((yt + 1) & 1);   // taps kt0, kt0 + ST, ...
  const int kh0 = (yh + 1) & 1;                   // taps kh0, kh0 + 2
  float acc[2][3] = {{0.f, 0.f, 0.f}, {0.f, 0.f, 0.f}};
#pragma unroll
  for (int a = 0; a < NKT; ++a) {
    const int kt = kt0 + a * ST;
    const int it = (yt + 3 - kt) / ST - (ST == 1 ? 2 : 1);
    const bool okt = it >= 0 && it < T;
    const float* plane = yT + (b * T + (okt ? it : 0)) * (64LL * Cout) * P;
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int kh = kh0 + 2 * e;
      const int ih = (yh + 3 - kh) / 2 - 1;
      const bool okh = okt && ih >= 0 && ih < H;
#pragma unroll
      for (int pw = 0; pw < 2; ++pw)
#pragma unroll
        for (int f = 0; f < 2; ++f) {
          const int kw = ((pw + 1) & 1) + 2 * f;
          const int iw = (2 * mw + pw + 3 - kw) / 2 - 1;
          const bool ok = okh && iw >= 0 && iw < W;
          const float* src = plane + static_cast<long long>(((kt * 4 + kh) * 4 + kw) * Cout) * P + (okh ? ih : 0) * W + (ok ? iw : 0);
#pragma unroll
          for (int c = 0; c < 3; ++c)
            if (c < Cout) acc[pw][c] += ok ? __ldg(src + c * P) : 0.f;
        }
    }
  }
#pragma unroll
  for (int c = 0; c < 3; ++c)
    if (c < Cout) {
      const float bc = bias != nullptr ? bias[c] : 0.f;
      float* dst = out + (((b * Cout + c) * To + yt) * Ho + yh) * Wo + 2LL * mw;
      *reinterpret_cast<float2*>(dst) = make_float2(acc[0][c] + bc, acc[1][c] + bc);
    }
}

}  // namespace dec
}  // namespace d3pm
