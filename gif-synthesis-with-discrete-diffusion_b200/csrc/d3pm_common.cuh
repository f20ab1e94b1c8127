// Shared device helpers for the D3PM reverse-step and training kernels (sm_100a only).
//
// Math notation follows DESIGN.md §3 / SURVEY.md §8(a8).  Reference lines are those of
// src/models/motionencoder/diffusion_transformer.py.
#pragma once

#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "d3pm_b200.h"

namespace d3pm {

constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;
constexpr float kClampLo = -70.0f;                // clamp floor of :236, :247, :283
constexpr float kPFloor = 3.975449735908647e-31f; // exp(-70)
constexpr float kLogTiny = -69.07755278982137f;   // log(1e-30): one-hot "zero" of :50, :258
constexpr float kTiny = 1e-30f;
constexpr float kTwoPowM24 = 5.9604644775390625e-8f;

// ---- coefficient table (one row of D3PM_COEF_STRIDE floats per timestep) -------------------
// With p_k = exp(log p(x0=k)), primes = cumulative schedule at t-1 (identity slot at t = 0):
//   masked x_t:    e^L = WM*sum(p) + 1e-30;  P_k = p_k*AM + BOM*e^L;  P_K = C1 + CP*e^L
//   unmasked x_t=j: e^L = WO*(sum(p)-p_j) + WS*p_j + 1e-30;
//                  P_k = p_k*AO + BOO*e^L (k!=j);  P_j = p_j*AS + BOS*e^L;  P_K = PK1*e^L
// and the posterior of :283 is clamp(log P, -70, 0).  The fused step knows sum(p) = 1 (p is a
// softmax), so its e^L needs only p_j.
enum Coef : int {
  C_AM = 0, C_BOM = 1, C_WM = 2, C_C1 = 3,
  C_CP = 4,
  C_AO = 8, C_AS = 9, C_BOO = 10, C_BOS = 11,
  C_WO = 12, C_WS = 13, C_PK1 = 14,
  C_COUNT = 16
};
static_assert(C_COUNT <= D3PM_COEF_STRIDE, "coefficient row too small");

struct RowCoef {  // what one token row needs, already specialised on masked / unmasked
  float A;     // multiplies p_k for k != x_t
  float BO;    // multiplies e^L for k != x_t
  float AS;    // multiplies p_j (unmasked only)
  float BOS;   // multiplies e^L for k == x_t (unmasked only)
  float W;     // weight of p_k in e^L (k != x_t)
  float WS;    // weight of p_j in e^L
  float PK0;   // P_K = PK0 + PK1 * e^L
  float PK1;
};

__device__ __forceinline__ float ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float lg2(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// exact residual of the fp32 product m*log2e (natural-log units -> log2 units)
__device__ __forceinline__ float to_log2_units(float m) { return __fmul_rn(m, kLog2e); }

// ln(sum_k exp(x_k - M)) from S = sum_k 2^(x_k*log2e - fl(M*log2e)): corrects the rounding of M*log2e
__device__ __forceinline__ float ln_rel_sum(float M, float S) {
  const float m2 = to_log2_units(M);
  const float delta = -fmaf(M, kLog2e, -m2);  // m2 - M*log2e, exact
  return kLn2 * (lg2(S) + delta);
}
// clamp(log P, -70, 0): the single place the posterior leaves the linear domain, shared by every
// sampling mode so that they agree bit for bit.
__device__ __forceinline__ float log_prob_clamped(float P) {
  return fminf(fmaxf(lg2(P) * kLn2, kClampLo), 0.0f);
}

// streaming 128-bit accesses: the logits are read exactly once, keep them out of L1
__device__ __forceinline__ float4 ld_stream4(const float* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ void st_stream4(float* p, float4 v) {
  asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
               : "memory");
}
// the 64-bit counterpart, for four 16-bit values
__device__ __forceinline__ void st_stream_b64(void* p, uint32_t lo, uint32_t hi) {
  asm volatile("st.global.cs.v2.b32 [%0], {%1,%2};" ::"l"(p), "r"(lo), "r"(hi) : "memory");
}

__device__ __forceinline__ float warp_max(float x) {
  float m;  // CREDUX.MAX.F32 on sm_100a: one instruction instead of five shuffles
  asm volatile("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(m) : "f"(x));
  return m;
}
__device__ __forceinline__ float warp_sum(float x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}
// Warp arg-max of (value, index) pairs with the first-index tie rule, as one orderable key: two CREDUX instead of a
// five-step 64-bit butterfly.  Every lane returns the warp's key.
__device__ __forceinline__ unsigned long long pack_key(float score, uint32_t k);
__device__ __forceinline__ unsigned long long warp_argmax_key(float v, uint32_t idx) {
  float vm;
  asm volatile("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(vm) : "f"(v));
  const uint32_t im = __reduce_min_sync(0xffffffffu, v == vm ? idx : 0xffffffffu);
  return pack_key(vm, im);
}
__device__ __forceinline__ unsigned long long warp_max_u64(unsigned long long x) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    unsigned long long y = __shfl_xor_sync(0xffffffffu, x, o);
    x = y > x ? y : x;
  }
  return x;
}

// (score, class) -> one 64-bit key whose integer order is "higher score, then lower class":
// exactly torch.argmax's first-maximal-index rule (:357).
__device__ __forceinline__ unsigned long long pack_key(float score, uint32_t k) {
  uint32_t b = __float_as_uint(score);
  b = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
  return (static_cast<unsigned long long>(b) << 32) | (0xffffffffu - k);
}
__device__ __forceinline__ uint32_t key_class(unsigned long long key) {
  return 0xffffffffu - static_cast<uint32_t>(key & 0xffffffffu);
}
__device__ __forceinline__ float key_score(unsigned long long key) {
  uint32_t b = static_cast<uint32_t>(key >> 32);
  b = (b & 0x80000000u) ? (b & 0x7fffffffu) : ~b;
  return __uint_as_float(b);
}

// ---- noise: Philox4x32-7 (Salmon et al. 2011) -----------------------------------------------------
// Every class k of every global token row draws a 23-bit integer m from a counter-based stream, so a
// row's noise does not depend on which GPU, CTA or kernel variant processes it:
//   * 16 high bits h from a COARSE call, counter (coarse_call(k), row, offset), eight 16-bit halves per
//     call.  The production kernel decides with h alone whether a class can still win the race.
//   * 7 low bits from a FINE call, counter (k >> 4, row, offset | 2^63), one byte per class; only classes
//     that survive the coarse test (and the verification paths) ever compute it.
// m = h << 7 | low7, v = (2m+1) / 2^24 in (0,1) is the "distance from 1" and u = 1 - v is the uniform
// torch.rand_like would have returned (:355); both are exact in fp32.
// A coarse call serves the two float4 chunks c and c+128 of a 1024-class block (the pair one thread of a
// 128-thread group owns): coarse_call = (c / 256) * 128 + c % 128, half = 4 * ((c / 128) % 2) + k % 4.
constexpr uint32_t kPhiloxM0 = 0xD2511F53u, kPhiloxM1 = 0xCD9E8D57u;
constexpr uint32_t kPhiloxW0 = 0x9E3779B9u, kPhiloxW1 = 0xBB67AE85u;
constexpr int kPhiloxRounds = 7;  // Philox4x32-7: the fewest rounds that pass BigCrush (Salmon et al., Table 2)

// Keys = where the 2 x 7 round keys live: NoiseKeysLocal derives them from the seed in registers; the stream kernel
// passes NoiseKeysParam, whose keys were expanded on the host into the kernel's parameter block, so that every round's
// key is a constant-bank operand of its LOP3 (no per-row key arithmetic, no registers).
struct NoiseKeysLocal {
  uint32_t rk0[kPhiloxRounds], rk1[kPhiloxRounds];
  __device__ __forceinline__ explicit NoiseKeysLocal(uint64_t seed) {
    uint32_t k0 = static_cast<uint32_t>(seed), k1 = static_cast<uint32_t>(seed >> 32);
#pragma unroll
    for (int r = 0; r < kPhiloxRounds; ++r) {
      rk0[r] = k0, rk1[r] = k1;
      k0 += kPhiloxW0, k1 += kPhiloxW1;
    }
  }
  __device__ __forceinline__ uint32_t key0(int r) const { return rk0[r]; }
  __device__ __forceinline__ uint32_t key1(int r) const { return rk1[r]; }
};
struct PhiloxRoundKeys {  // host-expanded keys (d3pm_api.cu fills them from the seed)
  uint32_t rk0[kPhiloxRounds + 1], rk1[kPhiloxRounds + 1];
};
inline void expand_round_keys(uint64_t seed, PhiloxRoundKeys& out) {
  uint32_t k0 = static_cast<uint32_t>(seed), k1 = static_cast<uint32_t>(seed >> 32);
  for (int r = 0; r <= kPhiloxRounds; ++r) {
    out.rk0[r] = k0, out.rk1[r] = k1;
    k0 += kPhiloxW0, k1 += kPhiloxW1;
  }
}
struct NoiseKeysParam {
  const PhiloxRoundKeys& k;
  __device__ __forceinline__ explicit NoiseKeysParam(const PhiloxRoundKeys& keys) : k(keys) {}
  __device__ __forceinline__ uint32_t key0(int r) const { return k.rk0[r]; }
  __device__ __forceinline__ uint32_t key1(int r) const { return k.rk1[r]; }
};

template <typename Keys>
struct NoiseStreamT {
  Keys keys;  // round keys (uniform across the grid)
  uint32_t off_lo, off_hi;

  __device__ __forceinline__ NoiseStreamT(const Keys& k, uint64_t offset)
      : keys(k), off_lo(static_cast<uint32_t>(offset)), off_hi(static_cast<uint32_t>(offset >> 32) & 0x7fffffffu) {}
  __device__ __forceinline__ uint4 philox(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) const {
#pragma unroll
    for (int r = 0; r < kPhiloxRounds; ++r) {
      const unsigned long long p0 = static_cast<unsigned long long>(kPhiloxM0) * c0;  // one IMAD.WIDE each
      const unsigned long long p1 = static_cast<unsigned long long>(kPhiloxM1) * c2;
      c0 = static_cast<uint32_t>(p1 >> 32) ^ c1 ^ keys.key0(r);
      c2 = static_cast<uint32_t>(p0 >> 32) ^ c3 ^ keys.key1(r);
      c1 = static_cast<uint32_t>(p1);
      c3 = static_cast<uint32_t>(p0);
    }
    return make_uint4(c0, c1, c2, c3);
  }
  __device__ __forceinline__ uint4 coarse(uint32_t call, uint64_t row) const {
    return philox(call, static_cast<uint32_t>(row), off_lo ^ static_cast<uint32_t>(row >> 32), off_hi);
  }
  __device__ __forceinline__ uint4 fine(uint32_t call, uint64_t row) const {
    return philox(call, static_cast<uint32_t>(row), off_lo ^ static_cast<uint32_t>(row >> 32), off_hi | 0x80000000u);
  }
  static __device__ __forceinline__ uint32_t coarse_call_of_chunk(uint32_t chunk) {
    return ((chunk >> 8) << 7) | (chunk & 127u);
  }
  static __device__ __forceinline__ uint32_t coarse_half_of(uint32_t k) { return (((k >> 9) & 1u) << 2) | (k & 3u); }
  // the 23-bit draw of class k (both calls; slow paths only)
  __device__ __forceinline__ uint32_t draw(uint32_t k, uint64_t row) const {
    const uint4 cw = coarse(coarse_call_of_chunk(k >> 2), row);
    const uint4 fw = fine(k >> 4, row);
    return (half_of(cw, coarse_half_of(k)) << 7) | low7_of(fw, k & 15u);
  }
  static __device__ __forceinline__ uint32_t word_of(const uint4& w, uint32_t i) {
    return i == 0 ? w.x : i == 1 ? w.y : i == 2 ? w.z : w.w;
  }
  static __device__ __forceinline__ uint32_t half_of(const uint4& w, uint32_t h) {
    const uint32_t x = word_of(w, h >> 1);
    return (h & 1u) ? (x >> 16) : (x & 0xffffu);
  }
  static __device__ __forceinline__ uint32_t low7_of(const uint4& w, uint32_t byte) {
    return (word_of(w, byte >> 2) >> (8u * (byte & 3u))) & 0x7fu;
  }
};
struct NoiseStream : NoiseStreamT<NoiseKeysLocal> {
  __device__ __forceinline__ NoiseStream(uint64_t seed, uint64_t offset) : NoiseStreamT<NoiseKeysLocal>(NoiseKeysLocal(seed), offset) {}
};
using ParamNoiseStream = NoiseStreamT<NoiseKeysParam>;

__device__ __forceinline__ float uniform_from_draw(uint32_t m) {
  return __uint2float_rn(0x1000000u - (2u * m + 1u)) * kTwoPowM24;
}
// Gumbel noise exactly as the reference forms it from u (:356), in accurate fp32.
__device__ __forceinline__ float gumbel_from_uniform(float u) {
  return -logf(-logf(u + kTiny) + kTiny);
}

constexpr int kRowThreads = 256;  // threads of the one-CTA-per-row kernels (step_rows_kernel, train_rows_kernel)

// ---- group reductions ------------------------------------------------------------------------
// All threads of a group (NW warps) call these together; `sync` is the group's barrier.
struct CtaSync {
  __device__ __forceinline__ void operator()() const { __syncthreads(); }
};

template <int NW, typename Sync>
__device__ __forceinline__ unsigned long long group_max_u64(unsigned long long key, unsigned long long* scratch,
                                                            Sync sync) {
  const int lane = threadIdx.x & 31, warp = (threadIdx.x >> 5) % NW;
  key = warp_max_u64(key);
  if (lane == 0) scratch[warp] = key;
  sync();
  unsigned long long best = scratch[0];
#pragma unroll
  for (int w = 1; w < NW; ++w) best = scratch[w] > best ? scratch[w] : best;
  return best;
}

template <int NW, typename Sync>
__device__ __forceinline__ float group_max_f32(float x, float* scratch, Sync sync) {
  const int lane = threadIdx.x & 31, warp = (threadIdx.x >> 5) % NW;
  x = warp_max(x);
  if (lane == 0) scratch[warp] = x;
  sync();
  float best = scratch[0];
#pragma unroll
  for (int w = 1; w < NW; ++w) best = fmaxf(best, scratch[w]);
  return best;
}

// Per-row coefficients from the table row of timestep t: the first 8 floats of a row serve masked tokens, floats
// 8..15 unmasked ones.  `lo`, `hi` are the two float4 of the half that applies.
__device__ __forceinline__ RowCoef row_coef_from(const float4& lo, const float4& hi, bool masked) {
  RowCoef r;
  if (masked) {
    r.A = lo.x;      // AM
    r.BO = lo.y;     // BOM
    r.AS = 0.f;
    r.BOS = 0.f;
    r.W = lo.z;      // WM
    r.WS = lo.z;
    r.PK0 = lo.w;    // C1
    r.PK1 = hi.x;    // CP
  } else {
    r.A = lo.x;      // AO
    r.AS = lo.y;     // AS
    r.BO = lo.z;     // BOO
    r.BOS = lo.w;    // BOS
    r.W = hi.x;      // WO
    r.WS = hi.y;     // WS
    r.PK0 = 0.f;
    r.PK1 = hi.z;    // PK1
  }
  return r;
}
__device__ __forceinline__ RowCoef load_row_coef(const float* __restrict__ table, int t, bool masked) {
  const float4* row = reinterpret_cast<const float4*>(table + static_cast<size_t>(t) * D3PM_COEF_STRIDE) + (masked ? 0 : 2);
  return row_coef_from(__ldg(row), __ldg(row + 1), masked);
}

}  // namespace d3pm
