// Plumbing shared by the two persistent kernels, the reverse step (d3pm_step_stream.cuh) and the training loss
// (d3pm_train_stream.cuh): the CTA shape, the group barrier, shared-memory read-backs, the 16-bit logit rows and the
// launcher.  Each kernel's own mathematics stays in its own file.
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <type_traits>

#include "d3pm_common.cuh"
#include "d3pm_host.h"

namespace d3pm {

constexpr int kStreamThreads = 512;  // one CTA per SM: 16 warps to hide a row's latency, up to 128 registers a thread
constexpr int kCoefSmemRows = 256;  // timesteps whose coefficients are staged in shared memory (16 KiB)

// barrier of a group of NW warps (named barrier `id`); a one-warp group only needs the warp to reconverge
template <int NW>
struct StreamSync {
  int id;
  __device__ __forceinline__ void operator()() const {
    if (NW == 1) __syncwarp();
    else asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(32 * NW) : "memory");
  }
};
__device__ __forceinline__ float4 lds4(const float* p) { return *reinterpret_cast<const float4*>(p); }
// Logit storage type of a stream-kernel instantiation.  LD = D3PM_LOGITS_F32: the stage holds fp32 rows.  F16 / BF16 (a
// denoiser run under autocast): the row is copied as it lies in HBM (half the bytes), a chunk of four classes is 8 bytes of
// the stage and is widened to fp32 in registers - exactly the values `logits.float()` would hold, without the 2 x 1 GB cast
// pass a caller would otherwise pay at config 2.  Everything downstream of the load is the fp32 code.
template <int LD>
struct LogitType {
  static constexpr uint32_t kBytes = LD == D3PM_LOGITS_F32 ? 4u : 2u;
  static __device__ __forceinline__ float2 widen(uint32_t pair) {
    if constexpr (LD == D3PM_LOGITS_BF16) {
      return make_float2(__uint_as_float(pair << 16), __uint_as_float(pair & 0xffff0000u));
    } else {
      return __half22float2(*reinterpret_cast<const __half2*>(&pair));
    }
  }
  // chunk q (classes 4q .. 4q+3) of a staged row: lo = classes (0, 1), hi = classes (2, 3)
  static __device__ __forceinline__ void chunk(const float* stage, int q, float2& lo, float2& hi) {
    if constexpr (LD == D3PM_LOGITS_F32) {
      const float4 a = lds4(stage + 4 * q);
      lo = make_float2(a.x, a.y), hi = make_float2(a.z, a.w);
    } else {
      const uint2 raw = *reinterpret_cast<const uint2*>(reinterpret_cast<const unsigned char*>(stage) + 8 * q);
      lo = widen(raw.x), hi = widen(raw.y);
    }
  }
  static __device__ __forceinline__ float one(const float* stage, uint32_t k) {
    if constexpr (LD == D3PM_LOGITS_F32) {
      return stage[k];
    } else {
      const uint32_t h = reinterpret_cast<const unsigned short*>(stage)[k];
      if constexpr (LD == D3PM_LOGITS_BF16) return __uint_as_float(h << 16);
      else return __half2float(__ushort_as_half(static_cast<unsigned short>(h)));
    }
  }
  static __device__ __forceinline__ const void* row(const float* base, unsigned long long elements) {
    return reinterpret_cast<const unsigned char*>(base) + elements * kBytes;
  }
  // Rows written in the logits' type (the training kernel's gradient): fp32 values narrowed with round-to-nearest-even,
  // which is what `tensor.to(torch.float16 / torch.bfloat16)` does, so a 16-bit row equals the fp32 row cast afterwards.
  using Elem = std::conditional_t<LD == D3PM_LOGITS_F32, float, unsigned short>;
  static __device__ __forceinline__ uint32_t narrow2(float lo, float hi) {
    uint32_t bits;
    if constexpr (LD == D3PM_LOGITS_BF16) {
      const __nv_bfloat162 v = __float22bfloat162_rn(make_float2(lo, hi));
      bits = *reinterpret_cast<const uint32_t*>(&v);
    } else {
      const __half2 v = __float22half2_rn(make_float2(lo, hi));
      bits = *reinterpret_cast<const uint32_t*>(&v);
    }
    return bits;
  }
  static __device__ __forceinline__ Elem narrow1(float v) {
    if constexpr (LD == D3PM_LOGITS_F32) return v;
    else if constexpr (LD == D3PM_LOGITS_BF16) return __bfloat16_as_ushort(__float2bfloat16_rn(v));
    else return __half_as_ushort(__float2half_rn(v));
  }
  // classes 4q .. 4q+3 of an output row, one streaming store (16 bytes for fp32, 8 for the 16-bit types)
  static __device__ __forceinline__ void store4(Elem* rowp, uint32_t q, const float (&o)[4]) {
    if constexpr (LD == D3PM_LOGITS_F32) {
      st_stream4(rowp + 4 * q, make_float4(o[0], o[1], o[2], o[3]));
    } else {
      st_stream_b64(rowp + 4 * q, narrow2(o[0], o[1]), narrow2(o[2], o[3]));
    }
  }
};
// the NW per-warp values of a reduction, read back in one shared-memory load (unused lanes of the float4 = neutral)
template <int NW>
__device__ __forceinline__ float4 lds_warps(const float* p, float neutral) {
  if (NW == 4) return lds4(p);
  const float2 a = *reinterpret_cast<const float2*>(p);
  return make_float4(a.x, a.y, neutral, neutral);
}

__device__ __forceinline__ float warp_min(float x) {
  float m;
  asm volatile("redux.sync.min.f32 %0, %1, 0xffffffff;" : "=f"(m) : "f"(x));
  return m;
}

// One CTA of `threads` threads per SM, `smem` bytes of dynamic shared memory.  D3PM_ERR_CUDA when the SM count cannot be
// queried or the shared-memory limit cannot be raised.
template <typename Params>
int launch_persistent(void (*kern)(Params), int threads, size_t smem, const Params& p, cudaStream_t s) {
  const int sms = host::sm_count();
  if (sms == 0) return D3PM_ERR_CUDA;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)) != cudaSuccess)
    return D3PM_ERR_CUDA;
  kern<<<static_cast<unsigned>(sms), threads, smem, s>>>(p);
  return D3PM_OK;
}

}  // namespace d3pm
