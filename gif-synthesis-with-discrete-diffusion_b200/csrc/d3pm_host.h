// Host-side helpers shared by the translation units of libd3pm_b200.so (not exported: hidden visibility).
#pragma once

#include <cuda_runtime.h>

#include "d3pm_b200.h"

namespace d3pm {
namespace host {

// sets the thread-local text d3pm_last_error() returns and hands `code` back
__attribute__((visibility("hidden"))) int fail(int code, const char* fmt, ...) __attribute__((format(printf, 2, 3)));
__attribute__((visibility("hidden"))) int check_launch(const char* what);

// SM count of the current device, 0 when it cannot be queried
__attribute__((visibility("hidden"))) inline int sm_count() {
  int dev = 0, sms = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
  return sms;
}

// The kernels launch on the CUDA *current* device; the caller's tensors (and stream) may live on another one
// (model on cuda:1 while cuda:0 is current).  Every entry point therefore makes the device that owns its first
// device pointer current for the duration of the call and restores the previous one on return.  The entry points
// of the host-step handle, which owns its buffers, name the device instead (the `int` constructor).
class __attribute__((visibility("hidden"))) DeviceGuard {
 public:
  explicit DeviceGuard(int device) {
    if (cudaGetDevice(&prev_) == cudaSuccess && prev_ != device) switched_ = cudaSetDevice(device) == cudaSuccess;
  }
  explicit DeviceGuard(const void* device_ptr) {
    if (cudaGetDevice(&prev_) != cudaSuccess) {
      cudaGetLastError();
      return;
    }
    cudaPointerAttributes attr;
    if (device_ptr == nullptr || cudaPointerGetAttributes(&attr, device_ptr) != cudaSuccess) {
      cudaGetLastError();  // not a CUDA allocation: the launch itself will report it
      return;
    }
    if ((attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged) && attr.device != prev_)
      switched_ = cudaSetDevice(attr.device) == cudaSuccess;
  }
  ~DeviceGuard() {
    if (switched_) cudaSetDevice(prev_);
  }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;

 private:
  int prev_ = 0;
  bool switched_ = false;
};

}  // namespace host
}  // namespace d3pm
