// common.cuh — shared helpers for libvrpx (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <stdint.h>
#include <stdio.h>

#include "vrpx.h"

namespace vrpx {

// ---------------------------------------------------------------- errors / accounting
void set_error(const char* fmt, ...);
void count_launch(int n = 1);

#define VRPX_CHECK_ARG(cond, msg)                                  \
  do {                                                             \
    if (!(cond)) {                                                 \
      vrpx::set_error("%s: %s", __func__, msg);                    \
      return VRPX_ERR_ARG;                                         \
    }                                                              \
  } while (0)

#define VRPX_CUDA(call)                                                                  \
  do {                                                                                   \
    cudaError_t e_ = (call);                                                             \
    if (e_ != cudaSuccess) {                                                             \
      vrpx::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
      return VRPX_ERR_CUDA;                                                              \
    }                                                                                    \
  } while (0)

#define VRPX_LAUNCH_CHECK()                 \
  do {                                      \
    vrpx::count_launch();                   \
    VRPX_CUDA(cudaGetLastError());          \
  } while (0)

int num_sms();  // multiprocessor count of the current device (cached)

// NVTX range around the host side of a phase (encoder / score tables / decode loop / backward): shows up in nsys / ncu
// timelines; costs nothing when no tool is attached (header-only NVTX v3, lazily bound).
struct NvtxRange {
  explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
  ~NvtxRange() { nvtxRangePop(); }
  NvtxRange(const NvtxRange&) = delete;
  NvtxRange& operator=(const NvtxRange&) = delete;
};

// Every launching entry point runs on the device that OWNS its buffers, not on whatever device happens to be current
// in the calling thread: the guard looks the owner of a device pointer up (cudaPointerGetAttributes), switches to it
// and restores the previous device on scope exit.  The stream the caller passes must belong to that device.
struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(const void* device_ptr) {
    cudaPointerAttributes a;
    err = cudaPointerGetAttributes(&a, device_ptr);
    if (err != cudaSuccess) return;
    if (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) {
      err = cudaErrorInvalidDevicePointer;
      return;
    }
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != a.device) {
      err = cudaSetDevice(a.device);
      switched = (err == cudaSuccess);
    }
  }
  ~DeviceGuard() {
    if (switched) cudaSetDevice(prev);
  }
  DeviceGuard(const DeviceGuard&) = delete;
  DeviceGuard& operator=(const DeviceGuard&) = delete;
};
#define VRPX_DEVICE_GUARD(ptr)                                                                       \
  vrpx::DeviceGuard device_guard_(ptr);                                                              \
  if (device_guard_.err != cudaSuccess) {                                                            \
    vrpx::set_error("%s: %s is not a device pointer this process can use (%s)", __func__, #ptr,      \
                    cudaGetErrorString(device_guard_.err));                                          \
    (void)cudaGetLastError();                                                                        \
    return VRPX_ERR_ARG;                                                                             \
  }

// ---------------------------------------------------------------- device helpers
constexpr int E = VRPX_EMB;      // 128
constexpr int NH = VRPX_HEADS;   // 8
constexpr int FF = VRPX_FF;      // 512

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Philox4x32-10 (Salmon et al. 2011), counter-based; one call = 4 x u32.
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0;
    key.y += W1;
  }
  return ctr;
}
// 53-bit uniform in [0,1) from two u32 (same construction as numpy's legacy random_sample).
__device__ __forceinline__ double u53(uint32_t a, uint32_t b) {
  return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
}
__device__ __forceinline__ float u24(uint32_t a) { return (float)(a >> 8) * (1.0f / 16777216.0f); }

}  // namespace vrpx
