// Internal (non-ABI) helpers shared by the translation units of libunipose_b200.so.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/unipose_b200.h"

namespace up {

// Records a thread-local message and returns `code` (so callers can `return fail(...)`).
int fail(int code, const char* fmt, ...);
int check_cuda(cudaError_t e, const char* what);

// Per-device facts and one-time kernel attributes (cudaFuncSetAttribute is per device): indexed by cudaGetDevice(), so
// a process that drives several GPUs - or a model on cuda:1 - gets the right SM count / shared-memory opt-in.
struct DeviceInfo {
  int sm_count = 0;
  size_t max_smem = 0;
  bool conv_attr = false;    // conv_tcgen05_kernel<*> MaxDynamicSharedMemorySize set on this device
  bool wgrad_attr = false;   // conv_wgrad_tcgen05_kernel
  bool chain_attr = false;   // wasp_chain_kernel
  bool bneck_attr = false;   // bneck_chain_kernel
  bool tail_attr = false;    // bneck_tail_kernel
  int max_clusters[5] = {0, 0, 0, 0, 0};   // cached cudaOccupancyMaxActiveClusters: [2], [4] conv kernel by cluster
                                           // size; [0] wasp chain, [1] bottleneck chain (both clusters of 2)
};
// Info of the CURRENT device (validated to be sm_100 class); nullptr + error message on failure.
DeviceInfo* device_info();

#define UP_CHECK_ARG(cond, ...)                                \
  do {                                                         \
    if (!(cond)) return ::up::fail(UP_ERR_INVALID, __VA_ARGS__); \
  } while (0)

#define UP_CHECK_LAUNCH(what)                                   \
  do {                                                          \
    int _rc = ::up::check_cuda(cudaGetLastError(), what);       \
    if (_rc != 0) return _rc;                                   \
  } while (0)

// ---- programmatic dependent launch ------------------------------------------------------------
// A kernel launched through launch_pdl may be SCHEDULED while its predecessor in the stream still runs (once every
// CTA of the predecessor has called pdl_enter or exited), so that launch latency and prologue overlap the
// predecessor's tail.  It must call pdl_enter() before touching anything the predecessor wrote: the wait returns when
// the predecessor has completed and its writes are visible.  UP_PDL=0 switches the attribute off.
__device__ __forceinline__ void pdl_enter() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}

inline bool pdl_enabled() {
  static const bool on = []() {
    const char* e = getenv("UP_PDL");
    return !(e && e[0] == '0');
  }();
  return on;
}

template <class... KArgs, class... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---- 16-bit storage <-> fp32 (device) -------------------------------------------------------
// kFmt: 0 = fp16, 1 = bf16 (matches the tcgen05 instruction-descriptor encoding).
template <int kFmt>
__device__ __forceinline__ float cvt16_to_f32(uint16_t v) {
  if constexpr (kFmt == 1) {
    return __uint_as_float(static_cast<uint32_t>(v) << 16);
  } else {
    return __half2float(__ushort_as_half(v));
  }
}
template <int kFmt>
__device__ __forceinline__ uint16_t cvt_f32_to16(float f) {
  if constexpr (kFmt == 1) {
    return __bfloat16_as_ushort(__float2bfloat16_rn(f));
  } else {
    return __half_as_ushort(__float2half_rn(f));
  }
}
__device__ __forceinline__ float cvt16_to_f32_rt(uint16_t v, int fmt) {
  return fmt == 1 ? cvt16_to_f32<1>(v) : cvt16_to_f32<0>(v);
}
__device__ __forceinline__ uint16_t cvt_f32_to16_rt(float f, int fmt) {
  return fmt == 1 ? cvt_f32_to16<1>(f) : cvt_f32_to16<0>(f);
}
// Pack two floats into one 32-bit word of two 16-bit values (a in the low half).
__device__ __forceinline__ uint32_t pack2_rt(float a, float b, int fmt) {
  return static_cast<uint32_t>(cvt_f32_to16_rt(a, fmt)) | (static_cast<uint32_t>(cvt_f32_to16_rt(b, fmt)) << 16);
}
// bf16 hi/lo split of an fp32 value: x ~= hi + lo with ~16 mantissa bits.
__device__ __forceinline__ void split_bf16(float x, uint16_t& hi, uint16_t& lo) {
  hi = cvt_f32_to16<1>(x);
  lo = cvt_f32_to16<1>(x - cvt16_to_f32<1>(hi));
}

inline int fmt_of_dtype(int dtype) { return dtype == UP_FP16 ? 0 : 1; }

// Eight fp32 values -> one 16-byte store of 16-bit values; kMode 0 = fp16, 1 = bf16, 2 = bf16 hi at p and lo at
// p + plane (UP_SPLIT).  The stem's space-to-depth input writers (data_pipeline.cu, image_prep.cu) share it.
template <int kMode>
__device__ __forceinline__ void store8_16(uint16_t* p, long long plane, const float (&v)[8]) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    if constexpr (kMode == 2) {
      uint16_t h0, l0, h1, l1;
      split_bf16(v[2 * e], h0, l0);
      split_bf16(v[2 * e + 1], h1, l1);
      h[e] = h0 | (static_cast<uint32_t>(h1) << 16);
      l[e] = l0 | (static_cast<uint32_t>(l1) << 16);
    } else {
      h[e] = cvt_f32_to16<kMode>(v[2 * e]) | (static_cast<uint32_t>(cvt_f32_to16<kMode>(v[2 * e + 1])) << 16);
    }
  }
  *reinterpret_cast<uint4*>(p) = make_uint4(h[0], h[1], h[2], h[3]);
  if constexpr (kMode == 2) *reinterpret_cast<uint4*>(p + plane) = make_uint4(l[0], l[1], l[2], l[3]);
}

}  // namespace up
