// Shared device/host helpers for the PFST sm_100a kernels.
// Everything in this library is written for B200 (sm_100a) only: no other
// -gencode is ever passed and there is no CPU fallback.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pfst_sm100.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "pfst_b200 kernels are written for sm_100a only"
#endif

namespace pfst {

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs

// ---- error plumbing -------------------------------------------------------
// Launchers never throw, never allocate and never synchronise the device; a
// CUDA launch error is stored per host thread for pfst_last_cuda_error().
void set_last_cuda_error(cudaError_t e, const char* where);

#define PFST_CHECK_LAUNCH(where)                          \
  do {                                                    \
    cudaError_t _e = cudaGetLastError();                  \
    if (_e != cudaSuccess) {                              \
      ::pfst::set_last_cuda_error(_e, where);             \
      return PFST_ERR_CUDA;                               \
    }                                                     \
  } while (0)

#define PFST_CUDA_TRY(expr, where)                        \
  do {                                                    \
    cudaError_t _e = (expr);                              \
    if (_e != cudaSuccess) {                              \
      ::pfst::set_last_cuda_error(_e, where);             \
      return PFST_ERR_CUDA;                               \
    }                                                     \
  } while (0)

__host__ __device__ static inline bool aligned16(const void* p) {
  return (reinterpret_cast<uintptr_t>(p) & 15u) == 0;
}
__host__ __device__ static inline bool aligned4(const void* p) {
  return (reinterpret_cast<uintptr_t>(p) & 3u) == 0;
}

// Label maps are int64 (the reference dtype) or uint8 (the dtype datasets store); the kernels that read
// or write them are templated on the element type, and the entry points take a PFST_DT_* tag.
template <class L> struct LabelDt;
template <> struct LabelDt<int64_t> { static constexpr int value = PFST_DT_I64; };
template <> struct LabelDt<uint8_t> { static constexpr int value = PFST_DT_U8; };
// Bytes of 4 consecutive labels as one vector access (int64: two 16-byte halves, uint8: one 32-bit
// word): the alignment the vectorised paths need.
template <class L>
__host__ __device__ static inline bool aligned_lbl4(const L* p) {
  return sizeof(L) == 8 ? aligned16(p) : aligned4(p);
}

// ---- streaming 128-bit global accesses ------------------------------------
// Inputs that are read exactly once bypass L1 (ld.global.nc.L1::no_allocate);
// outputs that are not re-read by the same kernel use plain vector stores.
__device__ __forceinline__ float4 ldg_stream_f4(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ int4 ldg_stream_i4(const void* p) {
  int4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ longlong2 ldg_stream_l2(const int64_t* p) {
  longlong2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.s64 {%0,%1}, [%2];"
               : "=l"(r.x), "=l"(r.y)
               : "l"(p));
  return r;
}
__device__ __forceinline__ uint32_t ldg_stream_u32(const void* p) {
  uint32_t r;
  asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ void stg_f4(float* p, float4 v) {
  *reinterpret_cast<float4*>(p) = v;
}
__device__ __forceinline__ void stg_l2(int64_t* p, longlong2 v) {
  *reinterpret_cast<longlong2*>(p) = v;
}

// ---- warp / block reductions ----------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ unsigned warp_sum(unsigned v) {
  return __reduce_add_sync(0xffffffffu, v);
}

// ---- nearest-resampled label lookup (F.interpolate(mode='nearest'), pfgst_loss.py:62) ----
__device__ __forceinline__ int pr_nearest(int dst, float scale, int in) {
  const int s = (int)floorf((float)dst * scale);
  return s < in - 1 ? s : in - 1;
}

// label of feature pixel p (0..h*w) of image b, 255 if outside [0,C) or masked out
template <class L>
__device__ __forceinline__ uint8_t pr_label(const L* __restrict__ labels, const float* __restrict__ conf,
                                            float conf_thr, int b, int p, int w, int lab_h, int lab_w,
                                            float sh, float sw, int C) {
  const int y = p / w, x = p - y * w;
  const int64_t o = ((int64_t)b * lab_h + pr_nearest(y, sh, lab_h)) * lab_w + pr_nearest(x, sw, lab_w);
  const int64_t l = labels[o];
  bool ok = l >= 0 && l < C;
  if (conf && ok) ok = conf[o] >= conf_thr;
  return ok ? (uint8_t)l : (uint8_t)255;
}

}  // namespace pfst
