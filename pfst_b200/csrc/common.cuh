// Shared device/host helpers for the PFST sm_100a kernels.
// Everything in this library is written for B200 (sm_100a) only: no other
// -gencode is ever passed and there is no CPU fallback.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
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

// Teacher outputs (the pseudo-label logits and the EMA features) are fp32, fp16 or bf16; the kernels that
// read them are templated on the element type and convert every value to fp32 once, on load (exact), so
// the arithmetic after the load is the fp32 code. The entry points take a PFST_DT_F* tag.
template <class T> struct FloatDt;
template <> struct FloatDt<float> { static constexpr int value = PFST_DT_F32; };
template <> struct FloatDt<__half> { static constexpr int value = PFST_DT_F16; };
template <> struct FloatDt<__nv_bfloat16> { static constexpr int value = PFST_DT_BF16; };

__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
template <class T> __device__ __forceinline__ float ldgf(const T* p) { return to_f32(__ldg(p)); }
// the low / high 16-bit element of a 32-bit word as fp32
template <class T> __device__ __forceinline__ float lo_f32(uint32_t w);
template <class T> __device__ __forceinline__ float hi_f32(uint32_t w);
template <> __device__ __forceinline__ float lo_f32<__nv_bfloat16>(uint32_t w) { return __uint_as_float(w << 16); }
template <> __device__ __forceinline__ float hi_f32<__nv_bfloat16>(uint32_t w) { return __uint_as_float(w & 0xffff0000u); }
template <> __device__ __forceinline__ float lo_f32<__half>(uint32_t w) {
  return __half2float(__ushort_as_half((unsigned short)(w & 0xffffu)));
}
template <> __device__ __forceinline__ float hi_f32<__half>(uint32_t w) {
  return __half2float(__ushort_as_half((unsigned short)(w >> 16)));
}
// four consecutive 16-bit elements (one 64-bit word) as fp32
template <class T> __device__ __forceinline__ float4 unpack4(uint2 v) {
  return make_float4(lo_f32<T>(v.x), hi_f32<T>(v.x), lo_f32<T>(v.y), hi_f32<T>(v.y));
}

// ---- dtype-tag dispatch of the entry points (host) -------------------------
// f(L{}) with L = int64_t or uint8_t for a PFST_DT_I64 / PFST_DT_U8 label tag; f(T{}) with T = float,
// __half or __nv_bfloat16 for a PFST_DT_F32 / F16 / BF16 float tag. Any other tag is
// PFST_ERR_UNSUPPORTED, returned before f runs (so before any argument check inside f).
template <class F>
static inline int with_label_dt(int32_t tag, F&& f) {
  if (tag == PFST_DT_I64) return f(int64_t{});
  if (tag == PFST_DT_U8) return f(uint8_t{});
  return PFST_ERR_UNSUPPORTED;
}
template <class F>
static inline int with_float_dt(int32_t tag, F&& f) {
  if (tag == PFST_DT_F32) return f(float{});
  if (tag == PFST_DT_F16) return f(__half{});
  if (tag == PFST_DT_BF16) return f(__nv_bfloat16{});
  return PFST_ERR_UNSUPPORTED;
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
// four consecutive elements as fp32: one 128-bit (fp32) or 64-bit (fp16 / bf16) streaming load
__device__ __forceinline__ float4 ldg_stream_4(const float* p) { return ldg_stream_f4(p); }
// (not volatile: a read-only load the compiler may schedule; with `volatile` ptxas spilled the C = 4 pseudo-label
// instantiation)
template <class T>
__device__ __forceinline__ float4 ldg_stream_4(const T* p) {
  uint2 r;
  asm("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
  return unpack4<T>(r);
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
