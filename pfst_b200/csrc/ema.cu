// E1/E2 — multi-tensor EMA mean-teacher update (one launch for all tensors).
//
// Reference: PFGST._update_ema, rsiseg/models/uda/pfgst.py:116-127
//   ema_param.data[:] = alpha_teacher * ema_param.data + (1 - alpha_teacher) * param.data
// torch evaluates this as three separately rounded fp32 ops:
//   fl( fl(a32*e) + fl(b32*p) ),  a32=(float)alpha_teacher, b32=(float)(1.0-alpha_teacher)
// An FMA-contracted version differs by up to 2.2e-5 relative on near-cancelling
// elements (SURVEY.md Appendix A), so the kernel uses __fmul_rn/__fadd_rn.
//
// HBM-bound: 12 B per parameter (read ema, read param, write ema).
// Layout: a device-resident chunk table maps blockIdx.x -> (tensor, offset);
// each 256-thread block streams one chunk of `chunk_elems` floats with
// 4 x 128-bit loads per operand in flight per thread.
#include "common.cuh"

namespace pfst {

constexpr int kEmaThreads = 256;
constexpr int kEmaVecPerThread = 4;                                  // float4s per operand per thread
constexpr int kEmaTile = kEmaThreads * kEmaVecPerThread * 4;         // 4096 floats per block pass

template <int MODE>
__device__ __forceinline__ float ema_op(float e, float p, float a, float b) {
  if (MODE == 1) return p;
  return __fadd_rn(__fmul_rn(a, e), __fmul_rn(b, p));
}

template <int MODE>
__device__ __forceinline__ void ema_span(float* __restrict__ e, const float* __restrict__ p,
                                         int64_t n, float a, float b) {
  // e/p point at the start of this block's span of n floats.
  const int tid = threadIdx.x;
  const bool vec_ok = ((reinterpret_cast<uintptr_t>(e) | reinterpret_cast<uintptr_t>(p)) & 15u) == 0;
  if (vec_ok) {
    const int64_t n4 = n >> 2;
    for (int64_t base = 0; base < n4; base += kEmaThreads * kEmaVecPerThread) {
      float4 ve[kEmaVecPerThread], vp[kEmaVecPerThread];
#pragma unroll
      for (int j = 0; j < kEmaVecPerThread; ++j) {
        const int64_t v = base + j * kEmaThreads + tid;
        if (v < n4) {
          vp[j] = __ldcs(reinterpret_cast<const float4*>(p) + v);
          if (MODE == 0) ve[j] = __ldcs(reinterpret_cast<const float4*>(e) + v);
        }
      }
#pragma unroll
      for (int j = 0; j < kEmaVecPerThread; ++j) {
        const int64_t v = base + j * kEmaThreads + tid;
        if (v < n4) {
          float4 r;
          r.x = ema_op<MODE>(ve[j].x, vp[j].x, a, b);
          r.y = ema_op<MODE>(ve[j].y, vp[j].y, a, b);
          r.z = ema_op<MODE>(ve[j].z, vp[j].z, a, b);
          r.w = ema_op<MODE>(ve[j].w, vp[j].w, a, b);
          __stcs(reinterpret_cast<float4*>(e) + v, r);
        }
      }
    }
    for (int64_t i = (n4 << 2) + tid; i < n; i += kEmaThreads) e[i] = ema_op<MODE>(e[i], p[i], a, b);
  } else {
    for (int64_t i = tid; i < n; i += kEmaThreads) e[i] = ema_op<MODE>(e[i], p[i], a, b);
  }
}

template <int MODE>
__global__ void __launch_bounds__(kEmaThreads)
ema_multi_kernel(float* const* __restrict__ ema_ptrs, const float* const* __restrict__ param_ptrs,
                 const int64_t* __restrict__ numel, const int32_t* __restrict__ chunk_tensor,
                 const int64_t* __restrict__ chunk_begin, int64_t n_chunks, int32_t chunk_elems,
                 float a, float b, const float* __restrict__ coefs_dev) {
  if (coefs_dev) {          // coefficients resident on the device: the launch is CUDA-graph capturable
    a = coefs_dev[0];
    b = coefs_dev[1];
  }
  for (int64_t c = blockIdx.x; c < n_chunks; c += gridDim.x) {
    const int32_t t = chunk_tensor[c];
    const int64_t begin = chunk_begin[c];
    const int64_t total = numel[t];
    int64_t n = total - begin;
    if (n > chunk_elems) n = chunk_elems;
    if (n <= 0) continue;
    ema_span<MODE>(ema_ptrs[t] + begin, param_ptrs[t] + begin, n, a, b);
  }
}

template <int MODE>
__global__ void __launch_bounds__(kEmaThreads)
ema_flat_kernel(float* __restrict__ ema, const float* __restrict__ param, int64_t n, float a, float b) {
  const int64_t n_tiles = (n + kEmaTile - 1) / kEmaTile;
  for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    const int64_t begin = t * kEmaTile;
    int64_t len = n - begin;
    if (len > kEmaTile) len = kEmaTile;
    ema_span<MODE>(ema + begin, param + begin, len, a, b);
  }
}

}  // namespace pfst

extern "C" {

int pfst_ema_coeffs(int64_t iter, double alpha, float* a32_host, float* b32_host) {
  if (!a32_host || !b32_host || iter < 0) return PFST_ERR_INVALID_ARG;
  // pfgst.py:117  alpha_teacher = min(1 - 1 / (iter + 1), self.alpha)   (python doubles)
  double a = 1.0 - 1.0 / (double)(iter + 1);
  if (alpha < a) a = alpha;
  *a32_host = (float)a;
  *b32_host = (float)(1.0 - a);
  return PFST_OK;
}

int pfst_ema_update_multi(float* const* ema_ptrs, const float* const* param_ptrs,
                          const int64_t* numel, const int32_t* chunk_tensor,
                          const int64_t* chunk_begin, int64_t n_chunks, int32_t chunk_elems,
                          float a32, float b32, int32_t mode, int32_t blocks_per_sm, void* stream) {
  if (n_chunks == 0) return PFST_OK;
  if (!ema_ptrs || !param_ptrs || !numel || !chunk_tensor || !chunk_begin || n_chunks < 0)
    return PFST_ERR_INVALID_ARG;
  if (chunk_elems <= 0 || (chunk_elems % 1024) != 0) return PFST_ERR_INVALID_ARG;
  if (mode != 0 && mode != 1) return PFST_ERR_INVALID_ARG;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // One block per chunk; capped so a pathological table still launches (the
  // kernel grid-strides over chunks). 148 SMs x 8 resident blocks = 1184 per wave.
  // blocks_per_sm > 0: a persistent grid of that many blocks per SM, so that the update can share
  // the SMs with kernels of other streams (it is independent of the rest of the step).
  if (blocks_per_sm < 0) return PFST_ERR_INVALID_ARG;
  const int64_t max_grid = blocks_per_sm > 0 ? (int64_t)pfst::kNumSMs * blocks_per_sm : (int64_t)pfst::kNumSMs * 8 * 64;
  const unsigned grid = (unsigned)(n_chunks < max_grid ? n_chunks : max_grid);
  if (mode == 0)
    pfst::ema_multi_kernel<0><<<grid, pfst::kEmaThreads, 0, s>>>(
        ema_ptrs, param_ptrs, numel, chunk_tensor, chunk_begin, n_chunks, chunk_elems, a32, b32, nullptr);
  else
    pfst::ema_multi_kernel<1><<<grid, pfst::kEmaThreads, 0, s>>>(
        ema_ptrs, param_ptrs, numel, chunk_tensor, chunk_begin, n_chunks, chunk_elems, a32, b32, nullptr);
  PFST_CHECK_LAUNCH("pfst_ema_update_multi");
  return PFST_OK;
}

int pfst_ema_update_multi_dev(float* const* ema_ptrs, const float* const* param_ptrs,
                              const int64_t* numel, const int32_t* chunk_tensor,
                              const int64_t* chunk_begin, int64_t n_chunks, int32_t chunk_elems,
                              const float* coefs_dev, int32_t blocks_per_sm, void* stream) {
  if (n_chunks == 0) return PFST_OK;
  if (!ema_ptrs || !param_ptrs || !numel || !chunk_tensor || !chunk_begin || !coefs_dev || n_chunks < 0)
    return PFST_ERR_INVALID_ARG;
  if (chunk_elems <= 0 || (chunk_elems % 1024) != 0 || blocks_per_sm < 0) return PFST_ERR_INVALID_ARG;
  const int64_t max_grid = blocks_per_sm > 0 ? (int64_t)pfst::kNumSMs * blocks_per_sm : (int64_t)pfst::kNumSMs * 8 * 64;
  const unsigned grid = (unsigned)(n_chunks < max_grid ? n_chunks : max_grid);
  pfst::ema_multi_kernel<0><<<grid, pfst::kEmaThreads, 0, static_cast<cudaStream_t>(stream)>>>(
      ema_ptrs, param_ptrs, numel, chunk_tensor, chunk_begin, n_chunks, chunk_elems, 0.f, 0.f, coefs_dev);
  PFST_CHECK_LAUNCH("pfst_ema_update_multi_dev");
  return PFST_OK;
}

int pfst_ema_update_flat(float* ema, const float* param, int64_t n, float a32, float b32,
                         int32_t mode, void* stream) {
  if (n == 0) return PFST_OK;
  if (!ema || !param || n < 0) return PFST_ERR_INVALID_ARG;
  if (mode != 0 && mode != 1) return PFST_ERR_INVALID_ARG;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int64_t n_tiles = (n + pfst::kEmaTile - 1) / pfst::kEmaTile;
  const int64_t max_grid = (int64_t)pfst::kNumSMs * 8 * 64;
  const unsigned grid = (unsigned)(n_tiles < max_grid ? n_tiles : max_grid);
  if (mode == 0)
    pfst::ema_flat_kernel<0><<<grid, pfst::kEmaThreads, 0, s>>>(ema, param, n, a32, b32);
  else
    pfst::ema_flat_kernel<1><<<grid, pfst::kEmaThreads, 0, s>>>(ema, param, n, a32, b32);
  PFST_CHECK_LAUNCH("pfst_ema_update_flat");
  return PFST_OK;
}

}  // extern "C"
