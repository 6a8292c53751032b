// S1/S2 — fused softmax / max-confidence / argmax / threshold / count.
//
// Reference: rsiseg/models/uda/pfgst.py:259-266
//   ema_softmax = torch.softmax(ema_logits.detach(), dim=1)
//   pseudo_prob, pseudo_label = torch.max(ema_softmax, dim=1)
//   ps_large_p = pseudo_prob.ge(self.pseudo_threshold).long() == 1
//   pseudo_weight = torch.sum(ps_large_p).item() / ps_size          ('all')
// The reference materialises the (B,C,H,W) softmax and runs 7 kernels and two
// host syncs; this is ONE pass over the NCHW logits: (4C + 12) bytes per pixel.
//
// Bit-parity rules (SURVEY.md §7 "hard parts"):
//   * softmax as torch computes it along a non-innermost dim: m = max_c x_c,
//     s = sum_c expf(x_c - m) accumulated in class order, out_c = expf(x_c-m)/s
//     (IEEE division). The winning probability is therefore 1.0f / s.
//   * torch.max returns the FIRST index of the maximum of the softmax OUTPUT.
//     That is the first index of the maximum logit unless an earlier class's
//     quotient rounds to the same float; that rare case is re-checked exactly.
//   * any NaN in the pixel's softmax makes every output NaN: label 0, conf NaN,
//     never confident.
//   * ge(thr) compares in fp32 against (float)thr.
#include <math.h>

#include "common.cuh"
#include "exp_exact.cuh"

namespace pfst {

constexpr int kPlThreads = 256;

struct PlOut {
  int label;
  float conf;
  bool confident;
};

// Slow path of the arg-max (kept out of line: it runs for a handful of pixels per
// image and would otherwise bloat the hot loop past the instruction cache). It
// re-reads the pixel's logits from memory so that the hot loop's register arrays
// never have their address taken.
__device__ __noinline__ int pl_tie_label(const float* __restrict__ px, int64_t HW, float m, float s,
                                         int am, float conf) {
  int label = am;
  for (int c = am - 1; c >= 0; --c) {
    const float d = px[(int64_t)c * HW] - m;
    if (d > -3.0e-4f && exp_exact(d) / s == conf) label = c;
  }
  return label;
}

// x[0..C) are the pixel's logits, held in registers (CMAX is a compile-time
// bound so the array never spills to local memory; EXACT means C == CMAX).
template <int CMAX, int MODE, bool EXACT>
__device__ __forceinline__ PlOut pl_pixel(const float (&x)[CMAX], int C, float thr,
                                          const float* __restrict__ thr_pc,
                                          const float* __restrict__ px, int64_t HW) {
  float m = x[0];
  int am = 0;
#pragma unroll
  for (int c = 1; c < CMAX; ++c)
    if ((EXACT || c < C) && x[c] > m) { m = x[c]; am = c; }
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < CMAX; ++c)
    if (EXACT || c < C) {
      const ExpParts e = exp_split(x[c] - m);
      s = __fmaf_rn(e.scale, e.mant, s);   // == `s += expf(x - m)` as nvcc contracts it
    }
  PlOut o;
  o.conf = 1.0f / s;  // IEEE-rounded: no -use_fast_math anywhere in this build
  o.label = am;
  if (s != s) {
    o.label = 0;  // all softmax outputs are NaN; torch.max returns the first
  } else if (s >= 1.9997f && am > 0) {
    // An EARLIER class whose quotient rounds to the same float wins torch.max's tie.
    // That needs a logit within ~1e-7 of the max; s >= 1.9997 is a cheap necessary
    // condition (exp > 0.9997), the compare loop the exact one, the call is rare.
    bool near = false;
#pragma unroll
    for (int c = 0; c < CMAX - 1; ++c)
      if ((EXACT || c < C) && c < am && (x[c] - m) > -3.0e-4f) near = true;
    if (near) o.label = pl_tie_label(px, HW, m, s, am, o.conf);
  }
  const float t = thr_pc ? thr_pc[o.label] : thr;
  if (MODE == 0) {
    o.confident = o.conf >= t;
  } else {
    // offline class-wise rule, loading.py:479-483: ent = -sum p*log(p+1e-8) < thr[pred]
    float ent = 0.f;
#pragma unroll
    for (int c = 0; c < CMAX; ++c)
      if (EXACT || c < C) {
        const float p = exp_exact(x[c] - m) / s;
        ent -= p * logf(p + 1e-8f);
      }
    o.confident = ent < t;
  }
  return o;
}

__device__ __forceinline__ void pl_block_count(unsigned local, unsigned long long* count) {
  __shared__ unsigned warp_counts[kPlThreads / 32];
  const unsigned w = warp_sum(local);
  if ((threadIdx.x & 31) == 0) warp_counts[threadIdx.x >> 5] = w;
  __syncthreads();
  if (threadIdx.x < 32) {
    unsigned v = threadIdx.x < kPlThreads / 32 ? warp_counts[threadIdx.x] : 0u;
    v = warp_sum(v);
    if (threadIdx.x == 0 && v) atomicAdd(count, (unsigned long long)v);
  }
}

// VEC consecutive pixels of one image plane per thread (VEC=4: 128-bit loads).
// Persistent grid (one resident wave) with a two-stage software pipeline: the
// loads of a thread's NEXT item are issued before the ~100 instructions/pixel of
// exp/divide work on the current one, so HBM never idles behind the math.
template <int VEC, int CMAX, bool EXACT>
__device__ __forceinline__ void pl_load(float (&x)[VEC][CMAX], const float* __restrict__ src, int C,
                                        int64_t HW) {
#pragma unroll
  for (int c = 0; c < CMAX; ++c)
    if (EXACT || c < C) {
      if (VEC == 4) {
        const float4 v = ldg_stream_f4(src);
        x[0][c] = v.x; x[1 % VEC][c] = v.y; x[2 % VEC][c] = v.z; x[3 % VEC][c] = v.w;
      } else {
        x[0][c] = __ldg(src);
      }
      src += HW;
    }
}

// L = uint8: one 32-bit store per 4 labels (the host guarantees C <= 255 and reject_label <= 255).
template <int VEC, int CMAX, int MODE, bool EXACT, class L>
__global__ void __launch_bounds__(kPlThreads)
pseudo_label_kernel(const float* __restrict__ logits, int64_t B, int C, int64_t HW, float thr,
                    const float* __restrict__ thr_per_class, int64_t reject_label,
                    L* __restrict__ label, float* __restrict__ conf,
                    float* __restrict__ weight_part, unsigned long long* __restrict__ count) {
  __shared__ float thr_s[CMAX];
  const float* thr_pc = nullptr;
  if (thr_per_class) {
    for (int c = threadIdx.x; c < C; c += kPlThreads) thr_s[c] = thr_per_class[c];
    __syncthreads();
    thr_pc = thr_s;
  }
  // item = VEC pixels; (b, i) = (image, item inside the image plane) is advanced
  // incrementally so the loop has no integer division.
  const unsigned per_img = (unsigned)(HW / VEC);
  const unsigned stride = gridDim.x * kPlThreads;
  const int64_t CHW = (int64_t)C * HW;
  unsigned local = 0;
  unsigned i = blockIdx.x * kPlThreads + threadIdx.x;
  int64_t b = i / per_img;
  i -= (unsigned)b * per_img;
  float cur[VEC][CMAX], nxt[VEC][CMAX];
  if (b < B) pl_load<VEC, CMAX, EXACT>(cur, logits + b * CHW + (int64_t)i * VEC, C, HW);
  while (b < B) {
    unsigned in = i + stride;
    int64_t bn = b;
    while (in >= per_img) { in -= per_img; ++bn; }
    if (bn < B) pl_load<VEC, CMAX, EXACT>(nxt, logits + bn * CHW + (int64_t)in * VEC, C, HW);

    PlOut o[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      o[k] = pl_pixel<CMAX, MODE, EXACT>(cur[k], C, thr, thr_pc,
                                           logits + b * CHW + (int64_t)i * VEC + k, HW);
      local += o[k].confident ? 1u : 0u;
    }
    const int64_t out = b * HW + (int64_t)i * VEC;
    int64_t lab[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k)
      lab[k] = (reject_label >= 0 && !o[k].confident) ? reject_label : (int64_t)o[k].label;
    if (VEC == 4) {
      if constexpr (sizeof(L) == 1) {
        *reinterpret_cast<uint32_t*>(label + out) =
            ((uint32_t)lab[0] & 255u) | (((uint32_t)lab[1 % VEC] & 255u) << 8) |
            (((uint32_t)lab[2 % VEC] & 255u) << 16) | ((uint32_t)lab[3 % VEC] << 24);
      } else {
        stg_l2(label + out, make_longlong2(lab[0], lab[1 % VEC]));
        stg_l2(label + out + 2, make_longlong2(lab[2 % VEC], lab[3 % VEC]));
      }
      stg_f4(conf + out, make_float4(o[0].conf, o[1 % VEC].conf, o[2 % VEC].conf, o[3 % VEC].conf));
      if (weight_part)
        stg_f4(weight_part + out,
               make_float4(o[0].confident ? 1.f : 0.f, o[1 % VEC].confident ? 1.f : 0.f,
                           o[2 % VEC].confident ? 1.f : 0.f, o[3 % VEC].confident ? 1.f : 0.f));
    } else {
      label[out] = (L)lab[0];
      conf[out] = o[0].conf;
      if (weight_part) weight_part[out] = o[0].confident ? 1.f : 0.f;
    }
#pragma unroll
    for (int k = 0; k < VEC; ++k)
#pragma unroll
      for (int c = 0; c < CMAX; ++c) cur[k][c] = nxt[k][c];
    b = bn;
    i = in;
  }
  pl_block_count(local, count);
}

// Any C: one pixel per thread, two passes over the pixel's logits (the second
// pass is served from L1/L2).
template <int MODE, class L>
__global__ void __launch_bounds__(kPlThreads)
pseudo_label_generic_kernel(const float* __restrict__ logits, int64_t B, int C, int64_t HW,
                            float thr, const float* __restrict__ thr_per_class,
                            int64_t reject_label, L* __restrict__ label,
                            float* __restrict__ conf, float* __restrict__ weight_part,
                            unsigned long long* __restrict__ count) {
  const int64_t total = B * HW;
  unsigned local = 0;
  for (int64_t i = (int64_t)blockIdx.x * kPlThreads + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * kPlThreads) {
    const int64_t b = i / HW;
    const int64_t p = i - b * HW;
    const float* src = logits + (b * C) * HW + p;
    float m = src[0];
    int am = 0;
    for (int c = 1; c < C; ++c) {
      const float v = src[(int64_t)c * HW];
      if (v > m) { m = v; am = c; }
    }
    float s = 0.f;
    for (int c = 0; c < C; ++c) {
      const ExpParts e = exp_split(src[(int64_t)c * HW] - m);
      s = __fmaf_rn(e.scale, e.mant, s);
    }
    const float cf = 1.0f / s;
    int lab = am;
    if (s != s) {
      lab = 0;
    } else {
      for (int c = am - 1; c >= 0; --c) {
        const float d = src[(int64_t)c * HW] - m;
        if (d > -3.0e-4f && exp_exact(d) / s == cf) lab = c;
      }
    }
    const float t = thr_per_class ? __ldg(thr_per_class + lab) : thr;
    bool confident;
    if (MODE == 0) {
      confident = cf >= t;
    } else {
      float ent = 0.f;
      for (int c = 0; c < C; ++c) {
        const float pc = exp_exact(src[(int64_t)c * HW] - m) / s;
        ent -= pc * logf(pc + 1e-8f);
      }
      confident = ent < t;
    }
    local += confident ? 1u : 0u;
    label[i] = (L)((reject_label >= 0 && !confident) ? reject_label : (int64_t)lab);
    conf[i] = cf;
    if (weight_part) weight_part[i] = confident ? 1.f : 0.f;
  }
  pl_block_count(local, count);
}

// thre_type='all': broadcast (float)(count/ps_size), zero the ignored rows.
__global__ void __launch_bounds__(256)
pseudo_weight_fill_kernel(float* __restrict__ weight, int64_t B, int64_t H, int64_t W,
                          const unsigned long long* __restrict__ count, int64_t ps_size,
                          int ignore_top, int ignore_bottom) {
  const float ratio = (float)((double)(*count) / (double)ps_size);
  const int64_t total = B * H * W;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t y = (i / W) % H;
    const bool zero = (y < ignore_top) || (y >= H - ignore_bottom);
    weight[i] = zero ? 0.f : ratio;
  }
}

// self-test: counts inputs for which the hand-split exp differs from expf
__global__ void exp_selftest_kernel(const float* __restrict__ x, int64_t n,
                                    unsigned long long* __restrict__ mismatches) {
  unsigned bad = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    const float a = exp_exact(x[i]), b = expf(x[i]);
    bad += (__float_as_uint(a) != __float_as_uint(b)) ? 1u : 0u;
  }
  bad = warp_sum(bad);
  if ((threadIdx.x & 31) == 0 && bad) atomicAdd(mismatches, (unsigned long long)bad);
}

template <int MODE, class L>
static int launch_pl(const float* logits, int64_t B, int C, int64_t HW, float thr,
                     const float* thr_pc, int64_t reject, L* label, float* conf,
                     float* wpart, unsigned long long* count, cudaStream_t s) {
  const bool vec4 = (HW % 4 == 0) && aligned16(logits) && aligned_lbl4(label) && aligned16(conf) &&
                    (!wpart || aligned16(wpart));
  if (HW > 0x7fffffffll || B * (HW / 4 + 1) > 0x7fffffffll * 2) return PFST_ERR_UNSUPPORTED;
  auto grid_flat = [](int64_t items) {
    int64_t g = (items + kPlThreads - 1) / kPlThreads;
    const int64_t cap = (int64_t)kNumSMs * 8 * 32;
    return (unsigned)(g < cap ? (g > 0 ? g : 1) : cap);
  };
#define PFST_PL_LAUNCH(VEC_, CMAX_, EXACT_)                                                      \
  do {                                                                                           \
    auto k = pseudo_label_kernel<VEC_, CMAX_, MODE, EXACT_, L>;                                     \
    int occ = 0;                                                                                 \
    PFST_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k, kPlThreads, 0),         \
                  "pfst_pseudo_label/occupancy");                                                \
    if (occ < 1) return PFST_ERR_UNSUPPORTED;                                                    \
    const int64_t items = B * (HW / VEC_);                                                       \
    int64_t g = (items + kPlThreads - 1) / kPlThreads;                                           \
    if (g > (int64_t)kNumSMs * occ) g = (int64_t)kNumSMs * occ;                                  \
    k<<<(unsigned)(g > 0 ? g : 1), kPlThreads, 0, s>>>(logits, B, C, HW, thr, thr_pc, reject,    \
                                                       label, conf, wpart, count);              \
  } while (0)
  if (C <= 8 && vec4 && MODE == 0) {
    // exact-C instantiations of the hot configuration (no per-class predicates); the uint8 build
    // does not instantiate the MODE 1 copies this branch never reaches
    if constexpr (MODE == 0 || sizeof(L) == 8) {
      switch (C) {
        case 2: PFST_PL_LAUNCH(4, 2, true); break;
        case 3: PFST_PL_LAUNCH(4, 3, true); break;
        case 4: PFST_PL_LAUNCH(4, 4, true); break;
        case 5: PFST_PL_LAUNCH(4, 5, true); break;
        case 6: PFST_PL_LAUNCH(4, 6, true); break;
        case 7: PFST_PL_LAUNCH(4, 7, true); break;
        case 8: PFST_PL_LAUNCH(4, 8, true); break;
        default: PFST_PL_LAUNCH(4, 8, false); break;
      }
    }
  } else if (C <= 8 && vec4) {
    PFST_PL_LAUNCH(4, 8, false);
  } else if (C <= 8) {
    PFST_PL_LAUNCH(1, 8, false);
  } else if (C == 33 && MODE == 0) {
    // round-2 candidate (SeasonNet, cfg4): exact-C instantiation — no per-class predicates, 66
    // instead of 80 pipeline registers; unverified on a GPU
    PFST_PL_LAUNCH(1, 33, true);
  } else if (C <= 40) {
    PFST_PL_LAUNCH(1, 40, false);
  } else {
    pseudo_label_generic_kernel<MODE, L><<<grid_flat(B * HW), kPlThreads, 0, s>>>(
        logits, B, C, HW, thr, thr_pc, reject, label, conf, wpart, count);
  }
#undef PFST_PL_LAUNCH
  PFST_CHECK_LAUNCH("pfst_pseudo_label");
  return PFST_OK;
}

}  // namespace pfst

extern "C" {

}  // extern "C"

namespace pfst {

template <class L>
static int pseudo_label(const float* logits, int64_t B, int32_t C, int64_t HW, float thr,
                        const float* thr_per_class, int32_t mode, int64_t reject_label, L* label,
                        float* conf, float* weight_part, unsigned long long* count, void* stream) {
  if (!logits || !label || !conf || !count) return PFST_ERR_INVALID_ARG;
  if (B < 0 || HW < 0 || C < 1) return PFST_ERR_INVALID_ARG;
  if (mode != 0 && mode != 1) return PFST_ERR_INVALID_ARG;
  if (sizeof(L) == 1 && (C > 255 || reject_label > 255)) return PFST_ERR_UNSUPPORTED;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PFST_CUDA_TRY(cudaMemsetAsync(count, 0, sizeof(unsigned long long), s), "pfst_pseudo_label/memset");
  if (B == 0 || HW == 0) return PFST_OK;
  if (mode == 0)
    return launch_pl<0>(logits, B, C, HW, thr, thr_per_class, reject_label, label, conf,
                        weight_part, count, s);
  return launch_pl<1>(logits, B, C, HW, thr, thr_per_class, reject_label, label, conf,
                      weight_part, count, s);
}

}  // namespace pfst

extern "C" {

int pfst_pseudo_label(const float* logits, int64_t B, int32_t C, int64_t HW, float thr,
                      const float* thr_per_class, int32_t mode, int64_t reject_label,
                      int64_t* label, float* conf, float* weight_part,
                      unsigned long long* count, void* stream) {
  return pfst::pseudo_label(logits, B, C, HW, thr, thr_per_class, mode, reject_label, label, conf,
                            weight_part, count, stream);
}

int pfst_pseudo_label_lbl(const float* logits, int64_t B, int32_t C, int64_t HW, float thr,
                          const float* thr_per_class, int32_t mode, int64_t reject_label,
                          void* label, int32_t label_dtype, float* conf, float* weight_part,
                          unsigned long long* count, void* stream) {
  if (label_dtype == PFST_DT_I64)
    return pfst::pseudo_label(logits, B, C, HW, thr, thr_per_class, mode, reject_label,
                              static_cast<int64_t*>(label), conf, weight_part, count, stream);
  if (label_dtype == PFST_DT_U8)
    return pfst::pseudo_label(logits, B, C, HW, thr, thr_per_class, mode, reject_label,
                              static_cast<uint8_t*>(label), conf, weight_part, count, stream);
  return PFST_ERR_UNSUPPORTED;
}

int pfst_selftest_exp(const float* x, int64_t n, unsigned long long* mismatches, void* stream) {
  if (!x || !mismatches || n < 0) return PFST_ERR_INVALID_ARG;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PFST_CUDA_TRY(cudaMemsetAsync(mismatches, 0, sizeof(unsigned long long), s), "pfst_selftest_exp/memset");
  if (n == 0) return PFST_OK;
  pfst::exp_selftest_kernel<<<pfst::kNumSMs * 8, 256, 0, s>>>(x, n, mismatches);
  PFST_CHECK_LAUNCH("pfst_selftest_exp");
  return PFST_OK;
}

int pfst_pseudo_weight_fill(float* weight, int64_t B, int64_t H, int64_t W,
                            const unsigned long long* count, int64_t ps_size,
                            int32_t ignore_top, int32_t ignore_bottom, void* stream) {
  if (!weight || !count || B < 0 || H < 0 || W < 0 || ps_size <= 0) return PFST_ERR_INVALID_ARG;
  if (ignore_top < 0 || ignore_bottom < 0) return PFST_ERR_INVALID_ARG;
  const int64_t total = B * H * W;
  if (total == 0) return PFST_OK;
  int64_t g = (total + 255) / 256;
  const int64_t cap = (int64_t)pfst::kNumSMs * 8 * 8;
  if (g > cap) g = cap;
  pfst::pseudo_weight_fill_kernel<<<(unsigned)g, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      weight, B, H, W, count, ps_size, ignore_top, ignore_bottom);
  PFST_CHECK_LAUNCH("pfst_pseudo_weight_fill");
  return PFST_OK;
}

}  // extern "C"
