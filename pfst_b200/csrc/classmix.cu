// M1/M2 — ClassMix: batch class presence, class masks and the fused mix of
// image / label / pixel weight.
//
// Reference: rsiseg/models/utils/dacs_transforms.py
//   get_class_masks :110-119   classes = torch.unique(labels)  (WHOLE batch, :113)
//                              np.random.choice(n, int((n + n%2)/2), replace=False)
//   generate_class_mask :122-126   label.eq(classes).sum(0)
//   one_mix :129-144               out = mask*a + (1-mask)*b
// and the per-image Python loop in rsiseg/models/uda/pfgst.py:287-300 that calls
// strong_transform twice per image (image+label, then weights).
//
// The host RNG draw stays on the host (it is part of the reference's observable
// behaviour); the device side is two HBM-bound passes:
//   presence: 8 B/px read of gt, 36-byte result (one tiny D2H);
//   mix:      read gt 8 + img 4c + trg 4c + pl 8 (+ w 4) ; write img 4c + lbl 8
//             + w 4 + mask 8 bytes per pixel  (84 B/px at c=3 with weight_in).
#include "common.cuh"

namespace pfst {

constexpr int kMixThreads = 256;

template <class L>
__global__ void __launch_bounds__(kMixThreads)
class_presence_kernel(const L* __restrict__ gt, int64_t n, uint32_t* __restrict__ presence) {
  __shared__ uint8_t seen[256];
  __shared__ int bad;
  const int tid = threadIdx.x;
  seen[tid] = 0;  // kMixThreads == 256
  if (tid == 0) bad = 0;
  __syncthreads();
  const bool vec = aligned16(gt);
  if constexpr (sizeof(L) == 1) {
    // uint8: 16 labels per 16-byte load, every value is in range (word 8 stays 0)
    const int64_t n16 = vec ? (n >> 4) : 0;
    const int64_t stride = (int64_t)gridDim.x * kMixThreads;
    for (int64_t i = (int64_t)blockIdx.x * kMixThreads + tid; i < n16; i += 4 * stride) {
      int4 v[4];
      bool ok[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        ok[u] = i + u * stride < n16;
        v[u] = ok[u] ? ldg_stream_i4(gt + 16 * (i + u * stride)) : make_int4(0, 0, 0, 0);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (!ok[u]) continue;
        const uint32_t words[4] = {(uint32_t)v[u].x, (uint32_t)v[u].y, (uint32_t)v[u].z, (uint32_t)v[u].w};
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
          for (int k = 0; k < 4; ++k) seen[(words[j] >> (8 * k)) & 255u] = 1;
      }
    }
    for (int64_t i = 16 * n16 + (int64_t)blockIdx.x * kMixThreads + tid; i < n;
         i += (int64_t)gridDim.x * kMixThreads)
      seen[gt[i]] = 1;
    __syncthreads();
    const unsigned word = __ballot_sync(0xffffffffu, seen[tid] != 0);
    if ((tid & 31) == 0 && word) atomicOr(&presence[tid >> 5], word);
    return;
  }
  const int64_t n2 = vec ? (n >> 1) : 0;
  // four 16-byte loads in flight per thread (one per pass kept the kernel at a quarter of the copy rate)
  const int64_t stride = (int64_t)gridDim.x * kMixThreads;
  for (int64_t i = (int64_t)blockIdx.x * kMixThreads + tid; i < n2; i += 4 * stride) {
    longlong2 v[4];
    bool ok[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      ok[u] = i + u * stride < n2;
      v[u] = ok[u] ? ldg_stream_l2(reinterpret_cast<const int64_t*>(gt) + 2 * (i + u * stride))
                   : make_longlong2(0, 0);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      if (!ok[u]) continue;
      if ((unsigned long long)v[u].x < 256ull) seen[v[u].x] = 1; else bad = 1;
      if ((unsigned long long)v[u].y < 256ull) seen[v[u].y] = 1; else bad = 1;
    }
  }
  for (int64_t i = 2 * n2 + (int64_t)blockIdx.x * kMixThreads + tid; i < n;
       i += (int64_t)gridDim.x * kMixThreads) {
    const int64_t v = gt[i];
    if ((unsigned long long)v < 256ull) seen[v] = 1; else bad = 1;
  }
  __syncthreads();
  const unsigned word = __ballot_sync(0xffffffffu, seen[tid] != 0);
  if ((tid & 31) == 0 && word) atomicOr(&presence[tid >> 5], word);
  if (tid == 0 && bad) atomicOr(&presence[8], 1u);
}

__device__ __forceinline__ float mix_f(float m, float a, float b) {
  // one_mix: stackedMask0 * data[0] + (1 - stackedMask0) * data[1], evaluated in
  // fp32 exactly as torch does (two multiplies, one add) so that signed zeros and
  // non-finite values propagate identically.
  return __fadd_rn(__fmul_rn(m, a), __fmul_rn(1.0f - m, b));
}

// L = uint8: the 4-pixel unit reads gt and the pseudo label as one 32-bit word each and writes
// the mixed label and the mask as one 32-bit word each.
template <int VEC, class L>
__global__ void __launch_bounds__(kMixThreads)
class_mix_kernel(const L* __restrict__ gt, const uint32_t* __restrict__ chosen,
                 const float* __restrict__ img, const float* __restrict__ trg,
                 const L* __restrict__ pl, const float* weight_in,
                 const unsigned long long* __restrict__ count, int64_t ps_size, int ignore_top,
                 int ignore_bottom, int64_t B, int channels, int64_t H, int64_t W,
                 float* __restrict__ mixed_img, L* __restrict__ mixed_lbl,
                 float* mixed_weight, L* __restrict__ mix_mask) {
  constexpr bool kU8 = sizeof(L) == 1;
  // grid = (tiles of the image plane, images): 32-bit pixel index, no 64-bit divisions
  const int64_t HW = H * W;
  const unsigned per_img = (unsigned)(HW / VEC);
  float ratio = 0.f;
  if (mixed_weight && !weight_in) ratio = (float)((double)(*count) / (double)ps_size);
  const unsigned i = blockIdx.x * kMixThreads + threadIdx.x;
  for (int64_t b = blockIdx.y; b < B && i < per_img; b += gridDim.y) {
    const int64_t p = (int64_t)i * VEC;
    const int64_t o = b * HW + p;
    int64_t g[VEC];
    if (VEC == 4 && kU8) {
      const uint32_t g4 = ldg_stream_u32(gt + o);
#pragma unroll
      for (int k = 0; k < VEC; ++k) g[k] = (g4 >> (8 * k)) & 255u;
    } else if (VEC == 4) {
      const longlong2 g0 = ldg_stream_l2(reinterpret_cast<const int64_t*>(gt) + o),
                      g1 = ldg_stream_l2(reinterpret_cast<const int64_t*>(gt) + o + 2);
      g[0] = g0.x; g[1 % VEC] = g0.y; g[2 % VEC] = g1.x; g[3 % VEC] = g1.y;
    } else {
      g[0] = gt[o];
    }
    const uint32_t* ch = chosen + b * 8;
    float m[VEC];
    bool mb[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      const unsigned long long v = (unsigned long long)g[k];
      mb[k] = v < 256ull && ((__ldg(ch + (v >> 5)) >> (v & 31)) & 1u);
      m[k] = mb[k] ? 1.f : 0.f;
    }
    if (mix_mask) {
      if (VEC == 4 && kU8) {
        *reinterpret_cast<uint32_t*>(mix_mask + o) = (uint32_t)mb[0] | ((uint32_t)mb[1 % VEC] << 8) |
                                                     ((uint32_t)mb[2 % VEC] << 16) | ((uint32_t)mb[3 % VEC] << 24);
      } else if (VEC == 4) {
        int64_t* mm = reinterpret_cast<int64_t*>(mix_mask);
        stg_l2(mm + o, make_longlong2(mb[0], mb[1 % VEC]));
        stg_l2(mm + o + 2, make_longlong2(mb[2 % VEC], mb[3 % VEC]));
      } else {
        mix_mask[o] = mb[0];
      }
    }
    if (mixed_img) {
      for (int c = 0; c < channels; ++c) {
        const int64_t oc = (b * channels + c) * HW + p;
        if (VEC == 4) {
          const float4 a = ldg_stream_f4(img + oc), t = ldg_stream_f4(trg + oc);
          stg_f4(mixed_img + oc, make_float4(mix_f(m[0], a.x, t.x), mix_f(m[1 % VEC], a.y, t.y),
                                             mix_f(m[2 % VEC], a.z, t.z), mix_f(m[3 % VEC], a.w, t.w)));
        } else {
          mixed_img[oc] = mix_f(m[0], img[oc], trg[oc]);
        }
      }
    }
    if (mixed_lbl) {
      if (VEC == 4 && kU8) {
        const uint32_t q4 = ldg_stream_u32(pl + o);
        uint32_t r = 0;
#pragma unroll
        for (int k = 0; k < VEC; ++k)
          r |= (mb[k] ? (uint32_t)g[k] : (q4 >> (8 * k)) & 255u) << (8 * k);
        *reinterpret_cast<uint32_t*>(mixed_lbl + o) = r;
      } else if (VEC == 4) {
        const int64_t* pl8 = reinterpret_cast<const int64_t*>(pl);
        int64_t* ml8 = reinterpret_cast<int64_t*>(mixed_lbl);
        const longlong2 q0 = ldg_stream_l2(pl8 + o), q1 = ldg_stream_l2(pl8 + o + 2);
        stg_l2(ml8 + o, make_longlong2(mb[0] ? g[0] : q0.x, mb[1 % VEC] ? g[1 % VEC] : q0.y));
        stg_l2(ml8 + o + 2,
               make_longlong2(mb[2 % VEC] ? g[2 % VEC] : q1.x, mb[3 % VEC] ? g[3 % VEC] : q1.y));
      } else {
        mixed_lbl[o] = mb[0] ? (L)g[0] : pl[o];
      }
    }
    if (mixed_weight) {
      float w[VEC];
      if (weight_in) {
        if (VEC == 4) {
          const float4 t = *reinterpret_cast<const float4*>(weight_in + o);
          w[0] = t.x; w[1 % VEC] = t.y; w[2 % VEC] = t.z; w[3 % VEC] = t.w;
        } else {
          w[0] = weight_in[o];
        }
      } else {
#pragma unroll
        for (int k = 0; k < VEC; ++k) w[k] = ratio;
      }
      if (ignore_top > 0 || ignore_bottom > 0) {
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
          const int64_t y = (int64_t)((unsigned)(p + k) / (unsigned)W);
          if (y < ignore_top || y >= H - ignore_bottom) w[k] = 0.f;
        }
      }
      // target=stack(gt_pixel_weight (ones), pseudo_weight): mask*1 + (1-mask)*w
      if (VEC == 4) {
        stg_f4(mixed_weight + o, make_float4(mix_f(m[0], 1.f, w[0]), mix_f(m[1 % VEC], 1.f, w[1 % VEC]),
                                             mix_f(m[2 % VEC], 1.f, w[2 % VEC]),
                                             mix_f(m[3 % VEC], 1.f, w[3 % VEC])));
      } else {
        mixed_weight[o] = mix_f(m[0], 1.f, w[0]);
      }
    }
  }
}

// Plain one_mix (dacs_transforms.py:129-144) for callers that already hold a mask
// tensor: out[c,p] = mask[p]*a[c,p] + (1-mask[p])*b[c,p]; mask is int64 {0,1}.
__global__ void __launch_bounds__(kMixThreads)
mask_mix_f32_kernel(const int64_t* __restrict__ mask, const float* __restrict__ a,
                    const float* __restrict__ b, float* __restrict__ out, int64_t channels,
                    int64_t HW) {
  const int64_t total = channels * HW;
  for (int64_t i = (int64_t)blockIdx.x * kMixThreads + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * kMixThreads) {
    const float m = (float)mask[i % HW];
    out[i] = mix_f(m, a[i], b[i]);
  }
}
__global__ void __launch_bounds__(kMixThreads)
mask_mix_i64_kernel(const int64_t* __restrict__ mask, const int64_t* __restrict__ a,
                    const int64_t* __restrict__ b, int64_t* __restrict__ out, int64_t channels,
                    int64_t HW) {
  const int64_t total = channels * HW;
  for (int64_t i = (int64_t)blockIdx.x * kMixThreads + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * kMixThreads) {
    const int64_t m = mask[i % HW];
    out[i] = m * a[i] + (1 - m) * b[i];
  }
}

}  // namespace pfst

extern "C" {

int pfst_mask_mix(const int64_t* mask, const void* a, const void* b, void* out, int32_t dtype,
                  int64_t channels, int64_t HW, void* stream) {
  if (channels < 0 || HW < 0) return PFST_ERR_INVALID_ARG;
  if (channels == 0 || HW == 0) return PFST_OK;
  if (!mask || !a || !b || !out) return PFST_ERR_INVALID_ARG;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int64_t g = (channels * HW + pfst::kMixThreads - 1) / pfst::kMixThreads;
  const int64_t cap = (int64_t)pfst::kNumSMs * 8 * 8;
  if (g > cap) g = cap;
  if (dtype == 0)
    pfst::mask_mix_f32_kernel<<<(unsigned)g, pfst::kMixThreads, 0, s>>>(
        mask, static_cast<const float*>(a), static_cast<const float*>(b), static_cast<float*>(out),
        channels, HW);
  else if (dtype == PFST_DT_I64)
    pfst::mask_mix_i64_kernel<<<(unsigned)g, pfst::kMixThreads, 0, s>>>(
        mask, static_cast<const int64_t*>(a), static_cast<const int64_t*>(b),
        static_cast<int64_t*>(out), channels, HW);
  else
    return PFST_ERR_INVALID_ARG;
  PFST_CHECK_LAUNCH("pfst_mask_mix");
  return PFST_OK;
}

}  // extern "C"

namespace pfst {

template <class L>
static int class_presence(const L* gt, int64_t n, uint32_t* presence, void* stream) {
  if (!presence || n < 0 || (n > 0 && !gt)) return PFST_ERR_INVALID_ARG;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PFST_CUDA_TRY(cudaMemsetAsync(presence, 0, 9 * sizeof(uint32_t), s), "pfst_class_presence/memset");
  if (n == 0) return PFST_OK;
  int64_t g = (n / (16 / sizeof(L)) + kMixThreads - 1) / kMixThreads;
  const int64_t cap = (int64_t)kNumSMs * 8;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  class_presence_kernel<L><<<(unsigned)g, kMixThreads, 0, s>>>(gt, n, presence);
  PFST_CHECK_LAUNCH("pfst_class_presence");
  return PFST_OK;
}

template <class L>
static int class_mix(const L* gt, const uint32_t* chosen, const float* img, const float* trg_img,
                     const L* pseudo_label, const float* weight_in, const unsigned long long* count,
                     int64_t ps_size, int32_t ignore_top, int32_t ignore_bottom, int64_t B,
                     int32_t img_channels, int64_t H, int64_t W, float* mixed_img, L* mixed_lbl,
                     float* mixed_weight, L* mix_mask, void* stream) {
  if (!gt || !chosen || B < 0 || H < 0 || W < 0 || img_channels < 0) return PFST_ERR_INVALID_ARG;
  if (mixed_img && (!img || !trg_img)) return PFST_ERR_INVALID_ARG;
  if (mixed_lbl && !pseudo_label) return PFST_ERR_INVALID_ARG;
  if (mixed_weight && !weight_in && (!count || ps_size <= 0)) return PFST_ERR_INVALID_ARG;
  if (ignore_top < 0 || ignore_bottom < 0) return PFST_ERR_INVALID_ARG;
  const int64_t HW = H * W;
  if (B == 0 || HW == 0) return PFST_OK;
  const bool vec4 = (HW % 4 == 0) && aligned_lbl4(gt) && (!mixed_img || (aligned16(img) && aligned16(trg_img) && aligned16(mixed_img))) &&
                    (!mixed_lbl || (aligned_lbl4(pseudo_label) && aligned_lbl4(mixed_lbl))) &&
                    (!mixed_weight || (aligned16(mixed_weight) && (!weight_in || aligned16(weight_in)))) &&
                    (!mix_mask || aligned_lbl4(mix_mask));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (HW > 0x7fffffffll) return PFST_ERR_UNSUPPORTED;
  const int64_t items = vec4 ? HW / 4 : HW;
  const dim3 g((unsigned)((items + kMixThreads - 1) / kMixThreads),
               (unsigned)(B < 65535 ? B : 65535), 1);
  if (vec4)
    class_mix_kernel<4, L><<<g, kMixThreads, 0, s>>>(
        gt, chosen, img, trg_img, pseudo_label, weight_in, count, ps_size, ignore_top, ignore_bottom,
        B, img_channels, H, W, mixed_img, mixed_lbl, mixed_weight, mix_mask);
  else
    class_mix_kernel<1, L><<<g, kMixThreads, 0, s>>>(
        gt, chosen, img, trg_img, pseudo_label, weight_in, count, ps_size, ignore_top, ignore_bottom,
        B, img_channels, H, W, mixed_img, mixed_lbl, mixed_weight, mix_mask);
  PFST_CHECK_LAUNCH("pfst_class_mix");
  return PFST_OK;
}

}  // namespace pfst

extern "C" {

int pfst_class_presence(const int64_t* gt, int64_t n, uint32_t* presence, void* stream) {
  return pfst::class_presence(gt, n, presence, stream);
}

int pfst_class_presence_lbl(const void* gt, int32_t label_dtype, int64_t n, uint32_t* presence,
                            void* stream) {
  if (label_dtype == PFST_DT_I64)
    return pfst::class_presence(static_cast<const int64_t*>(gt), n, presence, stream);
  if (label_dtype == PFST_DT_U8)
    return pfst::class_presence(static_cast<const uint8_t*>(gt), n, presence, stream);
  return PFST_ERR_UNSUPPORTED;
}

int pfst_class_mix(const int64_t* gt, const uint32_t* chosen, const float* img,
                   const float* trg_img, const int64_t* pseudo_label, const float* weight_in,
                   const unsigned long long* count, int64_t ps_size, int32_t ignore_top,
                   int32_t ignore_bottom, int64_t B, int32_t img_channels, int64_t H, int64_t W,
                   float* mixed_img, int64_t* mixed_lbl, float* mixed_weight, int64_t* mix_mask,
                   void* stream) {
  return pfst::class_mix(gt, chosen, img, trg_img, pseudo_label, weight_in, count, ps_size, ignore_top,
                         ignore_bottom, B, img_channels, H, W, mixed_img, mixed_lbl, mixed_weight, mix_mask,
                         stream);
}

int pfst_class_mix_lbl(const void* gt, const uint32_t* chosen, const float* img,
                       const float* trg_img, const void* pseudo_label, const float* weight_in,
                       const unsigned long long* count, int64_t ps_size, int32_t ignore_top,
                       int32_t ignore_bottom, int64_t B, int32_t img_channels, int64_t H, int64_t W,
                       float* mixed_img, void* mixed_lbl, float* mixed_weight, void* mix_mask,
                       int32_t label_dtype, void* stream) {
  if (label_dtype == PFST_DT_I64)
    return pfst::class_mix(static_cast<const int64_t*>(gt), chosen, img, trg_img,
                           static_cast<const int64_t*>(pseudo_label), weight_in, count, ps_size, ignore_top,
                           ignore_bottom, B, img_channels, H, W, mixed_img, static_cast<int64_t*>(mixed_lbl),
                           mixed_weight, static_cast<int64_t*>(mix_mask), stream);
  if (label_dtype == PFST_DT_U8)
    return pfst::class_mix(static_cast<const uint8_t*>(gt), chosen, img, trg_img,
                           static_cast<const uint8_t*>(pseudo_label), weight_in, count, ps_size, ignore_top,
                           ignore_bottom, B, img_channels, H, W, mixed_img, static_cast<uint8_t*>(mixed_lbl),
                           mixed_weight, static_cast<uint8_t*>(mix_mask), stream);
  return PFST_ERR_UNSUPPORTED;
}

}  // extern "C"
