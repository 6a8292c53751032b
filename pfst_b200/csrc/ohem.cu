// OHEM pixel sampler of a decode head: mmseg 0.x OHEMPixelSampler.sample, whose map replaces seg_weight in
// BaseDecodeHead.losses (rsiseg/models/decode_heads/decode_head.py:249-283). The 0/1 weight of every pixel
// of the (B,H,W) label map, on the device, without a host synchronisation:
//   valid = label != ignore_index, batch_kept = min_kept * B, n = #valid
//   thresh given: key = softmax(up)[label] (fp32), k = min(batch_kept, n - 1),
//                 threshold = max(k-th smallest valid key (0 when n == 0), fp32(thresh)),
//                 weight = valid & (key < threshold)
//   thresh None:  key = loss_weight * class_weight[label] * CE(up, label); the batch_kept valid pixels with
//                 the largest keys get weight 1 (a stable descending sort: on a tie at the boundary the lower
//                 flat index goes first)
// where up is the bilinear (align_corners=False) up-sampling of the low-resolution logits by an integer
// factor s >= 1 (s = 1: logits already at label resolution). The reference materialises the up-sampled
// logits, their soft-max and a full sort of the keys; here:
//   ohem_key_kernel        one thread per full-resolution pixel: the key, from the low-resolution logits
//                          with the CE kernel's bilinear weights (the up-sampled tensor never exists), as
//                          an order-preserving 32-bit pattern (0 = ignored pixel); counts the valid pixels
//   ohem_hist/scan_kernel  exact order statistic by a three-pass radix select on those patterns (11 + 11 +
//                          10 bit digits, the scheme of class_quantile.cu), its rank read from the device
//                          count: the k-th smallest key, or the batch_kept-th largest
//   ohem_tie_count_kernel  (top-k only) per chunk of 4096 pixels, the keys equal to the selected one;
//   ohem_tie_scan_kernel   exclusive prefix of those counts, so the tie fill takes the lowest indices
//   ohem_weight_kernel     the 0/1 map
// NaN keys order as torch.sort orders them: after every number (the largest). -0 and +0 are one key.
// Bytes: key pass B*H*W * (label size + 4) + the low-res logits; every other pass 4 B per pixel read
// (+ 4 B written by the weight pass).
#include <math.h>

#include <algorithm>

#include "common.cuh"

namespace pfst {

constexpr int kOhThreads = 256;
constexpr int kOhBins = 2048;
constexpr int kOhPer = 16;                          // keys per thread in the tie-count and weight passes
constexpr int kOhChunk = kOhThreads * kOhPer;       // pixels per block in those passes
constexpr int kOhScanThreads = 1024;

struct OhState {
  unsigned n;        // valid pixels (key pass)
  unsigned prefix;   // key bits fixed so far; after the last pass the selected key
  unsigned rank;     // residual ascending rank inside the prefix bucket
  unsigned eq;       // after the last pass: valid keys equal to the selected one
};

// torch upsample_bilinear2d, align_corners=False: the arithmetic of ce_src in weighted_ce.cu
__device__ __forceinline__ void oh_src(int dst, float scale, int in, int& i0, int& i1, float& l0, float& l1) {
  float r = scale * ((float)dst + 0.5f) - 0.5f;
  r = r < 0.f ? 0.f : r;
  i0 = (int)r;
  i1 = i0 + (i0 < in - 1 ? 1 : 0);
  l1 = r - (float)i0;
  l0 = 1.f - l1;
}

// unsigned order of the pattern = torch.sort order of the key: NaN largest, -0 == +0. No key maps to 0,
// which marks an ignored pixel (it would be a negative NaN, and NaNs map to 0xffffffff).
__device__ __forceinline__ unsigned oh_order(float v) {
  if (v != v) return 0xffffffffu;
  if (v == 0.f) return 0x80000000u;
  const unsigned u = __float_as_uint(v);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float oh_value(unsigned o) {
  return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}

template <class T, class L, bool TOPK>
__global__ void __launch_bounds__(kOhThreads)
ohem_key_kernel(const T* __restrict__ logits, const L* __restrict__ labels, const float* __restrict__ class_weight,
                int C, int lh, int lw, int H, int W, int64_t N, int64_t ignore_index, float loss_weight,
                unsigned* __restrict__ okeys, float* __restrict__ keys_out, OhState* __restrict__ st) {
  __shared__ unsigned red[kOhThreads / 32];
  const float sch = (float)lh / (float)H, scw = (float)lw / (float)W;
  const int64_t lplane = (int64_t)lh * lw;
  unsigned cnt = 0;
  for (int64_t p = (int64_t)blockIdx.x * kOhThreads + threadIdx.x; p < N; p += (int64_t)gridDim.x * kOhThreads) {
    const int x = (int)(p % W);
    const int64_t r = p / W;
    const int y = (int)(r % H);
    const int64_t b = r / H;
    int y0, y1, x0, x1;
    float hy0, hy1, wx0, wx1;
    oh_src(y, sch, lh, y0, y1, hy0, hy1);
    oh_src(x, scw, lw, x0, x1, wx0, wx1);
    const int64_t lab = (int64_t)labels[p];
    const bool valid = lab != ignore_index && lab >= 0 && lab < C;
    const int tgt = valid ? (int)lab : 0;                 // an ignored pixel gathers class 0
    const T* z = logits + b * C * lplane;
    const int o00 = y0 * lw + x0, o01 = y0 * lw + x1, o10 = y1 * lw + x0, o11 = y1 * lw + x1;
    auto up = [&](int c) {
      const T* zc = z + c * lplane;
      return hy0 * (wx0 * ldgf(zc + o00) + wx1 * ldgf(zc + o01)) + hy1 * (wx0 * ldgf(zc + o10) + wx1 * ldgf(zc + o11));
    };
    float m = -INFINITY, vt = 0.f;
    for (int c = 0; c < C; ++c) {
      const float v = up(c);
      m = v > m ? v : m;
      if (c == tgt) vt = v;
    }
    float sum = 0.f;
    for (int c = 0; c < C; ++c) sum += expf(up(c) - m);
    float key;
    if (TOPK) {   // CrossEntropyLoss(reduction_override='none', weight=None): 0 at an ignored pixel
      const float cw = class_weight ? class_weight[tgt] : 1.f;
      key = valid ? loss_weight * (cw * ((m + logf(sum)) - vt)) : 0.f;
    } else {
      key = expf(vt - m) / sum;
    }
    if (keys_out) keys_out[p] = key;
    okeys[p] = valid ? oh_order(key) : 0u;
    cnt += valid ? 1u : 0u;
  }
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = cnt;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned s = 0;
    for (int w = 0; w < kOhThreads / 32; ++w) s += red[w];
    if (s) atomicAdd(&st->n, s);
  }
}

// histogram of digit [shift, shift + bits) of the valid keys whose higher bits equal the prefix; lanes with
// the same digit are merged first (the first pass puts nearly every key of a soft-max into a few bins)
__global__ void __launch_bounds__(kOhThreads)
ohem_hist_kernel(const unsigned* __restrict__ okeys, int64_t N, const OhState* __restrict__ st, int shift, int bits,
                 unsigned hi_mask, unsigned* __restrict__ hist) {
  __shared__ unsigned h_s[kOhBins];
  if (st->n == 0) return;
  const unsigned prefix = st->prefix;
  for (int i = threadIdx.x; i < kOhBins; i += kOhThreads) h_s[i] = 0;
  __syncthreads();
  const unsigned dmask = (1u << bits) - 1u;
  for (int64_t base = (int64_t)blockIdx.x * kOhThreads; base < N; base += (int64_t)gridDim.x * kOhThreads) {
    const int64_t p = base + threadIdx.x;
    const unsigned k = p < N ? okeys[p] : 0u;
    const bool hit = k != 0u && (k & hi_mask) == prefix;
    const unsigned d = hit ? (k >> shift) & dmask : 0xffffffffu;
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    if (hit && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&h_s[d], (unsigned)__popc(peers));
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kOhBins; i += kOhThreads)
    if (h_s[i]) atomicAdd(&hist[i], h_s[i]);
}

// one block: the digit whose cumulative count passes the residual rank. The first pass sets the rank from
// the device count; the last writes the selected key's value to kth_out (0 when no pixel is valid).
__global__ void __launch_bounds__(kOhThreads)
ohem_scan_kernel(OhState* __restrict__ st, unsigned* __restrict__ hist, int shift, int bits, int first, int last,
                 int topk, int64_t batch_kept, float* __restrict__ kth_out) {
  __shared__ unsigned part[kOhThreads];
  const int nb = 1 << bits, per = (nb + kOhThreads - 1) / kOhThreads;
  unsigned local = 0;
  for (int j = 0; j < per; ++j) {
    const int bin = threadIdx.x * per + j;
    if (bin < nb) local += hist[bin];
  }
  part[threadIdx.x] = local;
  __syncthreads();
  OhState s = *st;
  if (threadIdx.x == 0 && s.n > 0) {
    if (first) {
      const int64_t n = s.n;
      s.rank = (unsigned)(topk ? (n > batch_kept ? n - batch_kept : 0) : (batch_kept < n - 1 ? batch_kept : n - 1));
    }
    unsigned cum = 0;
    int t = 0;
    for (; t < kOhThreads; ++t) {
      if (cum + part[t] > s.rank) break;
      cum += part[t];
    }
    if (t == kOhThreads) t = kOhThreads - 1;
    int bin = t * per;
    for (; bin < nb - 1 && bin < (t + 1) * per; ++bin) {
      if (cum + hist[bin] > s.rank) break;
      cum += hist[bin];
    }
    s.prefix |= (unsigned)bin << shift;
    s.rank -= cum;
    if (last) s.eq = hist[bin];
    *st = s;
  }
  __syncthreads();
  for (int j = threadIdx.x; j < nb; j += kOhThreads) hist[j] = 0;        // ready for the next pass
  if (last && threadIdx.x == 0 && kth_out) *kth_out = s.n > 0 ? oh_value(s.prefix) : 0.f;
}

// keys of chunk blockIdx.x in registers; thread t holds pixels chunk + i * kOhThreads + t, i < kOhPer
__device__ __forceinline__ void oh_load_chunk(const unsigned* __restrict__ okeys, int64_t N, unsigned (&k)[kOhPer]) {
  const int64_t base = (int64_t)blockIdx.x * kOhChunk + threadIdx.x;
#pragma unroll
  for (int i = 0; i < kOhPer; ++i) {
    const int64_t p = base + (int64_t)i * kOhThreads;
    k[i] = p < N ? okeys[p] : 0u;
  }
}

__global__ void __launch_bounds__(kOhThreads)
ohem_tie_count_kernel(const unsigned* __restrict__ okeys, int64_t N, const OhState* __restrict__ st,
                      unsigned* __restrict__ counts) {
  __shared__ unsigned red[kOhThreads / 32];
  const OhState s = *st;
  unsigned k[kOhPer];
  oh_load_chunk(okeys, N, k);
  unsigned c = 0;
#pragma unroll
  for (int i = 0; i < kOhPer; ++i) c += (s.n > 0 && k[i] == s.prefix) ? 1u : 0u;
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned t = 0;
    for (int w = 0; w < kOhThreads / 32; ++w) t += red[w];
    counts[blockIdx.x] = t;
  }
}

// one block: counts[0..nb) -> exclusive prefix sums, in place
__global__ void __launch_bounds__(kOhScanThreads) ohem_tie_scan_kernel(unsigned* __restrict__ counts, int nb) {
  __shared__ unsigned wsum[kOhScanThreads / 32];
  const int per = (nb + kOhScanThreads - 1) / kOhScanThreads;
  const int lo = threadIdx.x * per, hi = min(nb, lo + per);
  unsigned s = 0;
  for (int i = lo; i < hi; ++i) s += counts[i];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned inc = s;                                          // inclusive scan inside the warp
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned v = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += v;
  }
  if (lane == 31) wsum[warp] = inc;
  __syncthreads();
  unsigned before = inc - s;
  for (int w = 0; w < warp; ++w) before += wsum[w];
  for (int i = lo; i < hi; ++i) {
    const unsigned c = counts[i];
    counts[i] = before;
    before += c;
  }
}

// TOPK: weight = key > selected, or key == selected and among the first (eq - rank) such pixels in flat
// order (tie_base: that order's count before this chunk). Otherwise weight = valid & key < threshold.
template <bool TOPK>
__global__ void __launch_bounds__(kOhThreads)
ohem_weight_kernel(const unsigned* __restrict__ okeys, int64_t N, const OhState* __restrict__ st, float thresh,
                   const unsigned* __restrict__ tie_base, float* __restrict__ weight) {
  __shared__ unsigned wc[kOhPer][kOhThreads / 32];
  const OhState s = *st;
  unsigned k[kOhPer];
  oh_load_chunk(okeys, N, k);
  const int64_t base = (int64_t)blockIdx.x * kOhChunk + threadIdx.x;
  if (TOPK) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned lt = (1u << lane) - 1u;
    unsigned bal[kOhPer];
#pragma unroll
    for (int i = 0; i < kOhPer; ++i) {
      bal[i] = __ballot_sync(0xffffffffu, s.n > 0 && k[i] == s.prefix);
      if (lane == 0) wc[i][warp] = __popc(bal[i]);
    }
    __syncthreads();
    if (threadIdx.x == 0) {                                  // exclusive prefix in flat order: (i, warp)
      unsigned run = tie_base[blockIdx.x];
      for (int i = 0; i < kOhPer; ++i)
        for (int w = 0; w < kOhThreads / 32; ++w) {
          const unsigned c = wc[i][w];
          wc[i][w] = run;
          run += c;
        }
    }
    __syncthreads();
    const unsigned need = s.eq - s.rank;
#pragma unroll
    for (int i = 0; i < kOhPer; ++i) {
      const int64_t p = base + (int64_t)i * kOhThreads;
      if (p >= N) break;
      const bool eq = (bal[i] >> lane) & 1u;
      const bool on = s.n > 0 && (k[i] > s.prefix || (eq && wc[i][warp] + __popc(bal[i] & lt) < need));
      weight[p] = on ? 1.f : 0.f;
    }
  } else {
    // threshold = max(min_threshold, thresh) as Python's max evaluates it: thresh only if it is larger
    const float kth = s.n > 0 ? oh_value(s.prefix) : 0.f;
    const float th = thresh > kth ? thresh : kth;
#pragma unroll
    for (int i = 0; i < kOhPer; ++i) {
      const int64_t p = base + (int64_t)i * kOhThreads;
      if (p >= N) break;
      weight[p] = (k[i] != 0u && oh_value(k[i]) < th) ? 1.f : 0.f;
    }
  }
}

}  // namespace pfst

namespace {
struct OhLayout { size_t hist, counts, keys, total; int64_t chunks; };
inline size_t oh_up16(size_t v) { return (v + 15) / 16 * 16; }
// state | histogram u32[2048] | tie counts u32[chunks] | keys u32[N]
inline OhLayout oh_layout(int64_t N) {
  OhLayout L;
  L.chunks = (N + pfst::kOhChunk - 1) / pfst::kOhChunk;
  L.hist = oh_up16(sizeof(pfst::OhState));
  L.counts = L.hist + (size_t)pfst::kOhBins * 4;
  L.keys = oh_up16(L.counts + (size_t)L.chunks * 4);
  L.total = L.keys + (size_t)N * 4;
  return L;
}
constexpr int64_t kOhMaxPixels = (int64_t)1 << 31;   // counts and ranks are 32-bit

template <class T, class L>
int ohem_weight(const T* logits, const L* labels, const float* class_weight, int64_t B, int32_t C, int32_t lh,
                int32_t lw, int32_t H, int32_t W, int64_t ignore_index, float loss_weight, float thresh,
                int64_t min_kept, void* workspace, float* keys_out, float* kth_out, float* weight_out, void* stream) {
  if (B < 0 || C < 1 || lh < 1 || lw < 1 || H < 1 || W < 1 || min_kept < 2 || !workspace)
    return PFST_ERR_INVALID_ARG;
  // an empty batch reads and writes no pixel, so its (empty) tensors may have null data pointers
  if (B > 0 && (!logits || !labels || !weight_out)) return PFST_ERR_INVALID_ARG;
  if (H % lh != 0 || W % lw != 0 || H / lh != W / lw) return PFST_ERR_UNSUPPORTED;
  const int64_t N = B * H * W;
  if (N >= kOhMaxPixels || (int64_t)C * lh * lw >= kOhMaxPixels || !pfst::aligned16(workspace))
    return PFST_ERR_UNSUPPORTED;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  unsigned char* ws = static_cast<unsigned char*>(workspace);
  const OhLayout Ly = oh_layout(N);
  pfst::OhState* st = reinterpret_cast<pfst::OhState*>(ws);
  unsigned* hist = reinterpret_cast<unsigned*>(ws + Ly.hist);
  unsigned* counts = reinterpret_cast<unsigned*>(ws + Ly.counts);
  unsigned* okeys = reinterpret_cast<unsigned*>(ws + Ly.keys);
  PFST_CUDA_TRY(cudaMemsetAsync(ws, 0, Ly.counts, s), "pfst_ohem_weight/memset");
  if (N == 0) {
    if (kth_out) PFST_CUDA_TRY(cudaMemsetAsync(kth_out, 0, sizeof(float), s), "pfst_ohem_weight/empty");
    return PFST_OK;
  }
  const bool topk = thresh != thresh;
  const int64_t batch_kept = min_kept * B;
  using namespace pfst;
  const unsigned kgrid = (unsigned)std::min<int64_t>((N + kOhThreads - 1) / kOhThreads, (int64_t)kNumSMs * 16);
  if (topk)
    ohem_key_kernel<T, L, true><<<kgrid, kOhThreads, 0, s>>>(logits, labels, class_weight, C, lh, lw, H, W, N,
                                                             ignore_index, loss_weight, okeys, keys_out, st);
  else
    ohem_key_kernel<T, L, false><<<kgrid, kOhThreads, 0, s>>>(logits, labels, class_weight, C, lh, lw, H, W, N,
                                                              ignore_index, loss_weight, okeys, keys_out, st);
  PFST_CHECK_LAUNCH("pfst_ohem_weight/key");
  const unsigned hgrid = (unsigned)std::min<int64_t>((N + kOhThreads * 8 - 1) / (kOhThreads * 8), (int64_t)kNumSMs * 4);
  const int shifts[3] = {21, 10, 0}, bits[3] = {11, 11, 10};
  const unsigned hi_masks[3] = {0u, 0xffe00000u, 0xfffffc00u};
  for (int pass = 0; pass < 3; ++pass) {
    ohem_hist_kernel<<<hgrid, kOhThreads, 0, s>>>(okeys, N, st, shifts[pass], bits[pass], hi_masks[pass], hist);
    PFST_CHECK_LAUNCH("pfst_ohem_weight/hist");
    ohem_scan_kernel<<<1, kOhThreads, 0, s>>>(st, hist, shifts[pass], bits[pass], pass == 0, pass == 2, topk ? 1 : 0,
                                              batch_kept, kth_out);
    PFST_CHECK_LAUNCH("pfst_ohem_weight/scan");
  }
  const unsigned wgrid = (unsigned)Ly.chunks;
  if (topk) {
    ohem_tie_count_kernel<<<wgrid, kOhThreads, 0, s>>>(okeys, N, st, counts);
    PFST_CHECK_LAUNCH("pfst_ohem_weight/tie-count");
    ohem_tie_scan_kernel<<<1, kOhScanThreads, 0, s>>>(counts, (int)Ly.chunks);
    PFST_CHECK_LAUNCH("pfst_ohem_weight/tie-scan");
    ohem_weight_kernel<true><<<wgrid, kOhThreads, 0, s>>>(okeys, N, st, thresh, counts, weight_out);
  } else {
    ohem_weight_kernel<false><<<wgrid, kOhThreads, 0, s>>>(okeys, N, st, thresh, counts, weight_out);
  }
  PFST_CHECK_LAUNCH("pfst_ohem_weight/weight");
  return PFST_OK;
}
}  // namespace

extern "C" {

int64_t pfst_ohem_ws_bytes(int64_t B, int32_t H, int32_t W) {
  if (B < 0 || H < 1 || W < 1 || B * H * W >= kOhMaxPixels) return 0;
  return (int64_t)oh_layout(B * H * W).total;
}

int pfst_ohem_weight(const void* logits, int32_t logit_dtype, const void* labels, int32_t label_dtype,
                     const float* class_weight, int64_t B, int32_t C, int32_t lh, int32_t lw, int32_t H, int32_t W,
                     int64_t ignore_index, float loss_weight, float thresh, int64_t min_kept, void* workspace,
                     float* keys_out, float* kth_out, float* weight_out, void* stream) {
  return pfst::with_float_dt(logit_dtype, [&](auto t) {
    return pfst::with_label_dt(label_dtype, [&](auto l) {
      return ohem_weight(static_cast<const decltype(t)*>(logits), static_cast<const decltype(l)*>(labels),
                         class_weight, B, C, lh, lw, H, W, ignore_index, loss_weight, thresh, min_kept, workspace,
                         keys_out, kth_out, weight_out, stream);
    });
  });
}

}  // extern "C"
