// §8(f) rank 1 — pixel-weighted cross-entropy of a decode head, fused with the bilinear
// up-sampling of its logits, the top-1 accuracy and the gradient w.r.t. the LOW-resolution
// logits.
//
// Reference: BaseDecodeHead.losses, rsiseg/models/decode_heads/decode_head.py:249-283
//   seg_logit = resize(seg_logit, size=label.shape[2:], mode='bilinear', align_corners=False)
//   loss_ce   = loss_weight * mean_over_ALL_pixels( CE(seg_logit, label, ignore_index) * seg_weight )
//               (cross_entropy_loss.py:45-63 + utils.py:48-79: reduction 'mean', avg_non_ignore False)
//   acc_seg   = accuracy(seg_logit, label, ignore_index)           (accuracy.py:6-59, top-1)
// The reference materialises the (B,C,H,W) up-sampled logits (50 MB at cfg2), their
// log-softmax and, in backward, both gradients. Here one kernel reads the low-resolution
// logits (3 MB), the labels and the pixel weights once and produces the loss, the accuracy
// and d loss / d low-res logits: a block owns a 16x16 tile of low-res cells in shared memory,
// one thread per cell evaluates the s x s high-res pixels whose bilinear taps start there
// (torch's align_corners=False arithmetic, taps read from shared memory) and sums their
// per-class gradients privately; only the low-res tile (17*17*C values) goes to global
// memory with atomics.
// HBM-bound in principle: (8 + 4 [+4]) B per high-res pixel.
// The logits may be fp32, fp16 or bf16 (a student run under autocast): every value is converted to
// fp32 once, as the low-resolution tile is staged (exact), and all arithmetic after that is the fp32
// code. The gradient is always accumulated and written in fp32; scale_cast_kernel turns it into the
// logits' dtype in the backward.
#include <float.h>
#include <math.h>
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"

namespace pfst {

constexpr int kCeTile = 16;                      // low-res CELLS per tile side (one thread per cell)
constexpr int kCeHalo = kCeTile + 1;             // low-res pixels touched by a tile of cells
constexpr int kCeThreads = kCeTile * kCeTile;
constexpr int kCeMaxC = 64;
constexpr int kCeRegC = 8;                       // up to this many classes the up-sampled logits stay in registers

// The kernels' last template argument LT names the input types: a label type L (int64 or uint8) for fp32
// logits, Lp<L, T> for logits of type T = __half or __nv_bfloat16. Both families are one templated
// __global__ body each; the fp32 instantiations keep their names (weighted_ce_s4_kernel<6, ..., long>) and
// the 16-bit ones are their twins (weighted_ce_s4_kernel<6, ..., pfst::Lp<long, __half>>).
template <class L, class T> struct Lp {};
template <class LT> struct CeTypes { using label = LT; using logit = float; };
template <class L, class T> struct CeTypes<Lp<L, T>> { using label = L; using logit = T; };
template <class L, class T>
using CeIn = typename std::conditional<std::is_same<T, float>::value, L, Lp<L, T>>::type;

struct CeParams {
  const void* logits;        // (B, C, lh, lw), of the kernels' logits type T
  const void* labels;        // (B, H, W), int64 or uint8 (the kernels' L)
  const float* weight;       // (B, H, W) or null
  const float* class_weight; // (C) or null
  int B, C, lh, lw, H, W, s; // H = s * lh, W = s * lw
  int64_t ignore_index;
  float loss_weight;
  float* grad;               // (B, C, lh, lw) or null: d(loss_weight * mean loss) / d logits
  double* stats;             // [0] loss sum, [1] correct, [2] valid, [3] block counter
  float* out;                // [0] loss_weight * mean, [1] acc_seg
};

// torch upsample_bilinear2d, align_corners=False: src = max(scale * (dst + 0.5) - 0.5, 0)
__device__ __forceinline__ void ce_src(int dst, float scale, int in, int& i0, int& i1, float& l0, float& l1) {
  float r = scale * ((float)dst + 0.5f) - 0.5f;
  r = r < 0.f ? 0.f : r;
  i0 = (int)r;
  i1 = i0 + (i0 < in - 1 ? 1 : 0);
  l1 = r - (float)i0;
  l0 = 1.f - l1;
}

// One thread per low-resolution CELL (y0, x0): the high-res pixels whose bilinear taps start at
// that low-res pixel (s x s of them in the interior) all read and update the same four low-res
// corners, so their per-class gradients are summed in a private shared-memory accumulator
// ([class][corner][thread]: conflict-free, no atomics) and only four shared atomics per class and
// thread fold them into the block's low-res tile; the tile goes to global memory once.
template <bool REGC, bool PRIV, class LT>
__global__ void __launch_bounds__(kCeThreads)
weighted_ce_kernel(const CeParams P) {
  using L = typename CeTypes<LT>::label;
  using T = typename CeTypes<LT>::logit;
  extern __shared__ __align__(16) float ce_smem[];
  float* z_s = ce_smem;                                       // [C][kCeHalo*kCeHalo] low-res logits
  float* g_s = z_s + (size_t)P.C * kCeHalo * kCeHalo;           // same shape: gradient tile
  float* a_s = g_s + (size_t)P.C * kCeHalo * kCeHalo;           // [C][4][kCeThreads] private accumulators
  __shared__ double red[3][kCeThreads / 32];
  const int b = blockIdx.z;
  const int ly0 = blockIdx.y * kCeTile, lx0 = blockIdx.x * kCeTile;   // first cell of the tile
  const int64_t lplane = (int64_t)P.lh * P.lw;
  const T* zb = static_cast<const T*>(P.logits) + (int64_t)b * P.C * lplane;
  for (int i = threadIdx.x; i < P.C * kCeHalo * kCeHalo; i += kCeThreads) {
    const int c = i / (kCeHalo * kCeHalo), r = i - c * (kCeHalo * kCeHalo);
    const int ly = ly0 + r / kCeHalo, lx = lx0 + r % kCeHalo;
    z_s[i] = (ly < P.lh && lx < P.lw) ? to_f32(zb[c * lplane + (int64_t)ly * P.lw + lx]) : 0.f;
    g_s[i] = 0.f;
  }
  if (P.grad && PRIV)
    for (int i = threadIdx.x; i < P.C * 4 * kCeThreads; i += kCeThreads) a_s[i] = 0.f;
  __syncthreads();

  const int cy = threadIdx.x / kCeTile, cx = threadIdx.x % kCeTile;
  const int y0c = ly0 + cy, x0c = lx0 + cx;                         // this thread's cell
  const float sch = (float)P.lh / (float)P.H, scw = (float)P.lw / (float)P.W;
  const float gscale = P.loss_weight / (float)((double)P.B * P.H * P.W);
  double loss = 0.0, correct = 0.0, valid = 0.0;
  if (y0c < P.lh && x0c < P.lw) {
    // candidate high-res range of the cell (one extra pixel each side: the exact membership test
    // is torch's own fp32 source-index arithmetic, re-evaluated per pixel)
    const int ya = max(0, y0c * P.s + P.s / 2 - 1), yb = min(P.H - 1, (y0c + 1) * P.s + P.s / 2);
    const int xa = max(0, x0c * P.s + P.s / 2 - 1), xb = min(P.W - 1, (x0c + 1) * P.s + P.s / 2);
    const int i00 = cy * kCeHalo + cx;                               // the cell's corners inside the tile
    for (int y = (y0c == 0 ? 0 : ya); y <= yb; ++y) {
      int y0, y1;
      float hy0l, hy1l;
      ce_src(y, sch, P.lh, y0, y1, hy0l, hy1l);
      if (y0 != y0c) continue;
      const int dy = (y1 - y0) * kCeHalo;
      for (int x = (x0c == 0 ? 0 : xa); x <= xb; ++x) {
        int x0, x1;
        float wx0l, wx1l;
        ce_src(x, scw, P.lw, x0, x1, wx0l, wx1l);
        if (x0 != x0c) continue;
        const int dx = x1 - x0;
        const int64_t pix = ((int64_t)b * P.H + y) * P.W + x;
        const int64_t lab = static_cast<const L*>(P.labels)[pix];
        const float t00 = hy0l * wx0l, t01 = hy0l * wx1l, t10 = hy1l * wx0l, t11 = hy1l * wx1l;
        auto up = [&](int c) {
          const float* z = z_s + c * (kCeHalo * kCeHalo) + i00;
          return hy0l * (wx0l * z[0] + wx1l * z[dx]) + hy1l * (wx0l * z[dy] + wx1l * z[dy + dx]);
        };
        float vreg[REGC ? kCeRegC : 1];
        float m = -INFINITY;
        int arg = 0;
        if (REGC) {
#pragma unroll
          for (int c = 0; c < kCeRegC; ++c) {
            vreg[c] = c < P.C ? up(c) : -INFINITY;
            if (vreg[c] > m) { m = vreg[c]; arg = c; }        // first maximum wins
          }
        } else {
          for (int c = 0; c < P.C; ++c) {
            const float v = up(c);
            if (v > m) { m = v; arg = c; }
          }
        }
        const bool ign = lab == P.ignore_index || lab < 0 || lab >= P.C;
        if (ign) continue;
        valid += 1.0;
        if (arg == (int)lab) correct += 1.0;
        float sum = 0.f, vlab = 0.f;
        if (REGC) {
#pragma unroll
          for (int c = 0; c < kCeRegC; ++c) {
            if (c < P.C) {
              vreg[c] = expf(vreg[c] - m);
              sum += vreg[c];
              if (c == (int)lab) vlab = up(c);
            }
          }
        } else {
          for (int c = 0; c < P.C; ++c) {
            const float v = up(c);
            sum += expf(v - m);
            if (c == (int)lab) vlab = v;
          }
        }
        float wpx = P.weight ? P.weight[pix] : 1.f;
        if (P.class_weight) wpx *= P.class_weight[lab];
        loss += (double)(((m + logf(sum)) - vlab) * wpx);
        if (P.grad) {
          const float inv = 1.f / sum, k = gscale * wpx;
          float* acc = a_s + threadIdx.x;
          if (REGC) {
#pragma unroll
            for (int c = 0; c < kCeRegC; ++c) {
              if (c < P.C) {
                const float g = k * (vreg[c] * inv - (c == (int)lab ? 1.f : 0.f));
                float* q = acc + c * 4 * kCeThreads;
                q[0] += t00 * g; q[kCeThreads] += t01 * g; q[2 * kCeThreads] += t10 * g; q[3 * kCeThreads] += t11 * g;
              }
            }
          } else {
            for (int c = 0; c < P.C; ++c) {
              const float g = k * (expf(up(c) - m) * inv - (c == (int)lab ? 1.f : 0.f));
              if (PRIV) {
                float* q = acc + c * 4 * kCeThreads;
                q[0] += t00 * g; q[kCeThreads] += t01 * g; q[2 * kCeThreads] += t10 * g; q[3 * kCeThreads] += t11 * g;
              } else {      // many classes: the private accumulators do not fit, scatter into the tile directly
                float* gs = g_s + c * (kCeHalo * kCeHalo) + i00;
                atomicAdd(gs, t00 * g); atomicAdd(gs + dx, t01 * g);
                atomicAdd(gs + dy, t10 * g); atomicAdd(gs + dy + dx, t11 * g);
              }
            }
          }
        }
      }
    }
    // fold the cell's four corners into the block's low-res tile. The second tap of a clamped border
    // cell coincides with the first (x1 == x0 at the last column / y1 == y0 at the last row).
    if (P.grad && PRIV) {
      const int ddx = x0c < P.lw - 1 ? 1 : 0, ddy = (y0c < P.lh - 1 ? 1 : 0) * kCeHalo;
      for (int c = 0; c < P.C; ++c) {
        const float* q = a_s + c * 4 * kCeThreads + threadIdx.x;
        float* gs = g_s + c * (kCeHalo * kCeHalo) + i00;
        atomicAdd(gs, q[0]);
        atomicAdd(gs + ddx, q[kCeThreads]);
        atomicAdd(gs + ddy, q[2 * kCeThreads]);
        atomicAdd(gs + ddy + ddx, q[3 * kCeThreads]);
      }
    }
  }

  // gradient tile -> global (the last row / column of the tile belongs to the next tile too: atomics)
  __syncthreads();
  if (P.grad) {
    float* gb = P.grad + (int64_t)b * P.C * lplane;
    for (int i = threadIdx.x; i < P.C * kCeHalo * kCeHalo; i += kCeThreads) {
      const float v = g_s[i];
      if (v == 0.f) continue;
      const int c = i / (kCeHalo * kCeHalo), r = i - c * (kCeHalo * kCeHalo);
      const int ly = ly0 + r / kCeHalo, lx = lx0 + r % kCeHalo;
      if (ly < P.lh && lx < P.lw) atomicAdd(gb + c * lplane + (int64_t)ly * P.lw + lx, v);
    }
  }
  // statistics: block partials in fp64, last block finalises on the device
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  loss = warp_sum(loss); correct = warp_sum(correct); valid = warp_sum(valid);
  if (lane == 0) { red[0][warp] = loss; red[1][warp] = correct; red[2][warp] = valid; }
  __syncthreads();
  __shared__ bool is_last;
  if (threadIdx.x < 3) {
    double v = 0.0;
    for (int wv = 0; wv < kCeThreads / 32; ++wv) v += red[threadIdx.x][wv];
    if (v != 0.0) atomicAdd(&P.stats[threadIdx.x], v);
    __threadfence();
  }
  __syncthreads();
  if (threadIdx.x == 0)
    is_last = atomicAdd(reinterpret_cast<unsigned*>(P.stats + 3), 1u) == gridDim.x * gridDim.y * gridDim.z - 1;
  __syncthreads();
  if (is_last && threadIdx.x == 0) {
    __threadfence();
    const double s = *((volatile double*)&P.stats[0]);
    const double nc = *((volatile double*)&P.stats[1]), nv = *((volatile double*)&P.stats[2]);
    P.out[0] = P.loss_weight * (float)(s / ((double)P.B * P.H * P.W));
    // accuracy.py:50-58: (correct + eps) * (100 / (valid + eps)), eps = float32 epsilon
    const float eps = FLT_EPSILON;
    P.out[1] = ((float)nc + eps) * (float)(100.0 / (nv + (double)eps));
  }
}


// ---- factor-4 kernel (every shipped config: H/4 logits -> H) -----------------------------------
// With H = 4*lh the source coordinate 0.25*(dst+0.5)-0.5 is exact in fp32: the pixels x = 4k+2+j
// (j = 0..3) all interpolate between the low-res columns k and k+1 with the constant weights
// l1 = 0.125 + 0.25*j, and the two clamped pixels x = 0,1 sit on column 0 with l1 = 0. One thread
// owns one cell (k_y, k_x): its 4x4 pixels are loaded with 128-bit (labels) and 64-bit (weights)
// loads, all sixteen in flight; the four corner logits per class stay in registers; a column's
// horizontally interpolated pair (A0, A1) is formed once and reused down the four rows; the
// gradient is reduced over the rows first (S0, S1), then spread to the four corner accumulators,
// all in registers. The low-res halo is filled clamp-to-edge, so the last cell (x1 == x0) needs no
// special arithmetic and its "k+1" corner folds back onto k when the tile is written. No shared
// atomics anywhere (a float atomicAdd on shared memory is a CAS loop on sm_100a).
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// L = uint8: a cell row of 4 labels starts 2 pixels into a 4-pixel group (xb = 4 kx + 2), so it is
// read as two 16-bit halves, as the int64 kernel reads two 16-byte halves (2-byte aligned rows).
template <int CMAX, bool EXACT, bool FAST, bool GRAD, int TY, class LT>
__global__ void __launch_bounds__(kCeTile * TY, 512 / (kCeTile * TY))
weighted_ce_s4_kernel(const CeParams P) {
  using L = typename CeTypes<LT>::label;
  using T = typename CeTypes<LT>::logit;
  extern __shared__ __align__(16) float ce_smem[];
  constexpr int NT = kCeTile * TY;                    // threads = cells of the tile (16 wide, TY tall)
  constexpr int HH = kCeHalo * (TY + 1);              // low-res points under the tile
  const int C = EXACT ? CMAX : P.C;
  float* z_s = ce_smem;                               // [C][(TY+1)*17] low-res logits, clamp-to-edge halo
  float* a_s = z_s + (size_t)C * HH;                  // [C][4][NT] corner sums of every cell
  __shared__ double red[3][NT / 32];
  const int b = blockIdx.z;
  const int ly0 = blockIdx.y * TY, lx0 = blockIdx.x * kCeTile;
  const int64_t lplane = (int64_t)P.lh * P.lw;
  const T* zb = static_cast<const T*>(P.logits) + (int64_t)b * C * lplane;
  const int cy = threadIdx.x / kCeTile, cx = threadIdx.x % kCeTile;
  const int ky = ly0 + cy, kx = lx0 + cx;
  const bool active = ky < P.lh && kx < P.lw;
  const int xb = 4 * kx + 2, yb = 4 * ky + 2;
  const L* labp = static_cast<const L*>(P.labels) + (int64_t)b * P.H * P.W;
  const float* wp = P.weight ? P.weight + (int64_t)b * P.H * P.W : nullptr;

  // the cell's sixteen pixels first (all loads in flight before anything waits): labels as bytes
  // (255 = ignored / outside), weights (0 outside)
  unsigned lab4[4];
  float wv[4][4];
  auto lab_byte = [&](int64_t l) -> unsigned {
    return (l == P.ignore_index || l < 0 || l >= C) ? 255u : (unsigned)l;
  };
  longlong2 lraw[4][2];
  uint16_t lraw8[4][2];
  float2 wraw[4][2];
  {
    const bool right = xb + 3 < P.W;                  // false only in the last cell column (2 pixels)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int y = yb + i;
      const int64_t o = (int64_t)y * P.W + xb;
      const bool rowok = active && y < P.H;
      if constexpr (sizeof(L) == 1) {
        lraw8[i][0] = rowok ? *reinterpret_cast<const uint16_t*>(labp + o) : (uint16_t)0xffffu;
        lraw8[i][1] = rowok && right ? *reinterpret_cast<const uint16_t*>(labp + o + 2) : (uint16_t)0xffffu;
      } else {
        lraw[i][0] = rowok ? *reinterpret_cast<const longlong2*>(labp + o) : make_longlong2(-1, -1);
        lraw[i][1] = rowok && right ? *reinterpret_cast<const longlong2*>(labp + o + 2) : make_longlong2(-1, -1);
      }
      if (wp) {
        wraw[i][0] = rowok ? *reinterpret_cast<const float2*>(wp + o) : make_float2(0.f, 0.f);
        wraw[i][1] = rowok && right ? *reinterpret_cast<const float2*>(wp + o + 2) : make_float2(0.f, 0.f);
      } else {
        wraw[i][0] = wraw[i][1] = make_float2(1.f, 1.f);
      }
    }
  }
  {
    // low-res tile: thread -> halo points r = tid and r = NT + tid; 32-bit offsets inside one image
    const int lpl = P.lh * P.lw;
    const int r0 = threadIdx.x, r1 = NT + threadIdx.x;
    const int o0 = min(ly0 + r0 / kCeHalo, P.lh - 1) * P.lw + min(lx0 + r0 % kCeHalo, P.lw - 1);
    const int o1 = min(ly0 + r1 / kCeHalo, P.lh - 1) * P.lw + min(lx0 + r1 % kCeHalo, P.lw - 1);
    const bool two = r1 < HH;
    float t0[CMAX], t1[CMAX];
#pragma unroll
    for (int c = 0; c < CMAX; ++c) {
      t0[c] = c < C ? to_f32(zb[c * lpl + o0]) : 0.f;
      t1[c] = (c < C && two) ? to_f32(zb[c * lpl + o1]) : 0.f;
    }
#pragma unroll
    for (int c = 0; c < CMAX; ++c) {
      if (c < C) {
        z_s[c * HH + r0] = t0[c];
        if (two) z_s[c * HH + r1] = t1[c];
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if constexpr (sizeof(L) == 1)
      lab4[i] = lab_byte(lraw8[i][0] & 255u) | (lab_byte(lraw8[i][0] >> 8) << 8) |
                (lab_byte(lraw8[i][1] & 255u) << 16) | (lab_byte(lraw8[i][1] >> 8) << 24);
    else
      lab4[i] = lab_byte(lraw[i][0].x) | (lab_byte(lraw[i][0].y) << 8) | (lab_byte(lraw[i][1].x) << 16) |
                (lab_byte(lraw[i][1].y) << 24);
    wv[i][0] = wraw[i][0].x; wv[i][1] = wraw[i][0].y; wv[i][2] = wraw[i][1].x; wv[i][3] = wraw[i][1].y;
  }
  __syncthreads();

  float acc[CMAX][4];
#pragma unroll
  for (int c = 0; c < CMAX; ++c) acc[c][0] = acc[c][1] = acc[c][2] = acc[c][3] = 0.f;
  float loss_f = 0.f;
  int correct = 0, valid = 0;
  const float gscale = P.loss_weight / (float)((double)P.B * P.H * P.W);
  const float* zc = z_s + cy * kCeHalo + cx;

  // one column of pixels that interpolates between low-res columns (wx0, wx1), nrows rows with weights hy1[]
  auto column = [&](float wx0, float wx1, auto&& rowfn, int nrows) {
    float A0[CMAX], A1[CMAX], S0[CMAX], S1[CMAX];
#pragma unroll
    for (int c = 0; c < CMAX; ++c) {
      if (c < C) {
        const float* z = zc + c * HH;
        A0[c] = wx0 * z[0] + wx1 * z[1];
        A1[c] = wx0 * z[kCeHalo] + wx1 * z[kCeHalo + 1];
      } else {
        A0[c] = A1[c] = -INFINITY;
      }
      S0[c] = S1[c] = 0.f;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (i >= nrows) break;
      float hy0, hy1, w;
      unsigned lab;
      rowfn(i, hy0, hy1, lab, w);
      float v[CMAX];
      float m = -INFINITY;
      int arg = 0;
#pragma unroll
      for (int c = 0; c < CMAX; ++c) {
        v[c] = c < C ? hy0 * A0[c] + hy1 * A1[c] : -INFINITY;
        if (v[c] > m) { m = v[c]; arg = c; }                // first maximum wins
      }
      if (lab == 255u) continue;       // (a branch-free body was measured 12 % slower: register pressure)
      valid += 1;
      correct += arg == (int)lab ? 1 : 0;
      float sum = 0.f, vlab = 0.f;
#pragma unroll
      for (int c = 0; c < CMAX; ++c) {
        if (c < C) {
          vlab = c == (int)lab ? v[c] : vlab;
          v[c] = FAST ? ex2_approx((v[c] - m) * 1.4426950408889634f) : expf(v[c] - m);
          sum += v[c];
        }
      }
      if (P.class_weight) w *= P.class_weight[lab];
      loss_f += ((m + (FAST ? __logf(sum) : logf(sum))) - vlab) * w;
      if (GRAD) {
        const float k = gscale * w, kinv = FAST ? __fdividef(k, sum) : k / sum;
#pragma unroll
        for (int c = 0; c < CMAX; ++c) {
          if (c < C) {
            const float g = v[c] * kinv - (c == (int)lab ? k : 0.f);
            S0[c] += hy0 * g;
            S1[c] += hy1 * g;
          }
        }
      }
    }
    if (GRAD) {
#pragma unroll
      for (int c = 0; c < CMAX; ++c) {
        if (c < C) {
          acc[c][0] += wx0 * S0[c]; acc[c][1] += wx1 * S0[c];
          acc[c][2] += wx0 * S1[c]; acc[c][3] += wx1 * S1[c];
        }
      }
    }
  };

  if (active) {
    // the 4x4 pixels of the cell
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float wx1 = 0.125f + 0.25f * (float)j;
      column(1.f - wx1, wx1, [&](int i, float& hy0, float& hy1, unsigned& lab, float& w) {
        hy1 = 0.125f + 0.25f * (float)i; hy0 = 1.f - hy1;
        lab = (lab4[i] >> (8 * j)) & 255u; w = wv[i][j];
      }, 4);
    }
    // clamped border pixels: columns 0,1 belong to cell column 0 (l1 = 0), rows 0,1 to cell row 0
    auto load_px = [&](int y, int x, unsigned& lab, float& w) {
      if (y < P.H && x < P.W) {
        const int64_t o = (int64_t)y * P.W + x;
        lab = lab_byte(labp[o]); w = wp ? wp[o] : 1.f;
      } else {
        lab = 255u; w = 0.f;
      }
    };
    if (kx == 0) {
      for (int x = 0; x < 2; ++x)
        column(1.f, 0.f, [&](int i, float& hy0, float& hy1, unsigned& lab, float& w) {
          hy1 = 0.125f + 0.25f * (float)i; hy0 = 1.f - hy1;
          load_px(yb + i, x, lab, w);
        }, 4);
    }
    if (ky == 0) {
      for (int j = (kx == 0 ? -2 : 0); j < 4; ++j) {
        const int x = xb + j;
        const float wx1 = j < 0 ? 0.f : 0.125f + 0.25f * (float)j;
        column(1.f - wx1, wx1, [&](int i, float& hy0, float& hy1, unsigned& lab, float& w) {
          hy0 = 1.f; hy1 = 0.f;
          load_px(i, x, lab, w);
        }, 2);
      }
    }
  }

  // corner sums -> low-res gradient: point (py, px) collects corner 0 of cell (py, px), 1 of (py, px-1),
  // 2 of (py-1, px), 3 of (py-1, px-1); tile edges are shared with the neighbouring tiles (atomics);
  // indices past the last low-res row / column are the clamped taps and fold back onto it
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const double loss = warp_sum((double)loss_f), dcorrect = warp_sum((double)correct), dvalid = warp_sum((double)valid);
  if (lane == 0) { red[0][warp] = loss; red[1][warp] = dcorrect; red[2][warp] = dvalid; }
  if (GRAD) {
#pragma unroll
    for (int c = 0; c < CMAX; ++c) {
      if (c < C) {
        float* q = a_s + c * 4 * NT + threadIdx.x;
        q[0] = acc[c][0]; q[NT] = acc[c][1]; q[2 * NT] = acc[c][2]; q[3 * NT] = acc[c][3];
      }
    }
  }
  __syncthreads();
  if (GRAD) {
    float* gb = P.grad + (int64_t)b * C * lplane;
    const int lpl = P.lh * P.lw;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int r = h * NT + threadIdx.x;
      if (r >= HH) break;
      const int py = r / kCeHalo, px = r - py * kCeHalo;
      const int o = min(ly0 + py, P.lh - 1) * P.lw + min(lx0 + px, P.lw - 1);
      const bool p0 = py < TY && px < kCeTile, p1 = py < TY && px > 0, p2 = py > 0 && px < kCeTile,
                 p3 = py > 0 && px > 0;
      const int i0 = py * kCeTile + px;
#pragma unroll
      for (int c = 0; c < CMAX; ++c) {
        if (c < C) {
          const float* q = a_s + c * 4 * NT;
          float v = 0.f;
          if (p0) v += q[i0];
          if (p1) v += q[NT + i0 - 1];
          if (p2) v += q[2 * NT + i0 - kCeTile];
          if (p3) v += q[3 * NT + i0 - kCeTile - 1];
          if (v != 0.f) atomicAdd(gb + c * lpl + o, v);
        }
      }
    }
  }
  // statistics: block partials in fp64; only the first warp stays for the hand-off, the last block finalises
  if (warp != 0) return;
  if (lane < 3) {
    double v = 0.0;
#pragma unroll
    for (int wv2 = 0; wv2 < NT / 32; ++wv2) v += red[lane][wv2];
    if (v != 0.0) atomicAdd(&P.stats[lane], v);
    __threadfence();
  }
  __syncwarp();
  if (lane == 0) {
    const bool is_last = atomicAdd(reinterpret_cast<unsigned*>(P.stats + 3), 1u) == gridDim.x * gridDim.y * gridDim.z - 1;
    if (is_last) {
      __threadfence();
      const double s = *((volatile double*)&P.stats[0]);
      const double nc = *((volatile double*)&P.stats[1]), nv = *((volatile double*)&P.stats[2]);
      P.out[0] = P.loss_weight * (float)(s / ((double)P.B * P.H * P.W));
      const float eps = FLT_EPSILON;
      P.out[1] = ((float)nc + eps) * (float)(100.0 / (nv + (double)eps));
    }
  }
}

template <class L, class T>
static int weighted_ce(const T* logits, const L* labels, const float* weight, const float* class_weight,
                       int64_t B, int32_t C, int32_t lh, int32_t lw, int32_t H, int32_t W, int64_t ignore_index,
                       float loss_weight, float* grad_logits, double* stats, float* out2, void* stream) {
  // an empty batch reads nothing, so its (empty) tensors may have null data pointers
  if ((B > 0 && (!logits || !labels)) || !stats || !out2 || B < 0 || C < 1 || lh < 1 || lw < 1 || H < 1 || W < 1)
    return PFST_ERR_INVALID_ARG;
  if (C > pfst::kCeMaxC || B > 65535) return PFST_ERR_UNSUPPORTED;
  // the fused kernel covers integer up-sampling factors (H/4 logits -> H in every shipped config)
  if (H % lh != 0 || W % lw != 0 || H / lh != W / lw) return PFST_ERR_UNSUPPORTED;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  PFST_CUDA_TRY(cudaMemsetAsync(stats, 0, 4 * sizeof(double), s), "pfst_weighted_ce/memset");
  if (B == 0) {
    // the reference's mean over no pixels is NaN (all-ones bytes are a NaN) and accuracy.py returns 0
    // for an empty batch
    PFST_CUDA_TRY(cudaMemsetAsync(out2, 0xff, sizeof(float), s), "pfst_weighted_ce/empty-loss");
    PFST_CUDA_TRY(cudaMemsetAsync(out2 + 1, 0, sizeof(float), s), "pfst_weighted_ce/empty-acc");
    return PFST_OK;
  }
  if (grad_logits)
    PFST_CUDA_TRY(cudaMemsetAsync(grad_logits, 0, sizeof(float) * (size_t)B * C * lh * lw, s),
                  "pfst_weighted_ce/memset-grad");
  pfst::CeParams P{logits, labels, weight, class_weight, (int)B, C, lh, lw, H, W, H / lh,
                   ignore_index, loss_weight, grad_logits, stats, out2};
  // factor-4 up-sampling with few classes (every shipped config): cell-per-thread register kernel.
  // PFST_CE_V1=1 keeps the general kernel (A/B timing). The soft-max terms use ex2.approx / lg2.approx
  // (relative error ~2e-7 per term, inside the 1e-5 parity bound of the tests); PFST_CE_EXACT=1 selects
  // expf / logf / IEEE division instead
  static const bool force_v1 = getenv("PFST_CE_V1") != nullptr;
  static const bool fast = getenv("PFST_CE_EXACT") == nullptr;
  static const int ty = getenv("PFST_CE_TY") ? atoi(getenv("PFST_CE_TY")) : 8;
  // the factor-4 kernel reads a cell row of labels as two 16-byte (int64) or 2-byte (uint8) halves and
  // its weights as float2 (every row offset is even), so it needs maps aligned to that; other views,
  // such as a contiguous view at an odd storage offset, take the general kernel's scalar loads
  const bool rows_ok = reinterpret_cast<uintptr_t>(labels) % (sizeof(L) == 8 ? 16 : 2) == 0 &&
                       reinterpret_cast<uintptr_t>(weight) % 8 == 0;
  if (!force_v1 && C <= 8 && H == 4 * lh && W == 4 * lw && rows_ok) {
    const int TY = ty == 16 ? 16 : 8;
    const dim3 grid4((unsigned)((lw + pfst::kCeTile - 1) / pfst::kCeTile), (unsigned)((lh + TY - 1) / TY), (unsigned)B);
    if (grid4.y > 65535) return PFST_ERR_UNSUPPORTED;
    const size_t smem4 = ((size_t)C * pfst::kCeHalo * (TY + 1) + (size_t)C * 4 * pfst::kCeTile * TY) * sizeof(float);
    void (*k4)(const pfst::CeParams);
    using LT = pfst::CeIn<L, T>;
    const bool gr = grad_logits != nullptr;
#define PFST_CE_PICK2(CM, EX, F, G) (TY == 16 ? pfst::weighted_ce_s4_kernel<CM, EX, F, G, 16, LT> : pfst::weighted_ce_s4_kernel<CM, EX, F, G, 8, LT>)
#define PFST_CE_PICK(CM, EX)                                                       \
  (fast ? (gr ? PFST_CE_PICK2(CM, EX, true, true) : PFST_CE_PICK2(CM, EX, true, false)) \
        : (gr ? PFST_CE_PICK2(CM, EX, false, true) : PFST_CE_PICK2(CM, EX, false, false)))
    if (C == 6) k4 = PFST_CE_PICK(6, true);
    else if (C == 2) k4 = PFST_CE_PICK(2, true);
    else k4 = PFST_CE_PICK(8, false);
#undef PFST_CE_PICK
#undef PFST_CE_PICK2
    PFST_CUDA_TRY(cudaFuncSetAttribute(k4, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem4), "pfst_weighted_ce/attr4");
    k4<<<grid4, pfst::kCeTile * TY, smem4, s>>>(P);
    PFST_CHECK_LAUNCH("pfst_weighted_ce");
    return PFST_OK;
  }
  const dim3 grid((unsigned)((lw + pfst::kCeTile - 1) / pfst::kCeTile),
                  (unsigned)((lh + pfst::kCeTile - 1) / pfst::kCeTile), (unsigned)B);
  if (grid.y > 65535) return PFST_ERR_UNSUPPORTED;
  const size_t tile = (size_t)2 * C * pfst::kCeHalo * pfst::kCeHalo * sizeof(float);
  const size_t priv = grad_logits ? (size_t)C * 4 * pfst::kCeThreads * sizeof(float) : 0;
  const bool use_priv = tile + priv <= 100 * 1024;          // keeps two blocks per SM
  const size_t smem = tile + (use_priv ? priv : 0);
  if (smem > 200 * 1024) return PFST_ERR_UNSUPPORTED;
  using LT = pfst::CeIn<L, T>;
  auto k = C <= pfst::kCeRegC ? pfst::weighted_ce_kernel<true, true, LT>
                              : (use_priv ? pfst::weighted_ce_kernel<false, true, LT> : pfst::weighted_ce_kernel<false, false, LT>);
  PFST_CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "pfst_weighted_ce/attr");
  k<<<grid, pfst::kCeThreads, smem, s>>>(P);
  PFST_CHECK_LAUNCH("pfst_weighted_ce");
  return PFST_OK;
}

// ---- backward: the fp32 logits gradient times the upstream gradient, rounded once to the logits' dtype ----
// dst[i] = (T)(src[i] * *scale), an IEEE fp32 product (__fmul_rn: never fused into anything) and a
// round-to-nearest-even conversion: what autograd computes for `.float()` logits, where the upstream
// gradient multiplies the fp32 gradient and the cast's backward rounds the product. For T = float it
// is torch's `grad * grad_loss` bit for bit. `scale` stays on the device, so nothing waits for it.
__device__ __forceinline__ float from_f32(float v, float) { return v; }
__device__ __forceinline__ __half from_f32(float v, __half) { return __float2half_rn(v); }
__device__ __forceinline__ __nv_bfloat16 from_f32(float v, __nv_bfloat16) { return __float2bfloat16_rn(v); }

constexpr int kCastThreads = 256;

// VEC: src 16-byte and dst 4-element aligned, four elements per thread and step; the elements past the
// last whole group of four (and every element of an unaligned call) take the scalar loop
template <class T, bool VEC>
__global__ void __launch_bounds__(kCastThreads) scale_cast_kernel(const float* __restrict__ src,
                                                                  const float* __restrict__ scale, int64_t n,
                                                                  T* __restrict__ dst) {
  const float k = *scale;
  const int64_t stride = (int64_t)gridDim.x * kCastThreads;
  const int64_t t0 = (int64_t)blockIdx.x * kCastThreads + threadIdx.x;
  int64_t done = 0;
  if (VEC) {
    const int64_t n4 = n / 4;
    for (int64_t i = t0; i < n4; i += stride) {
      const float4 v = ldg_stream_f4(src + 4 * i);
      using V = typename std::conditional<sizeof(T) == 4, float4, uint2>::type;   // four elements of T
      alignas(sizeof(V)) const T r[4] = {from_f32(__fmul_rn(v.x, k), T{}), from_f32(__fmul_rn(v.y, k), T{}),
                                         from_f32(__fmul_rn(v.z, k), T{}), from_f32(__fmul_rn(v.w, k), T{})};
      *reinterpret_cast<V*>(dst + 4 * i) = *reinterpret_cast<const V*>(r);
    }
    done = 4 * n4;
  }
  for (int64_t i = done + t0; i < n; i += stride) dst[i] = from_f32(__fmul_rn(src[i], k), T{});
}

template <class T>
static int scale_cast(const float* src, const float* scale, int64_t n, T* dst, void* stream) {
  if (n < 0) return PFST_ERR_INVALID_ARG;
  if (n == 0) return PFST_OK;                     // an empty gradient: nothing is read, pointers may be null
  if (!src || !scale || !dst || !aligned4(src) || !aligned4(scale) ||
      reinterpret_cast<uintptr_t>(dst) % sizeof(T) != 0)
    return PFST_ERR_INVALID_ARG;
  const bool vec = aligned16(src) && reinterpret_cast<uintptr_t>(dst) % (4 * sizeof(T)) == 0;
  const int64_t work = vec ? (n + 3) / 4 : n;
  const unsigned blocks = (unsigned)std::min<int64_t>((work + kCastThreads - 1) / kCastThreads, 16 * kNumSMs);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (vec) scale_cast_kernel<T, true><<<blocks, kCastThreads, 0, s>>>(src, scale, n, dst);
  else scale_cast_kernel<T, false><<<blocks, kCastThreads, 0, s>>>(src, scale, n, dst);
  PFST_CHECK_LAUNCH("pfst_scale_cast");
  return PFST_OK;
}

}  // namespace pfst

extern "C" {

int pfst_weighted_ce_dt(const void* logits, int32_t logit_dtype, const void* labels, int32_t label_dtype,
                        const float* weight, const float* class_weight, int64_t B, int32_t C, int32_t lh, int32_t lw,
                        int32_t H, int32_t W, int64_t ignore_index, float loss_weight, float* grad_logits,
                        double* stats, float* out2, void* stream) {
  return pfst::with_float_dt(logit_dtype, [&](auto t) {
    return pfst::with_label_dt(label_dtype, [&](auto l) {
      return pfst::weighted_ce(static_cast<const decltype(t)*>(logits), static_cast<const decltype(l)*>(labels),
                               weight, class_weight, B, C, lh, lw, H, W, ignore_index, loss_weight, grad_logits,
                               stats, out2, stream);
    });
  });
}

int pfst_weighted_ce(const float* logits, const void* labels, int32_t label_dtype, const float* weight,
                     const float* class_weight, int64_t B, int32_t C, int32_t lh, int32_t lw, int32_t H, int32_t W,
                     int64_t ignore_index, float loss_weight, float* grad_logits, double* stats, float* out2,
                     void* stream) {
  return pfst_weighted_ce_dt(logits, PFST_DT_F32, labels, label_dtype, weight, class_weight, B, C, lh, lw, H, W,
                             ignore_index, loss_weight, grad_logits, stats, out2, stream);
}

int pfst_scale_cast(const float* src, const float* scale, int64_t n, void* dst, int32_t dst_dtype, void* stream) {
  return pfst::with_float_dt(dst_dtype, [&](auto t) {
    return pfst::scale_cast(src, scale, n, static_cast<decltype(t)*>(dst), stream);
  });
}

}  // extern "C"
