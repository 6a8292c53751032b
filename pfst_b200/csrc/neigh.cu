// L2 (+ its backward) — dilated 3x3 neighbourhood dot products of decoder features.
//
// Reference: PFGSTLoss.get_sim_feat, rsiseg/models/losses/pfgst_loss.py:181-201
//   unf = nn.Unfold(k=3, dilation=d, padding=d)(feats)      # materialises 9x the tensor
//   sim = F.cosine_similarity(unf, feats.unsqueeze(4), dim=1)
// (>90 % of the loss time in the reference: 604 MB of im2col per tensor, four
// full passes, col2im in backward.) Here the feature tensor is read ONCE:
//
//   forward  (pfst_neigh_dots): per pixel n the squared norm and the four
//            "forward" dot products x_n . x_{n+delta}, delta in {(0,+d), (+d,-d),
//            (+d,0), (+d,+d)}. cos(n, n+delta_k) for all nine taps follows from
//            these five maps by symmetry (cos(n,m) = cos(m,n)), so the loss kernel
//            gathers them; out-of-image taps are the unfold's zero padding.
//   backward (pfst_neigh_grad): grad_x[n,c] = sum_k coef[n,k] * x[n+delta_k, c],
//            the gather form of d(sum cos)/dx with per-pixel coefficients computed
//            by the loss backward kernel (no atomics, no col2im).
//
// Both are HBM-bound: 4*D bytes per pixel read (+ 4*D written in backward).
// Blackwell path: (W,H,D,B) TMA tensor map, 32x16-pixel tiles with the dilation
// halo (16-byte aligned box start), 8-channel boxes, hardware zero fill for the padding, 4-stage
// full/empty mbarrier ring, one producer warp + four consumer warps; each
// consumer thread owns a 1x4 pixel strip and reads shared memory as conflict-free
// 128-bit rows. Channel ranges are split across CTAs (ksplit) so that one
// resident wave covers the GPU; partial maps are summed by the consumer kernel in a
// fixed order (deterministic, no atomics).
// Shapes TMA cannot describe (W % 4 != 0, e.g. SeasonNet's 15x15 maps) take a
// plain coalesced kernel with the same outputs.
#include "common.cuh"
#include "tma.cuh"

namespace pfst {

constexpr int kNbTW = 32;          // tile width (pixels)
constexpr int kNbTH = 16;          // tile height
constexpr int kNbCH = 8;           // channels per TMA box / pipeline stage
constexpr int kNbStages = 4;
constexpr int kNbConsumers = 128;  // 4 warps, one 1x4 strip per thread
constexpr int kNbThreads = kNbConsumers + 32;

// TMA requires the box to start on a 16-byte boundary in the innermost dimension
// (x_start % 4 == 0 for fp32), so the left halo is always kNbHL = 4 columns wide
// (>= every supported dilation) and the box is 32 + 4 + 4 = 40 columns.
constexpr int kNbHL = 4;
template <int DIL>
struct NbGeom {
  static_assert(DIL <= kNbHL, "dilation larger than the aligned halo");
  static constexpr int RS = kNbTW + 2 * kNbHL;                // smem row stride = box width (40)
  static constexpr int FWD_ROWS = kNbTH + DIL;               // rows y0 .. y0+TH-1+d
  static constexpr int BWD_ROWS = kNbTH + 2 * DIL;           // rows y0-d .. y0+TH-1+d
};

struct NeighMaps {
  CUtensorMap m[2];
};

struct NbTile {
  int split, t, b, y0, x0, c_begin, c_end;
};

__device__ __forceinline__ NbTile nb_decode(int n_units, int B, int h, int w, int D, int ksplit) {
  // blockIdx.x -> (unit = tensor or 0, b, tile_y, tile_x, split)
  const int tiles_x = (w + kNbTW - 1) / kNbTW, tiles_y = (h + kNbTH - 1) / kNbTH;
  int idx = blockIdx.x;
  NbTile o;
  o.split = idx % ksplit; idx /= ksplit;
  o.x0 = (idx % tiles_x) * kNbTW; idx /= tiles_x;
  o.y0 = (idx % tiles_y) * kNbTH; idx /= tiles_y;
  o.b = idx % B;
  o.t = idx / B;
  const int chunks = (D + kNbCH - 1) / kNbCH;
  o.c_begin = (int)((int64_t)o.split * chunks / ksplit);
  o.c_end = (int)((int64_t)(o.split + 1) * chunks / ksplit);
  (void)n_units;
  return o;
}

__device__ __forceinline__ void nb_init_barriers(uint64_t* full_bar, uint64_t* empty_bar) {
  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < kNbStages; ++s) {
      mbar_init(&full_bar[s], 1);                  // producer's arrive.expect_tx
      mbar_init(&empty_bar[s], kNbConsumers / 32); // one arrive per consumer warp
    }
    mbar_fence_init();
  }
  __syncthreads();
}

template <int ROWS, int RS>
__device__ __forceinline__ void nb_produce(const CUtensorMap* map, float* stage_buf, uint64_t* full_bar,
                                           uint64_t* empty_bar, const NbTile& tl, int x_start,
                                           int y_start) {
  constexpr int kStageFloats = kNbCH * ROWS * RS;
  constexpr uint32_t kStageBytes = kStageFloats * sizeof(float);
  tma_prefetch_desc(map);
  int it = 0;
  for (int c = tl.c_begin; c < tl.c_end; ++c, ++it) {
    const int s = it % kNbStages;
    const uint32_t ph = (uint32_t)(it / kNbStages) & 1u;
    if (it >= kNbStages) mbar_wait(&empty_bar[s], ph ^ 1u);
    mbar_arrive_expect_tx(&full_bar[s], kStageBytes);
    tma_load_4d(stage_buf + (size_t)s * kStageFloats, map, &full_bar[s], x_start, y_start, c * kNbCH,
                tl.b);
  }
}

// ---------------------------------------------------------------- forward (TMA)
template <int DIL>
__global__ void __launch_bounds__(kNbThreads)
neigh_dots_tma_kernel(const __grid_constant__ NeighMaps maps, int n_tensors, int B, int D, int h, int w,
                      int ksplit, int slot0, int n_slots, float* __restrict__ dots) {
  using G = NbGeom<DIL>;
  constexpr int kStageFloats = kNbCH * G::FWD_ROWS * G::RS;
  extern __shared__ __align__(128) unsigned char nb_smem[];
  float* stage_buf = reinterpret_cast<float*>(nb_smem);
  __shared__ uint64_t full_bar[kNbStages], empty_bar[kNbStages];
  const NbTile tl = nb_decode(n_tensors, B, h, w, D, ksplit);
  nb_init_barriers(full_bar, empty_bar);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == kNbConsumers / 32) {
    if (lane == 0)
      nb_produce<G::FWD_ROWS, G::RS>(&maps.m[tl.t], stage_buf, full_bar, empty_bar, tl, tl.x0 - kNbHL, tl.y0);
    return;
  }
  // Each lane owns a CHAIN of four 1x4 pixel strips, rows r0 + k*DIL (k = 0..3): the row read
  // as "row y+d" of strip k is "row y" of strip k+1, so a channel costs 14 128-bit shared
  // loads per 16 pixels instead of 20 (the kernel is shared-memory-bandwidth bound). A warp
  // covers the whole 32x16 tile of one channel (8 lanes per row: conflict-free); the four
  // consumer warps take the stage's channels round-robin.
  const int lx = (lane & 7) * 4, chain = lane >> 3;
  const int r0 = (chain / DIL) * 4 * DIL + chain % DIL;
  float acc[5][4][4];
#pragma unroll
  for (int m = 0; m < 5; ++m)
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[m][k][i] = 0.f;

  int it = 0;
  for (int c = tl.c_begin; c < tl.c_end; ++c, ++it) {
    const int s = it % kNbStages;
    mbar_wait(&full_bar[s], (uint32_t)(it / kNbStages) & 1u);
    const float* buf = stage_buf + (size_t)s * kStageFloats + r0 * G::RS + lx;
#pragma unroll
    for (int cc = 0; cc < kNbCH / (kNbConsumers / 32); ++cc) {
      const int ch = warp + cc * (kNbConsumers / 32);
      // smem column of image column x is (x - x0 + 4); this strip's pixels sit at lx+4+i
      const float* row = buf + ch * G::FWD_ROWS * G::RS;
      float P[12], Q[12];                                  // P[j] = col lx+j of the current row
#pragma unroll
      for (int v = 1; v < 3; ++v) {
        const float4 f = *reinterpret_cast<const float4*>(row + 4 * v);
        P[4 * v] = f.x; P[4 * v + 1] = f.y; P[4 * v + 2] = f.z; P[4 * v + 3] = f.w;
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        row += DIL * G::RS;
#pragma unroll
        for (int v = 0; v < 3; ++v) {
          const float4 f = *reinterpret_cast<const float4*>(row + 4 * v);
          Q[4 * v] = f.x; Q[4 * v + 1] = f.y; Q[4 * v + 2] = f.z; Q[4 * v + 3] = f.w;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float a = P[4 + i];
          acc[0][k][i] = fmaf(a, a, acc[0][k][i]);
          acc[1][k][i] = fmaf(a, P[4 + i + DIL], acc[1][k][i]);      // ( 0, +d)
          acc[2][k][i] = fmaf(a, Q[4 + i - DIL], acc[2][k][i]);      // (+d, -d)
          acc[3][k][i] = fmaf(a, Q[4 + i], acc[3][k][i]);            // (+d,  0)
          acc[4][k][i] = fmaf(a, Q[4 + i + DIL], acc[4][k][i]);      // (+d, +d)
        }
#pragma unroll
        for (int j = 4; j < 12; ++j) P[j] = Q[j];
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty_bar[s]);
  }
  // The four warps hold partial sums over disjoint channels: merge through shared memory
  // (the stage ring is idle now) in a fixed order, then one warp-row-coalesced store per map.
  asm volatile("bar.sync 1, %0;" ::"n"(kNbConsumers) : "memory");
  float* red = stage_buf;                                   // [4 warps][5*16 values][32 lanes]
  if (warp > 0) {
#pragma unroll
    for (int m = 0; m < 5; ++m)
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int i = 0; i < 4; ++i) red[((warp * 80) + (m * 16 + k * 4 + i)) * 32 + lane] = acc[m][k][i];
  }
  asm volatile("bar.sync 1, %0;" ::"n"(kNbConsumers) : "memory");
  if (warp == 0) {
    const int x = tl.x0 + lx;
    float* out = dots + ((((int64_t)tl.split * n_slots + slot0 + tl.t) * B + tl.b) * 5) * h * w;
#pragma unroll
    for (int m = 0; m < 5; ++m)
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float o[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int e = m * 16 + k * 4 + i;
          o[i] = ((acc[m][k][i] + red[(80 + e) * 32 + lane]) + red[(160 + e) * 32 + lane]) + red[(240 + e) * 32 + lane];
        }
        const int y = tl.y0 + r0 + k * DIL;
        if (y < h && x < w)   // w % 4 == 0: a strip is entirely inside or outside
          *reinterpret_cast<float4*>(out + ((int64_t)m * h + y) * w + x) = make_float4(o[0], o[1], o[2], o[3]);
      }
  }
}

// --------------------------------------------------------------- backward (TMA)
// PROTO: the prototype-distance gradient (P3 backward, proto.cu) is added in the same pass,
//   grad[n,c] += g * (x[n,c] - mu[y_n,c]) / (dist_n * n_valid),
// so x_src is read once and grad_x written once for both losses.
template <class L>
struct ProtoBwdT {
  const L* labels;         // (B, lab_h, lab_w), int64 or uint8
  int lab_h, lab_w;
  const float* mu;         // (C, D)
  const uint8_t* seen;     // (C) or null
  int C;
  const float* dist;       // (B, h, w) from pfst_proto_dist_fwd
  const double* acc;       // acc[1] = number of valid pixels
  const float* grad_loss;  // device scalar
  int mu_stride;           // shared-memory row stride of the staged prototypes
};
using ProtoBwd = ProtoBwdT<int64_t>;

template <int DIL, bool PROTO, class L = int64_t>
__global__ void __launch_bounds__(kNbThreads)
neigh_grad_tma_kernel(const __grid_constant__ NeighMaps maps, const float* __restrict__ coef, int B, int D,
                      int h, int w, int ksplit, float* __restrict__ grad, const ProtoBwdT<L> pb) {
  using G = NbGeom<DIL>;
  constexpr int kStageFloats = kNbCH * G::BWD_ROWS * G::RS;
  extern __shared__ __align__(128) unsigned char nb_smem[];
  float* stage_buf = reinterpret_cast<float*>(nb_smem);
  float* mu_s = stage_buf + (size_t)kNbStages * kStageFloats;       // [C][mu_stride]  (PROTO only)
  __shared__ uint64_t full_bar[kNbStages], empty_bar[kNbStages];
  const NbTile tl = nb_decode(1, B, h, w, D, ksplit);
  if (PROTO) {   // this CTA's channel slice of the prototypes
    const int ch0 = tl.c_begin * kNbCH, nch = min(D, tl.c_end * kNbCH) - ch0;
    for (int i = threadIdx.x; i < pb.C * nch; i += kNbThreads) {
      const int c = i / nch, j = i - c * nch;
      mu_s[c * pb.mu_stride + j] = pb.mu[(int64_t)c * D + ch0 + j];
    }
  }
  nb_init_barriers(full_bar, empty_bar);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == kNbConsumers / 32) {
    if (lane == 0)
      nb_produce<G::BWD_ROWS, G::RS>(&maps.m[0], stage_buf, full_bar, empty_bar, tl, tl.x0 - kNbHL,
                                     tl.y0 - DIL);
    return;
  }
  // Each lane owns two 1x4 output strips, rows r and r+DIL: their 3x3 dilated windows share
  // two of the four input rows, so a channel costs 12 128-bit shared loads per 8 pixels
  // instead of 18 (shared-memory-bandwidth bound). Two warps cover the 32x16 tile of one
  // channel; warps {0,1} take the even channels of a stage, warps {2,3} the odd ones.
  const int lx = (lane & 7) * 4;
  const int pair = (warp & 1) * 4 + (lane >> 3);                 // 0..7
  const int r = (pair / DIL) * 2 * DIL + pair % DIL;             // first output row (tile-relative)
  const int half = warp >> 1;
  const int x = tl.x0 + lx;
  const int64_t plane = (int64_t)h * w;
  bool live[2];
  float K[2][9][4];
  // P3 backward: per-pixel coefficient and prototype row of the strips' pixels
  float pcoef[2][4];
  int prow[2][4];
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    const int y = tl.y0 + r + q * DIL;
    live[q] = (y < h) && (x < w);   // w % 4 == 0: a strip is entirely inside or outside
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (live[q]) v = *reinterpret_cast<const float4*>(coef + (((int64_t)tl.b * 9 + k) * h + y) * w + x);
      K[q][k][0] = v.x; K[q][k][1] = v.y; K[q][k][2] = v.z; K[q][k][3] = v.w;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) { pcoef[q][i] = 0.f; prow[q][i] = 0; }
    if (PROTO && live[q]) {
      const float g = pb.grad_loss[0];
      const float nvalid = (float)pb.acc[1];
      const float sh = (float)pb.lab_h / (float)h, sw = (float)pb.lab_w / (float)w;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int pp = y * w + x + i;
        uint8_t l = pr_label(pb.labels, nullptr, 0.f, tl.b, pp, w, pb.lab_h, pb.lab_w, sh, sw, pb.C);
        if (l != 255 && pb.seen && !pb.seen[l]) l = 255;
        const float dn = pb.dist[(int64_t)tl.b * plane + pp];
        pcoef[q][i] = (l != 255 && dn > 0.f) ? g / (dn * nvalid) : 0.f;   // torch.norm backward: 0 at 0
        prow[q][i] = (l != 255 ? (int)l : 0) * pb.mu_stride;
      }
    }
  }
  float* gout = grad + (((int64_t)tl.b * D) * h + tl.y0 + r) * w + x;

  int it = 0;
  for (int c = tl.c_begin; c < tl.c_end; ++c, ++it) {
    const int s = it % kNbStages;
    mbar_wait(&full_bar[s], (uint32_t)(it / kNbStages) & 1u);
    // smem row j holds image row y0 - DIL + j: output row r reads smem rows r, r+DIL, r+2*DIL
    const float* buf = stage_buf + (size_t)s * kStageFloats + r * G::RS + lx;
#pragma unroll
    for (int cc = 0; cc < kNbCH / 2; ++cc) {
      const int ch = cc * 2 + half;
      const float* row = buf + ch * G::BWD_ROWS * G::RS;
      float o[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
      float ctr[2][4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {                         // the four input rows of the two windows
        float R[12];                                        // R[e] = col lx+e  (pixel i at 4+i)
#pragma unroll
        for (int v = 0; v < 3; ++v) {
          const float4 f = *reinterpret_cast<const float4*>(row + j * DIL * G::RS + 4 * v);
          R[4 * v] = f.x; R[4 * v + 1] = f.y; R[4 * v + 2] = f.z; R[4 * v + 3] = f.w;
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
          const int ky = j - q;                             // tap row of window q that reads input row j
          if (ky < 0 || ky > 2) continue;
          if (ky == 1) {
#pragma unroll
            for (int i = 0; i < 4; ++i) ctr[q][i] = R[4 + i];
          }
#pragma unroll
          for (int kx = 0; kx < 3; ++kx)
#pragma unroll
            for (int i = 0; i < 4; ++i) o[q][i] = fmaf(K[q][ky * 3 + kx][i], R[4 + i + (kx - 1) * DIL], o[q][i]);
        }
      }
      const int cg = c * kNbCH + ch;
      if (PROTO) {
        const int cl = (c - tl.c_begin) * kNbCH + ch;
#pragma unroll
        for (int q = 0; q < 2; ++q)
#pragma unroll
          for (int i = 0; i < 4; ++i) o[q][i] = fmaf(pcoef[q][i], ctr[q][i] - mu_s[prow[q][i] + cl], o[q][i]);
      }
      if (cg < D) {
#pragma unroll
        for (int q = 0; q < 2; ++q)
          if (live[q])
            __stcs(reinterpret_cast<float4*>(gout + cg * plane + (int64_t)q * DIL * w),
                   make_float4(o[q][0], o[q][1], o[q][2], o[q][3]));
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty_bar[s]);
  }
}

// ------------------------------------------------- generic (any shape) kernels
__global__ void __launch_bounds__(128)
neigh_dots_generic_kernel(const float* __restrict__ xa, const float* __restrict__ xb, int n_tensors, int B,
                          int D, int h, int w, int dil, int ksplit, int slot0, int n_slots,
                          float* __restrict__ dots) {
  const int64_t plane = (int64_t)h * w;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  int z = blockIdx.y;
  const int split = z % ksplit; z /= ksplit;
  const int b = z % B, t = z / B;
  if (p >= plane) return;
  const int y = p / w, x = p - y * w;
  const int c_begin = (int)((int64_t)split * D / ksplit), c_end = (int)((int64_t)(split + 1) * D / ksplit);
  const float* src = (t == 0 ? xa : xb) + ((int64_t)b * D) * plane + p;
  const bool in1 = x + dil < w, inr = y + dil < h;
  const bool in2 = inr && x - dil >= 0, in4 = inr && x + dil < w;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, a4 = 0.f;
  for (int c = c_begin; c < c_end; ++c) {
    const float* q = src + (int64_t)c * plane;
    const float v = __ldg(q);
    a0 = fmaf(v, v, a0);
    if (in1) a1 = fmaf(v, __ldg(q + dil), a1);
    if (in2) a2 = fmaf(v, __ldg(q + (int64_t)dil * w - dil), a2);
    if (inr) a3 = fmaf(v, __ldg(q + (int64_t)dil * w), a3);
    if (in4) a4 = fmaf(v, __ldg(q + (int64_t)dil * w + dil), a4);
  }
  float* out = dots + ((((int64_t)split * n_slots + slot0 + t) * B + b) * 5) * plane + p;
  out[0] = a0; out[plane] = a1; out[2 * plane] = a2; out[3 * plane] = a3; out[4 * plane] = a4;
}

__global__ void __launch_bounds__(128)
neigh_grad_generic_kernel(const float* __restrict__ x, const float* __restrict__ coef, int B, int D, int h,
                          int w, int dil, float* __restrict__ grad) {
  const int64_t plane = (int64_t)h * w;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  const int b = blockIdx.y;
  if (p >= plane) return;
  const int y = p / w, xx = p - y * w;
  float K[9];
  int off[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    const int yy = y + (k / 3 - 1) * dil, xk = xx + (k % 3 - 1) * dil;
    const bool in = yy >= 0 && yy < h && xk >= 0 && xk < w;
    K[k] = in ? coef[((int64_t)b * 9 + k) * plane + p] : 0.f;
    off[k] = in ? (yy - y) * w + (xk - xx) : 0;
  }
  const float* src = x + ((int64_t)b * D) * plane + p;
  float* dst = grad + ((int64_t)b * D) * plane + p;
  for (int c = blockIdx.z; c < D; c += gridDim.z) {
    const float* q = src + (int64_t)c * plane;
    float o = 0.f;
#pragma unroll
    for (int k = 0; k < 9; ++k) o = fmaf(K[k], __ldg(q + off[k]), o);
    dst[(int64_t)c * plane] = o;
  }
}

// ------------------------------------------- small planes (any width): bulk-copy kernels
// Feature maps whose width is not a multiple of four (SeasonNet: 15x15) cannot be described by
// the TMA tensor map above, but a chunk of channels of one image, x[b, c:c+16], is ONE contiguous
// block of 16*h*w floats: it streams into shared memory with 1-D bulk async copies (mbarrier ring,
// one producer lane) and every thread owns one or two pixels, reading its taps from shared memory
// (consecutive threads -> consecutive addresses: conflict-free). HBM traffic = the tensor, once.
constexpr int kSpCH = 16;            // channels per stage
constexpr int kSpStages = 4;
constexpr int kSpConsumers = 256;
constexpr int kSpThreads = kSpConsumers + 32;
constexpr int kSpMaxHW = 400;        // 4 stages x 16 channels x 400 px x 4 B = 102 KB (two blocks per SM)
constexpr int kSpPix = (kSpMaxHW + kSpConsumers - 1) / kSpConsumers;   // pixels per thread (2)

__device__ __forceinline__ void sp_init(uint64_t* full_bar, uint64_t* empty_bar) {
  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < kSpStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], kSpConsumers / 32);
    }
    mbar_fence_init();
  }
  __syncthreads();
}

__device__ __forceinline__ void sp_produce(const float* src, int hw, int c_begin, int c_end, float* stage_buf,
                                           uint64_t* full_bar, uint64_t* empty_bar) {
  int it = 0;
  for (int c = c_begin; c < c_end; c += kSpCH, ++it) {
    const int s = it % kSpStages, n = min(kSpCH, c_end - c);
    if (it >= kSpStages) mbar_wait(&empty_bar[s], ((uint32_t)(it / kSpStages) & 1u) ^ 1u);
    const uint32_t bytes = (uint32_t)n * hw * sizeof(float);
    mbar_arrive_expect_tx(&full_bar[s], bytes);
    bulk_load_1d(stage_buf + (size_t)s * kSpCH * hw, src + (int64_t)c * hw, bytes, &full_bar[s]);
  }
}

__global__ void __launch_bounds__(kSpThreads)
neigh_dots_plane_kernel(const float* __restrict__ xa, const float* __restrict__ xb, int B, int D, int h, int w,
                        int dil, int ksplit, int slot0, int n_slots, float* __restrict__ dots) {
  extern __shared__ __align__(128) unsigned char sp_smem[];
  float* stage_buf = reinterpret_cast<float*>(sp_smem);
  __shared__ uint64_t full_bar[kSpStages], empty_bar[kSpStages];
  const int hw = h * w;
  int z = blockIdx.x;
  const int split = z % ksplit; z /= ksplit;
  const int b = z % B, t = z / B;
  const int c_begin = (int)((int64_t)split * D / ksplit), c_end = (int)((int64_t)(split + 1) * D / ksplit);
  const float* src = (t == 0 ? xa : xb) + (int64_t)b * D * hw;
  sp_init(full_bar, empty_bar);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == kSpConsumers / 32) {
    if (lane == 0) sp_produce(src, hw, c_begin, c_end, stage_buf, full_bar, empty_bar);
    return;
  }
  int off[kSpPix][4];
  bool ok[kSpPix][4], live[kSpPix];
  float acc[kSpPix][5];
#pragma unroll
  for (int q = 0; q < kSpPix; ++q) {
    const int p = threadIdx.x + q * kSpConsumers;
    live[q] = p < hw;
    const int y = p / w, x = p - y * w;
    ok[q][0] = live[q] && x + dil < w;                       // ( 0, +d)
    ok[q][1] = live[q] && y + dil < h && x - dil >= 0;       // (+d, -d)
    ok[q][2] = live[q] && y + dil < h;                       // (+d,  0)
    ok[q][3] = live[q] && y + dil < h && x + dil < w;        // (+d, +d)
    off[q][0] = dil; off[q][1] = dil * w - dil; off[q][2] = dil * w; off[q][3] = dil * w + dil;
#pragma unroll
    for (int k = 0; k < 5; ++k) acc[q][k] = 0.f;
  }
  int it = 0;
  for (int c = c_begin; c < c_end; c += kSpCH, ++it) {
    const int s = it % kSpStages, n = min(kSpCH, c_end - c);
    mbar_wait(&full_bar[s], (uint32_t)(it / kSpStages) & 1u);
    const float* buf = stage_buf + (size_t)s * kSpCH * hw;
#pragma unroll
    for (int q = 0; q < kSpPix; ++q) {
      if (!live[q]) continue;
      const float* pq = buf + threadIdx.x + q * kSpConsumers;
      for (int ch = 0; ch < n; ++ch) {
        const float* r = pq + ch * hw;
        const float v = r[0];
        acc[q][0] = fmaf(v, v, acc[q][0]);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (ok[q][k]) acc[q][k + 1] = fmaf(v, r[off[q][k]], acc[q][k + 1]);
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty_bar[s]);
  }
  float* out = dots + ((((int64_t)split * n_slots + slot0 + t) * B + b) * 5) * hw;
#pragma unroll
  for (int q = 0; q < kSpPix; ++q)
    if (live[q])
#pragma unroll
      for (int k = 0; k < 5; ++k) out[(int64_t)k * hw + threadIdx.x + q * kSpConsumers] = acc[q][k];
}

// grad[b,c,p] = sum_k coef[b,k,p] * x[b,c,p+delta_k]  (+ the prototype-distance term, as ProtoBwd above)
template <bool PROTO, class L = int64_t>
__global__ void __launch_bounds__(kSpThreads)
neigh_grad_plane_kernel(const float* __restrict__ x, const float* __restrict__ coef, int B, int D, int h, int w,
                        int dil, int ksplit, float* __restrict__ grad, const ProtoBwdT<L> pb) {
  extern __shared__ __align__(128) unsigned char sp_smem[];
  float* stage_buf = reinterpret_cast<float*>(sp_smem);
  __shared__ uint64_t full_bar[kSpStages], empty_bar[kSpStages];
  const int hw = h * w;
  float* mu_s = stage_buf + (size_t)kSpStages * kSpCH * hw;     // [C][mu_stride]  (PROTO only)
  const int split = blockIdx.x % ksplit, b = blockIdx.x / ksplit;
  const int c_begin = (int)((int64_t)split * D / ksplit), c_end = (int)((int64_t)(split + 1) * D / ksplit);
  if (PROTO) {
    const int nch = c_end - c_begin;
    for (int i = threadIdx.x; i < pb.C * nch; i += kSpThreads) {
      const int c = i / nch, j = i - c * nch;
      mu_s[c * pb.mu_stride + j] = pb.mu[(int64_t)c * D + c_begin + j];
    }
  }
  sp_init(full_bar, empty_bar);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == kSpConsumers / 32) {
    if (lane == 0) sp_produce(x + (int64_t)b * D * hw, hw, c_begin, c_end, stage_buf, full_bar, empty_bar);
    return;
  }
  float K[kSpPix][9], pcoef[kSpPix];
  int off[kSpPix][9], prow[kSpPix];
  bool live[kSpPix];
#pragma unroll
  for (int q = 0; q < kSpPix; ++q) {
    const int p = threadIdx.x + q * kSpConsumers;
    live[q] = p < hw;
    const int y = p / w, xx = p - y * w;
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      const int yy = y + (k / 3 - 1) * dil, xk = xx + (k % 3 - 1) * dil;
      const bool in = live[q] && yy >= 0 && yy < h && xk >= 0 && xk < w;
      K[q][k] = in ? coef[((int64_t)b * 9 + k) * hw + p] : 0.f;
      off[q][k] = in ? (yy - y) * w + (xk - xx) : 0;
    }
    pcoef[q] = 0.f;
    prow[q] = 0;
    if (PROTO && live[q]) {
      const float sh = (float)pb.lab_h / (float)h, sw = (float)pb.lab_w / (float)w;
      uint8_t l = pr_label(pb.labels, nullptr, 0.f, b, p, w, pb.lab_h, pb.lab_w, sh, sw, pb.C);
      if (l != 255 && pb.seen && !pb.seen[l]) l = 255;
      const float dn = pb.dist[(int64_t)b * hw + p];
      pcoef[q] = (l != 255 && dn > 0.f) ? pb.grad_loss[0] / (dn * (float)pb.acc[1]) : 0.f;
      prow[q] = (l != 255 ? (int)l : 0) * pb.mu_stride;
    }
  }
  float* gout = grad + (int64_t)b * D * hw;
  int it = 0;
  for (int c = c_begin; c < c_end; c += kSpCH, ++it) {
    const int s = it % kSpStages, n = min(kSpCH, c_end - c);
    mbar_wait(&full_bar[s], (uint32_t)(it / kSpStages) & 1u);
    const float* buf = stage_buf + (size_t)s * kSpCH * hw;
#pragma unroll
    for (int q = 0; q < kSpPix; ++q) {
      if (!live[q]) continue;
      const int p = threadIdx.x + q * kSpConsumers;
      for (int ch = 0; ch < n; ++ch) {
        const float* r = buf + ch * hw + p;
        float o = 0.f;
#pragma unroll
        for (int k = 0; k < 9; ++k) o = fmaf(K[q][k], r[off[q][k]], o);
        if (PROTO) o = fmaf(pcoef[q], r[0] - mu_s[prow[q] + (c - c_begin) + ch], o);
        gout[(int64_t)(c + ch) * hw + p] = o;
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty_bar[s]);
  }
}

// planes the bulk-copy kernels cover: small, 16-byte aligned channel chunks for every split
static bool sp_ok(const void* p0, const void* p1, int D, int h, int w, int ks) {
  const int hw = h * w;
  return hw <= kSpMaxHW && aligned16(p0) && (!p1 || aligned16(p1)) && D % (4 * ks) == 0;
}

static bool nb_tma_ok(const void* p0, const void* p1, int w, int dil) {
  return (w % 4 == 0) && aligned16(p0) && (!p1 || aligned16(p1)) && (dil == 1 || dil == 2 || dil == 4) &&
         get_encode_tiled() != nullptr;
}

static int nb_splits(int64_t units, int h, int w, int D) {
  const int64_t tiles = (int64_t)((w + kNbTW - 1) / kNbTW) * ((h + kNbTH - 1) / kNbTH);
  const int64_t items = units * tiles;
  const int chunks = (D + kNbCH - 1) / kNbCH;
  const int64_t slots = (int64_t)kNumSMs * 2;
  int ks = 1;
  while (ks < 8 && ks * 2 <= chunks && items * ks * 2 <= slots) ks *= 2;
  return ks;
}

template <int DIL>
static int launch_dots_tma(const float* xa, const float* xb, int T, int B, int D, int h, int w, int ks,
                           int slot0, int n_slots, float* dots, cudaStream_t s) {
  using G = NbGeom<DIL>;
  NeighMaps maps;
  if (!make_nchw_tensor_map(&maps.m[0], xa, B, D, h, w, G::RS, G::FWD_ROWS, kNbCH)) return PFST_ERR_CUDA;
  if (!make_nchw_tensor_map(&maps.m[1], xb ? xb : xa, B, D, h, w, G::RS, G::FWD_ROWS, kNbCH)) return PFST_ERR_CUDA;
  const size_t smem = (size_t)kNbStages * kNbCH * G::FWD_ROWS * G::RS * sizeof(float);
  auto k = neigh_dots_tma_kernel<DIL>;
  PFST_CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "pfst_neigh_dots/attr");
  const int64_t tiles = (int64_t)((w + kNbTW - 1) / kNbTW) * ((h + kNbTH - 1) / kNbTH);
  const int64_t grid = (int64_t)T * B * tiles * ks;
  k<<<(unsigned)grid, kNbThreads, smem, s>>>(maps, T, B, D, h, w, ks, slot0, n_slots, dots);
  PFST_CHECK_LAUNCH("pfst_neigh_dots");
  return PFST_OK;
}

// bytes of shared memory the fused prototype slice needs (0 = prototypes do not fit: unfused path)
static size_t nb_proto_smem(int C, int D, int ks, int* stride) {
  const int chunks = (D + kNbCH - 1) / kNbCH;
  const int nch = ((chunks + ks - 1) / ks) * kNbCH;
  *stride = nch + 1;                                   // +1: bank skew between prototype rows
  return (size_t)C * (nch + 1) * sizeof(float);
}

template <int DIL, bool PROTO, class L>
static int launch_grad_tma(const float* x, const float* coef, int B, int D, int h, int w, int ks, float* grad,
                           ProtoBwdT<L> pb, cudaStream_t s) {
  using G = NbGeom<DIL>;
  NeighMaps maps;
  if (!make_nchw_tensor_map(&maps.m[0], x, B, D, h, w, G::RS, G::BWD_ROWS, kNbCH)) return PFST_ERR_CUDA;
  maps.m[1] = maps.m[0];
  size_t smem = (size_t)kNbStages * kNbCH * G::BWD_ROWS * G::RS * sizeof(float);
  if (PROTO) smem += nb_proto_smem(pb.C, D, ks, &pb.mu_stride);
  auto k = neigh_grad_tma_kernel<DIL, PROTO, L>;
  PFST_CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "pfst_neigh_grad/attr");
  const int64_t tiles = (int64_t)((w + kNbTW - 1) / kNbTW) * ((h + kNbTH - 1) / kNbTH);
  const int64_t grid = (int64_t)B * tiles * ks;
  k<<<(unsigned)grid, kNbThreads, smem, s>>>(maps, coef, B, D, h, w, ks, grad, pb);
  PFST_CHECK_LAUNCH("pfst_neigh_grad");
  return PFST_OK;
}

template <bool PROTO, class L>
static int dispatch_grad_tma(int dilation, const float* x, const float* coef, int B, int D, int h, int w, int ks,
                             float* grad, const ProtoBwdT<L>& pb, cudaStream_t s) {
  switch (dilation) {
    case 1: return launch_grad_tma<1, PROTO, L>(x, coef, B, D, h, w, ks, grad, pb, s);
    case 2: return launch_grad_tma<2, PROTO, L>(x, coef, B, D, h, w, ks, grad, pb, s);
    default: return launch_grad_tma<4, PROTO, L>(x, coef, B, D, h, w, ks, grad, pb, s);
  }
}

static int launch_grad_generic(const float* x, const float* coef, int64_t B, int D, int h, int w, int dilation,
                               float* grad_x, cudaStream_t s) {
  const int64_t plane = (int64_t)h * w;
  const unsigned gx = (unsigned)((plane + 127) / 128);
  unsigned gz = (unsigned)(((int64_t)kNumSMs * 16) / ((int64_t)gx * B) + 1);
  if (gz > (unsigned)D) gz = (unsigned)D;
  if (gz > 64) gz = 64;
  neigh_grad_generic_kernel<<<dim3(gx, (unsigned)B, gz), 128, 0, s>>>(x, coef, (int)B, D, h, w, dilation, grad_x);
  PFST_CHECK_LAUNCH("pfst_neigh_grad");
  return PFST_OK;
}

// small-plane backward: channel splits so that about two blocks per SM are in flight
static int sp_grad_splits(int64_t B, int D) {
  int ks = (int)((2 * (int64_t)kNumSMs + B - 1) / B);
  if (ks > D / kSpCH) ks = D / kSpCH;
  if (ks < 1) ks = 1;
  while (ks > 1 && D % (4 * ks) != 0) --ks;
  return ks;
}

template <bool PROTO, class L>
static int launch_grad_plane(const float* x, const float* coef, int64_t B, int D, int h, int w, int dilation,
                             float* grad, ProtoBwdT<L> pb, int ks, cudaStream_t s) {
  size_t smem = (size_t)kSpStages * kSpCH * h * w * sizeof(float);
  if (PROTO) {
    pb.mu_stride = D / ks + 1;
    smem += (size_t)pb.C * pb.mu_stride * sizeof(float);
  }
  auto k = neigh_grad_plane_kernel<PROTO, L>;
  PFST_CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "pfst_neigh_grad/attr");
  k<<<(unsigned)(B * ks), kSpThreads, smem, s>>>(x, coef, (int)B, D, h, w, dilation, ks, grad, pb);
  PFST_CHECK_LAUNCH("pfst_neigh_grad");
  return PFST_OK;
}

}  // namespace pfst

extern "C" {

int32_t pfst_neigh_dots_splits(int64_t n_tensors, int64_t B, int32_t D, int32_t h, int32_t w) {
  if (n_tensors < 1 || B < 1 || D < 1 || h < 1 || w < 1) return 1;
  return pfst::nb_splits(n_tensors * B, h, w, D);
}

static int neigh_dots_impl(const float* x_a, const float* x_b, int64_t B, int32_t D, int32_t h, int32_t w,
                           int32_t dilation, int slot0, int n_slots, float* dots, cudaStream_t s) {
  const int T = x_b ? 2 : 1;
  const int ks = pfst::nb_splits((int64_t)T * B, h, w, D);
  if (pfst::nb_tma_ok(x_a, x_b, w, dilation)) {
    switch (dilation) {
      case 1: return pfst::launch_dots_tma<1>(x_a, x_b, T, (int)B, D, h, w, ks, slot0, n_slots, dots, s);
      case 2: return pfst::launch_dots_tma<2>(x_a, x_b, T, (int)B, D, h, w, ks, slot0, n_slots, dots, s);
      default: return pfst::launch_dots_tma<4>(x_a, x_b, T, (int)B, D, h, w, ks, slot0, n_slots, dots, s);
    }
  }
  if (pfst::sp_ok(x_a, x_b, D, h, w, ks) && (int64_t)T * B * ks <= 0x7fffffffll) {
    const size_t smem = (size_t)pfst::kSpStages * pfst::kSpCH * h * w * sizeof(float);
    PFST_CUDA_TRY(cudaFuncSetAttribute(pfst::neigh_dots_plane_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem), "pfst_neigh_dots/attr");
    pfst::neigh_dots_plane_kernel<<<(unsigned)(T * B * ks), pfst::kSpThreads, smem, s>>>(
        x_a, x_b, (int)B, D, h, w, dilation, ks, slot0, n_slots, dots);
    PFST_CHECK_LAUNCH("pfst_neigh_dots");
    return PFST_OK;
  }
  const int64_t plane = (int64_t)h * w;
  const dim3 grid((unsigned)((plane + 127) / 128), (unsigned)(T * B * ks), 1);
  if (grid.y > 65535) return PFST_ERR_UNSUPPORTED;
  pfst::neigh_dots_generic_kernel<<<grid, 128, 0, s>>>(x_a, x_b, T, (int)B, D, h, w, dilation, ks, slot0, n_slots,
                                                       dots);
  PFST_CHECK_LAUNCH("pfst_neigh_dots");
  return PFST_OK;
}

int pfst_neigh_dots(const float* x_a, const float* x_b, int64_t B, int32_t D, int32_t h, int32_t w,
                    int32_t dilation, float* dots, void* stream) {
  if (!x_a || !dots || B < 0 || D < 1 || h < 1 || w < 1 || dilation < 1) return PFST_ERR_INVALID_ARG;
  if (B == 0) return PFST_OK;
  if (B > 0x7fffffffll / 4) return PFST_ERR_UNSUPPORTED;
  return neigh_dots_impl(x_a, x_b, B, D, h, w, dilation, 0, x_b ? 2 : 1, dots, static_cast<cudaStream_t>(stream));
}

int pfst_neigh_dots_slot(const float* x, int64_t B, int32_t D, int32_t h, int32_t w, int32_t dilation,
                         int32_t slot, int32_t n_slots, float* dots, void* stream) {
  if (!x || !dots || B < 0 || D < 1 || h < 1 || w < 1 || dilation < 1 || n_slots < 1 || slot < 0 || slot >= n_slots)
    return PFST_ERR_INVALID_ARG;
  if (B == 0) return PFST_OK;
  if (B > 0x7fffffffll / 4) return PFST_ERR_UNSUPPORTED;
  return neigh_dots_impl(x, nullptr, B, D, h, w, dilation, slot, n_slots, dots, static_cast<cudaStream_t>(stream));
}

int pfst_neigh_grad(const float* x, const float* coef, int64_t B, int32_t D, int32_t h, int32_t w,
                    int32_t dilation, float* grad_x, void* stream) {
  if (!x || !coef || !grad_x || B < 0 || D < 1 || h < 1 || w < 1 || dilation < 1) return PFST_ERR_INVALID_ARG;
  if (B == 0) return PFST_OK;
  if (B > 65535) return PFST_ERR_UNSUPPORTED;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (pfst::nb_tma_ok(x, grad_x, w, dilation) && pfst::aligned16(coef)) {
    const int ks = pfst::nb_splits(B, h, w, D);
    return pfst::dispatch_grad_tma<false>(dilation, x, coef, (int)B, D, h, w, ks, grad_x, pfst::ProtoBwd{}, s);
  }
  const int ksp = pfst::sp_grad_splits(B, D);
  if (pfst::sp_ok(x, grad_x, D, h, w, ksp))
    return pfst::launch_grad_plane<false>(x, coef, B, D, h, w, dilation, grad_x, pfst::ProtoBwd{}, ksp, s);
  return pfst::launch_grad_generic(x, coef, B, D, h, w, dilation, grad_x, s);
}

}  // extern "C"

namespace pfst {

template <class L>
static int neigh_grad_proto(const float* x, const float* coef, int64_t B, int32_t D, int32_t h, int32_t w,
                            int32_t dilation, const L* labels, int32_t lab_h, int32_t lab_w, const float* mu,
                            const uint8_t* seen, int32_t C, const float* dist, const double* acc,
                            const float* grad_loss, float* grad_x, void* stream) {
  if (!x || !coef || !grad_x || !labels || !mu || !dist || !acc || !grad_loss || B < 0 || D < 1 || h < 1 ||
      w < 1 || dilation < 1 || lab_h < 1 || lab_w < 1 || C < 1)
    return PFST_ERR_INVALID_ARG;
  if (B == 0) return PFST_OK;
  if (B > 65535) return PFST_ERR_UNSUPPORTED;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (nb_tma_ok(x, grad_x, w, dilation) && aligned16(coef)) {
    const int ks = nb_splits(B, h, w, D);
    int stride = 0;
    if (nb_proto_smem(C, D, ks, &stride) <= 64 * 1024) {
      ProtoBwdT<L> pb{labels, lab_h, lab_w, mu, seen, C, dist, acc, grad_loss, stride};
      return dispatch_grad_tma<true>(dilation, x, coef, (int)B, D, h, w, ks, grad_x, pb, s);
    }
  }
  const int ksp = sp_grad_splits(B, D);
  if (sp_ok(x, grad_x, D, h, w, ksp) &&
      (size_t)kSpStages * kSpCH * h * w * 4 + (size_t)C * (D / ksp + 1) * 4 <= 200 * 1024) {
    ProtoBwdT<L> pb{labels, lab_h, lab_w, mu, seen, C, dist, acc, grad_loss, 0};
    return launch_grad_plane<true>(x, coef, B, D, h, w, dilation, grad_x, pb, ksp, s);
  }
  // shapes the fused kernels do not cover: two passes over grad_x
  const int rc = pfst_neigh_grad(x, coef, B, D, h, w, dilation, grad_x, stream);
  if (rc != PFST_OK) return rc;
  return pfst_proto_dist_bwd_lbl(x, B, D, h, w, labels, LabelDt<L>::value, lab_h, lab_w, mu, seen, C, dist, acc,
                                 grad_loss, grad_x, 1, stream);
}

}  // namespace pfst

extern "C" {

int pfst_neigh_grad_proto(const float* x, const float* coef, int64_t B, int32_t D, int32_t h, int32_t w,
                          int32_t dilation, const int64_t* labels, int32_t lab_h, int32_t lab_w,
                          const float* mu, const uint8_t* seen, int32_t C, const float* dist,
                          const double* acc, const float* grad_loss, float* grad_x, void* stream) {
  return pfst::neigh_grad_proto(x, coef, B, D, h, w, dilation, labels, lab_h, lab_w, mu, seen, C, dist, acc,
                                grad_loss, grad_x, stream);
}

int pfst_neigh_grad_proto_lbl(const float* x, const float* coef, int64_t B, int32_t D, int32_t h, int32_t w,
                              int32_t dilation, const void* labels, int32_t label_dtype, int32_t lab_h,
                              int32_t lab_w, const float* mu, const uint8_t* seen, int32_t C, const float* dist,
                              const double* acc, const float* grad_loss, float* grad_x, void* stream) {
  if (label_dtype == PFST_DT_I64)
    return pfst::neigh_grad_proto(x, coef, B, D, h, w, dilation, static_cast<const int64_t*>(labels), lab_h, lab_w,
                                  mu, seen, C, dist, acc, grad_loss, grad_x, stream);
  if (label_dtype == PFST_DT_U8)
    return pfst::neigh_grad_proto(x, coef, B, D, h, w, dilation, static_cast<const uint8_t*>(labels), lab_h, lab_w,
                                  mu, seen, C, dist, acc, grad_loss, grad_x, stream);
  return PFST_ERR_UNSUPPORTED;
}

}  // extern "C"
