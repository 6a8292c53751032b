// P1-P3 — class prototypes: masked segment-reduce of decoder features over
// (pseudo-)labels, prototype EMA, feature-to-prototype distance loss + backward.
//
// north_star extension: the reference ships no prototype code (SURVEY.md §0). The
// anchor is PFGST.masked_feat_dist, rsiseg/models/uda/pfgst.py:168-177
//   mean( ||f1 - f2||_2 over channels [mask] )           with f2 = mu[label].
// Label maps are nearest-resampled to the feature grid exactly as the loss does
// (pfgst_loss.py:62).
//
// All kernels are HBM-bound streams over the NCHW feature tensor:
//   accumulate  4*D B/pixel read   (sums (C,D) + counts merged with one atomic per
//               (warp, class, channel): per-lane private accumulators in shared
//               memory, acc[class][lane] — bank = lane, no atomics in the hot loop)
//   distance    fwd 4*D B/pixel read, bwd 4*D read + 4*D written
// The pixel x prototype contraction has arithmetic intensity 2C/4 flop/B (1, 3,
// 16.5 for C = 2, 6, 33) and must hold 1e-5 relative in fp32, which rules out
// TF32/BF16 MMA: it stays an FFMA bandwidth kernel (north_star: tensor cores only
// when D and C make it a real contraction).
#include <math.h>
#include <stdlib.h>

#include "common.cuh"
#include "tma.cuh"

namespace pfst {

constexpr int kPrThreads = 256;
constexpr int kPrWarps = kPrThreads / 32;
constexpr int kPrMaxC = 128;

// ---- P1: accumulate ------------------------------------------------------------------
// block = (channel group, pixel tile, image). The block first builds, ONCE, the list of its
// tile's pixel offsets sorted by class (a stable counting sort on warp match/ballot; every
// class segment is padded to a multiple of 32 with the offset of a zero slot). After that
// the segment-reduce of a channel plane is a branch-free gather: for each class, lanes
// stride over the class's segment of the list and add plane[offset] — one 16-bit and one
// 32-bit shared load plus one FADD per element, no label test, no atomics, no divergence;
// one warp reduction + one global RED per (class present, channel).
// Channel planes stream through a ring of shared-memory stages filled by 1-D bulk async
// copies (cp.async.bulk + mbarrier, one producer lane), so the HBM pipe holds
// kPaStages x 16 KB per SM regardless of how many warps are computing.
constexpr int kPaConsumers = 8;                       // consumer warps
constexpr int kPaThreads = (kPaConsumers + 1) * 32;   // + 1 producer warp
constexpr int kPaTile = 4096;                         // pixels per tile (16 KB per plane)
constexpr int kPaMaxStages = 12;
constexpr int kPaUnroll = 8;

struct PaLayout {      // dynamic shared memory carve-up (host and device agree through this)
  int tile, stages, plane_stride;   // plane_stride: floats per stage (tile + 4: zero slot, 16 B aligned)
  size_t off_order, off_grp, off_rows, off_seg, total;
};
__host__ __device__ inline PaLayout pa_layout(int tile, int stages, int C) {
  PaLayout L;
  L.tile = tile; L.stages = stages; L.plane_stride = ((tile + 3) / 4) * 4 + 4;
  size_t o = (size_t)stages * L.plane_stride * sizeof(float);
  L.off_order = o; o += ((size_t)(tile + 32 * C + 256) * 2 + 15) / 16 * 16;  // u16 offsets (+ a padding block of rows)
  L.off_grp = o;   o += ((size_t)((tile + 31) / 32) * C * 2 + 15) / 16 * 16;  // u16 [groups][C]
  L.off_rows = o;  o += ((size_t)((tile + 31) / 32 + C + 8) + 15) / 16 * 16;   // u8 class of every 32-entry row
  L.off_seg = o;   o += ((size_t)(2 * C + 2) * sizeof(int) + 15) / 16 * 16;   // seg[C+1], tot[C]
  L.total = o;
  return L;
}

__device__ __forceinline__ void pa_sync_consumers() {
  asm volatile("bar.sync 1, %0;" ::"n"(kPaConsumers * 32) : "memory");
}

// MODE 0: self-contained (sort + stream). MODE 1: sort only — one block per (image, tile) writes
// the class-sorted lists to `ws` (and the pixel counts to `counts`). MODE 2: stream only — the
// lists are copied from `ws`, so the ~18 us sort prologue is paid by 8 blocks once instead of by
// every one of the 144 streaming blocks.
template <int MODE, class LabelT = int64_t>
__global__ void __launch_bounds__(kPaThreads)
proto_accum_kernel(const float* __restrict__ feats, int B, int D, int h, int w,
                   const LabelT* __restrict__ labels, const float* __restrict__ conf, float conf_thr,
                   int lab_h, int lab_w, int C, int groups, int tile, int stages, int use_bulk,
                   float* __restrict__ packed, float* __restrict__ counts, unsigned char* __restrict__ ws) {
  extern __shared__ __align__(128) unsigned char pa_smem[];
  __shared__ uint64_t full_bar[kPaMaxStages], empty_bar[kPaMaxStages];
  __shared__ int issued;          // number of planes the producer has issued so far
  const PaLayout L = pa_layout(tile, stages, C);
  float* planes = reinterpret_cast<float*>(pa_smem);
  uint16_t* order = reinterpret_cast<uint16_t*>(pa_smem + L.off_order);
  uint16_t* grp = reinterpret_cast<uint16_t*>(pa_smem + L.off_grp);
  uint8_t* rowcls = pa_smem + L.off_rows;
  int* seg = reinterpret_cast<int*>(pa_smem + L.off_seg);
  int* tot = seg + C + 1;

  const int hw = h * w;
  const int n_tiles = (hw + tile - 1) / tile;
  const int grp_id = blockIdx.x % groups;
  const int tile_id = (blockIdx.x / groups) % n_tiles;
  const int b = blockIdx.x / (groups * n_tiles);
  const int p0 = tile_id * tile;
  const int np = min(tile, hw - p0);
  const int ch0 = (int)((int64_t)grp_id * D / groups), ch1 = (int)((int64_t)(grp_id + 1) * D / groups);
  const int n_items = ch1 - ch0;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* base = feats + ((int64_t)b * D + ch0) * hw + p0;

  const size_t list_bytes = L.total - L.off_order;           // order | grp | rowcls | seg, tot
  unsigned char* ws_tile = ws ? ws + ((size_t)b * n_tiles + tile_id) * list_bytes : nullptr;
  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_fence_init();
    issued = 0;
  }
  for (int s = threadIdx.x; s < stages; s += kPaThreads) planes[(size_t)s * L.plane_stride + np] = 0.f;  // zero slot
  __syncthreads();

  if (warp == kPaConsumers) {          // ---- producer: stream the channel planes
    if (MODE != 1 && lane == 0 && use_bulk) {
      const uint32_t bytes = (uint32_t)np * sizeof(float);
      for (int i = 0; i < n_items; ++i) {
        const int s = i % stages;
        if (i >= stages) mbar_wait(&empty_bar[s], (uint32_t)((i / stages) & 1) ^ 1u);
        mbar_arrive_expect_tx(&full_bar[s], bytes);
        bulk_load_1d(planes + (size_t)s * L.plane_stride, base + (int64_t)i * hw, bytes, &full_bar[s]);
        *reinterpret_cast<volatile int*>(&issued) = i + 1;
      }
    }
    return;
  }

  if (MODE == 2) {      // ---- the lists were built by the MODE 1 launch: copy them in
    const uint4* src = reinterpret_cast<const uint4*>(ws_tile);
    uint4* dst = reinterpret_cast<uint4*>(pa_smem + L.off_order);
    for (int i = threadIdx.x; i < (int)(list_bytes / 16); i += kPaConsumers * 32) dst[i] = src[i];
    pa_sync_consumers();
  } else {
    // ---- consumers: class-sorted offset list of this tile (stable counting sort) ----------
    const int ng = (np + 31) / 32;                    // 32-pixel groups, <= kPaTile / 32
    constexpr int kGroupsPerWarp = kPaTile / 32 / kPaConsumers;
    const float sh = (float)lab_h / (float)h, sw = (float)lab_w / (float)w;
    for (int i = threadIdx.x; i < ng * C; i += kPaConsumers * 32) grp[i] = 0;
    // all label gathers of this warp's groups in flight at once (one memory latency, not 16)
    unsigned lv[kGroupsPerWarp];
    if constexpr (sizeof(LabelT) == 1) {
      // uint8: 32-bit offsets inside this image's map (the host keeps lab_h * lab_w below 2^31) and
      // byte-sized label registers, so the gathers fit next to the sort without spilling
      const LabelT* lb = labels + (int64_t)b * lab_h * lab_w;
      const float* cb = conf ? conf + (int64_t)b * lab_h * lab_w : nullptr;
      int off[kGroupsPerWarp];
      unsigned raw[kGroupsPerWarp];
  #pragma unroll
      for (int u = 0; u < kGroupsPerWarp; ++u) {
        const int p = p0 + (warp + u * kPaConsumers) * 32 + lane;
        const int y = p / w, x = p - y * w;
        off[u] = pr_nearest(y, sh, lab_h) * lab_w + pr_nearest(x, sw, lab_w);
      }
  #pragma unroll
      for (int u = 0; u < kGroupsPerWarp; ++u)
        raw[u] = (warp + u * kPaConsumers) * 32 + lane < np ? (unsigned)__ldg(lb + off[u]) : 255u;
  #pragma unroll
      for (int u = 0; u < kGroupsPerWarp; ++u) {
        bool ok = raw[u] < (unsigned)C;
        if (cb && ok) ok = __ldg(cb + off[u]) >= conf_thr;
        lv[u] = ok ? raw[u] : 255u;
      }
    } else {
      int64_t off[kGroupsPerWarp], raw[kGroupsPerWarp];
  #pragma unroll
      for (int u = 0; u < kGroupsPerWarp; ++u) {           // addresses first ...
        const int p = p0 + (warp + u * kPaConsumers) * 32 + lane;
        const int y = p / w, x = p - y * w;
        off[u] = ((int64_t)b * lab_h + pr_nearest(y, sh, lab_h)) * lab_w + pr_nearest(x, sw, lab_w);
      }
  #pragma unroll
      for (int u = 0; u < kGroupsPerWarp; ++u)             // ... then every load back to back
        raw[u] = (warp + u * kPaConsumers) * 32 + lane < np ? __ldg(labels + off[u]) : (int64_t)-1;
  #pragma unroll
      for (int u = 0; u < kGroupsPerWarp; ++u) {
        bool ok = raw[u] >= 0 && raw[u] < C;
        if (conf && ok) ok = __ldg(conf + off[u]) >= conf_thr;
        lv[u] = ok ? (unsigned)raw[u] : 255u;
      }
    }
    pa_sync_consumers();
  #pragma unroll
    for (int u = 0; u < kGroupsPerWarp; ++u) {
      const int g = warp + u * kPaConsumers;
      if (g < ng) {                                    // warp-uniform
        const unsigned m = __match_any_sync(0xffffffffu, lv[u]);
        if (lv[u] != 255u && lane == __ffs(m) - 1) grp[g * C + lv[u]] = (uint16_t)__popc(m);
      }
    }
    pa_sync_consumers();
    // exclusive scan over the groups, one warp per class: lane owns 4 consecutive groups
    for (int c = warp; c < C; c += kPaConsumers) {
      int v[4], run = 0;
  #pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int g = lane * 4 + k;
        v[k] = g < ng ? grp[g * C + c] : 0;
        run += v[k];
      }
      int incl = run;
  #pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      int excl = incl - run;
  #pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int g = lane * 4 + k;
        if (g < ng) grp[g * C + c] = (uint16_t)excl;
        excl += v[k];
      }
      if (lane == 31) tot[c] = incl;
    }
    pa_sync_consumers();
    if (warp == 0) {                                   // padded segment offsets: scan over the classes
      int carry = 0;
      for (int c0 = 0; c0 < C; c0 += 32) {
        const int c = c0 + lane;
        const int len = c < C ? (tot[c] + 31) & ~31 : 0;
        int incl = len;
  #pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int t = __shfl_up_sync(0xffffffffu, incl, o);
          if (lane >= o) incl += t;
        }
        if (c < C) seg[c] = carry + incl - len;
        carry += __shfl_sync(0xffffffffu, incl, 31);
      }
      if (lane == 0) seg[C] = carry;
    }
    pa_sync_consumers();
  #pragma unroll
    for (int u = 0; u < kGroupsPerWarp; ++u) {
      const int g = warp + u * kPaConsumers;
      if (g < ng) {
        const unsigned l = lv[u];
        const unsigned m = __match_any_sync(0xffffffffu, l);
        if (l != 255u) order[seg[l] + grp[g * C + l] + __popc(m & ((1u << lane) - 1u))] = (uint16_t)(g * 32 + lane);
      }
    }
    for (int c = warp; c < C; c += kPaConsumers) {              // pad every segment with the zero slot
      const int j = seg[c] + tot[c] + lane;
      if (j < seg[c + 1]) order[j] = (uint16_t)np;
      for (int r = seg[c] / 32 + lane; r < seg[c + 1] / 32; r += 32) rowcls[r] = (uint8_t)c;
    }
    {   // rows are consumed eight at a time: pad the list to a multiple of 8 rows (class 255, zero slot)
      const int n_rows = seg[C] / 32, n_pad = ((n_rows + 7) & ~7) - n_rows;
      for (int i = threadIdx.x; i < n_pad * 32; i += kPaConsumers * 32) order[n_rows * 32 + i] = (uint16_t)np;
      if (threadIdx.x < n_pad) rowcls[n_rows + threadIdx.x] = 255;
    }
    // pixel counts: once per (image, tile), by channel group 0
    if (grp_id == 0 && counts)
      for (int c = threadIdx.x; c < C; c += kPaConsumers * 32)
        if (tot[c]) atomicAdd(&counts[c], (float)tot[c]);
    pa_sync_consumers();

    if (MODE == 1) {    // ---- sort-only launch: publish the lists
      const uint4* src = reinterpret_cast<const uint4*>(pa_smem + L.off_order);
      uint4* dst = reinterpret_cast<uint4*>(ws_tile);
      for (int i = threadIdx.x; i < (int)(list_bytes / 16); i += kPaConsumers * 32) dst[i] = src[i];
      return;
    }
  }
  // ---- consumers: one channel plane per warp per turn ------------------------------------
  for (int i = warp; i < n_items; i += kPaConsumers) {
    const int s = use_bulk ? i % stages : warp;
    float* pl = planes + (size_t)s * L.plane_stride;
    if (use_bulk) {
      // A stage is consumed by a different warp on every revolution of the ring, and a parity
      // wait is only meaningful within one phase of the barrier: this warp may get here before
      // the PREVIOUS plane of the stage has even landed, and would then take that barrier's
      // older phase for its own. Plane i is issued only after that previous plane was consumed,
      // so wait for the issue first.
      while (*reinterpret_cast<volatile int*>(&issued) <= i) {}
      mbar_wait(&full_bar[s], (uint32_t)((i / stages) & 1));
    } else {                             // planes a bulk copy cannot describe: the warp stages its own
      const float* src = base + (int64_t)i * hw;
      for (int e0 = lane; e0 < np; e0 += 32 * kPaUnroll) {
        float v[kPaUnroll];
#pragma unroll
        for (int u = 0; u < kPaUnroll; ++u)
          if (e0 + u * 32 < np) v[u] = __ldg(src + e0 + u * 32);
#pragma unroll
        for (int u = 0; u < kPaUnroll; ++u)
          if (e0 + u * 32 < np) pl[e0 + u * 32] = v[u];
      }
      __syncwarp();
    }
    float* dst = packed + ch0 + i;
    // walk the class-sorted list 8 rows (256 offsets) at a time: 16 independent shared loads in
    // flight per lane, the class of a row is warp-uniform, a class boundary costs one reduction
    const int n_rows8 = (seg[C] / 32 + 7) / 8;
    unsigned cur = 255u;
    float run = 0.f;
    for (int r8 = 0; r8 < n_rows8; ++r8) {
      const uint2 cls = *reinterpret_cast<const uint2*>(rowcls + r8 * 8);
      const uint16_t* op = order + r8 * 256 + lane;
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = pl[op[32 * u]];
      const unsigned same = cur * 0x01010101u;
      if (cls.x == same && cls.y == same) {
        run += ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
      } else {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const unsigned c = ((u < 4 ? cls.x : cls.y) >> (8 * (u & 3))) & 0xffu;
          if (c != cur) {                                  // warp-uniform
            if (cur != 255u) {
              const float t = warp_sum(run);
              if (lane == 0) atomicAdd(dst + (int64_t)cur * D, t);
            }
            cur = c;
            run = 0.f;
          }
          run += v[u];
        }
      }
    }
    if (cur != 255u) {
      const float t = warp_sum(run);
      if (lane == 0) atomicAdd(dst + (int64_t)cur * D, t);
    }
    __syncwarp();
    if (use_bulk && lane == 0) mbar_arrive(&empty_bar[s]);
  }
}

// ---- few classes (C <= 8): masked accumulation, no sort ------------------------------------------
// With a handful of classes the class test is cheaper than the sorted gather's list handling: a
// block stages the label bytes of its (image, tile) once (16 gathers per thread, all in flight), then
// every warp streams channel planes straight from global memory with 128-bit loads (eight in flight
// per lane) and adds each value to the register accumulator of its class — 2 predicated instructions
// per class and value, NC accumulators per lane, one warp reduction and one RED per (class, channel).
// No sort kernel, no workspace, one launch; and the step no longer has a kernel that must be kept
// away from the TMA kernels (DESIGN.md 3.2).
constexpr int kPmThreads = 256;
constexpr int kPmTile = 4096;

template <int NC, bool FULL, class L>
__global__ void __launch_bounds__(kPmThreads, 2)
proto_accum_masked_kernel(const float* __restrict__ feats, int D, int h, int w, const L* __restrict__ labels,
                          const float* __restrict__ conf, float conf_thr, int lab_h, int lab_w, int groups,
                          float* __restrict__ packed, float* __restrict__ counts) {
  __shared__ __align__(16) uint8_t lab_s[kPmTile];
  const int hw = h * w;
  const int n_tiles = (hw + kPmTile - 1) / kPmTile;
  const int grp_id = blockIdx.x % groups;
  const int tile_id = (blockIdx.x / groups) % n_tiles;
  const int b = blockIdx.x / (groups * n_tiles);
  const int p0 = tile_id * kPmTile;
  const int np = min(kPmTile, hw - p0);                 // multiple of 4 (host checks hw % 4 == 0)
  const int ch0 = (int)((int64_t)grp_id * D / groups), ch1 = (int)((int64_t)(grp_id + 1) * D / groups);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // A warp owns the channel planes ch0 + warp + 8 i and accumulates them TWO at a time: the class tests
  // of a pixel (the bulk of the instructions) are shared by both planes. Work = chunks of 4 float4 per
  // lane and plane; two chunks are in flight: the first is requested BEFORE the label staging below (it
  // does not need the labels), then chunk t+1 is requested while chunk t is accumulated.
  // FULL: the tile is a whole number of 128-float4 chunks (no bounds tests in the loop).
  const int nvec = np / 4;                              // float4 groups of the tile
  const int cpp = (nvec + 127) / 128;                   // chunks per plane pair
  const int n_planes = ch1 - ch0 > warp ? (ch1 - ch0 - warp + 7) / 8 : 0;
  const int n_pairs = (n_planes + 1) / 2;
  const int total = n_pairs * cpp;
  const float* base = feats + ((int64_t)b * D) * hw + p0;
  struct Buf { float4 a[4], b[4]; };
  auto issue = [&](int pair_i, int chunk_i, Buf& q) {
    const int ch = ch0 + warp + 16 * pair_i;
    const bool has_b = ch + 8 < ch1;
    const float4* pa = reinterpret_cast<const float4*>(base + (int64_t)ch * hw) + lane + 128 * chunk_i;
    const float4* pb = reinterpret_cast<const float4*>(base + (int64_t)(ch + (has_b ? 8 : 0)) * hw) + lane + 128 * chunk_i;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const bool ok = FULL || lane + 128 * chunk_i + 32 * u < nvec;
      q.a[u] = ok ? __ldcs(pa + 32 * u) : make_float4(0.f, 0.f, 0.f, 0.f);
      q.b[u] = (ok && has_b) ? __ldcs(pb + 32 * u) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  Buf va, vb;
  if (total > 0) issue(0, 0, va);
  {
    const float sh = (float)lab_h / (float)h, sw = (float)lab_w / (float)w;
    constexpr int kPer = kPmTile / kPmThreads;          // 16 label gathers per thread, issued back to back
    uint8_t l[kPer];
#pragma unroll
    for (int u = 0; u < kPer; ++u) {
      const int e = threadIdx.x + u * kPmThreads;
      l[u] = e < np ? pr_label(labels, conf, conf_thr, b, p0 + e, w, lab_h, lab_w, sh, sw, NC) : (uint8_t)255;
    }
#pragma unroll
    for (int u = 0; u < kPer; ++u) lab_s[threadIdx.x + u * kPmThreads] = l[u];
  }
  __syncthreads();
  if (grp_id == 0 && counts) {                          // pixel counts: once per (image, tile)
    unsigned cnt[NC];
#pragma unroll
    for (int c = 0; c < NC; ++c) cnt[c] = 0;
    for (int e = threadIdx.x; e < np; e += kPmThreads) {
      const unsigned lv = lab_s[e];
#pragma unroll
      for (int c = 0; c < NC; ++c) cnt[c] += lv == (unsigned)c ? 1u : 0u;
    }
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const unsigned t = warp_sum(cnt[c]);
      if (lane == 0 && t) atomicAdd(&counts[c], (float)t);
    }
  }
  const uint32_t* lab_w4 = reinterpret_cast<const uint32_t*>(lab_s) + lane;
  float acc_a[NC], acc_b[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) acc_a[c] = acc_b[c] = 0.f;
  int pair_i = 0, chunk_i = 0;                          // position of the chunk being accumulated
  auto process = [&](const Buf& q) {
    const uint32_t* lp = lab_w4 + 128 * chunk_i;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const uint32_t lw = (FULL || lane + 128 * chunk_i + 32 * u < nvec) ? lp[32 * u] : 0xffffffffu;
      const unsigned l0 = __byte_perm(lw, 0, 0x4440), l1 = __byte_perm(lw, 0, 0x4441),
                     l2 = __byte_perm(lw, 0, 0x4442), l3 = __byte_perm(lw, 0, 0x4443);
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        if (l0 == (unsigned)c) { acc_a[c] += q.a[u].x; acc_b[c] += q.b[u].x; }
        if (l1 == (unsigned)c) { acc_a[c] += q.a[u].y; acc_b[c] += q.b[u].y; }
        if (l2 == (unsigned)c) { acc_a[c] += q.a[u].z; acc_b[c] += q.b[u].z; }
        if (l3 == (unsigned)c) { acc_a[c] += q.a[u].w; acc_b[c] += q.b[u].w; }
      }
    }
    if (++chunk_i == cpp) {                             // the plane pair is complete: one RED per class and plane
      const int ch = ch0 + warp + 16 * pair_i;
      const bool has_b = ch + 8 < ch1;
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        const float ta = warp_sum(acc_a[c]), tb = warp_sum(acc_b[c]);
        if (lane == 0 && ta != 0.f) atomicAdd(packed + (int64_t)c * D + ch, ta);
        if (lane == 0 && has_b && tb != 0.f) atomicAdd(packed + (int64_t)c * D + ch + 8, tb);
        acc_a[c] = acc_b[c] = 0.f;
      }
      chunk_i = 0;
      ++pair_i;
    }
  };
  // request position: one chunk ahead of the accumulate position
  int rp = 0, rc = 1;
  if (rc == cpp) { rc = 0; rp = 1; }
  for (int t = 0; t < total; t += 2) {
    if (t + 1 < total) {
      issue(rp, rc, vb);
      if (++rc == cpp) { rc = 0; ++rp; }
    }
    process(va);
    if (t + 2 < total) {
      issue(rp, rc, va);
      if (++rc == cpp) { rc = 0; ++rp; }
    }
    if (t + 1 < total) process(vb);
  }
}

// ---- small planes (h*w <= kPsMaxHw, e.g. SeasonNet's 15x15): one block per (image, 32-channel chunk) --
// The tile machinery above is built for 4096-pixel tiles: with 225 pixels and 33 classes every class
// segment is padded to a 32-lane row (a 5x longer walk) and every (class, channel) costs a warp reduction
// and a global RED. Here the block stages its 32 channel planes — contiguous in NCHW, one coalesced
// copy — with an odd row stride, rebuilds the per-pixel class from the sorted list of the MODE 1 launch,
// and each warp adds whole pixels into a warp-private [class][channel] tile (lane = channel: no bank
// conflicts, no atomics); the eight tiles are merged in fixed order and one RED per (class present,
// channel) goes to `packed`.
constexpr int kPsCh = 32;
constexpr int kPsThreads = 256;
constexpr int kPsMaxHw = 576;

__host__ __device__ inline size_t ps_smem_bytes(int hw, int C) {
  const size_t stride = (size_t)(hw | 1);
  return ((size_t)kPsCh * stride + (size_t)(kPsThreads / 32) * C * kPsCh) * sizeof(float) + (size_t)((hw + 15) / 16) * 16;
}

__global__ void __launch_bounds__(kPsThreads)
proto_accum_small_kernel(const float* __restrict__ feats, int D, int hw, int C, const unsigned char* __restrict__ ws,
                         size_t list_bytes, size_t off_rows, size_t off_seg, float* __restrict__ packed) {
  extern __shared__ __align__(16) unsigned char ps_smem[];
  const int stride = hw | 1;
  float* F = reinterpret_cast<float*>(ps_smem);                          // [32][stride]
  float* acc = F + (size_t)kPsCh * stride;                               // [8 warps][C][32]
  uint8_t* lab = reinterpret_cast<uint8_t*>(acc + (size_t)(kPsThreads / 32) * C * kPsCh);
  const int chunks = (D + kPsCh - 1) / kPsCh;
  const int b = blockIdx.x / chunks, c0 = (blockIdx.x - b * chunks) * kPsCh;
  const int nch = min(kPsCh, D - c0);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // stage the chunk: nch planes of hw floats, contiguous in global memory
  const float* src = feats + ((int64_t)b * D + c0) * hw;
  for (int e = threadIdx.x; e < nch * hw; e += kPsThreads) {
    const int ch = e / hw, px = e - ch * hw;
    F[ch * stride + px] = __ldg(src + e);
  }
  for (int i = threadIdx.x; i < (kPsThreads / 32) * C * kPsCh; i += kPsThreads) acc[i] = 0.f;
  for (int i = threadIdx.x; i < hw; i += kPsThreads) lab[i] = 255;
  __syncthreads();
  // per-pixel class from the class-sorted list: row r (32 entries) belongs to class rowcls[r]
  const unsigned char* list = ws + (size_t)b * list_bytes;
  const uint16_t* order = reinterpret_cast<const uint16_t*>(list);
  const uint8_t* rowcls = list + off_rows;
  const int n_entries = reinterpret_cast<const int*>(list + off_seg)[C];
  for (int i = threadIdx.x; i < n_entries; i += kPsThreads) {
    const unsigned px = order[i];
    if (px < (unsigned)hw) lab[px] = rowcls[i >> 5];
  }
  __syncthreads();
  float* mine = acc + (size_t)warp * C * kPsCh;
  if (lane < nch)
    for (int px = warp; px < hw; px += kPsThreads / 32) {
      const unsigned c = lab[px];
      if (c != 255u) mine[c * kPsCh + lane] += F[lane * stride + px];
    }
  __syncthreads();
  for (int i = threadIdx.x; i < C * kPsCh; i += kPsThreads) {
    float t = 0.f;
#pragma unroll
    for (int wv = 0; wv < kPsThreads / 32; ++wv) t += acc[(size_t)wv * C * kPsCh + i];
    const int c = i / kPsCh, ch = i - c * kPsCh;
    if (t != 0.f && ch < nch) atomicAdd(packed + (int64_t)c * D + c0 + ch, t);
  }
}

// iter_state (nullable): device int64[2] = {prototype-bank iteration, block-completion counter}.
// When given, the EMA coefficients are derived from the device-resident iteration with the
// E2 rule (pfgst.py:117, in fp64 like the host) and the last block to finish advances it —
// the launch then has no per-step host argument and can live inside a CUDA graph.
__global__ void proto_finalize_kernel(float* __restrict__ packed, int C, int D,
                                      const float* mu_prev, const uint8_t* seen_prev,
                                      float a32, float b32, double alpha, long long* iter_state,
                                      float* mu_out, int64_t* __restrict__ cnt_out, uint8_t* seen_out,
                                      int reset) {
  // mu_out may alias mu_prev and seen_out may alias seen_prev (in-place bank update): every
  // element is read and written by the same thread, the per-class flags after a barrier.
  const int c = blockIdx.x;
  long long it = 0;
  if (iter_state) {
    it = *reinterpret_cast<volatile long long*>(iter_state);
    if (it > 0) {
      double a = 1.0 - 1.0 / (double)(it + 1);
      if (alpha < a) a = alpha;
      a32 = (float)a;
      b32 = (float)(1.0 - a);
    } else {
      a32 = 0.f;
      b32 = 1.f;
    }
  }
  const float cnt = packed[(int64_t)C * D + c];
  const bool has = cnt > 0.f;
  const bool seen = seen_prev ? seen_prev[c] != 0 : false;
  const float denom = fmaxf(cnt, 1.f);
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    const float mean = packed[(int64_t)c * D + d] / denom;
    const float prev = mu_prev ? mu_prev[(int64_t)c * D + d] : 0.f;
    float out = prev;
    if (has) out = seen ? __fadd_rn(__fmul_rn(a32, prev), __fmul_rn(b32, mean)) : mean;
    mu_out[(int64_t)c * D + d] = out;
    if (reset) packed[(int64_t)c * D + d] = 0.f;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (cnt_out) cnt_out[c] = (int64_t)cnt;
    if (seen_out) seen_out[c] = (has || seen) ? 1 : 0;
    if (reset) packed[(int64_t)C * D + c] = 0.f;
    if (iter_state) {
      __threadfence();
      if (atomicAdd(reinterpret_cast<unsigned long long*>(iter_state + 1), 1ull) == gridDim.x - 1) {
        iter_state[1] = 0;
        iter_state[0] = it + 1;      // every block has read `it` before it could finish
      }
    }
  }
}

// ---- distance: block = 128 consecutive pixels of one image x all channels -------
constexpr int kPdPix = 128;
constexpr int kPdUnroll = 8;    // channel planes in flight per warp (backward: + grad read)
constexpr int kPdUnrollFwd = 16;

// four consecutive pixels of one channel plane (128-bit when the plane allows it)
template <bool READ_ONLY = true>
__device__ __forceinline__ void pd_load4(const float* p, bool vec, int pix, int hw, float (&v)[4]) {
  if (vec) {
    const float4 t = READ_ONLY ? ldg_stream_f4(p) : *reinterpret_cast<const float4*>(p);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = (pix + i < hw) ? (READ_ONLY ? __ldg(p + i) : p[i]) : 0.f;
  }
}

struct PdCtx {
  int b, p0, hw;
  uint8_t lab[4];
};

// BWD = false: dist[n] = ||f_n - mu_y||, block sums -> acc[0] (sum dist), acc[1] (n valid)
// BWD = true : grad[n,d] = g * (f - mu_y) / (dist * n_valid)
template <bool BWD, class L>
__global__ void __launch_bounds__(kPrThreads)
proto_dist_kernel(const float* __restrict__ feats, int B, int D, int h, int w,
                  const L* __restrict__ labels, int lab_h, int lab_w, const float* __restrict__ mu,
                  const uint8_t* __restrict__ seen, int C, float* __restrict__ dist, double* __restrict__ acc,
                  float* __restrict__ loss, const float* __restrict__ grad_loss, float* __restrict__ grad,
                  unsigned* __restrict__ done_counter, int accumulate) {
  extern __shared__ __align__(16) unsigned char pd_smem[];
  float* mu_s = reinterpret_cast<float*>(pd_smem);                 // [C][D+1]  (+1: bank skew)
  float* part = mu_s + (size_t)C * (D + 1);                        // [warps][128]
  const int hw = h * w;
  const int tiles = (hw + kPdPix - 1) / kPdPix;
  const int b = blockIdx.x / tiles, p0 = (blockIdx.x - b * tiles) * kPdPix;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < C * D; i += kPrThreads) mu_s[(i / D) * (D + 1) + (i % D)] = mu[i];
  const float sh = (float)lab_h / (float)h, sw = (float)lab_w / (float)w;
  // this lane's four pixels
  int lab[4];
  bool ok[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int p = p0 + lane * 4 + i;
    uint8_t l = 255;
    if (p < hw) l = pr_label(labels, nullptr, 0.f, b, p, w, lab_h, lab_w, sh, sw, C);
    if (l != 255 && seen && !seen[l]) l = 255;
    ok[i] = l != 255;
    lab[i] = ok[i] ? l : 0;
  }
  __syncthreads();
  const float* src = feats + (int64_t)b * D * hw + p0 + lane * 4;
  const bool vec = (hw % 4 == 0) && ((reinterpret_cast<uintptr_t>(feats) & 15u) == 0);
  const bool any_px = p0 + lane * 4 < hw;

  if (!BWD) {
    float ss[4] = {0.f, 0.f, 0.f, 0.f};
    if (any_px)
      for (int d0 = warp; d0 < D; d0 += kPrWarps * kPdUnrollFwd) {
        float v[kPdUnrollFwd][4];
#pragma unroll
        for (int u = 0; u < kPdUnrollFwd; ++u) {
          const int d = d0 + u * kPrWarps;
          if (d < D) pd_load4(src + (int64_t)d * hw, vec, p0 + lane * 4, hw, v[u]);
        }
#pragma unroll
        for (int u = 0; u < kPdUnrollFwd; ++u) {
          const int d = d0 + u * kPrWarps;
          if (d < D) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float df = v[u][i] - mu_s[lab[i] * (D + 1) + d];
              ss[i] = fmaf(df, df, ss[i]);
            }
          }
        }
      }
#pragma unroll
    for (int i = 0; i < 4; ++i) part[warp * kPdPix + lane * 4 + i] = ss[i];
    __syncthreads();
    double bsum = 0.0, bcnt = 0.0;
    if (warp == 0) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float s = 0.f;
        for (int wv = 0; wv < kPrWarps; ++wv) s += part[wv * kPdPix + lane * 4 + i];
        const float dn = ok[i] ? sqrtf(s) : 0.f;
        const int p = p0 + lane * 4 + i;
        if (p < hw) dist[(int64_t)b * hw + p] = dn;
        if (ok[i]) { bsum += (double)dn; bcnt += 1.0; }
      }
      bsum = warp_sum(bsum);
      bcnt = warp_sum(bcnt);
      if (lane == 0) {
        if (bcnt != 0.0) { atomicAdd(&acc[0], bsum); atomicAdd(&acc[1], bcnt); }
        __threadfence();
        if (atomicAdd(done_counter, 1u) == gridDim.x - 1) {
          __threadfence();
          const double s = *((volatile double*)&acc[0]), n = *((volatile double*)&acc[1]);
          loss[0] = (float)(s / n);   // mean of an empty selection is NaN, as torch.mean
        }
      }
    }
  } else {
    const float g = grad_loss[0];
    const float nvalid = (float)acc[1];
    float coef[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int p = p0 + lane * 4 + i;
      const float dn = (p < hw) ? dist[(int64_t)b * hw + p] : 0.f;
      coef[i] = (ok[i] && dn > 0.f) ? g / (dn * nvalid) : 0.f;   // torch.norm backward: 0 at 0
    }
    float* dst = grad + (int64_t)b * D * hw + p0 + lane * 4;
    if (any_px)
      for (int d0 = warp; d0 < D; d0 += kPrWarps * kPdUnroll) {
        float v[kPdUnroll][4], o[kPdUnroll][4];
#pragma unroll
        for (int u = 0; u < kPdUnroll; ++u) {
          const int d = d0 + u * kPrWarps;
          if (d < D) {
            pd_load4(src + (int64_t)d * hw, vec, p0 + lane * 4, hw, v[u]);
            if (accumulate) {   // grad += ... : the PFGST loss gradient is already in the buffer
              pd_load4<false>(dst + (int64_t)d * hw, vec, p0 + lane * 4, hw, o[u]);
            } else {
#pragma unroll
              for (int i = 0; i < 4; ++i) o[u][i] = 0.f;
            }
          }
        }
#pragma unroll
        for (int u = 0; u < kPdUnroll; ++u) {
          const int d = d0 + u * kPrWarps;
          if (d < D) {
#pragma unroll
            for (int i = 0; i < 4; ++i) o[u][i] = fmaf(coef[i], v[u][i] - mu_s[lab[i] * (D + 1) + d], o[u][i]);
            if (vec) {
              __stcs(reinterpret_cast<float4*>(dst + (int64_t)d * hw), make_float4(o[u][0], o[u][1], o[u][2], o[u][3]));
            } else {
#pragma unroll
              for (int i = 0; i < 4; ++i)
                if (p0 + lane * 4 + i < hw) dst[(int64_t)d * hw + i] = o[u][i];
            }
          }
        }
      }
  }
}

// ---- forward distance for planes a float4 cannot address (h*w % 4 != 0, e.g. SeasonNet's 15x15) --------
// The kernel above then falls back to four guarded scalar loads per lane and, with 128-pixel tiles, to two
// blocks per 225-pixel image (128 blocks on 148 SMs), each staging all C*D prototypes (67 KB at C = 33).
// Here a block owns 32 consecutive pixels of one image (one per lane: a plane row of a warp is one
// coalesced 128-byte request) and its eight warps split the channels, sixteen planes in flight per lane;
// the prototype value of a pixel's class comes through L1 (the table is <= 67 KB and shared by every block
// of the SM). The eight channel partials of a pixel are summed in warp order: deterministic like the kernel above.
constexpr int kPdsUnroll = 16;

template <class L>
__global__ void __launch_bounds__(kPrThreads)
proto_dist_small_kernel(const float* __restrict__ feats, int D, int h, int w, const L* __restrict__ labels,
                        int lab_h, int lab_w, const float* __restrict__ mu, const uint8_t* __restrict__ seen, int C,
                        float* __restrict__ dist, double* __restrict__ acc, float* __restrict__ loss,
                        unsigned* __restrict__ done_counter) {
  __shared__ float part[kPrWarps][32];
  const int hw = h * w;
  const int tiles = (hw + 31) / 32;
  const int b = blockIdx.x / tiles, p0 = (blockIdx.x - b * tiles) * 32;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int p = p0 + lane;
  const bool in = p < hw;
  uint8_t l = 255;
  if (in) l = pr_label(labels, nullptr, 0.f, b, p, w, lab_h, lab_w, (float)lab_h / (float)h, (float)lab_w / (float)w, C);
  if (l != 255 && seen && !seen[l]) l = 255;
  const bool ok = l != 255;
  const float* src = feats + (int64_t)b * D * hw + p;
  const float* mrow = mu + (int64_t)(ok ? l : 0) * D;
  float ss = 0.f;
  if (in)
    for (int d0 = warp; d0 < D; d0 += kPrWarps * kPdsUnroll) {
      float v[kPdsUnroll], m[kPdsUnroll];
#pragma unroll
      for (int u = 0; u < kPdsUnroll; ++u) {
        const int d = d0 + u * kPrWarps;
        v[u] = d < D ? __ldg(src + (int64_t)d * hw) : 0.f;
        m[u] = d < D ? __ldg(mrow + d) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < kPdsUnroll; ++u) {
        const float df = v[u] - m[u];
        ss = fmaf(df, df, ss);
      }
    }
  part[warp][lane] = ss;
  __syncthreads();
  if (warp == 0) {
    float t = 0.f;
#pragma unroll
    for (int wv = 0; wv < kPrWarps; ++wv) t += part[wv][lane];
    const float dn = ok ? sqrtf(t) : 0.f;
    if (in) dist[(int64_t)b * hw + p] = dn;
    const double bsum = warp_sum(ok ? (double)dn : 0.0), bcnt = warp_sum(ok ? 1.0 : 0.0);
    if (lane == 0) {
      if (bcnt != 0.0) { atomicAdd(&acc[0], bsum); atomicAdd(&acc[1], bcnt); }
      __threadfence();
      if (atomicAdd(done_counter, 1u) == gridDim.x - 1) {
        __threadfence();
        const double sd = *((volatile double*)&acc[0]), n = *((volatile double*)&acc[1]);
        loss[0] = (float)(sd / n);   // mean of an empty selection is NaN, as torch.mean
      }
    }
  }
}

// all-class distances: out[b,c,n] = ||f_n - mu_c||_2
__global__ void __launch_bounds__(kPrThreads)
proto_dist_all_kernel(const float* __restrict__ feats, int B, int D, int h, int w,
                      const float* __restrict__ mu, int C, float* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char pall_smem[];
  float* mu_s = reinterpret_cast<float*>(pall_smem);     // [C][D]
  const int hw = h * w;
  for (int i = threadIdx.x; i < C * D; i += kPrThreads) mu_s[i] = mu[i];
  __syncthreads();
  const int64_t total = (int64_t)B * hw;
  for (int64_t n = (int64_t)blockIdx.x * kPrThreads + threadIdx.x; n < total;
       n += (int64_t)gridDim.x * kPrThreads) {
    const int b = (int)(n / hw);
    const int p = (int)(n - (int64_t)b * hw);
    const float* src = feats + (int64_t)b * D * hw + p;
    for (int c0 = 0; c0 < C; c0 += 8) {
      float ss[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      for (int d = 0; d < D; ++d) {
        const float v = __ldg(src + (int64_t)d * hw);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (c0 + j < C) {
            const float df = v - mu_s[(c0 + j) * D + d];
            ss[j] = fmaf(df, df, ss[j]);
          }
      }
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (c0 + j < C) out[((int64_t)b * C + c0 + j) * hw + p] = sqrtf(ss[j]);
    }
  }
}

}  // namespace pfst

namespace {

struct PaPlan {
  int tile, n_tiles, stages, use_bulk;
  int64_t groups;
  pfst::PaLayout L;
  size_t list_bytes;
};

// Launch geometry shared by the three accumulate entry points (stream = with plane stages).
int pa_plan(PaPlan& P, const float* feats, int64_t B, int32_t D, int32_t h, int32_t w, int32_t C, bool stream) {
  const int64_t hw = (int64_t)h * w;
  P.tile = (int)(hw < pfst::kPaTile ? hw : pfst::kPaTile);
  P.n_tiles = (int)((hw + P.tile - 1) / P.tile);
  // bulk async copies need 16-byte aligned planes whose tiles are multiples of 16 bytes
  P.use_bulk = (hw % 4 == 0) && (!feats || pfst::aligned16(feats)) ? 1 : 0;
  if (getenv("PFST_ACCUM_NO_BULK")) P.use_bulk = 0;   // debugging aid
  P.stages = 0;
  if (stream) {   // stages: as many as fit next to the sort buffers, at least one per consumer warp + 1
    P.stages = pfst::kPaMaxStages;
    while (P.stages > pfst::kPaConsumers + 1 && pfst::pa_layout(P.tile, P.stages, C).total > 200 * 1024) --P.stages;
  }
  P.L = pfst::pa_layout(P.tile, P.stages, C);
  if (P.L.total > 200 * 1024) return PFST_ERR_UNSUPPORTED;
  P.list_bytes = P.L.total - P.L.off_order;
  // channel groups: fill every SM's shared memory with blocks, keep >= 2 planes per consumer warp
  int per_sm = (int)((220 * 1024) / (P.L.total + 1024));
  if (per_sm < 1) per_sm = 1;
  if (per_sm > 6) per_sm = 6;
  P.groups = ((int64_t)pfst::kNumSMs * per_sm) / (B * P.n_tiles);
  const int64_t max_groups = (D + 2 * pfst::kPaConsumers - 1) / (2 * pfst::kPaConsumers);
  if (P.groups > max_groups) P.groups = max_groups;
  if (P.groups < 1) P.groups = 1;
  if (B * P.n_tiles * P.groups > 0x7fffffffll) return PFST_ERR_UNSUPPORTED;
  return PFST_OK;
}

template <int MODE, class L>
int pa_launch(const PaPlan& P, const float* feats, int64_t B, int32_t D, int32_t h, int32_t w,
              const L* labels, int32_t lab_h, int32_t lab_w, const float* conf, float conf_thr, int32_t C,
              float* packed, float* counts, unsigned char* ws, cudaStream_t s, const char* what) {
  auto k = pfst::proto_accum_kernel<MODE, L>;
  PFST_CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)P.L.total), what);
  const int64_t groups = MODE == 1 ? 1 : P.groups;
  k<<<(unsigned)(B * P.n_tiles * groups), pfst::kPaThreads, P.L.total, s>>>(
      feats, (int)B, D, h, w, labels, conf, conf_thr, lab_h, lab_w, C, (int)groups, P.tile, P.stages, P.use_bulk,
      packed, counts, ws);
  PFST_CHECK_LAUNCH(what);
  return PFST_OK;
}

}  // namespace

extern "C" {

int pfst_proto_accum_is_masked(int32_t C, int32_t h, int32_t w) {
  static const bool off = getenv("PFST_ACCUM_NO_MASKED") != nullptr;     // A/B switch
  return (!off && C >= 1 && C <= 8 && ((int64_t)h * w) % 4 == 0 && (int64_t)h * w > pfst::kPsMaxHw) ? 1 : 0;
}

}  // extern "C"

namespace {

template <class L>
int proto_accum(const float* feats, int64_t B, int32_t D, int32_t h, int32_t w, const L* labels, int32_t lab_h,
                int32_t lab_w, const float* conf, float conf_thr, int32_t C, float* packed, void* stream) {
  if (sizeof(L) == 1 && (int64_t)lab_h * lab_w > 0x7fffffffll) return PFST_ERR_UNSUPPORTED;   // 32-bit gathers
  if (!feats || !labels || !packed || B < 0 || D < 1 || h < 1 || w < 1 || lab_h < 1 || lab_w < 1 || C < 1)
    return PFST_ERR_INVALID_ARG;
  if (C > pfst::kPrMaxC) return PFST_ERR_UNSUPPORTED;
  if (B == 0) return PFST_OK;
  const int64_t hw = (int64_t)h * w;
  if (pfst_proto_accum_is_masked(C, h, w) && pfst::aligned16(feats)) {
    // few classes: masked accumulation straight from global memory, no sort (see proto_accum_masked_kernel)
    const int64_t n_tiles = (hw + pfst::kPmTile - 1) / pfst::kPmTile;
    int64_t groups = ((int64_t)pfst::kNumSMs * 2) / (B * n_tiles);
    const int64_t max_groups = (D + 15) / 16;                     // >= 2 planes per warp
    if (groups > max_groups) groups = max_groups;
    if (groups < 1) groups = 1;
    const int64_t grid = B * n_tiles * groups;
    if (grid > 0x7fffffffll) return PFST_ERR_UNSUPPORTED;
    void (*k)(const float*, int, int, int, const L*, const float*, float, int, int, int, float*, float*);
    // whole 128-float4 chunks in every tile: no bounds tests in the streaming loop
    const bool full = hw % 512 == 0;
#define PFST_PM_PICK(N) (full ? pfst::proto_accum_masked_kernel<N, true, L> : pfst::proto_accum_masked_kernel<N, false, L>)
    switch (C) {
      case 1: k = PFST_PM_PICK(1); break;
      case 2: k = PFST_PM_PICK(2); break;
      case 3: k = PFST_PM_PICK(3); break;
      case 4: k = PFST_PM_PICK(4); break;
      case 5: k = PFST_PM_PICK(5); break;
      case 6: k = PFST_PM_PICK(6); break;
      case 7: k = PFST_PM_PICK(7); break;
      default: k = PFST_PM_PICK(8); break;
    }
#undef PFST_PM_PICK
    k<<<(unsigned)grid, pfst::kPmThreads, 0, static_cast<cudaStream_t>(stream)>>>(
        feats, D, h, w, labels, conf, conf_thr, lab_h, lab_w, (int)groups, packed, packed + (int64_t)C * D);
    PFST_CHECK_LAUNCH("pfst_proto_accum/masked");
    return PFST_OK;
  }
  PaPlan P;
  const int rc = pa_plan(P, feats, B, D, h, w, C, true);
  if (rc != PFST_OK) return rc;
  return pa_launch<0>(P, feats, B, D, h, w, labels, lab_h, lab_w, conf, conf_thr, C, packed,
                      packed + (int64_t)C * D, nullptr, static_cast<cudaStream_t>(stream), "pfst_proto_accum");
}

}  // namespace

extern "C" {

int pfst_proto_accum(const float* feats, int64_t B, int32_t D, int32_t h, int32_t w,
                     const int64_t* labels, int32_t lab_h, int32_t lab_w, const float* conf,
                     float conf_thr, int32_t C, float* packed, void* stream) {
  return proto_accum(feats, B, D, h, w, labels, lab_h, lab_w, conf, conf_thr, C, packed, stream);
}

int pfst_proto_accum_lbl(const float* feats, int64_t B, int32_t D, int32_t h, int32_t w,
                         const void* labels, int32_t label_dtype, int32_t lab_h, int32_t lab_w,
                         const float* conf, float conf_thr, int32_t C, float* packed, void* stream) {
  if (label_dtype == PFST_DT_I64)
    return proto_accum(feats, B, D, h, w, static_cast<const int64_t*>(labels), lab_h, lab_w, conf, conf_thr, C,
                       packed, stream);
  if (label_dtype == PFST_DT_U8)
    return proto_accum(feats, B, D, h, w, static_cast<const uint8_t*>(labels), lab_h, lab_w, conf, conf_thr, C,
                       packed, stream);
  return PFST_ERR_UNSUPPORTED;
}

int64_t pfst_proto_order_ws_bytes(int64_t B, int32_t h, int32_t w, int32_t C) {
  if (B < 1 || h < 1 || w < 1 || C < 1 || C > pfst::kPrMaxC) return 0;
  PaPlan P;
  if (pa_plan(P, nullptr, B, 1, h, w, C, false) != PFST_OK) return 0;
  return (int64_t)(B * P.n_tiles * P.list_bytes);
}

}  // extern "C"

namespace {

template <class L>
int proto_order(const L* labels, int64_t B, int32_t h, int32_t w, int32_t lab_h, int32_t lab_w,
                const float* conf, float conf_thr, int32_t C, float* counts, void* workspace, void* stream) {
  if (sizeof(L) == 1 && (int64_t)lab_h * lab_w > 0x7fffffffll) return PFST_ERR_UNSUPPORTED;   // 32-bit gathers
  if (!labels || !workspace || B < 0 || h < 1 || w < 1 || lab_h < 1 || lab_w < 1 || C < 1)
    return PFST_ERR_INVALID_ARG;
  if (C > pfst::kPrMaxC || !pfst::aligned16(workspace)) return PFST_ERR_UNSUPPORTED;
  if (B == 0) return PFST_OK;
  PaPlan P;
  const int rc = pa_plan(P, nullptr, B, 1, h, w, C, false);
  if (rc != PFST_OK) return rc;
  return pa_launch<1>(P, nullptr, B, 1, h, w, labels, lab_h, lab_w, conf, conf_thr, C, nullptr, counts,
                      static_cast<unsigned char*>(workspace), static_cast<cudaStream_t>(stream), "pfst_proto_order");
}

}  // namespace

extern "C" {

int pfst_proto_order(const int64_t* labels, int64_t B, int32_t h, int32_t w, int32_t lab_h, int32_t lab_w,
                     const float* conf, float conf_thr, int32_t C, float* counts, void* workspace,
                     void* stream) {
  return proto_order(labels, B, h, w, lab_h, lab_w, conf, conf_thr, C, counts, workspace, stream);
}

int pfst_proto_order_lbl(const void* labels, int32_t label_dtype, int64_t B, int32_t h, int32_t w, int32_t lab_h,
                         int32_t lab_w, const float* conf, float conf_thr, int32_t C, float* counts,
                         void* workspace, void* stream) {
  if (label_dtype == PFST_DT_I64)
    return proto_order(static_cast<const int64_t*>(labels), B, h, w, lab_h, lab_w, conf, conf_thr, C, counts,
                       workspace, stream);
  if (label_dtype == PFST_DT_U8)
    return proto_order(static_cast<const uint8_t*>(labels), B, h, w, lab_h, lab_w, conf, conf_thr, C, counts,
                       workspace, stream);
  return PFST_ERR_UNSUPPORTED;
}

int pfst_proto_accum_ordered(const float* feats, int64_t B, int32_t D, int32_t h, int32_t w, int32_t C,
                             const void* workspace, float* packed, void* stream) {
  if (!feats || !workspace || !packed || B < 0 || D < 1 || h < 1 || w < 1 || C < 1) return PFST_ERR_INVALID_ARG;
  if (C > pfst::kPrMaxC || !pfst::aligned16(workspace)) return PFST_ERR_UNSUPPORTED;
  if (B == 0) return PFST_OK;
  PaPlan P;
  const int hw = h * w;
  if (hw <= pfst::kPsMaxHw && pfst::ps_smem_bytes(hw, C) <= 200 * 1024 && !getenv("PFST_ACCUM_NO_SMALL")) {
    // small planes: one block per (image, 32-channel chunk), lists from the MODE 1 launch
    if (pa_plan(P, nullptr, B, 1, h, w, C, false) != PFST_OK) return PFST_ERR_UNSUPPORTED;
    const size_t smem = pfst::ps_smem_bytes(hw, C);
    PFST_CUDA_TRY(cudaFuncSetAttribute(pfst::proto_accum_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem), "pfst_proto_accum_ordered/attr");
    const int64_t grid = B * ((D + pfst::kPsCh - 1) / pfst::kPsCh);
    if (grid > 0x7fffffffll) return PFST_ERR_UNSUPPORTED;
    pfst::proto_accum_small_kernel<<<(unsigned)grid, pfst::kPsThreads, smem, static_cast<cudaStream_t>(stream)>>>(
        feats, D, hw, C, static_cast<const unsigned char*>(workspace), P.list_bytes, P.L.off_rows - P.L.off_order,
        P.L.off_seg - P.L.off_order, packed);
    PFST_CHECK_LAUNCH("pfst_proto_accum_ordered/small");
    return PFST_OK;
  }
  const int rc = pa_plan(P, feats, B, D, h, w, C, true);
  if (rc != PFST_OK) return rc;
  return pa_launch<2>(P, feats, B, D, h, w, (const int64_t*)nullptr, 1, 1, nullptr, 0.f, C, packed, nullptr,
                      static_cast<unsigned char*>(const_cast<void*>(workspace)), static_cast<cudaStream_t>(stream),
                      "pfst_proto_accum_ordered");
}

int pfst_proto_finalize(float* packed, int32_t C, int32_t D, const float* mu_prev,
                        const uint8_t* seen_prev, float a32, float b32, float* mu_out, int64_t* cnt_out,
                        uint8_t* seen_out, int32_t reset_packed, void* stream) {
  if (!packed || !mu_out || C < 1 || D < 1) return PFST_ERR_INVALID_ARG;
  pfst::proto_finalize_kernel<<<(unsigned)C, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      packed, C, D, mu_prev, seen_prev, a32, b32, 0.0, nullptr, mu_out, cnt_out, seen_out, reset_packed);
  PFST_CHECK_LAUNCH("pfst_proto_finalize");
  return PFST_OK;
}

int pfst_proto_finalize_dev(float* packed, int32_t C, int32_t D, const float* mu_prev,
                            const uint8_t* seen_prev, double alpha, int64_t* iter_state, float* mu_out,
                            int64_t* cnt_out, uint8_t* seen_out, int32_t reset_packed, void* stream) {
  if (!packed || !mu_out || !iter_state || C < 1 || D < 1) return PFST_ERR_INVALID_ARG;
  pfst::proto_finalize_kernel<<<(unsigned)C, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      packed, C, D, mu_prev, seen_prev, 0.f, 1.f, alpha, reinterpret_cast<long long*>(iter_state), mu_out, cnt_out,
      seen_out, reset_packed);
  PFST_CHECK_LAUNCH("pfst_proto_finalize_dev");
  return PFST_OK;
}

}  // extern "C"

template <class L>
static int proto_dist_common(bool bwd, const float* feats, int64_t B, int32_t D, int32_t h, int32_t w,
                             const L* labels, int32_t lab_h, int32_t lab_w, const float* mu,
                             const uint8_t* seen, int32_t C, float* dist, double* acc, float* loss,
                             const float* grad_loss, float* grad, int accumulate, cudaStream_t s) {
  if (!feats || !labels || !mu || !dist || !acc || B < 0 || D < 1 || h < 1 || w < 1 || C < 1)
    return PFST_ERR_INVALID_ARG;
  if (C > pfst::kPrMaxC) return PFST_ERR_UNSUPPORTED;
  const size_t smem = ((size_t)C * (D + 1) + (size_t)pfst::kPrWarps * pfst::kPdPix) * sizeof(float);
  if (smem > 200 * 1024) return PFST_ERR_UNSUPPORTED;
  const int hw = h * w;
  const int64_t grid = B * ((hw + pfst::kPdPix - 1) / pfst::kPdPix);
  if (grid == 0) return PFST_OK;
  if (!bwd) {
    if (!loss) return PFST_ERR_INVALID_ARG;
    PFST_CUDA_TRY(cudaMemsetAsync(acc, 0, 4 * sizeof(double), s), "pfst_proto_dist_fwd/memset");
    static const bool no_small = getenv("PFST_DIST_NO_SMALL") != nullptr;       // A/B switch
    if (hw % 4 != 0 && !no_small) {
      const int64_t grid_s = B * ((hw + 31) / 32);
      if (grid_s > 0x7fffffffll) return PFST_ERR_UNSUPPORTED;
      pfst::proto_dist_small_kernel<L><<<(unsigned)grid_s, pfst::kPrThreads, 0, s>>>(
          feats, D, h, w, labels, lab_h, lab_w, mu, seen, C, dist, acc, loss, reinterpret_cast<unsigned*>(acc + 3));
      PFST_CHECK_LAUNCH("pfst_proto_dist_fwd/small");
      return PFST_OK;
    }
    auto k = pfst::proto_dist_kernel<false, L>;
    PFST_CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "pfst_proto_dist_fwd/attr");
    k<<<(unsigned)grid, pfst::kPrThreads, smem, s>>>(feats, (int)B, D, h, w, labels, lab_h, lab_w, mu, seen, C, dist,
                                                     acc, loss, nullptr, nullptr,
                                                     reinterpret_cast<unsigned*>(acc + 3), 0);
  } else {
    if (!grad_loss || !grad) return PFST_ERR_INVALID_ARG;
    auto k = pfst::proto_dist_kernel<true, L>;
    PFST_CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "pfst_proto_dist_bwd/attr");
    k<<<(unsigned)grid, pfst::kPrThreads, smem, s>>>(feats, (int)B, D, h, w, labels, lab_h, lab_w, mu, seen, C, dist,
                                                     acc, nullptr, grad_loss, grad, nullptr, accumulate);
  }
  PFST_CHECK_LAUNCH(bwd ? "pfst_proto_dist_bwd" : "pfst_proto_dist_fwd");
  return PFST_OK;
}

extern "C" {

int pfst_proto_dist_fwd(const float* feats, int64_t B, int32_t D, int32_t h, int32_t w,
                        const int64_t* labels, int32_t lab_h, int32_t lab_w, const float* mu,
                        const uint8_t* seen, int32_t C, float* dist, double* acc, float* loss, void* stream) {
  return proto_dist_common(false, feats, B, D, h, w, labels, lab_h, lab_w, mu, seen, C, dist, acc, loss, nullptr,
                           nullptr, 0, static_cast<cudaStream_t>(stream));
}

int pfst_proto_dist_bwd(const float* feats, int64_t B, int32_t D, int32_t h, int32_t w,
                        const int64_t* labels, int32_t lab_h, int32_t lab_w, const float* mu,
                        const uint8_t* seen, int32_t C, const float* dist, const double* acc,
                        const float* grad_loss, float* grad_feats, int32_t accumulate, void* stream) {
  return proto_dist_common(true, feats, B, D, h, w, labels, lab_h, lab_w, mu, seen, C, const_cast<float*>(dist),
                           const_cast<double*>(acc), nullptr, grad_loss, grad_feats, accumulate,
                           static_cast<cudaStream_t>(stream));
}

int pfst_proto_dist_fwd_lbl(const float* feats, int64_t B, int32_t D, int32_t h, int32_t w,
                            const void* labels, int32_t label_dtype, int32_t lab_h, int32_t lab_w, const float* mu,
                            const uint8_t* seen, int32_t C, float* dist, double* acc, float* loss, void* stream) {
  if (label_dtype == PFST_DT_I64)
    return pfst_proto_dist_fwd(feats, B, D, h, w, static_cast<const int64_t*>(labels), lab_h, lab_w, mu, seen, C,
                               dist, acc, loss, stream);
  if (label_dtype == PFST_DT_U8)
    return proto_dist_common(false, feats, B, D, h, w, static_cast<const uint8_t*>(labels), lab_h, lab_w, mu, seen,
                             C, dist, acc, loss, nullptr, nullptr, 0, static_cast<cudaStream_t>(stream));
  return PFST_ERR_UNSUPPORTED;
}

int pfst_proto_dist_bwd_lbl(const float* feats, int64_t B, int32_t D, int32_t h, int32_t w,
                            const void* labels, int32_t label_dtype, int32_t lab_h, int32_t lab_w, const float* mu,
                            const uint8_t* seen, int32_t C, const float* dist, const double* acc,
                            const float* grad_loss, float* grad_feats, int32_t accumulate, void* stream) {
  if (label_dtype == PFST_DT_I64)
    return pfst_proto_dist_bwd(feats, B, D, h, w, static_cast<const int64_t*>(labels), lab_h, lab_w, mu, seen, C,
                               dist, acc, grad_loss, grad_feats, accumulate, stream);
  if (label_dtype == PFST_DT_U8)
    return proto_dist_common(true, feats, B, D, h, w, static_cast<const uint8_t*>(labels), lab_h, lab_w, mu, seen,
                             C, const_cast<float*>(dist), const_cast<double*>(acc), nullptr, grad_loss, grad_feats,
                             accumulate, static_cast<cudaStream_t>(stream));
  return PFST_ERR_UNSUPPORTED;
}

int pfst_proto_dist_all(const float* feats, int64_t B, int32_t D, int32_t h, int32_t w, const float* mu,
                        int32_t C, float* out, void* stream) {
  if (!feats || !mu || !out || B < 0 || D < 1 || h < 1 || w < 1 || C < 1) return PFST_ERR_INVALID_ARG;
  const size_t smem = (size_t)C * D * sizeof(float);
  if (smem > 200 * 1024) return PFST_ERR_UNSUPPORTED;
  const int64_t total = B * h * w;
  if (total == 0) return PFST_OK;
  PFST_CUDA_TRY(cudaFuncSetAttribute(pfst::proto_dist_all_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)smem), "pfst_proto_dist_all/attr");
  int64_t grid = (total + pfst::kPrThreads - 1) / pfst::kPrThreads;
  const int64_t cap = (int64_t)pfst::kNumSMs * 4;
  if (grid > cap) grid = cap;
  pfst::proto_dist_all_kernel<<<(unsigned)grid, pfst::kPrThreads, smem, static_cast<cudaStream_t>(stream)>>>(
      feats, (int)B, D, h, w, mu, C, out);
  PFST_CHECK_LAUNCH("pfst_proto_dist_all");
  return PFST_OK;
}

}  // extern "C"
