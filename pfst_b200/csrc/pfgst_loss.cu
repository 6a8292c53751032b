// L1, L3-L6 — the per-pixel part of PFGSTLoss, forward statistics and backward maps.
//
// Reference: rsiseg/models/losses/pfgst_loss.py
//   forward :44-140, get_cross_prob_map_diag :142-159, get_sim_losses :203-234
// (SURVEY.md Appendix B restates it per pixel). The reference runs ~60 ATen
// kernels with 3+ host syncs (boolean-mask gathers, `if ignore_mask.sum() > 1`);
// here ONE kernel reduces everything into 9 fp64 sums (the last block turns them
// into the six losses on the device) and ONE backward kernel produces
//   * coef (B,9,fh,fw): per-pixel coefficients of the gather-form gradient of the
//     source cosine statistics w.r.t. x_src (consumed by pfst_neigh_grad), and
//   * grad_logits: d(loss_sim_pos + loss_sim_neg)/d logits_trg through p only
//     (q is detached: detach_unfold=True, configs/pfst/*.py:44).
//
// Everything here works on maps of (B, few, g, g) floats — a few MB; the cost is
// launch latency, not bandwidth. The heavy tensors are touched by neigh.cu only.
#include <math.h>
#include <stdlib.h>

#include "common.cuh"

namespace pfst {

constexpr int kMaxC = 64;   // classes held in registers per pixel

struct LossParams {
  // neighbourhood dot maps from pfst_neigh_dots: (ksplit, 2, B, 5, fh, fw); tensor 0 = x_ema, 1 = x_src
  const float* dots;
  int ksplit;
  int B, fh, fw, up;          // feature grid, loss grid = feature grid * up
  const float* logits;        // (B, C, lh, lw) student logits on the mixed image
  int C, lh, lw;
  float lscale_h, lscale_w;   // torch nearest: src = min(floor(dst * scale), in - 1)
  const void* gt;             // (B,1,gt_h,gt_w) source labels, int64 or uint8 (prep kernel's L)
  const void* mix;            // (B,1,gt_h,gt_w) ClassMix masks, same dtype
  int gt_h, gt_w;
  float gscale_h, gscale_w;
  int gh, gw;                 // loss grid
  int dil;                    // dilation on the loss grid (feature-grid dilation = dil / up)
  int top_k;
  float w_src_pos, w_src_neg, w_src_pos_std, w_src_neg_std, w_sim_pos, w_sim_neg;
  // workspace written by the prep kernel, read by the statistics / backward kernels
  float* dm;                  // (2, B, 5, fh, fw)  dots summed over the channel splits
  float* invn;                // (2, B, fh, fw)     1 / max(|x|, 1e-8)
  float* prob;                // (B, C, gh, gw)     softmax of the resampled logits
  uint8_t* lab;               // (B, gh, gw)        resampled source label (0..255)
  uint8_t* flags;             // (B, gh, gw)        bit0 = gt != 255, bit1 = target pixel (mix mask == 0)
  long long* raw;             // [16] integer accumulators of the statistics kernel (see kFix) + block counter
  // options beyond the shipped configuration (pfgst_loss.py:16-18)
  int gauss;                  // sim_type: 0 = 'cosine', 1 = 'gaussian' exp(-|x_n - x_m|^2 / sigma^2) (:189-191)
  float inv_sigma2;           // 1 / sigma^2
  const float* logits_q;      // cross_prob_type='ema' (:161-178): teacher logits (B,C,gh,gw) or null
  float* prob_q;              // (B,C,gh,gw) softmax of logits_q (workspace) or null: q = unfold(prob_q)
  float* dcp;                 // detach_unfold=False (:148-149): (B,9,gh,gw) d loss / d cross-prob (workspace) or null
  int n_top, n_bot;           // taps kept by the two top-k selections: top_k + 1 / top_k, or 9 / 9 for top_k=None (:215-217)
  int src_mode;               // src_loss_type (:110-135): 0 'mean_std', 1 'margin', 2 'margin2'
  float margin_pos, margin_neg;
  int zfill;                  // backward: L > 0 = the logits are exactly L x the loss grid; every loss pixel then writes
                              // its whole L x L cell of grad_logits (value at the sampled logit, zeros elsewhere): no memset
};

__device__ __forceinline__ int nearest_src(int dst, float scale, int in) {
  const int s = (int)floorf((float)dst * scale);
  return s < in - 1 ? s : in - 1;
}

__host__ __device__ inline size_t ws_floats(int B, int C, int fh, int fw, int up) {
  const size_t fplane = (size_t)fh * fw, gplane = fplane * up * up;
  return (size_t)2 * B * 5 * fplane + (size_t)2 * B * fplane + (size_t)B * C * gplane;
}

// ---- prep: everything that is per-pixel (not per-neighbourhood), computed once --------
// Two independent block ranges in one launch: [0, blocks_a) merge the channel-split dot
// maps (one thread per (tensor, image, map, pixel); map 0 also yields the inverse norm),
// the rest resample labels / masks and take the softmax (one thread per loss-grid pixel).
constexpr int kPrepThreads = 128;

template <int CMAX, class L>
__global__ void __launch_bounds__(kPrepThreads)
pfgst_loss_prep_kernel(const LossParams P, int blocks_a) {
  const int fplane = P.fh * P.fw, gplane = P.gh * P.gw;       // per-image planes: 32-bit offsets
  if (blockIdx.x == 0 && threadIdx.x < 16) P.raw[threadIdx.x] = 0;     // the statistics kernel starts from zero
  if ((int)blockIdx.x < blocks_a) {
    const int64_t n_a = (int64_t)2 * P.B * 5 * fplane;
    const int64_t i = (int64_t)blockIdx.x * kPrepThreads + threadIdx.x;
    if (i >= n_a) return;
    // i = ((tensor*B + image)*5 + map)*fplane + pixel: the same offset in every split
    const float* src = P.dots + i;
    float a = 0.f;
    if (P.ksplit == 8) {                                      // all partial maps in flight, summed in fixed order
      float v[8];
#pragma unroll
      for (int sp = 0; sp < 8; ++sp) v[sp] = src[sp * n_a];
#pragma unroll
      for (int sp = 0; sp < 8; ++sp) a += v[sp];
    } else {
#pragma unroll 4
      for (int sp = 0; sp < P.ksplit; ++sp) a += src[sp * n_a];   // fixed order: deterministic
    }
    P.dm[i] = a;
    const int64_t tbk = i / fplane;
    if (tbk % 5 == 0) P.invn[(tbk / 5) * fplane + (i - tbk * fplane)] = 1.f / fmaxf(sqrtf(a), 1e-8f);
    return;
  }
  const int64_t i = (int64_t)(blockIdx.x - blocks_a) * kPrepThreads + threadIdx.x;
  if (i >= (int64_t)P.B * gplane) return;
  const int b = (int)(i / gplane);
  const int r = (int)(i - (int64_t)b * gplane);
  const int y = r / P.gw, x = r - y * P.gw;
  const int sy = nearest_src(y, P.gscale_h, P.gt_h), sx = nearest_src(x, P.gscale_w, P.gt_w);
  const int64_t go = ((int64_t)b * P.gt_h + sy) * P.gt_w + sx;
  const int64_t g = static_cast<const L*>(P.gt)[go];
  const int64_t mx = static_cast<const L*>(P.mix)[go];
  // softmax of the nearest-resampled logits (pfgst_loss.py:57, 145): every class plane of the pixel
  // is requested before the first value is used (one memory round trip instead of three per class)
  const int ly = nearest_src(y, P.lscale_h, P.lh), lx = nearest_src(x, P.lscale_w, P.lw);
  const int lplane = P.lh * P.lw;
  const float* z = P.logits + (int64_t)b * P.C * lplane + ly * P.lw + lx;
  float* po = P.prob + (int64_t)b * P.C * gplane + r;
  float zr[CMAX];
#pragma unroll
  for (int c = 0; c < CMAX; ++c) zr[c] = c < P.C ? z[c * lplane] : -INFINITY;
  float m = -INFINITY;
#pragma unroll
  for (int c = 0; c < CMAX; ++c) m = fmaxf(m, zr[c]);
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < CMAX; ++c) {
    if (c < P.C) { zr[c] = expf(zr[c] - m); s += zr[c]; }
  }
  const float inv = 1.f / s;
#pragma unroll
  for (int c = 0; c < CMAX; ++c)
    if (c < P.C) po[c * gplane] = zr[c] * inv;
  P.lab[i] = (uint8_t)(g < 0 ? 0 : (g > 255 ? 255 : g));
  P.flags[i] = (uint8_t)((g != 255 ? 1 : 0) | (mx <= 0 ? 2 : 0));   // (1 - mix) > 0.5
  if (P.logits_q) {     // cross_prob_type='ema': q comes from the teacher's logits, already on the loss grid
    const float* zq = P.logits_q + (int64_t)b * P.C * gplane + r;
    float* pq = P.prob_q + (int64_t)b * P.C * gplane + r;
#pragma unroll
    for (int c = 0; c < CMAX; ++c) zr[c] = c < P.C ? zq[c * gplane] : -INFINITY;
    m = -INFINITY;
#pragma unroll
    for (int c = 0; c < CMAX; ++c) m = fmaxf(m, zr[c]);
    s = 0.f;
#pragma unroll
    for (int c = 0; c < CMAX; ++c) {
      if (c < P.C) { zr[c] = expf(zr[c] - m); s += zr[c]; }
    }
    const float invq = 1.f / s;
#pragma unroll
    for (int c = 0; c < CMAX; ++c)
      if (c < P.C) pq[c * gplane] = zr[c] * invq;
  }
}

// ---- one (tap, pixel) thread: warp = tap k (0..8), lane = pixel of the block's 32 ---------
// The maps are tiny (a few MB); with one thread per pixel the GPU holds ~7 warps per SM and
// the kernels are pure latency. Spreading the nine taps of a pixel over nine warps gives 9x
// the parallelism, coalesced map reads along x, warp-uniform tap branches and no per-thread
// arrays; the taps of a pixel meet in shared memory ([tap][pixel], bank = pixel).
constexpr int kLpPix = 32;                 // pixels per block
constexpr int kLpThreads = 9 * kLpPix;     // nine tap-warps

struct Tap {
  bool in;            // tap inside the loss grid
  float s_ema, s_src; // cos(x[n], x[n+delta_k]) of the teacher / source features, 0 outside
  float inv_m_src;    // 1 / max(|x_src[n+delta_k]|, eps), 0 outside
  bool pos_pair;      // unfold(gt)[k] == gt[n]  (zero padding reads as class 0)
  bool nb_valid;      // gt != 255 at the in-bounds neighbour
  bool trg;           // neighbour is a target pixel (mix mask == 0)
  int gm;             // loss-grid offset of the neighbour inside the image plane
};

struct Center {
  int b, y, x;
  bool valid_src;     // gt != 255
  float inv_n_src;
};

__device__ __forceinline__ void load_tap(const LossParams& P, int k, int b, int y, int x, Center& c, Tap& t) {
  const int64_t fplane = (int64_t)P.fh * P.fw, gplane = (int64_t)P.gh * P.gw;
  const int fy = P.up == 1 ? y : y / P.up, fx = P.up == 1 ? x : x / P.up, fd = P.up == 1 ? P.dil : P.dil / P.up;
  const int fn = fy * P.fw + fx;
  const float* dme = P.dm + ((int64_t)(0 * P.B + b) * 5) * fplane;
  const float* dms = P.dm + ((int64_t)(1 * P.B + b) * 5) * fplane;
  const float* ine = P.invn + (int64_t)(0 * P.B + b) * fplane;
  const float* ins = P.invn + (int64_t)(1 * P.B + b) * fplane;
  const uint8_t* lab = P.lab + (int64_t)b * gplane;
  const uint8_t* flg = P.flags + (int64_t)b * gplane;
  const int gn = y * P.gw + x;
  c.b = b; c.y = y; c.x = x;
  c.valid_src = (flg[gn] & 1) != 0;
  c.inv_n_src = ins[fn];
  const int g0 = lab[gn];
  const int oy = k / 3 - 1, ox = k % 3 - 1;
  const int yy = y + oy * P.dil, xx = x + ox * P.dil;
  t.in = yy >= 0 && yy < P.gh && xx >= 0 && xx < P.gw;
  t.s_ema = 0.f; t.s_src = 0.f; t.inv_m_src = 0.f;
  t.nb_valid = false; t.trg = false; t.gm = 0;
  int gk = 0;          // zero padding of unfold(gt.float())
  if (t.in) {
    const int fm = (fy + oy * fd) * P.fw + (fx + ox * fd);
    float de, ds;
    if (k == 4)      { de = dme[fn]; ds = dms[fn]; }
    // forward taps (k > 4) are stored at n, backward taps at the neighbour (symmetry)
    else if (k > 4)  { de = dme[(k - 4) * fplane + fn]; ds = dms[(k - 4) * fplane + fn]; }
    else             { de = dme[(4 - k) * fplane + fm]; ds = dms[(4 - k) * fplane + fm]; }
    if (P.gauss) {    // exp(-|x_n - x_m|^2 / sigma^2), |x_n - x_m|^2 = |x_n|^2 + |x_m|^2 - 2 x_n.x_m  (>= 0)
      t.s_ema = expf(-fmaxf(dme[fn] + dme[fm] - 2.f * de, 0.f) * P.inv_sigma2);
      t.s_src = expf(-fmaxf(dms[fn] + dms[fm] - 2.f * ds, 0.f) * P.inv_sigma2);
    } else {
      t.inv_m_src = ins[fm];
      t.s_ema = de * (ine[fn] * ine[fm]);
      t.s_src = ds * (c.inv_n_src * t.inv_m_src);
    }
    t.gm = yy * P.gw + xx;
    gk = lab[t.gm];
    const unsigned f = flg[t.gm];
    t.nb_valid = (f & 1u) != 0;
    t.trg = (f & 2u) != 0;
  }
  else if (P.gauss) {   // zero padding of the unfold: the neighbour is the zero vector (cosine: similarity 0)
    t.s_ema = expf(-dme[fn] * P.inv_sigma2);
    t.s_src = expf(-dms[fn] * P.inv_sigma2);
  }
  t.pos_pair = gk == g0;
}

// rank of tap k among the nine similarities of pixel p (column p of s[9][kLpPix]): number of
// taps strictly "before" it in descending / ascending order, ties broken by the lower index.
__device__ __forceinline__ void tap_rank(const float (*s)[kLpPix], int p, int k, int& rank_desc, int& rank_asc) {
  const float sk = s[k][p];
  int rd = 0, ra = 0;
#pragma unroll
  for (int j = 0; j < 9; ++j) {
    const float sj = s[j][p];
    const bool first = j < k;
    rd += (j != k && (sj > sk || (sj == sk && first))) ? 1 : 0;
    ra += (j != k && (sj < sk || (sj == sk && first))) ? 1 : 0;
  }
  rank_desc = rd;
  rank_asc = ra;
}

// stats layout (fp64): 0 n_pos, 1 sum_pos, 2 sumsq_pos, 3 n_neg, 4 sum_neg, 5 sumsq_neg,
//                      6 |Mk|, 7 sum loc_pos, 8 sum loc_neg
constexpr int kNumStats = 9;

__device__ __forceinline__ void finalize_losses(const LossParams& P, const double* st, float* losses) {
  const double n_pos = st[0], n_neg = st[3], mk = st[6];
  const double mean_pos = st[1] / n_pos, mean_neg = st[4] / n_neg;
  const double var_pos = (st[2] - n_pos * mean_pos * mean_pos) / (n_pos - 1.0);
  const double var_neg = (st[5] - n_neg * mean_neg * mean_neg) / (n_neg - 1.0);
  if (P.src_mode == 0) {
    losses[0] = (float)(-mean_pos) * P.w_src_pos;
    losses[1] = (float)(mean_neg) * P.w_src_neg;
    losses[2] = (float)sqrt(var_pos > 0.0 || var_pos != var_pos ? var_pos : 0.0) * P.w_src_pos_std;
    losses[3] = (float)sqrt(var_neg > 0.0 || var_neg != var_neg ? var_neg : 0.0) * P.w_src_neg_std;
  } else {      // margin / margin2 (:117-133): st[1], st[4] hold the sums of the hinge terms; two losses only
    losses[0] = (float)mean_pos * P.w_src_pos;
    losses[1] = (float)mean_neg * P.w_src_neg;
    losses[2] = 0.f;
    losses[3] = 0.f;
  }
  const bool any = mk > 1.0;   // pfgst_loss.py:227  `if ignore_mask.sum() > 1`
  losses[4] = any ? (float)(st[7] / (mk * (double)P.n_top)) * P.w_sim_pos : 0.f;
  losses[5] = any ? (float)(st[8] / (mk * (double)P.n_bot)) * P.w_sim_neg : 0.f;
}

// The nine statistics are accumulated as INTEGERS: counts exactly, sums in fixed point with
// 2^-24 resolution (|value| <= 2, so a warp's 32 values fit an int32 and one REDUX instruction
// reduces them; blocks merge with 64-bit integer atomics). Integer addition is associative: the
// statistics — and with them the six losses — are bit-identical from run to run, and the
// reduction costs 9 instructions per warp instead of ~135 for fp64 shuffles. Rounding error:
// <= 3e-8 absolute per term, i.e. ~1e-10 relative on sums over 10^5 terms.
constexpr float kFix = 16777216.f;              // 2^24
constexpr double kUnfix = 1.0 / 16777216.0;

__device__ __forceinline__ int to_fix(float v, bool& bad) {
  if (!(fabsf(v) <= 4.f)) { bad = true; return 0; }      // NaN / Inf / out of range: reported, not summed
  return __float2int_rn(v * kFix);
}

__global__ void __launch_bounds__(kLpThreads)
pfgst_loss_fwd_kernel(const LossParams P, double* __restrict__ stats, float* __restrict__ losses,
                      float* __restrict__ density, uint8_t* __restrict__ eroded_out) {
  __shared__ float s_se[9][kLpPix];
  __shared__ uint8_t s_ok[9][kLpPix];        // tap in bounds and on a target pixel (erosion)
  __shared__ long long red[kNumStats + 1][9];
  const int k = threadIdx.x >> 5, p = threadIdx.x & 31;     // warp = tap, lane = pixel
  const int64_t plane = (int64_t)P.gh * P.gw;
  // grid = (row segments of 32 pixels, rows, images): no index divisions
  const int b = blockIdx.z, y = blockIdx.y, x = blockIdx.x * kLpPix + p;
  const bool live = x < P.gw;
  const int64_t n = (int64_t)b * plane + (int64_t)y * P.gw + x;
  bool is_pos = false, is_neg = false, in_mk_center = false, bad = false;
  float s_val = 0.f, lp = 0.f, ln = 0.f;

  Center c;
  Tap t;
  if (live) {
    load_tap(P, k, b, y, x, c, t);
    // L4: source pair statistics (pfgst_loss.py:85-113)
    if (c.valid_src) {
      is_pos = t.pos_pair;
      is_neg = !t.pos_pair;
      s_val = t.s_src;
    }
    s_se[k][p] = t.s_ema;
    s_ok[k][p] = (t.in && t.trg) ? 1 : 0;
  } else {
    s_se[k][p] = 0.f;
    s_ok[k][p] = 0;
  }
  __syncthreads();
  if (live) {
    bool er = true;
#pragma unroll
    for (int j = 0; j < 9; ++j) er = er && s_ok[j][p] != 0;
    if (k == 0) {
      float mean_e = 0.f;
#pragma unroll
      for (int j = 0; j < 9; ++j) mean_e += s_se[j][p];
      if (density) density[n] = 1.f - mean_e / 9.f;
      if (eroded_out) eroded_out[n] = er ? 1 : 0;
    }
    // L3 + L5: target consistency terms on Mk (every tap of an Mk pixel is in bounds)
    if (er && c.valid_src) {
      int rd, ra;
      tap_rank(s_se, p, k, rd, ra);
      const bool top = rd < P.n_top, bot = ra < P.n_bot;
      if (top || bot) {
        const float* pn = P.prob + (int64_t)c.b * P.C * plane + (int64_t)c.y * P.gw + c.x;
        const float* pm = (P.prob_q ? P.prob_q : P.prob) + (int64_t)c.b * P.C * plane + t.gm;
        float cp = 0.f;
        {
          const int pl = (int)plane;
          int cc = 0;
          for (; cc + 16 <= P.C; cc += 16) {               // sixteen class planes of both pixels in flight
            float a[16], q[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) { a[u] = pn[(cc + u) * pl]; q[u] = pm[(cc + u) * pl]; }
#pragma unroll
            for (int u = 0; u < 16; ++u) cp = fmaf(a[u], q[u], cp);
          }
          for (; cc + 8 <= P.C; cc += 8) {
            float a[8], q[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) { a[u] = pn[(cc + u) * pl]; q[u] = pm[(cc + u) * pl]; }
#pragma unroll
            for (int u = 0; u < 8; ++u) cp = fmaf(a[u], q[u], cp);
          }
          float a[8], q[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const bool on = cc + u < P.C;
            a[u] = on ? pn[(cc + u) * pl] : 0.f; q[u] = on ? pm[(cc + u) * pl] : 0.f;
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) cp = fmaf(a[u], q[u], cp);
        }
        if (top) lp = t.s_ema * (-cp);
        if (bot) ln = (1.f - t.s_ema) * (-(1.f - cp));
      }
      in_mk_center = k == 4;
    }
  }

  // warp reductions: three ballots and six integer REDUX
  const unsigned full = 0xffffffffu;
  float v1 = s_val, v2 = s_val * s_val;
  if (P.src_mode) {        // hinge terms instead of the similarity itself (margin: linear, margin2: squared)
    const float h = is_pos ? fmaxf(P.margin_pos - s_val, 0.f) : (is_neg ? fmaxf(s_val - P.margin_neg, 0.f) : 0.f);
    v1 = P.src_mode == 2 ? h * h : h;
    v2 = 0.f;
  }
  const int f_s = to_fix(v1, bad), f_s2 = to_fix(v2, bad);
  long long w[kNumStats + 1];
  w[0] = __popc(__ballot_sync(full, is_pos));
  w[1] = __reduce_add_sync(full, is_pos ? f_s : 0);
  w[2] = __reduce_add_sync(full, is_pos ? f_s2 : 0);
  w[3] = __popc(__ballot_sync(full, is_neg));
  w[4] = __reduce_add_sync(full, is_neg ? f_s : 0);
  w[5] = __reduce_add_sync(full, is_neg ? f_s2 : 0);
  w[6] = __popc(__ballot_sync(full, in_mk_center));
  w[7] = __reduce_add_sync(full, to_fix(lp, bad));
  w[8] = __reduce_add_sync(full, to_fix(ln, bad));
  w[9] = __any_sync(full, bad) ? 1 : 0;
  if (p == 0) {
#pragma unroll
    for (int i = 0; i <= kNumStats; ++i) red[i][k] = w[i];
  }
  __syncthreads();
  if (threadIdx.x <= kNumStats) {
    long long v = 0;
    for (int wv = 0; wv < 9; ++wv) v += red[threadIdx.x][wv];
    if (v != 0) atomicAdd(reinterpret_cast<unsigned long long*>(&P.raw[threadIdx.x]), (unsigned long long)v);
    __threadfence();
  }
  // last block converts the integer sums and finalises the six losses on the device
  __shared__ bool is_last;
  __syncthreads();
  if (threadIdx.x == 0)
    is_last = atomicAdd(reinterpret_cast<unsigned long long*>(&P.raw[15]), 1ull) ==
              (unsigned long long)gridDim.x * gridDim.y * gridDim.z - 1;
  __syncthreads();
  if (is_last && threadIdx.x == 0) {
    __threadfence();
    double st[kNumStats];
    for (int i = 0; i < kNumStats; ++i) {
      const long long r = *((volatile long long*)&P.raw[i]);
      st[i] = (i == 0 || i == 3 || i == 6) ? (double)r : (double)r * kUnfix;
    }
    if (*((volatile long long*)&P.raw[kNumStats]) != 0)      // a non-finite similarity: NaN like the reference
      for (int i = 1; i < kNumStats; ++i)
        if (i != 3 && i != 6) st[i] = __longlong_as_double(0x7ff8000000000000ll);
    for (int i = 0; i < kNumStats; ++i) stats[i] = st[i];      // fp64 copy for the backward kernel
    finalize_losses(P, st, losses);
  }
}

// Block = 32 FEATURE-grid pixels x nine taps; loops over the up x up loss-grid pixels of a
// feature pixel (up = 1 unless the features are coarser than the loss grid).
constexpr int kLpMaxOwn = (kMaxC + 8) / 9;     // classes a tap-thread owns in the logits gradient

// UP2 = false: lane = feature pixel, the up x up loss pixels of a feature pixel in a serial loop (any up).
// UP2 = true (up == 2, SeasonNet): lane = LOSS pixel of one row, the two loss rows of a feature row on two
// groups of nine tap-warps, so the four loss pixels of a feature pixel run in parallel; their coefficient
// contributions meet in shared memory and are summed in the serial loop's order (uy, ux).
template <bool UP2>
__global__ void __launch_bounds__(kLpThreads * (UP2 ? 2 : 1), UP2 ? 2 : 3)
pfgst_loss_bwd_kernel(const LossParams P, const double* __restrict__ stats, const float* __restrict__ gout,
                      float* __restrict__ coef, float* __restrict__ grad_logits) {
  constexpr int NR = UP2 ? 2 : 1;
  __shared__ float s_se_[NR][9][kLpPix];
  __shared__ uint8_t s_ok_[NR][9][kLpPix];
  __shared__ float s_bs_[NR][9][kLpPix];           // W * S of every tap (centre-tap coefficient)
  __shared__ float s_dcp_[NR][9][kLpPix];          // d loss / d cross-prob of every tap
  __shared__ int s_gm_[NR][9][kLpPix];             // neighbour offsets (for the class-parallel pass)
  __shared__ float s_dot_[NR][9][kLpPix];
  const int wid = threadIdx.x >> 5, p = threadIdx.x & 31;
  const int ry = UP2 ? wid / 9 : 0, k = UP2 ? wid % 9 : wid;
  float (*s_se)[kLpPix] = s_se_[ry];
  uint8_t (*s_ok)[kLpPix] = s_ok_[ry];
  float (*s_bs)[kLpPix] = s_bs_[ry];
  float (*s_dcp)[kLpPix] = s_dcp_[ry];
  int (*s_gm)[kLpPix] = s_gm_[ry];
  float (*s_dot)[kLpPix] = s_dot_[ry];
  const int64_t fplane = (int64_t)P.fh * P.fw, gplane = (int64_t)P.gh * P.gw;
  // grid = (row segments of 32 feature pixels [UP2: 32 loss pixels], feature rows, images)
  const int b = blockIdx.z, fy = blockIdx.y;
  const int xl = blockIdx.x * kLpPix + p;                     // UP2: loss-grid column; else feature column
  const int fx = UP2 ? xl >> 1 : xl;
  const bool live = UP2 ? xl < P.gw : fx < P.fw;
  const int r = fy * P.fw + fx;

  // the backward constants (fp64 divisions and square roots) once per block, not per thread
  __shared__ float s_k[8];
  __shared__ int s_any;
  if (threadIdx.x == 0) {
    const double n_pos = stats[0], n_neg = stats[3], mk = stats[6];
    const double mean_pos = stats[1] / n_pos, mean_neg = stats[4] / n_neg;
    const double std_pos = sqrt(fmax((stats[2] - n_pos * mean_pos * mean_pos) / (n_pos - 1.0), 0.0));
    const double std_neg = sqrt(fmax((stats[5] - n_neg * mean_neg * mean_neg) / (n_neg - 1.0), 0.0));
    const bool any_ = mk > 1.0;
    // d loss / d S for a positive / negative source pair:  a + c * (S - mean)
    s_k[0] = (float)(-(double)gout[0] * P.w_src_pos / n_pos);
    s_k[1] = (float)((double)gout[2] * P.w_src_pos_std / ((n_pos - 1.0) * std_pos));
    s_k[2] = (float)((double)gout[1] * P.w_src_neg / n_neg);
    s_k[3] = (float)((double)gout[3] * P.w_src_neg_std / ((n_neg - 1.0) * std_neg));
    s_k[4] = (float)mean_pos;
    s_k[5] = (float)mean_neg;
    if (P.src_mode) {       // hinge losses: d loss / d S = -/+ a [* 2 relu] (applied per pair below)
      s_k[0] = (float)((double)gout[0] * P.w_src_pos / n_pos);
      s_k[2] = (float)((double)gout[1] * P.w_src_neg / n_neg);
      s_k[1] = s_k[3] = 0.f;
    }
    s_k[6] = any_ ? (float)((double)gout[4] * P.w_sim_pos / (mk * (double)P.n_top)) : 0.f;
    s_k[7] = any_ ? (float)((double)gout[5] * P.w_sim_neg / (mk * (double)P.n_bot)) : 0.f;
    s_any = any_ ? 1 : 0;
  }
  // (no barrier yet: the first pixel's map loads are issued while thread 0 does the fp64 arithmetic)
  float a_pos = 0.f, c_pos = 0.f, a_neg = 0.f, c_neg = 0.f, fmean_pos = 0.f, fmean_neg = 0.f, g_pos = 0.f, g_neg = 0.f;
  bool want_logits = false;     // block-uniform

  float cf = 0.f;
  const int n_u = UP2 ? 1 : P.up;
  for (int uy = 0; uy < n_u; ++uy)
    for (int ux = 0; ux < n_u; ++ux) {
      const int y = UP2 ? fy * 2 + ry : fy * P.up + uy, x = UP2 ? xl : fx * P.up + ux;
      Center c;
      Tap t;
      float bs = 0.f;
      c.valid_src = false; c.inv_n_src = 0.f; c.b = b; c.y = y; c.x = x;
      t.in = false; t.s_ema = 0.f; t.trg = false; t.gm = 0;
      if (live) load_tap(P, k, b, y, x, c, t);
      if (uy == 0 && ux == 0) {
        __syncthreads();
        a_pos = s_k[0]; c_pos = s_k[1]; a_neg = s_k[2]; c_neg = s_k[3];
        fmean_pos = s_k[4]; fmean_neg = s_k[5]; g_pos = s_k[6]; g_neg = s_k[7];
        // (detach_unfold=False: the d loss / d cross-prob maps are always written, zeros included)
        want_logits = P.dcp ? true : (grad_logits != nullptr && (s_any != 0 || P.zfill));
      }
      if (live) {
        // --- x_src: gather-form coefficients (SURVEY.md Appendix B step 6) ---
        if (k != 4 && (t.in || P.gauss)) {
          const float S = t.s_src;
          float g;
          if (P.src_mode == 0) {
            g = t.pos_pair ? a_pos + c_pos * (S - fmean_pos) : a_neg + c_neg * (S - fmean_neg);
          } else {          // relu'(0) = 0 as torch
            const float h = t.pos_pair ? P.margin_pos - S : S - P.margin_neg;
            const float d = h > 0.f ? (P.src_mode == 2 ? 2.f * h : 1.f) : 0.f;
            g = t.pos_pair ? -a_pos * d : a_neg * d;
          }
          // the pair (n, m) is counted once from n (if n is valid) and once from m (if m is valid);
          // a padded (zero-vector) neighbour only from n, and only the Gaussian similarity depends on x_n then
          const float W = g * ((c.valid_src ? 1.f : 0.f) + ((t.in && t.nb_valid) ? 1.f : 0.f));
          // cosine: dS/dx_n = x_m / (|n||m|) - S x_n / |n|^2;  gaussian: dS/dx_n = (2/sigma^2) S (x_m - x_n)
          if (t.in) cf += P.gauss ? W * S * (2.f * P.inv_sigma2) : W * c.inv_n_src * t.inv_m_src;
          bs = W * S;
        }
      }
      s_bs[k][p] = bs;
      s_se[k][p] = t.s_ema;
      s_ok[k][p] = (live && t.in && t.trg) ? 1 : 0;
      s_gm[k][p] = t.gm;
      __syncthreads();
      if (live && k == 4) {
        float bsum = 0.f;
#pragma unroll
        for (int j = 0; j < 9; ++j) bsum += s_bs[j][p];
        cf -= P.gauss ? bsum * (2.f * P.inv_sigma2) : bsum * c.inv_n_src * c.inv_n_src;
      }
      if (want_logits) {
        // --- logits_trg: through p only (q detached) ---
        bool er = live;
#pragma unroll
        for (int j = 0; j < 9; ++j) er = er && s_ok[j][p] != 0;
        const bool in_mk = er && c.valid_src;
        float dcp = 0.f;
        if (in_mk) {
          int rd, ra;
          tap_rank(s_se, p, k, rd, ra);
          const bool top = rd < P.n_top, bot = ra < P.n_bot;
          // d/dcp of  -S*cp  and of  -(1-S)*(1-cp)
          dcp = (top ? -t.s_ema * g_pos : 0.f) + (bot ? (1.f - t.s_ema) * g_neg : 0.f);
        }
        s_dcp[k][p] = dcp;
        if (P.dcp && live) P.dcp[((int64_t)b * 9 + k) * gplane + y * P.gw + x] = dcp;
        __syncthreads();
        // class-parallel: this thread owns classes k, k+9, ... of pixel p
        float dp[kLpMaxOwn], pc[kLpMaxOwn];
        float part = 0.f;
        const float* pb = P.prob + (int64_t)b * P.C * gplane;
        const float* pbq = (P.prob_q ? P.prob_q : P.prob) + (int64_t)b * P.C * gplane;   // q = neighbours' distribution
        if (in_mk && !P.dcp) {
#pragma unroll
          for (int j = 0; j < kLpMaxOwn; ++j) {
            const int cc = k + 9 * j;
            dp[j] = 0.f; pc[j] = 0.f;
            if (cc < P.C) {
              // all nine neighbour probabilities requested at once (zero-weight taps read a valid
              // address and are dropped by the select: 0 * NaN must not leak)
              const float* pcl = pbq + (int64_t)cc * gplane;
              float q[9];
#pragma unroll
              for (int kk = 0; kk < 9; ++kk) q[kk] = pcl[s_gm[kk][p]];
              pc[j] = pb[(int64_t)cc * gplane + y * P.gw + x];
              float d = 0.f;
#pragma unroll
              for (int kk = 0; kk < 9; ++kk) {
                const float w = s_dcp[kk][p];
                d = w != 0.f ? fmaf(w, q[kk], d) : d;
              }
              dp[j] = d;
              part = fmaf(pc[j], d, part);
            }
          }
        }
        s_dot[k][p] = part;
        __syncthreads();
        if (P.zfill && live) {
          // the whole L x L logit cell of this loss pixel (nearest sampling reads its first element)
          float dot = 0.f;
#pragma unroll
          for (int j = 0; j < 9; ++j) dot += s_dot[j][p];
          const int L = P.zfill;
          float* gz = grad_logits + ((int64_t)b * P.C * P.lh + L * y) * P.lw + L * x;
          const int lplane = P.lh * P.lw;
#pragma unroll
          for (int j = 0; j < kLpMaxOwn; ++j) {
            const int cc = k + 9 * j;
            if (cc < P.C) {
              const float v = in_mk ? pc[j] * (dp[j] - dot) : 0.f;
              for (int dy = 0; dy < L; ++dy)
                for (int dx = 0; dx < L; ++dx) gz[cc * lplane + dy * P.lw + dx] = (dy | dx) == 0 ? v : 0.f;
            }
          }
        } else if (in_mk && !P.dcp) {
          float dot = 0.f;
#pragma unroll
          for (int j = 0; j < 9; ++j) dot += s_dot[j][p];
          const int sy = nearest_src(y, P.lscale_h, P.lh), sx = nearest_src(x, P.lscale_w, P.lw);
          float* gz = grad_logits + ((int64_t)b * P.C * P.lh + sy) * P.lw + sx;
          const int64_t lplane = (int64_t)P.lh * P.lw;
          // several loss pixels can map to one logit only when the logits are UP-sampled
          // (lscale < 1); accumulate then, plain store otherwise
          const bool shared_src = P.lscale_h < 1.f || P.lscale_w < 1.f;
#pragma unroll
          for (int j = 0; j < kLpMaxOwn; ++j) {
            const int cc = k + 9 * j;
            if (cc < P.C) {
              const float v = pc[j] * (dp[j] - dot);
              if (shared_src) atomicAdd(gz + cc * lplane, v); else gz[cc * lplane] = v;
            }
          }
        }
      }
      __syncthreads();     // the shared arrays are rewritten by the next loss pixel
    }
  if (UP2) {
    // the four loss pixels of a feature pixel: (uy, ux) order of the serial loop
    s_dot_[ry][k][p] = cf;
    __syncthreads();
    if (ry == 0 && (p & 1) == 0 && live && coef)
      coef[((int64_t)b * 9 + k) * fplane + r] =
          ((s_dot_[0][k][p] + s_dot_[0][k][p + 1]) + s_dot_[1][k][p]) + s_dot_[1][k][p + 1];
  } else {
    if (live && coef) coef[((int64_t)b * 9 + k) * fplane + r] = cf;
  }
}

// ---- detach_unfold=False (pfgst_loss.py:148-149 not taken): cross_prob = p * unfold(p) sends gradient
// through BOTH factors. With D_k(n) = d loss / d cross_prob_k(n) (written by the kernel above),
//   d loss / d p_m[c] = sum_k D_k(m) p_{m+delta_k}[c]  +  sum_k D_k(m-delta_k) p_{m-delta_k}[c]
// (the second sum is the pixel's role as somebody's neighbour; padded neighbours carry no gradient),
// followed by the soft-max backward. One thread per loss pixel; off the shipped path.
template <int CMAX>
__global__ void __launch_bounds__(128)
pfgst_loss_unfold_grad_kernel(const LossParams P, float* __restrict__ grad_logits) {
  const int gplane = P.gh * P.gw;
  const int64_t i = (int64_t)blockIdx.x * 128 + threadIdx.x;
  if (i >= (int64_t)P.B * gplane) return;
  const int b = (int)(i / gplane), r = (int)(i - (int64_t)b * gplane);
  const int y = r / P.gw, x = r - y * P.gw;
  const float* pb = P.prob + (int64_t)b * P.C * gplane;
  const float* db = P.dcp + (int64_t)b * 9 * gplane;
  float dp[CMAX];
#pragma unroll
  for (int c = 0; c < CMAX; ++c) dp[c] = 0.f;
  bool touched = false;
  for (int k = 0; k < 9; ++k) {
    const int oy = (k / 3 - 1) * P.dil, ox = (k % 3 - 1) * P.dil;
#pragma unroll
    for (int side = 0; side < 2; ++side) {
      // side 0: this pixel as the centre of its own tap k; side 1: as the neighbour of the pixel at -delta_k
      const int sy = side == 0 ? y : y - oy, sx = side == 0 ? x : x - ox;   // pixel whose D_k is used
      const int py = side == 0 ? y + oy : sy, px = side == 0 ? x + ox : sx; // pixel whose p multiplies it
      if (sy < 0 || sy >= P.gh || sx < 0 || sx >= P.gw || py < 0 || py >= P.gh || px < 0 || px >= P.gw) continue;
      const float w = db[k * gplane + sy * P.gw + sx];
      if (w == 0.f) continue;
      touched = true;
      const float* pp = pb + py * P.gw + px;
#pragma unroll
      for (int c = 0; c < CMAX; ++c)
        if (c < P.C) dp[c] = fmaf(w, pp[c * gplane], dp[c]);
    }
  }
  if (!touched) return;      // grad_logits was zero-filled
  float pc[CMAX], dot = 0.f;
#pragma unroll
  for (int c = 0; c < CMAX; ++c) {
    pc[c] = c < P.C ? pb[c * gplane + r] : 0.f;
    dot = fmaf(pc[c], dp[c], dot);
  }
  const int ly = nearest_src(y, P.lscale_h, P.lh), lx = nearest_src(x, P.lscale_w, P.lw);
  const int lplane = P.lh * P.lw;
  float* gz = grad_logits + (int64_t)b * P.C * lplane + ly * P.lw + lx;
  const bool shared_src = P.lscale_h < 1.f || P.lscale_w < 1.f;
#pragma unroll
  for (int c = 0; c < CMAX; ++c) {
    if (c < P.C) {
      const float v = pc[c] * (dp[c] - dot);
      if (shared_src) atomicAdd(gz + c * lplane, v); else gz[c * lplane] = v;
    }
  }
}

// bits of the `options` argument of pfst_pfgst_loss_ws_bytes / _fwd / _bwd
constexpr int kOptGauss = 1, kOptProbEma = 2, kOptUnfoldGrad = 4, kOptMargin = 8, kOptMargin2 = 16;

static int fill_params(LossParams& P, const float* dots, int ksplit, int64_t B, int fh, int fw, int up,
                       const float* logits, int C, int lh, int lw, float lsh, float lsw, const void* gt,
                       const void* mix, int gt_h, int gt_w, int dil, int top_k, const float* w6, void* ws) {
  if (!dots || !logits || !gt || !mix || !w6 || !ws) return PFST_ERR_INVALID_ARG;
  if (B < 0 || B > 0x7fffffff || fh < 1 || fw < 1 || up < 1 || C < 1 || lh < 1 || lw < 1 || gt_h < 1 || gt_w < 1)
    return PFST_ERR_INVALID_ARG;
  if (C > kMaxC) return PFST_ERR_UNSUPPORTED;
  if (dil < 1 || dil % up != 0 || top_k < 0 || top_k > 4 || ksplit < 1) return PFST_ERR_INVALID_ARG;   // top_k 0 = None
  P.dots = dots; P.ksplit = ksplit; P.B = (int)B; P.fh = fh; P.fw = fw; P.up = up;
  P.logits = logits; P.C = C; P.lh = lh; P.lw = lw; P.lscale_h = lsh; P.lscale_w = lsw;
  P.gt = gt; P.mix = mix; P.gt_h = gt_h; P.gt_w = gt_w;
  P.gh = fh * up; P.gw = fw * up;
  // F.interpolate(size=...) nearest: scale = (float)in / out
  P.gscale_h = (float)gt_h / (float)P.gh; P.gscale_w = (float)gt_w / (float)P.gw;
  P.dil = dil; P.top_k = top_k;
  P.w_src_pos = w6[0]; P.w_src_neg = w6[1]; P.w_src_pos_std = w6[2]; P.w_src_neg_std = w6[3];
  P.w_sim_pos = w6[4]; P.w_sim_neg = w6[5];
  const size_t fplane = (size_t)fh * fw, gplane = (size_t)P.gh * P.gw;
  P.dm = static_cast<float*>(ws);
  P.invn = P.dm + (size_t)2 * B * 5 * fplane;
  P.prob = P.invn + (size_t)2 * B * fplane;
  P.lab = reinterpret_cast<uint8_t*>(P.prob + (size_t)B * C * gplane);
  P.flags = P.lab + (size_t)B * gplane;
  P.raw = reinterpret_cast<long long*>((reinterpret_cast<uintptr_t>(P.flags + (size_t)B * gplane) + 15) & ~(uintptr_t)15);
  P.gauss = 0; P.inv_sigma2 = 0.f; P.logits_q = nullptr; P.prob_q = nullptr; P.dcp = nullptr; P.zfill = 0;
  P.n_top = top_k ? top_k + 1 : 9; P.n_bot = top_k ? top_k : 9;
  P.src_mode = 0; P.margin_pos = 0.f; P.margin_neg = 0.f;
  return PFST_OK;
}

// the optional regions follow the 16 accumulators: prob_q (B,C,gh,gw), then dcp (B,9,gh,gw)
static int apply_options(LossParams& P, int options, float sigma, const float* logits_ema, const float* margin) {
  if (options & ~(kOptGauss | kOptProbEma | kOptUnfoldGrad | kOptMargin | kOptMargin2)) return PFST_ERR_INVALID_ARG;
  if (options & (kOptMargin | kOptMargin2)) {
    if (!margin || ((options & kOptMargin) && (options & kOptMargin2))) return PFST_ERR_INVALID_ARG;
    // the hinge terms are summed in 2^-24 fixed point with |value| <= 4: similarities lie in [-1, 1]
    if (!(fabsf(margin[0]) <= 1.f) || !(fabsf(margin[1]) <= 1.f)) return PFST_ERR_UNSUPPORTED;
    P.src_mode = (options & kOptMargin2) ? 2 : 1;
    P.margin_pos = margin[0];
    P.margin_neg = margin[1];
  }
  float* extra = reinterpret_cast<float*>(P.raw + 16);
  const size_t gplane = (size_t)P.gh * P.gw;
  if (options & kOptGauss) {
    if (!(sigma > 0.f)) return PFST_ERR_INVALID_ARG;
    P.gauss = 1;
    P.inv_sigma2 = 1.f / (sigma * sigma);
  }
  if (options & kOptProbEma) {
    if (!logits_ema) return PFST_ERR_INVALID_ARG;
    P.logits_q = logits_ema;
    P.prob_q = extra;
    extra += (size_t)P.B * P.C * gplane;
  }
  // q from the teacher carries no gradient: detach_unfold is irrelevant then (pfgst_loss.py:161-178)
  if ((options & kOptUnfoldGrad) && !(options & kOptProbEma)) P.dcp = extra;
  return PFST_OK;
}

}  // namespace pfst

extern "C" {

int64_t pfst_pfgst_loss_ws_bytes(int64_t B, int32_t C, int32_t fh, int32_t fw, int32_t up, int32_t options) {
  if (B < 0 || C < 1 || fh < 1 || fw < 1 || up < 1) return 0;
  const size_t gplane = (size_t)fh * fw * up * up;
  size_t extra = 0;
  if (options & pfst::kOptProbEma) extra += (size_t)B * C * gplane * sizeof(float);
  else if (options & pfst::kOptUnfoldGrad) extra += (size_t)B * 9 * gplane * sizeof(float);
  return (int64_t)(pfst::ws_floats((int)B, C, fh, fw, up) * sizeof(float) + 2 * (size_t)B * gplane + 16 +
                   16 * sizeof(long long) + 16 + extra);
}

int pfst_pfgst_loss_fwd(const float* dots, int32_t ksplit, int64_t B, int32_t fh, int32_t fw, int32_t up,
                        const float* logits, int32_t C, int32_t lh, int32_t lw, float lscale_h,
                        float lscale_w, const void* gt, const void* mix, int32_t gt_h, int32_t gt_w,
                        int32_t dilation, int32_t top_k, const float* weights6_host, void* workspace,
                        double* stats, float* losses, float* density, uint8_t* eroded, int32_t options,
                        float sigma, const float* logits_ema, const float* margin_host, int32_t label_dtype,
                        void* stream) {
  return pfst::with_label_dt(label_dtype, [&](auto l) {
    using L = decltype(l);
    pfst::LossParams P;
    int rc = pfst::fill_params(P, dots, ksplit, B, fh, fw, up, logits, C, lh, lw, lscale_h, lscale_w, gt,
                               mix, gt_h, gt_w, dilation, top_k, weights6_host, workspace);
    if (rc != PFST_OK) return rc;
    rc = pfst::apply_options(P, options, sigma, logits_ema, margin_host);
    if (rc != PFST_OK) return rc;
    if (!stats || !losses) return PFST_ERR_INVALID_ARG;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    // (the prep kernel zeroes the integer accumulators: no memset node between the kernels)
    const int64_t total = (int64_t)P.B * P.gh * P.gw;
    if (total == 0) return PFST_OK;
    {
      const int64_t n_a = (int64_t)2 * P.B * 5 * fh * fw;
      const int64_t blocks_a = (n_a + pfst::kPrepThreads - 1) / pfst::kPrepThreads;
      const int64_t blocks_b = (total + pfst::kPrepThreads - 1) / pfst::kPrepThreads;
      if (blocks_a + blocks_b > 0x7fffffffll) return PFST_ERR_UNSUPPORTED;
      auto prep = C <= 8 ? pfst::pfgst_loss_prep_kernel<8, L>
                         : (C <= 40 ? pfst::pfgst_loss_prep_kernel<40, L> : pfst::pfgst_loss_prep_kernel<pfst::kMaxC, L>);
      prep<<<(unsigned)(blocks_a + blocks_b), pfst::kPrepThreads, 0, s>>>(P, (int)blocks_a);
      PFST_CHECK_LAUNCH("pfst_pfgst_loss_fwd/prep");
    }
    if (P.gh > 65535 || P.B > 65535) return PFST_ERR_UNSUPPORTED;
    const dim3 grid((unsigned)((P.gw + pfst::kLpPix - 1) / pfst::kLpPix), (unsigned)P.gh, (unsigned)P.B);
    pfst::pfgst_loss_fwd_kernel<<<grid, pfst::kLpThreads, 0, s>>>(
        P, stats, losses, density, eroded);
    PFST_CHECK_LAUNCH("pfst_pfgst_loss_fwd");
    return PFST_OK;
  });
}

// The backward reads the per-pixel label classes the forward's prep kernel left in the workspace, never gt
// or mix themselves: the label dtype is only validated here.
int pfst_pfgst_loss_bwd(const float* dots, int32_t ksplit, int64_t B, int32_t fh, int32_t fw, int32_t up,
                        const float* logits, int32_t C, int32_t lh, int32_t lw, float lscale_h,
                        float lscale_w, const void* gt, const void* mix, int32_t gt_h, int32_t gt_w,
                        int32_t dilation, int32_t top_k, const float* weights6_host, const void* workspace,
                        const double* stats, const float* grad_losses, float* coef, float* grad_logits,
                        int32_t options, float sigma, const float* logits_ema, const float* margin_host,
                        int32_t label_dtype, void* stream) {
  const int tag_rc = pfst::with_label_dt(label_dtype, [](auto) { return PFST_OK; });
  if (tag_rc != PFST_OK) return tag_rc;
  pfst::LossParams P;
  int rc = pfst::fill_params(P, dots, ksplit, B, fh, fw, up, logits, C, lh, lw, lscale_h, lscale_w, gt,
                             mix, gt_h, gt_w, dilation, top_k, weights6_host, const_cast<void*>(workspace));
  if (rc != PFST_OK) return rc;
  rc = pfst::apply_options(P, options, sigma, logits_ema, margin_host);
  if (rc != PFST_OK) return rc;
  if (!grad_logits) P.dcp = nullptr;        // nothing consumes the d loss / d cross-prob maps then
  {
    // logits exactly L x the loss grid (the shipped configs: L = 2, or 1 without downscale): the kernel covers
    // every element of grad_logits itself and the memset node in front of it is dropped
    const int L = (int)lscale_h;
    if (grad_logits && !P.dcp && L >= 1 && L <= 4 && (float)L == lscale_h && lscale_w == lscale_h &&
        lh == L * P.gh && lw == L * P.gw)
      P.zfill = L;
  }
  if (!stats || !grad_losses || (!coef && !grad_logits)) return PFST_ERR_INVALID_ARG;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (grad_logits && !P.zfill)
    PFST_CUDA_TRY(cudaMemsetAsync(grad_logits, 0, sizeof(float) * (size_t)P.B * C * lh * lw, s),
                  "pfst_pfgst_loss_bwd/memset");
  const int64_t total = (int64_t)P.B * fh * fw;
  if (total == 0) return PFST_OK;
  if (fh > 65535 || P.B > 65535) return PFST_ERR_UNSUPPORTED;
  static const bool no_up2 = getenv("PFST_LOSS_NO_UP2") != nullptr;       // A/B switch
  if (up == 2 && !no_up2) {
    const dim3 grid2((unsigned)((P.gw + pfst::kLpPix - 1) / pfst::kLpPix), (unsigned)fh, (unsigned)P.B);
    pfst::pfgst_loss_bwd_kernel<true><<<grid2, 2 * pfst::kLpThreads, 0, s>>>(P, stats, grad_losses, coef, grad_logits);
  } else {
    const dim3 grid((unsigned)((fw + pfst::kLpPix - 1) / pfst::kLpPix), (unsigned)fh, (unsigned)P.B);
    pfst::pfgst_loss_bwd_kernel<false><<<grid, pfst::kLpThreads, 0, s>>>(P, stats, grad_losses, coef, grad_logits);
  }
  PFST_CHECK_LAUNCH("pfst_pfgst_loss_bwd");
  if (P.dcp) {      // detach_unfold=False: the logits gradient needs every pixel's d loss / d cross-prob map
    const int64_t n = (int64_t)P.B * P.gh * P.gw;
    auto k2 = C <= 8 ? pfst::pfgst_loss_unfold_grad_kernel<8>
                     : (C <= 40 ? pfst::pfgst_loss_unfold_grad_kernel<40> : pfst::pfgst_loss_unfold_grad_kernel<pfst::kMaxC>);
    k2<<<(unsigned)((n + 127) / 128), 128, 0, s>>>(P, grad_logits);
    PFST_CHECK_LAUNCH("pfst_pfgst_loss_bwd/unfold_grad");
  }
  return PFST_OK;
}

}  // extern "C"
