/*
 * pfst_sm100.h — C ABI of libpfst_sm100.so: hand-written sm_100a (B200) CUDA
 * kernels for the per-iteration self-training hot path of zhu-xlab/PFST.
 *
 * The reference has NO foreign-function interface (it is pure Python/PyTorch);
 * every entry point below names the reference Python code (file:line under the
 * reference checkout) whose arithmetic it replaces. INTEGRATION.md shows the
 * ctypes binding a maintainer of the reference would add.
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes only; all data pointers are DEVICE pointers on
 *     the current CUDA device unless the parameter comment says "host";
 *   - tensors are dense, row-major, in the reference's layouts (NCHW logits /
 *     features, (B,1,H,W) label maps); every entry point that takes label maps takes them as
 *     void* plus an int32 label_dtype tag, PFST_DT_I64 (the reference dtype) or PFST_DT_U8 (the
 *     dtype datasets store); one call's label maps share that dtype. The entry points that read
 *     the EMA teacher's outputs take them as void* plus a float tag, PFST_DT_F32, PFST_DT_F16 or
 *     PFST_DT_BF16. Any other tag returns PFST_ERR_UNSUPPORTED before any other argument check;
 *   - `stream` is a cudaStream_t passed as void*; work is enqueued
 *     asynchronously on it; nothing here synchronises the device, allocates
 *     device memory or throws;
 *   - return value: PFST_OK (0) or a negative PFST_ERR_* code. A failed CUDA
 *     launch leaves its text in pfst_last_cuda_error() (per host thread);
 *   - there is no CPU fallback: on a machine without an sm_100 device the
 *     compute entry points return PFST_ERR_NO_DEVICE / PFST_ERR_CUDA.
 */
#ifndef PFST_SM100_H_
#define PFST_SM100_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PFST_OK 0
#define PFST_ERR_INVALID_ARG (-1)
#define PFST_ERR_UNSUPPORTED (-2)
#define PFST_ERR_CUDA (-3)
#define PFST_ERR_NO_DEVICE (-4)

/* dtype tags for the label-map entry points */
#define PFST_DT_U8 0
#define PFST_DT_I32 1
#define PFST_DT_I64 2
/* dtype tags for the teacher outputs: the EMA teacher's logits and features may be fp32, fp16 or
 * bf16 (a teacher pass run under autocast). Converting fp16 / bf16 to fp32 is exact, so every
 * output equals the fp32 output on the upcast tensor. */
#define PFST_DT_F32 16
#define PFST_DT_F16 17
#define PFST_DT_BF16 18

/* ---- library ------------------------------------------------------------ */
const char* pfst_version(void);
const char* pfst_error_string(int code);
const char* pfst_last_cuda_error(void);
/* PFST_OK iff the current device is compute capability 10.x (B200). */
int pfst_device_check(void);
/* cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, stream): the two tiny transfers of M1 (36 B of
 * class-presence bits to pinned host memory, 32 B per image of chosen-class masks back) on an explicit
 * stream, without a host-side stream switch. Host buffers must be pinned for the copy to be async. */
int pfst_copy_async(void* dst, const void* src, int64_t bytes, void* stream);
/* M1, host side (no device work): the per-image class draw of get_class_masks
 * (rsiseg/models/utils/dacs_transforms.py:110-126: `np.random.choice(n, int((n + n % 2) / 2), replace=False)`
 * once per image, n = number of classes present in the batch) replayed from RAW 32-bit outputs of the same
 * numpy MT19937 stream. numpy's legacy choice(replace=False) is permutation(n)[:k], and permutation is a
 * Fisher-Yates shuffle whose index draws are masked rejection samples of successive 32-bit outputs
 * (`RandomState.bytes` / the MT19937 bit generator's `random_raw` hand out exactly those words; one per
 * uint64 element, low 32 bits, as `random_raw` returns them). Resumable: `state` (258 int32: image index,
 * swap index, permutation) starts as zeros; each call consumes ALL `n_words` new words. If they run out,
 * *words_missing is the least number of further words the batch still needs (the caller draws exactly that
 * many and calls again with the same state: the stream is never over-consumed); when *words_missing = 0
 * the batch is complete and masks (batch x 8 uint32, 256 class bits per image) holds the chosen classes. */
int pfst_classmix_draw(const uint64_t* words, int64_t n_words, const int64_t* classes, int32_t n_classes,
                       int32_t batch, uint32_t* masks, int32_t* state, int64_t* words_missing);

/* ---- E1/E2: EMA mean-teacher update ---------------------------------------
 * Replaces PFGST._init_ema_weights / PFGST._update_ema
 * (rsiseg/models/uda/pfgst.py:105-114, 116-127): a Python loop of
 * `ema[:] = a*ema + (1-a)*p` over ~214 parameter tensors (3 ATen launches
 * each). One launch updates every tensor; arithmetic is the reference's
 * separately-rounded fl(fl(a32*e) + fl(b32*p)) (no FMA contraction).          */

/* a = min(1 - 1/(iter+1), alpha) in double; a32=(float)a, b32=(float)(1.0-a)
 * (pfgst.py:117 + torch's python-scalar -> fp32 conversion). Host only.       */
int pfst_ema_coeffs(int64_t iter, double alpha, float* a32_host, float* b32_host);

/* mode 0: ema = a32*ema + b32*param ; mode 1: ema = param (E1, bit copy).
 * ema_ptrs/param_ptrs/numel: device arrays of n_tensors entries.
 * chunk_tensor/chunk_begin: device arrays of n_chunks entries; chunk i covers
 * elements [chunk_begin[i], min(chunk_begin[i]+chunk_elems, numel[t])) of
 * tensor t = chunk_tensor[i]. chunk_elems must be a multiple of 1024.
 * blocks_per_sm > 0 launches a bounded, persistent grid of 148 * blocks_per_sm blocks that
 * stride over the chunk table (0 = one block per chunk). A small grid leaves registers and
 * issue slots for kernels of other streams: the EMA update is independent of the rest of the
 * step and overlaps its latency-bound kernels.                                  */
int pfst_ema_update_multi(float* const* ema_ptrs, const float* const* param_ptrs,
                          const int64_t* numel, const int32_t* chunk_tensor,
                          const int64_t* chunk_begin, int64_t n_chunks,
                          int32_t chunk_elems, float a32, float b32, int32_t mode,
                          int32_t blocks_per_sm, void* stream);

/* pfst_ema_update_multi's mode 0 arithmetic with the two coefficients read from DEVICE memory
 * (coefs_dev = float[2] {a32, b32}, e.g. uploaded from pinned memory before a graph launch):
 * no per-step host argument, so the launch can sit at any point of a captured CUDA graph. */
int pfst_ema_update_multi_dev(float* const* ema_ptrs, const float* const* param_ptrs,
                              const int64_t* numel, const int32_t* chunk_tensor,
                              const int64_t* chunk_begin, int64_t n_chunks,
                              int32_t chunk_elems, const float* coefs_dev,
                              int32_t blocks_per_sm, void* stream);

/* Same arithmetic over one flat buffer (e.g. a flattened parameter bucket).   */
int pfst_ema_update_flat(float* ema, const float* param, int64_t n, float a32,
                         float b32, int32_t mode, void* stream);

/* ---- S1/S2: pseudo-label generation ----------------------------------------
 * Replaces pfgst.py:259-262 (softmax -> max -> ge(thr)) and the count used for
 * the pseudo-weight at pfgst.py:264-266. One pass over NCHW logits of logit_dtype
 * (PFST_DT_F32, PFST_DT_F16 or PFST_DT_BF16: the teacher pass may run under autocast;
 * torch.softmax is on autocast's fp32 list, so the reference upcasts first). Every value
 * is converted to fp32 once, on load: the outputs equal the fp32 outputs on the upcast logits.
 *   label[b,p] = argmax_c softmax(logits[b,:,p])  (first index on ties, label_dtype)
 *   conf[b,p]  = max_c softmax(...)               (fp32, = 1/sum exp(x-max))
 *   confident  = mode 0: conf >= thr[label]  (reference online rule; thr is one
 *                        scalar broadcast, or a per-class vector)
 *                mode 1: entropy(softmax) < thr[label] (offline class-wise rule,
 *                        rsiseg/datasets/pipelines/loading.py:474-487)
 *   *count     = number of confident pixels (zeroed here, then accumulated)
 *   weight_part (nullable) = confident ? 1.f : 0.f   (thre_type='part', :267-268)
 *   If reject_label >= 0, label is replaced by reject_label where not confident
 *   (loading.py:484 writes 255).
 * thr_per_class: device pointer to C floats, or NULL to use the scalar `thr`.
 * label: PFST_DT_I64 or PFST_DT_U8; uint8 labels need C <= 255 and reject_label <= 255
 * (otherwise PFST_ERR_UNSUPPORTED). An unknown logit_dtype or label_dtype returns
 * PFST_ERR_UNSUPPORTED.                                                         */
int pfst_pseudo_label(const void* logits, int32_t logit_dtype, int64_t B, int32_t C, int64_t HW,
                      float thr, const float* thr_per_class, int32_t mode, int64_t reject_label,
                      void* label, int32_t label_dtype, float* conf, float* weight_part,
                      unsigned long long* count, void* stream);

/* Self-test of the kernel's hand-scheduled exp: *mismatches = number of x[i]
 * (x[i] <= 0) for which it differs bitwise from CUDA's expf. Must be 0.       */
int pfst_selftest_exp(const float* x, int64_t n, unsigned long long* mismatches,
                      void* stream);

/* thre_type='all' (pfgst.py:264-266, 273-276): weight[b,y,x] =
 * (float)((double)*count / (double)ps_size), rows [0,ignore_top) and
 * [H-ignore_bottom,H) zeroed. `count` is read on the device (no host sync).    */
int pfst_pseudo_weight_fill(float* weight, int64_t B, int64_t H, int64_t W,
                            const unsigned long long* count, int64_t ps_size,
                            int32_t ignore_top, int32_t ignore_bottom, void* stream);

/* ---- M1/M2: ClassMix ---------------------------------------------------------
 * Replaces get_class_masks / generate_class_mask / one_mix
 * (rsiseg/models/utils/dacs_transforms.py:110-144) and the per-image mixing
 * loop pfgst.py:287-300.                                                        */

/* presence: device uint32[9]; words 0..7 = bitmask of label values 0..255 that
 * occur anywhere in gt[0..n) (torch.unique of the whole batch, :113); word 8 is
 * set non-zero if any label lies outside [0,255] (never for a uint8 map). Zeroed here.
 * gt: label_dtype PFST_DT_I64 or PFST_DT_U8, else PFST_ERR_UNSUPPORTED.         */
int pfst_class_presence(const void* gt, int32_t label_dtype, int64_t n, uint32_t* presence,
                        void* stream);

/* chosen: device uint32[B*8], per-image bitmask of the classes drawn by the
 * host RNG (np.random.choice, :115-117).
 *   mask        = chosen[b] has bit gt[b,p]                      -> mix_mask
 *   mixed_img   = mask*img + (1-mask)*trg_img  (fp32 arithmetic as one_mix)
 *   mixed_lbl   = mask ? gt : pseudo_label
 *   mixed_weight= mask*1 + (1-mask)*w, w = weight_in[b,p] if weight_in != NULL,
 *                 else the thre_type='all' ratio (float)(count/ps_size) with the
 *                 ignore_top/bottom rows zeroed (pfgst.py:264-277, 295-298).
 * gt, pseudo_label, mixed_lbl and mix_mask are all of label_dtype (PFST_DT_I64 or
 * PFST_DT_U8, else PFST_ERR_UNSUPPORTED).
 * Any output pointer may be NULL to skip it. weight_in may alias mixed_weight.  */
int pfst_class_mix(const void* gt, const uint32_t* chosen, const float* img,
                   const float* trg_img, const void* pseudo_label, const float* weight_in,
                   const unsigned long long* count, int64_t ps_size, int32_t ignore_top,
                   int32_t ignore_bottom, int64_t B, int32_t img_channels, int64_t H, int64_t W,
                   float* mixed_img, void* mixed_lbl, float* mixed_weight, void* mix_mask,
                   int32_t label_dtype, void* stream);

/* one_mix for a caller-supplied mask (dacs_transforms.py:129-144), one image:
 * out[c,p] = mask[p]*a[c,p] + (1-mask[p])*b[c,p]; mask int64 {0,1} of HW entries;
 * dtype 0 = fp32 operands, PFST_DT_I64 = int64 operands.                        */
int pfst_mask_mix(const int64_t* mask, const void* a, const void* b, void* out,
                  int32_t dtype, int64_t channels, int64_t HW, void* stream);

/* ---- L1-L6: PFGST auxiliary loss ----------------------------------------------
 * Replaces PFGSTLoss.forward and its autograd backward
 * (rsiseg/models/losses/pfgst_loss.py:44-234) for the shipped configuration:
 * sim_type='cosine', kernel_size=3, cross_prob_type='trg', src_loss_type='mean_std',
 * detach_unfold=True, feat_level=None. Four launches replace ~60 ATen kernels, two
 * 604 MB im2col buffers and 3+ host syncs:
 *   pfst_neigh_dots      x_ema, x_src  -> five dot-product maps per tensor (:181-201)
 *   pfst_pfgst_loss_fwd  maps, logits, gt, mix masks -> six losses on the device
 *   pfst_pfgst_loss_bwd  upstream grads -> coef maps + grad of logits_trg
 *   pfst_neigh_grad      coef, x_src -> grad of x_src                              */

/* Number of channel splits pfst_neigh_dots uses for this shape (>= 1); the caller
 * sizes `dots` as float[splits][n_tensors][B][5][h][w]. Host only.                 */
int32_t pfst_neigh_dots_splits(int64_t n_tensors, int64_t B, int32_t D, int32_t h,
                               int32_t w);

/* x_a, x_b: (B,D,h,w) fp32 NCHW features (x_b may be NULL: one tensor). For every
 * pixel n: dots[...,0,n] = |x_n|^2 and dots[...,1..4,n] = x_n . x_{n+delta} for
 * delta = (0,+d), (+d,-d), (+d,0), (+d,+d) (rows, cols), 0 outside the image.      */
int pfst_neigh_dots(const float* x_a, const float* x_b, int64_t B, int32_t D, int32_t h,
                    int32_t w, int32_t dilation, float* dots, void* stream);

/* grad_x[b,c,n] = sum_{k=0..8} coef[b,k,n] * x[b,c,n+delta_k], delta_k =
 * ((k/3-1)*d, (k%3-1)*d), zero outside the image. coef: (B,9,h,w).                 */
int pfst_neigh_grad(const float* x, const float* coef, int64_t B, int32_t D, int32_t h,
                    int32_t w, int32_t dilation, float* grad_x, void* stream);

/* pfst_neigh_dots for ONE tensor written into slot `slot` of an `n_slots`-tensor dots
 * buffer of pfst_neigh_dots_splits(1,B,D,h,w) channel splits (the loss reads slot 0 =
 * x_ema, slot 1 = x_src), so the two feature tensors can be processed at different
 * points of the step (x_ema next to the prototype accumulation, x_src next to the
 * prototype distance: the second kernel of each pair then hits the 126 MB L2).
 * x: x_dtype PFST_DT_F32, PFST_DT_F16 or PFST_DT_BF16 (the EMA features of a teacher run
 * under autocast; get_sim_feat pfgst_loss.py:181-201, cosine_similarity is on autocast's
 * fp32 list), else PFST_ERR_UNSUPPORTED. A 16-bit x gives the dot maps of its fp32 upcast
 * bit for bit: the same channel splits, the same per-warp channel order and the same merge
 * order, on every path (TMA, small-plane bulk copy, generic).                          */
int pfst_neigh_dots_slot(const void* x, int32_t x_dtype, int64_t B, int32_t D, int32_t h, int32_t w,
                         int32_t dilation, int32_t slot, int32_t n_slots, float* dots, void* stream);

/* pfst_neigh_grad and pfst_proto_dist_bwd (below) in one pass over x: grad_x =
 * neighbourhood-cosine gradient + grad_loss * (x - mu[label]) / (dist * n_valid)
 * (pfgst_loss.py:181-201 backward + pfgst.py:168-177 backward).
 * x is read once and grad_x written once for both losses (8*D B/pixel instead of
 * 20*D). Same argument meaning as the two entry points it fuses; labels of label_dtype
 * (PFST_DT_I64 or PFST_DT_U8, else PFST_ERR_UNSUPPORTED).                              */
int pfst_neigh_grad_proto(const float* x, const float* coef, int64_t B, int32_t D, int32_t h,
                          int32_t w, int32_t dilation, const void* labels, int32_t label_dtype,
                          int32_t lab_h, int32_t lab_w, const float* mu, const uint8_t* seen,
                          int32_t C, const float* dist, const double* acc,
                          const float* grad_loss, float* grad_x, void* stream);

/* PFGSTLoss.forward and its backward (pfgst_loss.py:44-234). `options` is a bit set of the
 * PFGSTLoss options outside the shipped configuration (pfgst_loss.py:16-18); 0 = the shipped
 * configuration:
 *   PFST_LOSS_SIM_GAUSSIAN   sim_type='gaussian' (:189-191): exp(-|x_n - x_m|^2 / sigma^2), formed from the
 *                            same five dot maps as the cosine (|x_n|^2 + |x_m|^2 - 2 x_n.x_m); the zero
 *                            padding of the unfold is the zero vector (similarity exp(-|x_n|^2 / sigma^2));
 *   PFST_LOSS_CROSS_PROB_EMA cross_prob_type='ema' (:161-178): q = unfold(softmax(logits_ema)), logits_ema
 *                            (B,C,fh*up,fw*up) on the loss grid as the reference requires;
 *   PFST_LOSS_UNFOLD_GRAD    detach_unfold=False (:148-149 not taken): the logits gradient also flows through
 *                            the unfolded factor (one more launch in the backward).
 *   PFST_LOSS_SRC_MARGIN / PFST_LOSS_SRC_MARGIN2  src_loss_type='margin' / 'margin2' (:117-133): the source
 *                            statistics are hinge terms relu(margin[0] - S) over positive pairs and
 *                            relu(S - margin[1]) over negative pairs (margin2: squared); margin_host = HOST
 *                            float[2], |margin| <= 1. losses[0], losses[1] = loss_src_pos, loss_src_neg;
 *                            losses[2], losses[3] = 0.
 * top_k = 0 stands for the reference's top_k=None (:218-220): every tap enters both consistency terms.   */
#define PFST_LOSS_SIM_GAUSSIAN 1
#define PFST_LOSS_CROSS_PROB_EMA 2
#define PFST_LOSS_UNFOLD_GRAD 4
#define PFST_LOSS_SRC_MARGIN 8
#define PFST_LOSS_SRC_MARGIN2 16

/* Bytes of the `workspace` pfst_pfgst_loss_fwd / _bwd share for these `options` (per-pixel
 * maps written by the forward's prep kernel and re-read by the backward). Host only.   */
int64_t pfst_pfgst_loss_ws_bytes(int64_t B, int32_t C, int32_t fh, int32_t fw, int32_t up,
                                 int32_t options);

/* dots: output of pfst_neigh_dots(x_ema, x_src) on the (fh,fw) feature grid with
 * dilation `dilation/up`; the loss grid is (fh*up, fw*up) (features nearest-
 * upsampled by the integer factor `up`, pfgst_loss.py:58-59).
 * logits: (B,C,lh,lw), sampled at src = min(floor(dst*lscale), in-1) (nearest
 * down-scaling by `downscale`, :57; lscale = 1/downscale).
 * gt, mix: (B,1,gt_h,gt_w) source labels / ClassMix masks of label_dtype (PFST_DT_I64 or
 * PFST_DT_U8, else PFST_ERR_UNSUPPORTED), nearest-sampled to the loss grid (:62-67).
 * weights6 (host): src_pos, src_neg, src_pos_std, src_neg_std, sim_pos, sim_neg (:110-135).
 * workspace: device buffer of pfst_pfgst_loss_ws_bytes(..., options) bytes, 16-byte aligned,
 * kept (with stats) for the backward. stats: device double[16] (first nine written here).
 * losses: device float[6] = loss_src_pos_mean, loss_src_neg_mean, loss_src_pos_std,
 * loss_src_neg_std, loss_sim_pos, loss_sim_neg. density (nullable): (B,fh*up,fw*up)
 * = 1 - mean_k cos_ema ('vis|density_sim_feat', :136); eroded (nullable): uint8 of
 * the eroded target mask (:69-71). options / sigma / logits_ema / margin_host: above
 * (0, 0, NULL, NULL for the shipped configuration).                                 */
int pfst_pfgst_loss_fwd(const float* dots, int32_t ksplit, int64_t B, int32_t fh,
                        int32_t fw, int32_t up, const float* logits, int32_t C,
                        int32_t lh, int32_t lw, float lscale_h, float lscale_w,
                        const void* gt, const void* mix, int32_t gt_h,
                        int32_t gt_w, int32_t dilation, int32_t top_k,
                        const float* weights6_host, void* workspace, double* stats,
                        float* losses, float* density, uint8_t* eroded, int32_t options,
                        float sigma, const float* logits_ema, const float* margin_host,
                        int32_t label_dtype, void* stream);

/* The arguments the forward took, plus: grad_losses: device float[6], upstream gradient of
 * each loss. coef (nullable): (B,9,fh,fw) for pfst_neigh_grad(x_src, dilation/up).
 * grad_logits (nullable): (B,C,lh,lw), zero-filled here, gradient of the two loss_sim
 * terms. At least one of the two outputs; two launches (coef only / grad_logits only) let
 * the coefficient maps — the only part the x_src gradient pass waits for — leave the
 * critical path early. gt and mix are not read (the forward left their classes in the
 * workspace); label_dtype is still validated.                                        */
int pfst_pfgst_loss_bwd(const float* dots, int32_t ksplit, int64_t B, int32_t fh,
                        int32_t fw, int32_t up, const float* logits, int32_t C,
                        int32_t lh, int32_t lw, float lscale_h, float lscale_w,
                        const void* gt, const void* mix, int32_t gt_h,
                        int32_t gt_w, int32_t dilation, int32_t top_k,
                        const float* weights6_host, const void* workspace,
                        const double* stats, const float* grad_losses, float* coef,
                        float* grad_logits, int32_t options, float sigma,
                        const float* logits_ema, const float* margin_host,
                        int32_t label_dtype, void* stream);

/* ---- P1-P3: class prototypes (north_star extension; no reference code) ----------
 * Anchor: PFGST.masked_feat_dist, rsiseg/models/uda/pfgst.py:168-177. Labels are
 * nearest-resampled to the feature grid as pfgst_loss.py:62 does.                  */

/* 1 when pfst_proto_accum(feats with these shapes) runs as ONE masked-accumulation launch (few classes,
 * no label sort: nothing to order against the TMA kernels, DESIGN.md 3.2) — schedulers then call
 * pfst_proto_accum directly instead of pfst_proto_order + pfst_proto_accum_ordered. Host only.        */
int pfst_proto_accum_is_masked(int32_t C, int32_t h, int32_t w);

/* packed: float[C*D + C], ACCUMULATED INTO (caller zeroes it; it is the NCCL
 * all-reduce buffer): packed[c*D+d] += sum of feats[b,d,n] over pixels n with
 * label c (0 <= label < C, and conf >= conf_thr when conf != NULL);
 * packed[C*D+c] += number of such pixels. labels: (B,lab_h,lab_w) of label_dtype
 * (PFST_DT_I64 or PFST_DT_U8), conf: (B,lab_h,lab_w) fp32 or NULL. feats: feat_dtype
 * PFST_DT_F32, PFST_DT_F16 or PFST_DT_BF16 (the EMA features of a teacher run under
 * autocast), every value converted to fp32 on load; the sums are float atomics.
 * An unknown feat_dtype or label_dtype returns PFST_ERR_UNSUPPORTED.                */
int pfst_proto_accum(const void* feats, int32_t feat_dtype, int64_t B, int32_t D, int32_t h, int32_t w,
                     const void* labels, int32_t label_dtype, int32_t lab_h, int32_t lab_w,
                     const float* conf, float conf_thr, int32_t C, float* packed, void* stream);

/* pfst_proto_accum split in two, so that the label sort is done ONCE per (image, tile) and
 * not by every streaming block:
 *   pfst_proto_order          builds, per 4096-pixel tile of every image, the list of pixel
 *                             offsets sorted by class (labels of label_dtype, PFST_DT_I64 or
 *                             PFST_DT_U8, nearest-resampled to (h,w), confidence mask applied)
 *                             into `workspace` (pfst_proto_order_ws_bytes() bytes, 16-byte
 *                             aligned) and adds the per-class pixel counts to counts[C]
 *                             (nullable; pass packed + C*D). The lists do not depend on the
 *                             label dtype;
 *   pfst_proto_accum_ordered  streams the feature planes (feat_dtype PFST_DT_F32, PFST_DT_F16
 *                             or PFST_DT_BF16) against those lists:
 *                             packed[c*D+d] += sum of feats over the pixels of class c.
 * Together they equal pfst_proto_accum. An unknown tag returns PFST_ERR_UNSUPPORTED.   */
int64_t pfst_proto_order_ws_bytes(int64_t B, int32_t h, int32_t w, int32_t C);
int pfst_proto_order(const void* labels, int32_t label_dtype, int64_t B, int32_t h, int32_t w,
                     int32_t lab_h, int32_t lab_w, const float* conf, float conf_thr, int32_t C,
                     float* counts, void* workspace, void* stream);
int pfst_proto_accum_ordered(const void* feats, int32_t feat_dtype, int64_t B, int32_t D, int32_t h,
                             int32_t w, int32_t C, const void* workspace, float* packed, void* stream);

/* mu_out[c] = packed sums / max(count,1) for classes with pixels; classes already
 * seen (seen_prev[c] != 0) are EMA-updated fl(fl(a32*mu_prev)+fl(b32*mean)) (the E2
 * rule); classes without pixels keep mu_prev. mu_prev / seen_prev may be NULL
 * (first call) and may alias mu_out / seen_out (in-place bank update). cnt_out
 * int64[C], seen_out uint8[C] may be NULL. reset_packed != 0 zeroes `packed` after it
 * has been consumed (ready for the next step's accumulation; no separate memset).
 * The bank iteration is kept ON THE DEVICE: iter_state = int64[2] {iteration (0 on the
 * first call), internal block counter (0)}. The kernel derives a = min(1 - 1/(iter+1), alpha),
 * b = 1 - a in fp64 exactly as pfst_ema_coeffs does (a32 = (float)a, b32 = (float)b; iter 0:
 * plain mean) and advances the iteration itself, so the launch carries no per-step host
 * argument and can be captured in a CUDA graph.                                        */
int pfst_proto_finalize(float* packed, int32_t C, int32_t D, const float* mu_prev,
                        const uint8_t* seen_prev, double alpha, int64_t* iter_state,
                        float* mu_out, int64_t* cnt_out, uint8_t* seen_out,
                        int32_t reset_packed, void* stream);

/* ---- G1: PFGST.masked_feat_dist (rsiseg/models/uda/pfgst.py:168-177) -----------------------
 * loss = mean over the selected pixels of ||f1[:,n] - f2[:,n]||_2; selected = mask[n] != 0
 * (mask: (B,1,h,w) uint8 / bool bytes, NULL = every pixel). f1, f2: (B,D,h,w) fp32.
 * dist: (B,h,w) per-pixel norms (0 where not selected), acc: device double[4] workspace (zeroed
 * here; acc[1] = number of selected pixels) — both kept for the backward. An empty selection
 * gives NaN like torch.mean. Backward: grad_f1 = g (f1-f2) / (dist n), 0 where dist = 0 or the
 * pixel is not selected; grad_f2 = -grad_f1 (either may be NULL).                            */
int pfst_feat_dist_fwd(const float* f1, const float* f2, const uint8_t* mask, int64_t B, int32_t D,
                       int32_t h, int32_t w, float* dist, double* acc, float* loss, void* stream);
int pfst_feat_dist_bwd(const float* f1, const float* f2, const uint8_t* mask, int64_t B, int32_t D,
                       int32_t h, int32_t w, const float* dist, const double* acc,
                       const float* grad_loss, float* grad_f1, float* grad_f2, void* stream);

/* ---- P2 across ranks: one-shot all-reduce over NVLink peer memory, fused into the finalise ----
 * north_star: "only the prototype sums and counts ... are reduced" across the data-parallel
 * ranks. The reference's only cross-rank reduction of per-iteration quantities is
 * BaseSegmentor._parse_losses' dist.all_reduce (rsiseg/models/segmentors/base.py:214-218);
 * prototypes are the north_star extension (P1-P3). Instead of a collective call between
 * two kernels, every rank owns a "board" (inbox[2][nranks][stride] fp32 + flags[nranks][C]
 * u64) that all peers map through a CUDA IPC handle; pfst_proto_finalize_peer pushes this
 * rank's packed [sums|counts] into every board, waits for the peers' step tokens and sums the
 * inbox in rank order (bit-identical prototypes on every rank), then finalises like
 * pfst_proto_finalize (which it equals for nranks = 1).
 *
 * Set-up entry points (called once; these DO allocate / synchronise):
 *   pfst_peer_board_bytes  size of a board; also returns the inbox stride (floats) and the
 *                          byte offset of the flags;
 *   pfst_peer_alloc        cudaMalloc + zero + IPC handle (64 bytes, host) of a board;
 *   pfst_peer_open/close   map / unmap a peer's board from its IPC handle;
 *   pfst_peer_free         release a board obtained from pfst_peer_alloc.                  */
int64_t pfst_peer_board_bytes(int32_t C, int32_t D, int32_t nranks, int64_t* stride_out,
                              int64_t* flag_offset_out);
int pfst_peer_alloc(int64_t bytes, void** ptr_out, void* ipc_handle64_host);
int pfst_peer_open(const void* ipc_handle64_host, void** ptr_out);
int pfst_peer_close(void* ptr);
int pfst_peer_free(void* ptr);

/* boards: device uint64[nranks] = base address of every rank's board as mapped in THIS
 * process (entry `rank` = the local board). status: device int64[2] = {1 if a wait for a peer
 * exceeded timeout_ns (that step's prototypes are invalid), last completed token}.
 * Asynchronous, no allocation, graph-capturable; every rank must launch it once per step.  */
int pfst_proto_finalize_peer(float* packed, int32_t C, int32_t D, const float* mu_prev,
                             const uint8_t* seen_prev, double alpha, int64_t* iter_state,
                             float* mu_out, int64_t* cnt_out, uint8_t* seen_out,
                             const uint64_t* boards, int32_t rank, int32_t nranks,
                             int64_t* status, int64_t timeout_ns, void* stream);

/* loss = mean over valid pixels of ||feats[:,n] - mu[label_n]||_2 (masked_feat_dist,
 * pfgst.py:168-177, with f2 = mu[label]); valid = label in [0,C) and seen[label] (seen may
 * be NULL). labels: (B,lab_h,lab_w) of label_dtype (PFST_DT_I64 or PFST_DT_U8, else
 * PFST_ERR_UNSUPPORTED), nearest-resampled to (h,w).
 * dist: (B,h,w) per-pixel distances (0 where invalid), kept for the backward.
 * acc: device double[4] workspace (zeroed here; acc[1] = number of valid pixels).  */
int pfst_proto_dist_fwd(const float* feats, int64_t B, int32_t D, int32_t h, int32_t w,
                        const void* labels, int32_t label_dtype, int32_t lab_h, int32_t lab_w,
                        const float* mu, const uint8_t* seen, int32_t C, float* dist,
                        double* acc, float* loss, void* stream);

/* grad_feats[b,d,n] (+)= grad_loss * (f - mu[label]) / (dist * n_valid), 0 where
 * invalid; accumulate != 0 adds into grad_feats (e.g. on top of pfst_neigh_grad).
 * labels and label_dtype as in pfst_proto_dist_fwd.                                 */
int pfst_proto_dist_bwd(const float* feats, int64_t B, int32_t D, int32_t h, int32_t w,
                        const void* labels, int32_t label_dtype, int32_t lab_h, int32_t lab_w,
                        const float* mu, const uint8_t* seen, int32_t C,
                        const float* dist, const double* acc, const float* grad_loss,
                        float* grad_feats, int32_t accumulate, void* stream);

/* out[b,c,n] = ||feats[b,:,n] - mu[c]||_2 for every class: (B,C,h,w).               */
int pfst_proto_dist_all(const float* feats, int64_t B, int32_t D, int32_t h, int32_t w,
                        const float* mu, int32_t C, float* out, void* stream);

/* ---- next row (SURVEY.md §8f rank 1): decode-head loss ------------------------------
 * Replaces BaseDecodeHead.losses (rsiseg/models/decode_heads/decode_head.py:249-283) with
 * CrossEntropyLoss (cross_entropy_loss.py:12-65, utils.py:48-79) and accuracy (accuracy.py:6-59):
 *   up   = bilinear(logits -> (H,W), align_corners=False)
 *   out2[0] = loss_weight * mean over ALL B*H*W pixels of CE(up, label; ignore_index)
 *             * weight[pixel] (nullable) * class_weight[label] (nullable)
 *   out2[1] = top-1 accuracy in percent over the non-ignored pixels
 *   grad_logits (nullable, (B,C,lh,lw), zeroed here) = d out2[0] / d logits
 * in ONE pass: the up-sampled logits are never materialised. Integer up-sampling factors
 * only (H = s*lh, W = s*lw). stats: device double[4] workspace (zeroed here).
 * labels: (B,H,W) of label_dtype (PFST_DT_I64 or PFST_DT_U8, else PFST_ERR_UNSUPPORTED).
 * labels and weight may start at any element alignment. B = 0 reads nothing (logits and
 * labels may be null) and writes out2 = {NaN, 0}, the reference's mean and accuracy.       */
int pfst_weighted_ce(const float* logits, const void* labels, int32_t label_dtype,
                     const float* weight, const float* class_weight, int64_t B, int32_t C,
                     int32_t lh, int32_t lw, int32_t H, int32_t W, int64_t ignore_index,
                     float loss_weight, float* grad_logits, double* stats, float* out2,
                     void* stream);

/* pfst_weighted_ce for logits of logit_dtype: PFST_DT_F32, or PFST_DT_F16 / PFST_DT_BF16 (a decode
 * head run under autocast); any other tag returns PFST_ERR_UNSUPPORTED before any other argument
 * check. pfst_weighted_ce(...) is pfst_weighted_ce_dt with PFST_DT_F32. The result is what mmseg's
 * @force_fp32 losses compute on logits.float(): each logit is converted to fp32 once, on load
 * (exact), so out2 and grad_logits equal the fp32 call's on the upcast logits (up to the order of
 * the float atomics). grad_logits stays an fp32 buffer: pfst_scale_cast turns it into the logits'
 * dtype. A 16-bit view may start at any element; it takes the same kernel as its fp32 upcast.
 *
 * pfst_scale_cast: dst[i] = (dst_dtype)(src[i] * *scale) for i < n, an IEEE fp32 product rounded
 * ONCE to dst_dtype (PFST_DT_F32, PFST_DT_F16 or PFST_DT_BF16, round to nearest even; any other tag
 * returns PFST_ERR_UNSUPPORTED before any other argument check). This is the backward of
 * `loss(logits.float())`: the fp32 gradient times the upstream gradient, then the cast's backward.
 * Rounding the gradient to 16 bits first and multiplying after would round twice. scale: device
 * float[1] (the upstream gradient; read on the device, nothing synchronises). src, scale: 4-byte
 * aligned; dst: aligned to its element. n = 0 reads and writes nothing (pointers may be null). */
int pfst_weighted_ce_dt(const void* logits, int32_t logit_dtype, const void* labels,
                        int32_t label_dtype, const float* weight, const float* class_weight,
                        int64_t B, int32_t C, int32_t lh, int32_t lw, int32_t H, int32_t W,
                        int64_t ignore_index, float loss_weight, float* grad_logits,
                        double* stats, float* out2, void* stream);
int pfst_scale_cast(const float* src, const float* scale, int64_t n, void* dst, int32_t dst_dtype,
                    void* stream);

/* ---- OHEM pixel sampler of the decode-head loss ------------------------------------------
 * mmseg 0.x OHEMPixelSampler.sample(seg_logit, seg_label), whose map replaces seg_weight in
 * BaseDecodeHead.losses (decode_head.py:249-283), with seg_logit the bilinear (align_corners=False)
 * up-sampling of logits (B,C,lh,lw) to the labels' (H,W) by an integer factor s >= 1 (H = s*lh,
 * W = s*lw; s = 1 is the sampler on already up-sampled logits). valid = label != ignore_index (and in
 * [0, C)), n = #valid, batch_kept = min_kept * B:
 *   thresh not NaN: key = softmax(up)[label] (fp32); kth = k-th smallest valid key, k = min(batch_kept,
 *                   n - 1) (0 when n == 0); weight = valid & (key < max(kth, thresh)), where thresh wins
 *                   only if it is larger (Python's max(min_threshold, thresh));
 *   thresh NaN:     key = loss_weight * class_weight[label] * CE(up, label) (0 at ignored pixels); kth =
 *                   the batch_kept-th largest valid key (the smallest when batch_kept >= n); the
 *                   min(batch_kept, n) valid pixels with the largest keys get weight 1, and at a tie on
 *                   kth the lower flat index goes first (a stable descending sort).
 * Keys order as torch.sort orders them: NaN after every number. The up-sampled logits are never
 * materialised and nothing synchronises the host: the order statistic is an exact radix select whose
 * rank is read from the device count. logits: logit_dtype PFST_DT_F32 / F16 / BF16; labels (B,H,W):
 * label_dtype PFST_DT_I64 / PFST_DT_U8 (an unknown tag returns PFST_ERR_UNSUPPORTED before any other
 * check). class_weight: (C) fp32 or NULL. min_kept >= 2 (mmseg asserts min_kept > 1).
 * workspace: pfst_ohem_ws_bytes(B, H, W) bytes, 16-byte aligned. Outputs: weight_out (B,H,W) fp32 0/1;
 * keys_out (B,H,W) fp32 or NULL (ignored pixels: softmax(up)[0] with a thresh, 0 without); kth_out
 * device float[1] or NULL. B = 0 reads nothing, writes kth_out = 0 (logits, labels, weight_out may be
 * NULL); no valid pixel gives a zero map. B*H*W and C*lh*lw must be below 2^31. */
int64_t pfst_ohem_ws_bytes(int64_t B, int32_t H, int32_t W);
int pfst_ohem_weight(const void* logits, int32_t logit_dtype, const void* labels, int32_t label_dtype,
                     const float* class_weight, int64_t B, int32_t C, int32_t lh, int32_t lw, int32_t H,
                     int32_t W, int64_t ignore_index, float loss_weight, float thresh, int64_t min_kept,
                     void* workspace, float* keys_out, float* kth_out, float* weight_out, void* stream);

/* ---- next row (SURVEY.md §8f rank 4): offline class-wise thresholds -------------------
 * Replaces PseudoLabelingHookV4._cal_threshold
 * (rsiseg/core/hook/pseudo_labeling_hookv4.py:173-205): for the n sampled pixels idx[] (row
 * indices of the (B*HW, C) pixel-major view; NULL = all pixels in order) compute pred = argmax
 * softmax, ent = sum -p*log(p), and for every class c and ratio r
 *   thr_out[c*R + r] = (n_c == 0) ? 0 : sorted(ent[pred == c])[int(n_c * ratios[r])]
 * — an exact order statistic by radix select, no sort. ratios_dev: device double[R].
 * workspace: pfst_class_quantile_ws_bytes(n, C, R) bytes, 16-byte aligned.                */
int64_t pfst_class_quantile_ws_bytes(int64_t n, int32_t C, int32_t R);
int pfst_class_quantile(const float* logits, int64_t B, int32_t C, int64_t HW, const int64_t* idx,
                        int64_t n, const double* ratios_dev, int32_t R, void* workspace,
                        float* thr_out, void* stream);

/* ---- V1/V4: confusion matrix / area histograms -------------------------------
 * Replaces intersect_and_union (rsiseg/core/evaluation/metrics.py:26-86, three
 * float32 torch.histc per image on the CPU) and the integer confusion matrix of
 * tools/confusion_matrix.py:46-65 / tests/test_metrics.py:9-28.
 * For every image i (n_images maps of `pixels` each):
 *   lab = lut ? lut[label] : label   (label_map, metrics.py:66-68; uint8 domain)
 *   reduce_zero_label as metrics.py:69-72; pixels with lab == ignore_index drop.
 *   row = lab in [0,C) ? lab : C ; col = pred in [0,C) ? pred : C
 *   conf[slot(i)][row][col] += 1   with slot(i) = per_image ? i : 0
 * conf is int64 [(per_image ? n_images : 1)][C+1][C+1], accumulated INTO (the
 * caller zeroes it), so sweeps can be chained. The C x C top-left block is the
 * confusion matrix; histc areas follow as
 *   intersect[c]=conf[c][c], label[c]=sum_j conf[c][j], pred[c]=sum_i conf[i][c].
 * lut: device uint8[256] or NULL.                                               */
int pfst_confusion_accum(const void* pred, int32_t pred_dtype, const void* label,
                         int32_t label_dtype, int64_t n_images, int64_t pixels,
                         int32_t C, int64_t ignore_index, int32_t reduce_zero_label,
                         const uint8_t* lut, int64_t* conf, int32_t per_image,
                         void* stream);

/* ---- V0+V1: on-device evaluation input path (SURVEY.md 8f-4) ------------------
 * Replaces, for a batch of n_images logit maps that are already on the GPU,
 *   output   = F.softmax(seg_logit, dim=1)            encoder_decoder.py:311
 *   seg_pred = output.argmax(dim=1).cpu().numpy()     encoder_decoder.py:329-338
 *   intersect_and_union(seg_pred[i], gt[i], ...)      custom.py:644-682, metrics.py:26-86
 * by one pass over logits (n_images, C, pixels) fp32 NCHW and label (n_images, pixels):
 * pred = first index of the maximum of the softmax as torch CUDA computes it (ties in
 * softmax space go to the lowest class; a NaN anywhere in the pixel's softmax gives 0),
 * then conf[slot(i)][row][col] += 1 exactly as pfst_confusion_accum (same label_map LUT,
 * reduce_zero_label, ignore_index, out-of-range row C; accumulated INTO conf).
 * pred_out (nullable): the arg-max map itself, uint8 or int64 (pred_dtype), for callers
 * that keep simple_test's return value. conf and label may both be NULL (arg-max only).  */
int pfst_argmax_confusion(const float* logits, int64_t n_images, int32_t C, int64_t pixels,
                          const void* label, int32_t label_dtype, int64_t ignore_index,
                          int32_t reduce_zero_label, const uint8_t* lut, int64_t* conf,
                          int32_t per_image, void* pred_out, int32_t pred_dtype, void* stream);

/* ---- V0: test-time sliding-window accumulation and flip ---------------------------
 * The tensor arithmetic of EncoderDecoder.slide_inference / inference
 * (rsiseg/models/segmentors/encoder_decoder.py:220-263, 312-324); the network pass on each crop
 * stays with the caller.
 *   pfst_slide_add       preds[:, :, y1:y1+ch, x1:x1+cw] += crop      (:245-249: `preds += F.pad(crop_seg_logit, ...)`,
 *                        a full-size padded copy and a full-size add per window in the reference)
 *   pfst_slide_finalize  out = flip(preds / count)                    (:255 `preds / count_mat`, :316-321 the flips;
 *                        a flip commutes with the per-pixel soft-max of :311)
 * The windows are a product of row and column intervals, so count_mat(y, x) = cnt_y[y] * cnt_x[x]
 * (device float vectors of H and W entries built by the caller; both NULL = no division). preds / out:
 * (B, C, H, W) fp32, crop: (B, C, ch, cw) fp32. out may equal preds when no flip is requested.
 * Bit-exact with the reference: same additions in the same window order, IEEE division.              */
int pfst_slide_add(float* preds, const float* crop, int64_t B, int32_t C, int32_t H, int32_t W,
                   int32_t y1, int32_t x1, int32_t ch, int32_t cw, void* stream);
int pfst_slide_finalize(const float* preds, const float* cnt_y, const float* cnt_x, int64_t B,
                        int32_t C, int32_t H, int32_t W, int32_t flip_h, int32_t flip_v, float* out,
                        void* stream);

/* aug_test (encoder_decoder.py:355-373): `seg_logit = inference(imgs[0]); seg_logit += inference(imgs[i])...;
 * seg_logit /= len(imgs); seg_pred = seg_logit.argmax(dim=1)` where `inference` returns the soft-max.
 *   pfst_softmax_accum  acc (+)= softmax(logits) per pixel, torch CUDA's arithmetic (max, sum of expf in class
 *                       order, IEEE division); first != 0 overwrites acc. logits / acc: (n_images, C, pixels) fp32.
 *   pfst_div_argmax     pred = argmax_c (acc / divisor): first maximum wins, NaN counts as maximum (torch.argmax).
 * The soft-max tensors of the augmentations never exist.                                                      */
int pfst_softmax_accum(const float* logits, float* acc, int64_t n_images, int32_t C, int64_t pixels,
                       int32_t first, void* stream);
int pfst_div_argmax(const float* acc, int64_t n_images, int32_t C, int64_t pixels, float divisor,
                    int64_t* pred, void* stream);

/* ---- strong augmentation: Gaussian blur of the mixed image (SURVEY.md 8f-3) -----
 * Replaces gaussian_blur, rsiseg/models/utils/dacs_transforms.py:88-107:
 *   kornia.filters.GaussianBlur2d(kernel_size=(ksize_y,ksize_x), sigma=(s,s))(data)
 * (kornia: third-party, unpinned; published algorithm = normalised 1-D Gaussians
 * exp(-x^2/(2 s^2)), x = t - k/2, 'reflect' border, per-channel correlation).
 * in/out: (n_images, C, H, W) fp32, out != in. ksize_*: odd, ksize/2 < size (reflect).
 * sigma_host: HOST array of n_images floats (one sigma per image, both axes, as the call
 * site draws them); it is copied into the launch parameters, so the call is asynchronous
 * and needs no staging buffer. Taps below 2^-30 of the centre weight are not evaluated.   */
int pfst_gaussian_blur(const float* in, float* out, int64_t n_images, int32_t C, int32_t H,
                       int32_t W, int32_t ksize_y, int32_t ksize_x, const float* sigma_host,
                       void* stream);

/* ---- strong augmentation: photometric distortion of uint8 images (SURVEY.md 8f-3) ------
 * Replaces StrongAugmentation.__call__, rsiseg/datasets/pipelines/transforms.py:1062-1145
 * (brightness / contrast = convert(alpha, beta), saturation and hue through mmcv.bgr2hsv /
 * hsv2bgr = cv2.cvtColor on uint8), given the distortions the host drew: for image i the ops
 * op_codes_host[4 i + k], k = 0..3, are applied in order (0 = none) with parameters
 * op_params_host[2 (4 i + k) + {0, 1}] = (alpha, beta) for PFST_SA_CONVERT, (alpha, -) for
 * PFST_SA_SATURATION, (integer hue delta, -) for PFST_SA_HUE. in/out: (n_images, H, W, 3) uint8
 * BGR, HWC as the pipeline holds them; in == out is allowed. Both HOST arrays are copied into the
 * launch parameters (asynchronous, no staging buffer). Results are bit-identical to OpenCV 4.13's
 * uint8 conversions, including its layout dependence: HSV->BGR truncates inside the simd_width-pixel
 * blocks of a row and rounds in the row's tail (simd_width = 32 on AVX2 hosts; 0 = no tail).     */
#define PFST_SA_CONVERT 1
#define PFST_SA_SATURATION 2
#define PFST_SA_HUE 3
int pfst_photometric_u8(const uint8_t* in, uint8_t* out, int64_t n_images, int32_t H, int32_t W,
                        const int32_t* op_codes_host, const float* op_params_host,
                        int32_t simd_width, void* stream);

/* ---- strong augmentation: colour jitter of the mixed image (SURVEY.md 8f-3) -------------
 * Replaces color_jitter, rsiseg/models/utils/dacs_transforms.py:56-85:
 *   denorm_(data, mean, std); kornia.augmentation.ColorJitter(s, s, s, s)(data); renorm_(...)
 * given the factors and the order the host drew (kornia: third-party, unpinned; 0.6-series
 * arithmetic restated in oracle/strong_aug.py, parity unpinned). in/out: (n_images, 3, HW) fp32
 * planar, in == out allowed. factors_host[4 i + {0,1,2,3}] = brightness, contrast, saturation, hue
 * factor of image i; order_host[4 i + k] = k-th transform to apply (0 brightness, 1 contrast,
 * 2 saturation, 3 hue, -1 none). denorm = 1: (x*std + mean)/255 before and (x*255 - mean)/std after
 * (mean_host/std_host: 3 floats), 0: data already in [0,1]. HOST arrays travel in the launch
 * parameters (asynchronous, no staging buffer).                                              */
int pfst_color_jitter(const float* in, float* out, int64_t n_images, int64_t HW,
                      const float* factors_host, const int32_t* order_host,
                      const float* mean_host, const float* std_host, int32_t denorm, void* stream);

/* ---- offline class-wise pseudo-labelling, remaining pieces (SURVEY.md §8f rank 4) -------------
 * pfst_loc_dis: PseudoLabelingHookV4._cal_loc_dis (rsiseg/core/hook/pseudo_labeling_hookv4.py:208-230)
 *   out[b,y,x,k] = sum_c (feats[b,c,y+dy_k*d,x+dx_k*d] - feats[b,c,y,x])^2, k over the 3x3 taps,
 *   zero padding (an out-of-image tap reads 0). feats (B,C,H,W) fp32 -> out (B,H,W,9) fp32; the
 *   nn.Unfold copy (9x the feature map) never exists.
 * pfst_gather_rows: dst[i,:] = src[idx[i],:] — the random pixel subset `cur_tensor[idx, :]` (:255-256),
 *   idx drawn on the host from the numpy stream.
 * pfst_sigma_bisect: the binary search of _cal_sigmas (:262-275) for ONE mean_sim: `steps` times
 *   sigma = (left+right)/2; mean(exp(-dis / sigma^2)) < mean_sim ? left = sigma : right = sigma
 *   (the reference's `while abs(left-right) > 1e-6` from [0,1000] is exactly 30 steps). The interval
 *   lives in state = device double[4] {left, right, scratch, scratch}: one launch per step, no host
 *   sync inside the search. dis: n fp32 values, 16-byte aligned. Result: state[0] (left).
 * pfst_loader_pseudo_labels: the label rule of LoadAnnotationsPseudoLabelsV2.__call__
 *   (rsiseg/datasets/pipelines/loading.py:474-487) for N maps at once: pred = argmax_c logits;
 *   p = exp(logits)/sum exp(logits) (no max shift, as the loader); H = -sum p log(p + 1e-8);
 *   label = H < thres[pred] ? pred : 255; reduce_zero_label: 0 -> 255, label-1, 254 -> 255.
 *   logits (N,C,HW) fp32, thres C fp32 (device) -> labels (N,HW) uint8.                          */
int pfst_loc_dis(const float* feats, int64_t B, int32_t C, int32_t H, int32_t W, int32_t dilation,
                 float* out, void* stream);
int pfst_gather_rows(const float* src, const int64_t* idx, int64_t n, int32_t row_floats, float* dst,
                     void* stream);
int pfst_sigma_bisect(const float* dis, int64_t n, float mean_sim, double left0, double right0,
                      int32_t steps, double* state, void* stream);
int pfst_loader_pseudo_labels(const float* logits, int64_t N, int32_t C, int64_t HW,
                              const float* thres, int32_t reduce_zero_label, uint8_t* labels,
                              void* stream);

/* ---- log variables without host round trips (SURVEY.md §8f-2) ------------------------------
 * Replaces the arithmetic of BaseSegmentor._parse_losses
 * (rsiseg/models/segmentors/base.py:177-222): `loss = sum(v for k, v in log_vars if 'loss' in k)`
 * (left-to-right fp32 adds from 0), and per variable `v.div_(world)` before the all-reduce and
 * `.item()`. ptrs_host: HOST array of n <= 32 DEVICE pointers to fp32 scalars; weights_host:
 * HOST array of n multipliers applied inside the sum (NULL = all 1). row_out (nullable):
 * row_out[i] = v_i / divisor, row_out[n] = sum / divisor. total_out (nullable): the undivided
 * sum over the entries whose bit is set in sum_mask. One single-thread launch.               */
int pfst_gather_scalars(const float* const* ptrs_host, const float* weights_host, int32_t n,
                        uint32_t sum_mask, float divisor, float* row_out, float* total_out,
                        void* stream);

/* All _parse_losses calls of one PFGST.forward_train iteration in ONE launch. Entry i (n <= 32)
 * belongs to the current segment (= one call, entries in call order); flags_host[i] bit0: its key
 * contains 'loss' (it enters the segment's sum), bit1: last entry of the segment. row_out receives
 * every entry / divisor and, behind the last entry of each segment, the segment's sum / divisor
 * (that call's 'loss' log variable): n + (number of segments) floats. total_out (nullable) =
 * 0 + sum over segments of weights_host[last entry of the segment] * segment sum, left to right
 * in fp32 — total_loss of rsiseg/models/uda/pfgst.py:237,310,342.                             */
int pfst_gather_segments(const float* const* ptrs_host, const float* weights_host,
                         const uint8_t* flags_host, int32_t n, float divisor, float* row_out,
                         float* total_out, void* stream);

/* out[i] = *ptrs_host[i] * weights_host[i] (0 where the pointer is NULL; weights NULL = 1),
 * i < n <= 32: packs separate 0-dim device scalars — e.g. the upstream gradients autograd hands
 * to the backward of the six PFGSTLoss terms and the prototype distance — into one vector.  */
int pfst_pack_scalars(const float* const* ptrs_host, const float* weights_host, int32_t n,
                      float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PFST_SM100_H_ */
