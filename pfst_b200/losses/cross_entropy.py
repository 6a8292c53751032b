"""Decode-head loss — drop-in for BaseDecodeHead.losses
(rsiseg/models/decode_heads/decode_head.py:249-283) with its configured CrossEntropyLoss
(rsiseg/models/losses/cross_entropy_loss.py:12-65, reduction='mean', avg_non_ignore=False) and
`accuracy` (rsiseg/models/losses/accuracy.py:6-59): SURVEY.md §8(f) rank 1.

The reference up-samples the (B,C,H/4,W/4) logits to (B,C,H,W), takes a log-softmax, gathers,
multiplies by the pixel weights, averages over all pixels and computes the top-1 accuracy —
about ten ATen kernels moving the 50 MB up-sampled tensor several times, forward and backward.
`pfst_weighted_ce_dt` (csrc/weighted_ce.cu) does all of it in one pass over the low-resolution
logits, labels and weights, and also leaves d loss / d logits behind, so the backward is a scalar
multiply.

The logits may be fp32, fp16 or bf16 (a decode head run under autocast). The result is what mmseg's
`@force_fp32(apply_to=('seg_logit',))` losses compute on `seg_logit.float()`: the loss and the accuracy
are fp32 and equal the fp32 path's on the upcast logits, and the logits' gradient has their dtype and
equals the fp32 gradient times the upstream gradient, rounded once (`pfst_scale_cast`). There is no
`.float()` copy in the forward and no multiply-and-cast pair in the backward.
"""
from __future__ import annotations

from typing import Optional

import torch

from .. import _lib, ops
from .._lib import PfstError


LOGIT_DTYPES = (torch.float32, torch.float16, torch.bfloat16)


class _UpsampleCE(torch.autograd.Function):
    @staticmethod
    def forward(ctx, seg_logit, labels, seg_weight, class_weight, ignore_index, loss_weight):
        B, C, lh, lw = seg_logit.shape
        H, W = labels.shape[-2:]
        if H % lh or W % lw or H // lh != W // lw:
            raise PfstError(f"decode_head_losses: {lh}x{lw} logits -> {H}x{W} labels is not an integer "
                            "up-sampling factor (unsupported resampling)")
        dev = seg_logit.device
        need_grad = seg_logit.requires_grad
        # the gradient is accumulated in fp32 whatever the logits' dtype; the backward rounds it once
        grad = torch.empty_like(seg_logit, dtype=torch.float32) if need_grad else None
        stats = torch.empty(4, dtype=torch.float64, device=dev)
        out2 = torch.empty(2, dtype=torch.float32, device=dev)
        tag = ops._FLOAT2DT[seg_logit.dtype]
        _lib.call("pfst_weighted_ce_dt", ops._dev(seg_logit, "seg_logit"), tag,
                  labels.data_ptr(), ops._labels(labels, "seg_label"), ops._opt(seg_weight, "seg_weight", torch.float32),
                  ops._opt(class_weight, "class_weight", torch.float32), B, C, lh, lw, H, W, int(ignore_index),
                  float(loss_weight), None if grad is None else grad.data_ptr(), stats.data_ptr(), out2.data_ptr(),
                  ops._stream())
        ctx.save_for_backward(grad)
        ctx.logit_dtype = seg_logit.dtype
        ctx.set_materialize_grads(False)            # acc_seg has no gradient: no zero tensor is filled for it
        loss, acc = out2[0], out2[1:2]
        ctx.mark_non_differentiable(acc)
        return loss, acc

    @staticmethod
    def backward(ctx, grad_loss, _grad_acc):
        (grad,) = ctx.saved_tensors
        if grad is None or grad_loss is None:
            return None, None, None, None, None, None
        if ctx.logit_dtype == torch.float32:        # the same bits as pfst_scale_cast, less host time per call
            return grad * grad_loss, None, None, None, None, None
        # 16-bit logits: (fp32 gradient * upstream) rounded once to their dtype, in one launch
        scale = grad_loss.float()
        out = torch.empty(grad.shape, dtype=ctx.logit_dtype, device=grad.device)
        _lib.call("pfst_scale_cast", grad.data_ptr(), scale.data_ptr(), grad.numel(), out.data_ptr(),
                  ops._FLOAT2DT[ctx.logit_dtype], ops._stream())
        return out, None, None, None, None, None


def upsample_cross_entropy(seg_logit: torch.Tensor, seg_label: torch.Tensor, seg_weight: Optional[torch.Tensor] = None,
                           class_weight: Optional[torch.Tensor] = None, ignore_index: int = 255,
                           loss_weight: float = 1.0):
    """-> (loss 0-dim fp32, acc_seg (1,) fp32). seg_logit (B,C,lh,lw) fp32, fp16 or bf16 (its gradient has its
    dtype); seg_label (B,1,H,W) or (B,H,W) int64 or uint8; seg_weight (B,H,W) fp32 or None; class_weight (C,)
    fp32 or None."""
    if isinstance(seg_logit, torch.Tensor) and seg_logit.dtype not in LOGIT_DTYPES:
        raise TypeError(f"seg_logit: decode-head logits must be torch.float32, torch.float16 or torch.bfloat16, "
                        f"got {seg_logit.dtype}")
    if seg_label.dim() == 4:
        seg_label = seg_label[:, 0]
    seg_logit = seg_logit.contiguous()
    seg_label = seg_label.contiguous()
    if seg_weight is not None:
        seg_weight = seg_weight.float().contiguous()                       # cross_entropy_loss.py:58-59
        if seg_weight.numel() != seg_label.numel():
            raise ValueError("seg_weight must hold one weight per label pixel")
    if class_weight is not None:
        class_weight = torch.as_tensor(class_weight, dtype=torch.float32, device=seg_logit.device).contiguous()
        if class_weight.numel() != seg_logit.shape[1]:
            raise ValueError("class_weight must have one entry per class")
    return _UpsampleCE.apply(seg_logit, seg_label, seg_weight, class_weight, ignore_index, loss_weight)


def decode_head_losses(seg_logit, seg_label, seg_weight=None, *, ignore_index: int = 255, loss_weight: float = 1.0,
                       class_weight=None, align_corners: bool = False, loss_name: str = "loss_ce",
                       sampler=None) -> dict:
    """Body of BaseDecodeHead.losses (decode_head.py:249-283) with one CrossEntropyLoss:
    {loss_name: loss, 'acc_seg': accuracy}. sampler: the head's pixel sampler (an OHEMPixelSampler) or None;
    as in the reference its map replaces seg_weight. It is computed from the low-resolution seg_logit on the
    device (pfst_ohem_weight) and fed to the fused loss."""
    if align_corners:
        raise PfstError("decode_head_losses: align_corners=True is not covered by the fused kernel "
                        "(every shipped config uses align_corners=False)")
    if sampler is not None:
        seg_weight = sampler.weight_map(seg_logit, seg_label)
    loss, acc = upsample_cross_entropy(seg_logit, seg_label, seg_weight, class_weight, ignore_index, loss_weight)
    return {loss_name: loss, "acc_seg": acc}
