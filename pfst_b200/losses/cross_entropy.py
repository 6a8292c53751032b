"""Decode-head loss — drop-in for BaseDecodeHead.losses
(rsiseg/models/decode_heads/decode_head.py:249-283) with its configured CrossEntropyLoss
(rsiseg/models/losses/cross_entropy_loss.py:12-65, reduction='mean', avg_non_ignore=False) and
`accuracy` (rsiseg/models/losses/accuracy.py:6-59): SURVEY.md §8(f) rank 1.

The reference up-samples the (B,C,H/4,W/4) logits to (B,C,H,W), takes a log-softmax, gathers,
multiplies by the pixel weights, averages over all pixels and computes the top-1 accuracy —
about ten ATen kernels moving the 50 MB up-sampled tensor several times, forward and backward.
`pfst_weighted_ce` (csrc/weighted_ce.cu) does all of it in one pass over the low-resolution
logits, labels and weights, and also leaves d loss / d logits behind, so the backward is a scalar
multiply.
"""
from __future__ import annotations

from typing import Optional

import torch

from .. import _lib, ops
from .._lib import PfstError


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
        grad = torch.empty_like(seg_logit) if need_grad else None
        stats = torch.empty(4, dtype=torch.float64, device=dev)
        out2 = torch.empty(2, dtype=torch.float32, device=dev)
        _lib.call("pfst_weighted_ce", ops._dev(seg_logit, "seg_logit", torch.float32),
                  labels.data_ptr(), ops._labels(labels, "seg_label"), ops._opt(seg_weight, "seg_weight", torch.float32),
                  ops._opt(class_weight, "class_weight", torch.float32), B, C, lh, lw, H, W, int(ignore_index),
                  float(loss_weight), None if grad is None else grad.data_ptr(), stats.data_ptr(), out2.data_ptr(),
                  ops._stream())
        ctx.save_for_backward(grad)
        loss, acc = out2[0], out2[1:2]
        ctx.mark_non_differentiable(acc)
        return loss, acc

    @staticmethod
    def backward(ctx, grad_loss, _grad_acc):
        (grad,) = ctx.saved_tensors
        return (None if grad is None else grad * grad_loss), None, None, None, None, None


def upsample_cross_entropy(seg_logit: torch.Tensor, seg_label: torch.Tensor, seg_weight: Optional[torch.Tensor] = None,
                           class_weight: Optional[torch.Tensor] = None, ignore_index: int = 255,
                           loss_weight: float = 1.0):
    """-> (loss 0-dim, acc_seg (1,)). seg_logit (B,C,lh,lw) fp32; seg_label (B,1,H,W) or (B,H,W) int64 or uint8;
    seg_weight (B,H,W) fp32 or None; class_weight (C,) fp32 or None."""
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
                       class_weight=None, align_corners: bool = False, loss_name: str = "loss_ce") -> dict:
    """Body of BaseDecodeHead.losses (decode_head.py:249-283) for the shipped configuration
    (one CrossEntropyLoss, no OHEM sampler): {loss_name: loss, 'acc_seg': accuracy}."""
    if align_corners:
        raise PfstError("decode_head_losses: align_corners=True is not covered by the fused kernel "
                        "(every shipped config uses align_corners=False)")
    loss, acc = upsample_cross_entropy(seg_logit, seg_label, seg_weight, class_weight, ignore_index, loss_weight)
    return {loss_name: loss, "acc_seg": acc}
