"""CPU oracle (TEST INFRASTRUCTURE, see oracle/__init__.py) for the OHEM pixel sampler of a decode head.

The reference configures it with `decode_head.sampler=dict(type='OHEMPixelSampler', thresh=..., min_kept=...)`
and ships mmseg 0.x's class under rsiseg/core/seg (SURVEY.md §2 row 14); BaseDecodeHead.losses
(rsiseg/models/decode_heads/decode_head.py:249-283) replaces `seg_weight` with its output:
    seg_logit = resize(seg_logit, size=seg_label.shape[2:], mode='bilinear', align_corners=self.align_corners)
    if self.sampler is not None:
        seg_weight = self.sampler.sample(seg_logit, seg_label)
What follows restates the published mmseg 0.x source of `OHEMPixelSampler`
(mmseg/core/seg/sampler/ohem_pixel_sampler.py, v0.11-v0.30; the single-`loss_decode` form) line for line, and
the part of mmseg's `CrossEntropyLoss` (mmseg/models/losses/cross_entropy_loss.py, use_sigmoid=False) that
the sampler calls with `reduction_override='none'`. Pinned bit for bit against the reference's own class
when PFST_REFERENCE names a checkout (tests/test_ohem_oracle.py); otherwise parity is unpinned.
"""
from __future__ import annotations

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import weighted_ce as WC


class CrossEntropyLoss(nn.Module):
    """mmseg CrossEntropyLoss(use_sigmoid=False, use_mask=False) for the sampler's call:
    loss_weight * F.cross_entropy(score, label, weight=class_weight, reduction='none', ignore_index)."""

    def __init__(self, loss_weight=1.0, class_weight=None, loss_name='loss_ce'):
        super().__init__()
        self.use_sigmoid = False
        self.loss_weight = loss_weight
        self.class_weight = class_weight
        self.loss_name = loss_name

    def forward(self, cls_score, label, weight=None, avg_factor=None, reduction_override=None, ignore_index=255):
        assert reduction_override == 'none' and weight is None and avg_factor is None
        class_weight = cls_score.new_tensor(self.class_weight) if self.class_weight is not None else None
        loss = F.cross_entropy(cls_score, label, weight=class_weight, reduction='none', ignore_index=ignore_index)
        return self.loss_weight * loss


class OHEMPixelSampler:
    """mmseg 0.x OHEMPixelSampler: context is the decode head (ignore_index, loss_decode)."""

    def __init__(self, context, thresh=None, min_kept=100000):
        self.context = context
        assert min_kept > 1
        self.thresh = thresh
        self.min_kept = min_kept

    def sample(self, seg_logit, seg_label):
        with torch.no_grad():
            assert seg_logit.shape[2:] == seg_label.shape[2:]
            assert seg_label.shape[1] == 1
            seg_label = seg_label.squeeze(1).long()
            batch_kept = self.min_kept * seg_label.size(0)
            valid_mask = seg_label != self.context.ignore_index
            seg_weight = seg_logit.new_zeros(size=seg_label.size())
            valid_seg_weight = seg_weight[valid_mask]
            if self.thresh is not None:
                seg_prob = F.softmax(seg_logit, dim=1)

                tmp_seg_label = seg_label.clone().unsqueeze(1)
                tmp_seg_label[tmp_seg_label == self.context.ignore_index] = 0
                seg_prob = seg_prob.gather(1, tmp_seg_label).squeeze(1)
                sort_prob, sort_indices = seg_prob[valid_mask].sort()

                if sort_prob.numel() > 0:
                    min_threshold = sort_prob[min(batch_kept, sort_prob.numel() - 1)]
                else:
                    min_threshold = 0.0
                threshold = max(min_threshold, self.thresh)
                valid_seg_weight[seg_prob[valid_mask] < threshold] = 1.
            else:
                losses = self.context.loss_decode(
                    seg_logit,
                    seg_label,
                    weight=None,
                    ignore_index=self.context.ignore_index,
                    reduction_override='none')
                # faster than topk according to https://github.com/pytorch/pytorch/issues/22812  # noqa
                _, sort_indices = losses[valid_mask].sort(descending=True)
                valid_seg_weight[sort_indices[:batch_kept]] = 1.

            seg_weight[valid_mask] = valid_seg_weight

            return seg_weight


class Head:
    """The attributes of a decode head the sampler reads."""

    def __init__(self, ignore_index=255, loss_weight=1.0, class_weight=None):
        self.ignore_index = ignore_index
        self.loss_decode = CrossEntropyLoss(loss_weight, class_weight)


def decode_head_losses(seg_logit, seg_label, sampler, class_weight=None, ignore_index=255, loss_weight=1.0):
    """decode_head.py:249-283 with a sampler: resize -> sampler.sample -> the loss with seg_weight = its map
    -> accuracy. -> (loss_ce 0-dim, acc_seg (1,), seg_weight (B,H,W))."""
    up = F.interpolate(seg_logit, seg_label.shape[2:], None, 'bilinear', False)     # ops/wrappers.py:28
    seg_weight = sampler.sample(up, seg_label)
    label = seg_label.squeeze(1)
    loss = F.cross_entropy(up, label, weight=class_weight, reduction='none', ignore_index=ignore_index)
    loss = loss_weight * (loss * seg_weight).mean()
    return loss, WC.accuracy(up, label, ignore_index), seg_weight
