"""OHEM pixel sampler of a decode head — drop-in for mmseg 0.x `OHEMPixelSampler`
(mmseg/core/seg/sampler/ohem_pixel_sampler.py; the reference ships it under rsiseg/core/seg), configured as
`decode_head.sampler=dict(type='OHEMPixelSampler', thresh=..., min_kept=...)`. Its map replaces `seg_weight`
in BaseDecodeHead.losses (decode_head.py:249-283).

The reference takes the soft-max of the up-sampled logits (or the per-pixel loss), sorts every valid key and,
with a `thresh`, compares a device value with a Python float (a host synchronisation). Here `pfst_ohem_weight`
(csrc/ohem.cu) computes each pixel's key from the LOW-resolution logits with the bilinear weights of the fused
loss and finds the order statistic by an exact radix select whose rank is read from the device: no up-sampled
tensor, no sort, nothing waits, so a decode-head loss with the sampler can be captured in a CUDA graph.

Rules the reference leaves to torch: keys order as `torch.sort` orders them (NaN after every number); without
a `thresh`, a tie at the boundary of the `min_kept * B` kept pixels goes to the lower flat index (a stable
descending sort; torch promises no order there).
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn as nn

from .. import ops
from .._lib import PfstError
from ..registry import PIXEL_SAMPLERS


@PIXEL_SAMPLERS.register_module()
class OHEMPixelSampler:
    """context: the decode head (its `ignore_index` and `loss_decode`, one softmax CrossEntropyLoss with
    `loss_weight` and `class_weight`). thresh: None (keep the `min_kept * B` pixels of largest loss) or the
    probability below which a pixel is hard. min_kept > 1."""

    def __init__(self, context, thresh: Optional[float] = None, min_kept: int = 100000):
        if int(min_kept) <= 1:
            raise ValueError(f"OHEMPixelSampler: min_kept must be > 1, got {min_kept}")
        self.context = context
        self.thresh = thresh
        self.min_kept = int(min_kept)
        self._class_weight: dict = {}            # (device, class weights) -> fp32 device tensor

    def _loss_params(self, device):
        loss = getattr(self.context, "loss_decode", None)
        if isinstance(loss, (nn.ModuleList, list, tuple)):
            raise PfstError("OHEMPixelSampler: several loss_decode modules are not supported (only a single "
                            "softmax cross-entropy)")
        if getattr(loss, "use_sigmoid", False):
            raise PfstError("OHEMPixelSampler: a sigmoid loss_decode is not supported (only a single softmax "
                            "cross-entropy)")
        cw = getattr(loss, "class_weight", None)
        if cw is not None:
            if isinstance(cw, torch.Tensor):
                cw = cw.to(device=device, dtype=torch.float32).contiguous()
            else:                                 # mmseg keeps a list: one host-to-device copy per device
                key = (device, tuple(float(v) for v in cw))
                if key not in self._class_weight:
                    self._class_weight[key] = torch.tensor(key[1], dtype=torch.float32, device=device)
                cw = self._class_weight[key]
        return float(getattr(loss, "loss_weight", 1.0)), cw

    def weight_map(self, seg_logit: torch.Tensor, seg_label: torch.Tensor) -> torch.Tensor:
        """The map `sample` returns for the bilinear (align_corners=False) up-sampling of seg_logit (B,C,lh,lw)
        to the labels' size, computed from seg_logit itself: an integer factor H/lh = W/lw >= 1."""
        loss_weight, class_weight = self._loss_params(seg_logit.device)
        with torch.no_grad():
            weight, _, _ = ops.ohem_weight(seg_logit.detach().contiguous(), seg_label.contiguous(),
                                           thresh=self.thresh, min_kept=self.min_kept,
                                           ignore_index=self.context.ignore_index, class_weight=class_weight,
                                           loss_weight=loss_weight)
        return weight

    def sample(self, seg_logit: torch.Tensor, seg_label: torch.Tensor) -> torch.Tensor:
        """mmseg `sample`: seg_logit (B,C,H,W) already at label resolution, seg_label (B,1,H,W)
        -> seg_weight (B,H,W) fp32 of 0 and 1."""
        if seg_logit.shape[2:] != seg_label.shape[2:] or seg_label.dim() != 4 or seg_label.shape[1] != 1:
            raise ValueError(f"OHEMPixelSampler.sample: seg_logit {tuple(seg_logit.shape)} and seg_label "
                             f"{tuple(seg_label.shape)} must be (B,C,H,W) and (B,1,H,W)")
        return self.weight_map(seg_logit, seg_label)
