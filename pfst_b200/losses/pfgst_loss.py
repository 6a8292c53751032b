"""PFGSTLoss — drop-in for rsiseg/models/losses/pfgst_loss.py:12-234.

Same constructor arguments, same `forward(tensors) -> dict` contract (six
autograd-connected 0-dim `loss_*` tensors + the 'vis|density_sim_feat' tuple),
computed by four sm_100a kernels (csrc/neigh.cu, csrc/pfgst_loss.cu) instead of
~60 ATen kernels, two 604 MB im2col buffers and 3+ host syncs. Besides the branch the
shipped configs use (configs/pfst/*.py:34-47: cosine, cross_prob_type='trg',
detach_unfold=True) the kernels cover sim_type='gaussian' (:189-191),
cross_prob_type='ema' (:161-178), detach_unfold=False (:148-149), src_loss_type='margin' /
'margin2' (:117-133) and top_k=None (:218-220); the remaining options (src_perc, proj_net_cfg,
kernel_size != 3) raise instead of silently computing something else.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from .. import ops
from .._lib import PfstError
from ..registry import LOSSES

LOSS_KEYS = ("loss_src_pos_mean", "loss_src_neg_mean", "loss_src_pos_std", "loss_src_neg_std",
             "loss_sim_pos", "loss_sim_neg")


class _PFGSTLossFn(torch.autograd.Function):
    """losses[6] = f(logits_trg, x_src | x_ema, gt_src, mix_masks). Gradients flow to
    logits_trg (through p only, q detached) and x_src, exactly as in the reference."""

    @staticmethod
    def forward(ctx, logits_trg, x_src, x_ema, gt_src, mix_masks, cfg, logits_ema=None):
        logits_trg = logits_trg.contiguous()
        x_src = x_src.contiguous()
        x_ema = x_ema.contiguous()
        gt_src = gt_src.contiguous()
        mix_masks = mix_masks.contiguous()
        geo = ops.LossGeometry(logits_trg.shape, x_src.shape, gt_src.shape, cfg["downscale"], cfg["dilation"])
        if x_ema.shape != x_src.shape:
            raise PfstError("PFGSTLoss: x_ema / x_src shape mismatch")
        for name, t in (("logits_trg", logits_trg), ("x_src", x_src), ("logits_ema", logits_ema)):
            if t is not None and t.dtype != torch.float32:
                raise TypeError(f"PFGSTLoss: {name} must be torch.float32, got {t.dtype} (only the teacher's "
                                "x_ema may be fp16 / bf16: the student's tensors carry gradients, and the loss's "
                                "second soft-max of logits_ema is fp32 only)")
        dots, ks = ops.neigh_dots(x_ema, x_src, geo.dilation // geo.up)
        opts, sigma = cfg.get("options", 0), cfg.get("sigma", 30.0)
        if logits_ema is not None:
            logits_ema = logits_ema.detach().contiguous()
        losses, stats, density, eroded = ops.pfgst_loss_fwd(dots, ks, geo, logits_trg, gt_src, mix_masks,
                                                            cfg["top_k"], cfg["w6"], options=opts, sigma=sigma,
                                                            logits_ema=logits_ema, margin=cfg.get("margin"))
        ctx.logits_ema = logits_ema
        ctx.save_for_backward(logits_trg, x_src, gt_src, mix_masks, dots, stats[0], stats[1])
        ctx.geo, ctx.ks, ctx.cfg = geo, ks, cfg
        ctx.mark_non_differentiable(density, eroded)
        return losses, density, eroded

    @staticmethod
    def backward(ctx, grad_losses, _gd, _ge):
        logits_trg, x_src, gt_src, mix_masks, dots, st, ws = ctx.saved_tensors
        stats = (st, ws)
        geo, cfg = ctx.geo, ctx.cfg
        need_logits, need_x = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        coef, glog = ops.pfgst_loss_bwd(dots, ctx.ks, geo, logits_trg, gt_src, mix_masks, cfg["top_k"], cfg["w6"],
                                        stats, grad_losses.contiguous().float(), want_logits_grad=need_logits,
                                        options=cfg.get("options", 0), sigma=cfg.get("sigma", 30.0),
                                        logits_ema=ctx.logits_ema, margin=cfg.get("margin"))
        gx = ops.neigh_grad(x_src, coef, geo.dilation // geo.up) if need_x else None
        return glog, gx, None, None, None, None, None


@LOSSES.register_module()
class PFGSTLoss(nn.Module):

    def __init__(self, top_k, dilation, kernel_size, weights, sigma=30, mean_sim=0.6, feat_level=2,
                 sim_type='gaussian', num_bins=100, apply_ignore=False, src_perc=None,
                 proj_net_cfg=None, src_loss_type='mean_std', margin=[0.5, 0.5],
                 detach_unfold=False, cross_prob_type='trg', downscale=None):
        super().__init__()
        unsupported = []
        if sim_type not in ('cosine', 'gaussian'):
            raise ValueError()                      # pfgst_loss.py:198-199
        if sim_type == 'gaussian' and not float(sigma) > 0:
            unsupported.append(f"sigma={sigma} (must be positive)")
        if kernel_size != 3:
            unsupported.append(f"kernel_size={kernel_size} (only 3)")
        if top_k is not None and not (1 <= int(top_k) <= 4):
            unsupported.append(f"top_k={top_k} (1..4 or None)")
        if src_perc is not None:
            unsupported.append("src_perc")
        if proj_net_cfg is not None:
            unsupported.append("proj_net_cfg")
        if src_loss_type not in ('mean_std', 'margin', 'margin2'):
            unsupported.append(f"src_loss_type={src_loss_type!r} ('mean_std', 'margin', 'margin2')")
        elif src_loss_type != 'mean_std' and not all(abs(float(m)) <= 1.0 for m in margin):
            unsupported.append(f"margin={margin} (|margin| <= 1: similarities lie in [-1, 1])")
        if cross_prob_type not in ('trg', 'ema'):
            unsupported.append(f"cross_prob_type={cross_prob_type!r} ('trg' or 'ema')")
        if unsupported:
            raise PfstError("PFGSTLoss (B200 path) does not implement: " + "; ".join(unsupported))
        if not isinstance(weights, dict):
            raise PfstError("PFGSTLoss: `weights` must be the dict form used by configs/pfst/*.py")
        self.top_k = None if top_k is None else int(top_k)
        self.margin = margin
        self.dilation = int(dilation)
        self.kernel_size = kernel_size
        self.weights = weights
        self.sim_type = sim_type
        self.sigma = sigma
        self.feat_level = feat_level
        self.detach_unfold = detach_unfold
        self.cross_prob_type = cross_prob_type
        self.downscale = downscale
        self.src_loss_type = src_loss_type
        options = ((ops.LOSS_SIM_GAUSSIAN if sim_type == 'gaussian' else 0) |
                   (ops.LOSS_CROSS_PROB_EMA if cross_prob_type == 'ema' else 0) |
                   (0 if detach_unfold else ops.LOSS_UNFOLD_GRAD) |
                   {'mean_std': 0, 'margin': ops.LOSS_SRC_MARGIN, 'margin2': ops.LOSS_SRC_MARGIN2}[src_loss_type])
        # top_k=None (pfgst_loss.py:218-220) travels as 0; the margin losses read no *_std weights (:117-133)
        self._cfg = dict(top_k=self.top_k or 0, dilation=self.dilation, downscale=downscale,
                         w6=(weights['src_pos'], weights['src_neg'], weights.get('src_pos_std', 0.0),
                             weights.get('src_neg_std', 0.0), weights['sim_pos'], weights['sim_neg']),
                         options=options, sigma=float(sigma),
                         margin=None if src_loss_type == 'mean_std' else (float(margin[0]), float(margin[1])))

    @property
    def shipped_branch(self) -> bool:
        """True for the configuration the fused launch groups of PluginEngine / SelfTrainingStep are built for."""
        return self._cfg["options"] == 0 and self.top_k is not None

    def forward(self, tensors):
        logits_trg = tensors['logits_trg']
        gt_src = tensors['gt_src']
        x_ema = tensors['x_ema'][self.feat_level] if self.feat_level is not None else tensors['x_ema']
        x_src = tensors['x_src'][self.feat_level] if self.feat_level is not None else tensors['x_src']
        logits_ema = tensors['logits_ema'] if self.cross_prob_type == 'ema' else None
        losses, density, eroded = _PFGSTLossFn.apply(logits_trg, x_src, x_ema.detach(), gt_src,
                                                     tensors['mix_masks'], self._cfg, logits_ema)
        if self.src_loss_type == 'mean_std':
            out = {k: losses[i] for i, k in enumerate(LOSS_KEYS)}
        else:                                   # pfgst_loss.py:117-133: two source losses, no std terms
            out = {'loss_src_pos': losses[0], 'loss_src_neg': losses[1], 'loss_sim_pos': losses[4],
                   'loss_sim_neg': losses[5]}
        out['vis|density_sim_feat'] = (tensors.get('img_trg'), density, eroded.bool())
        return out
