"""PFGST — drop-in for rsiseg/models/uda/pfgst.py:53-368 (the UDA trainer selected
by `uda.type='PFGST'`, configs/_base_/uda/pfst.py:8).

Same constructor keys, same `train_step` / `forward_train` / `_init_ema_weights` /
`_update_ema` / `get_model` / `get_ema_model` / `get_imnet_model` API, same
`log_vars` keys and `vis|…` states, same host RNG consumption (python `random` for
the jitter/blur draws, the global numpy stream for ClassMix). The three segmentor
passes are the caller's network (cuDNN); everything between them runs in the
sm_100a kernels of this package:

  reference (pfgst.py)                                   here
  ------------------------------------------------------------------------------
  :105-127  per-tensor Python EMA loop (~850 launches)   EmaTable.update, 1 launch
  :259-266  softmax/max/ge/sum/.item()/.cpu()            ops.pseudo_label, 1 launch,
                                                         count stays on the device
  :282      torch.unique + np.random.choice + eq/sum     ClassMixPlan (presence kernel,
                                                         36-byte D2H, host draw)
  :287-300  2B strong_transform calls in a Python loop   ops.class_mix, 1 launch
            + kornia GaussianBlur2d per image (51x51)    ops.gaussian_blur, 1 launch
  :333-342  PFGSTLoss (~60 ATen kernels, 3+ syncs)       losses.PFGSTLoss, 2+2 launches
  optional  --                                           PrototypeBank / proto_dist_loss
                                                         (north_star P1-P3, cfg 'prototypes')
"""
from __future__ import annotations

import random
import warnings
from copy import deepcopy

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F
from torch.nn.modules.dropout import _DropoutNd

from .. import losses as _losses  # noqa: F401  (registers PFGSTLoss in LOSSES)
from .. import ops
from .._lib import PfstError
from ..engine import LOSS_KEYS, PluginEngine, StepTotalFn
from ..losses.pfgst_loss import PFGSTLoss
from ..prototypes import PrototypeBank, masked_feat_dist as _masked_feat_dist, proto_dist_loss
from ..registry import UDA, build_loss
from ..utils.dacs_transforms import ClassMixPlan, draw_color_jitter, gaussian_blur_batch, get_mean_std
from .log_ledger import StepRecord, ledger_for
from .uda_decorator import UDADecorator, build_model, get_module


def add_prefix(inputs, prefix):
    """rsiseg/core/utils/misc.py:2-18."""
    return {f'{prefix}.{name}': value for name, value in inputs.items()}


def _params_equal(ema_model, model):
    """pfgst.py:33-39."""
    for ema_param, param in zip(ema_model.named_parameters(), model.named_parameters()):
        if not torch.equal(ema_param[1].data, param[1].data):
            return False
    return True


@UDA.register_module()
class PFGST(UDADecorator):

    def __init__(self, **cfg):
        super().__init__(**cfg)
        self.local_iter = 0
        self.max_iters = cfg['max_iters']
        self.alpha = cfg['alpha']
        self.pseudo_threshold = cfg['pseudo_threshold']
        self.psweight_ignore_top = cfg['pseudo_weight_ignore_top']
        self.psweight_ignore_bottom = cfg['pseudo_weight_ignore_bottom']
        self.fdist_lambda = cfg['imnet_feature_dist_lambda']
        self.fdist_classes = cfg['imnet_feature_dist_classes']
        self.fdist_scale_min_ratio = cfg['imnet_feature_dist_scale_min_ratio']
        self.enable_fdist = self.fdist_lambda > 0
        self.mix = cfg['mix']
        self.blur = cfg['blur']
        self.color_jitter_s = cfg['color_jitter_strength']
        self.color_jitter_p = cfg['color_jitter_probability']
        self.print_grad_magnitude = cfg['print_grad_magnitude']
        self.trg_loss_weight = cfg.get('trg_loss_weight', 1.)
        self.use_decoded_feats = cfg.get('use_decoded_feats', False)
        self.thre_type = cfg.get('thre_type', 'all')
        self.strong_aug_denorm_type = cfg.get('strong_aug_denorm_type', 'mean_std')
        self.apply_no_mix = cfg.get('apply_no_mix', False)
        assert self.mix == 'class'
        if self.thre_type not in ('all', 'part'):
            raise ValueError(f"thre_type {self.thre_type!r}")
        # B200-path extras (absent keys = reference behaviour)
        self.pseudo_threshold_per_class = cfg.get('pseudo_threshold_per_class', None)   # north_star S2'
        # kornia's ColorJitter in strong_transform (dacs_transforms.py:56-85): 'builtin' (default) runs the
        # in-tree restatement of kornia 0.6 (parity unpinned: kornia is not installed where this was
        # built), 'skip' leaves the image unjittered, 'error' raises when the branch is drawn
        self.kornia_aug = cfg.get('kornia_aug', 'builtin')
        if self.kornia_aug not in ('builtin', 'skip', 'error'):
            raise ValueError(f"kornia_aug {self.kornia_aug!r}")
        if self.kornia_aug == 'builtin' and self.color_jitter_p < 1.0:
            warnings.warn("PFGST (B200 path): the colour jitter of strong_transform runs the built-in restatement of "
                          "kornia.augmentation.ColorJitter (0.6 series); it has not been compared with an installed "
                          "kornia (kornia_aug='error' refuses the branch instead, 'skip' drops it)", stacklevel=2)
        self.compute_vis = cfg.get('compute_vis', True)
        proto_cfg = cfg.get('prototypes', None)

        self.class_probs = {}
        self.ema_model = build_model(cfg['model'])
        # pfgst.py:84-87: with imnet_feature_dist_lambda > 0 the reference builds a third (ImageNet) copy of
        # the segmentor — and never uses it: PFGST.forward_train has no feature-distance term
        self.imnet_model = build_model(cfg['model']) if self.enable_fdist else None

        aux_losses = cfg.get('aux_losses', None)
        self.apply_aux = False
        if aux_losses is not None:
            self.apply_aux = True
            if not type(aux_losses) == list:
                aux_losses = [aux_losses]
            aux_losses = [l if isinstance(l, nn.Module) else build_loss(l) for l in aux_losses]
            self.aux_losses = nn.ModuleList(aux_losses)

        self._ema_table = None
        self._mix_plan = None
        self._thr_vec = None
        self.proto_cfg = proto_cfg
        self.proto_bank = None
        self._engine = None            # PluginEngine: the fused launch groups (built on first use)
        self._aux_stream = None        # high-priority stream of the class-presence read
        self._teacher_eval_modules = None
        self._geo_cache = {}
        self.fused = cfg.get('fused_hot_path', True)

    # ------------------------------------------------------------------ accessors
    def get_ema_model(self):
        return get_module(self.ema_model)

    def get_imnet_model(self):
        return get_module(self.imnet_model)

    # ------------------------------------------------------------------------ EMA
    TABLE_RECHECK = 64     # iterations between full pointer checks of the 2 x 214 parameter tensors

    def _table(self):
        """The (teacher, student) pointer table of the multi-tensor EMA kernel. Parameter objects and
        their storage are stable while an optimizer updates them in place, so the table is built once;
        every call spot-checks the first and last tensor, every TABLE_RECHECK-th call (and any call
        after the module was moved or cast through `_apply`) re-walks all parameters."""
        t = self._ema_table
        self._table_calls = getattr(self, "_table_calls", 0) + 1
        if t is not None and self._table_calls % self.TABLE_RECHECK:
            (e0, e1), (p0, p1) = self._table_spot
            if (e0.data_ptr(), e1.data_ptr(), p0.data_ptr(), p1.data_ptr()) == self._table_spot_ptrs:
                return t
        ema_p = list(self.get_ema_model().parameters())
        stu_p = list(self.get_model().parameters())
        if t is None or t.stale(ema_p, stu_p):
            self._ema_table = t = ops.EmaTable(ema_p, stu_p)
        self._table_spot = ((ema_p[0], ema_p[-1]), (stu_p[0], stu_p[-1]))
        self._table_spot_ptrs = (ema_p[0].data_ptr(), ema_p[-1].data_ptr(), stu_p[0].data_ptr(), stu_p[-1].data_ptr())
        return t

    def _apply(self, fn, *args, **kwargs):
        self._ema_table = None          # .to() / .cuda() / .half() re-allocate the parameters
        return super()._apply(fn, *args, **kwargs)

    def _init_ema_weights(self):
        """pfgst.py:105-114 — teacher <- student, one launch."""
        for param in self.get_ema_model().parameters():
            param.detach_()
        self._table().update(0.0, 1.0, mode=1)

    def _update_ema(self, iter):
        """pfgst.py:116-127 — one launch, fl(fl(a*ema)+fl((1-a)*p)) per element."""
        a32, b32 = ops.ema_coeffs(iter, self.alpha)
        self._table().update(a32, b32, mode=0)

    # ----------------------------------------------------------------- train step
    def train_step(self, data_batch, optimizer, **kwargs):
        """pfgst.py:129-166."""
        optimizer.zero_grad()
        log_vars, vis_states = self(**data_batch)
        optimizer.step()
        log_vars.pop('loss', None)
        return dict(log_vars=log_vars, num_samples=len(data_batch['img_metas']), states=vis_states)

    def masked_feat_dist(self, f1, f2, mask=None):
        """pfgst.py:168-177 (no caller in the reference's PFGST either): one fused launch each way."""
        return _masked_feat_dist(f1, f2, mask)

    def _threshold_args(self, dev):
        if self.pseudo_threshold_per_class is None:
            return float(self.pseudo_threshold), None
        if self._thr_vec is None or self._thr_vec.device != dev:
            self._thr_vec = torch.tensor(list(self.pseudo_threshold_per_class), dtype=torch.float32, device=dev)
        return 0.0, self._thr_vec

    def _check_kornia(self, color_jitter):
        """-> True when the built-in colour jitter must run for this iteration."""
        if not (color_jitter > self.color_jitter_p):
            return False
        if self.kornia_aug == 'builtin':
            return True
        msg = ("the kornia ColorJitter branch of strong_transform is third-party arithmetic with its own random "
               "sampler (SURVEY.md §8c): kornia_aug='builtin' runs the built-in restatement (parity unpinned), "
               "color_jitter_probability=1.0 disables the branch")
        if self.kornia_aug == 'skip':
            warnings.warn(msg + "; skipped (kornia_aug='skip')", stacklevel=3)
            return False
        raise PfstError(msg)

    # ------------------------------------------------------------------ fused launch groups
    def _fused_loss_module(self):
        """The PFGSTLoss module when the auxiliary-loss section can run as the engine's fused launch
        groups (exactly one PFGSTLoss on a single decoded-feature map), else None -> generic path."""
        if not self.fused or not self.apply_aux or len(self.aux_losses) != 1:
            return None
        mod = self.aux_losses[0]
        return mod if type(mod) is PFGSTLoss and mod.feat_level is None and mod.shipped_branch else None

    def _get_engine(self, dev, loss_module) -> PluginEngine:
        if self._engine is None or self._engine.device != dev:
            self._engine = PluginEngine(dev, self.num_classes, None if loss_module is None else loss_module._cfg,
                                        self.proto_cfg, alpha=self.alpha)
        return self._engine

    def _freeze_teacher_dropout(self):
        """pfgst.py:247-251; the module list is collected once (the model structure is static)."""
        if self._teacher_eval_modules is None:
            self._teacher_eval_modules = [m for m in self.get_ema_model().modules()
                                          if isinstance(m, _DropoutNd) or type(m).__name__ == 'DropPath']
        for m in self._teacher_eval_modules:
            m.training = False

    def d2h_bytes(self) -> int:
        """Bytes this module has copied device->host so far (log-variable ledger reads + the
        36-byte class-presence reads of ClassMix)."""
        n = 0
        for p in self.parameters():
            n = ledger_for(p.device).d2h_bytes
            break
        return n + (0 if self._mix_plan is None else 36 * self._mix_plan._started)

    def close(self) -> None:
        """Collective on multi-rank runs, before destroy_process_group(): drops the captured graphs
        and unmaps the NVLink peer boards of the prototype exchange."""
        if self._engine is not None:
            self._engine.close()
            self._engine = None

    def forward_train(self, img, img_metas, gt_semantic_seg, target_img, target_img_metas,
                      target_img_strong_aug):
        """pfgst.py:179-356. gt_semantic_seg: int64 or uint8; the iteration's pseudo labels, ClassMix labels
        and masks follow its dtype (the student's forward_train receives source and mixed labels in it)."""
        if gt_semantic_seg.dtype not in ops.LABEL_DTYPES:     # before any launch or RNG draw
            raise TypeError(f"gt_semantic_seg: label maps must be torch.int64 or torch.uint8, got {gt_semantic_seg.dtype}")
        log_vars = {}
        vis_states = {}
        batch_size = img.shape[0]
        dev = img.device
        loss_mod = self._fused_loss_module()
        eng = self._get_engine(dev, loss_mod)
        ledger = ledger_for(dev)
        ledger.begin()
        parts, part_w = [], []

        # ① EMA teacher (pfgst.py:203-208): own stream, joined right before the teacher pass ④
        if self.local_iter == 0:
            for param in self.get_ema_model().parameters():
                param.detach_()
        eng.launch_ema(self._table(), self.local_iter)

        # ② host RNG draws, in the reference's order (pfgst.py:212-222)
        color_jitter = random.uniform(0, 1)
        blur = random.uniform(0, 1) if self.blur else 0
        jitter = self._check_kornia(color_jitter)

        # ClassMix needs the batch's class set: presence kernel + 36-byte D2H on a high-priority
        # stream now, read after the two network passes have been enqueued (SURVEY.md §7)
        gt_semantic_seg = gt_semantic_seg.contiguous()
        if self._mix_plan is None or self._mix_plan.device != dev or batch_size > self._mix_plan._chosen.shape[0]:
            self._mix_plan = ClassMixPlan(dev, max_batch=max(batch_size, 64))
            self._aux_stream = torch.cuda.Stream(device=dev, priority=-1)
        self._mix_plan.drop_pending()          # an exception in an earlier iteration must not shift the FIFO
        self._aux_stream.wait_stream(torch.cuda.current_stream())
        self._mix_plan.start(gt_semantic_seg, self._aux_stream)

        # ③ student on source (pfgst.py:225-236)
        clean_losses = self.get_model().forward_train(
            img, img_metas, gt_semantic_seg, return_feats=True, return_logits=True,
            return_decoded_feats=self.use_decoded_feats)
        src_feats = clean_losses.pop('features')
        if self.use_decoded_feats:
            src_feats = clean_losses.pop('decoded_features')
        src_logits = clean_losses.pop('logits')
        single_feats = isinstance(src_feats, torch.Tensor)
        fused = loss_mod is not None and single_feats
        rec = StepRecord(ledger) if fused else None     # fused path: ONE gather launch for the whole iteration
        if fused:
            log_vars.update(rec.add(clean_losses, 1.0))
        else:
            clean_loss, clean_log_vars = self._parse_losses(clean_losses)
            log_vars.update(clean_log_vars)
            parts.append(clean_loss); part_w.append(1.0)

        # ④ teacher on target (pfgst.py:247-257) — after the EMA update of this iteration
        self._freeze_teacher_dropout()
        eng.wait_ema()
        ema_logits, ema_states = self.get_ema_model().encode_decode(target_img, target_img_metas)
        ema_feats = ema_states['feats']
        if self.use_decoded_feats:
            ema_feats = ema_states['decoded_features']

        # ⑤ pseudo labels (pfgst.py:259-277) ║ neighbourhood dots of x_ema -> prototypes (P1/P2)
        thr, thr_vec = self._threshold_args(dev)
        single_feats = single_feats and isinstance(ema_feats, torch.Tensor)
        if fused and not single_feats:
            raise PfstError("PFGSTLoss(feat_level=None) needs single feature maps from both passes")
        if self.proto_cfg is not None and not single_feats:
            raise PfstError("prototypes need use_decoded_feats=True (a single (B,D,h,w) feature map)")
        geo = None
        if fused:
            gkey = (src_logits.shape, src_feats.shape, gt_semantic_seg.shape)
            geo = self._geo_cache.get(gkey)
            if geo is None:
                geo = self._geo_cache[gkey] = ops.LossGeometry(src_logits.shape, src_feats.shape,
                                                               gt_semantic_seg.shape, loss_mod.downscale,
                                                               loss_mod.dilation)
            if ema_feats.shape != src_feats.shape:
                raise PfstError("PFGSTLoss: x_ema / x_src shape mismatch")
        x_ema = ema_feats.detach().contiguous() if (fused or self.proto_cfg is not None) else None
        pseudo_label, pseudo_prob, count, weight_part = eng.teacher_outputs(
            ema_logits.detach().contiguous(), x_ema, thr, thr_vec,
            self.thre_type == 'part', geo, label_dtype=gt_semantic_seg.dtype)
        ps_size = pseudo_label.numel()

        # ⑥⑦ ClassMix (pfgst.py:281-300): host draw, then ONE fused launch
        chosen = self._mix_plan.choose()
        if self.apply_no_mix:
            chosen = torch.zeros_like(chosen)
        trg_img = target_img if self.apply_no_mix else target_img_strong_aug
        mixed_img, mixed_lbl, pseudo_weight, mix_masks = ops.class_mix(
            gt_semantic_seg, chosen, img.contiguous(), trg_img.contiguous(), pseudo_label,
            weight_in=weight_part, count=count, ps_size=ps_size,
            ignore_top=self.psweight_ignore_top, ignore_bottom=self.psweight_ignore_bottom)
        # gaussian_blur of strong_transform (dacs_transforms.py:88-107): B sigma draws in image
        # order on the global numpy stream (after the ClassMix draws, as in the reference loop)
        if jitter:
            # color_jitter of strong_transform (dacs_transforms.py:56-85): one kornia-style draw per image
            # from the torch CPU generator, in image order; denorm/renorm with the first image's statistics
            # like the reference (`means[0]`, pfgst.py:218-219)
            draws = [draw_color_jitter(self.color_jitter_s) for _ in range(batch_size)]
            dn = self.strong_aug_denorm_type == 'mean_std'
            if self.strong_aug_denorm_type not in ('mean_std', 'none'):
                raise ValueError('No such denorm type!')
            mixed_img = ops.color_jitter(mixed_img, [d[0] for d in draws], [d[1] for d in draws],
                                         img_metas[0]['img_norm_cfg']['mean'] if dn else None,
                                         img_metas[0]['img_norm_cfg']['std'] if dn else None)
        mixed_img = gaussian_blur_batch(blur, mixed_img)

        # ⑧ student on the mixed batch (pfgst.py:303-310)
        mix_losses = self.get_model().forward_train(
            mixed_img, img_metas, mixed_lbl, pseudo_weight, return_feats=True, return_logits=True)
        mixed_feats = mix_losses.pop('features')
        mixed_logits = mix_losses.pop('logits')
        mix_losses = add_prefix(mix_losses, 'mix')
        if fused:
            log_vars.update(rec.add(mix_losses, float(self.trg_loss_weight)))
        else:
            mix_loss, mix_log_vars = self._parse_losses(mix_losses)
            log_vars.update(mix_log_vars)
            parts.append(mix_loss); part_w.append(float(self.trg_loss_weight))

        # ⑨ auxiliary losses (pfgst.py:333-342) + P3
        if fused:
            mixed_logits_c, src_feats_c = mixed_logits.contiguous(), src_feats.contiguous()
            plan = eng.aux_plan(mixed_logits_c, src_feats_c, gt_semantic_seg, mix_masks, geo, self.compute_vis)
            fb = plan["b"]
            log_vars.update(rec.add(dict(zip(LOSS_KEYS, fb["loss_views"])), 1.0))
            if self.proto_cfg is not None:
                self.proto_bank = eng.bank
                log_vars.update(rec.add({'loss_proto_dist': fb["ploss_view"]}, 1.0))
            # ⑩ total = 0 + clean + mix*w + aux (+ proto) (pfgst.py:237,310,342): one autograd node whose
            # forward is the auxiliary launch group + ONE gather launch for every log variable
            idx = [i for i, t in enumerate(rec.tensors) if t.requires_grad]
            total_loss = StepTotalFn.apply(eng, rec, plan, gt_semantic_seg, idx, mixed_logits_c, src_feats_c,
                                           *[rec.tensors[i] for i in idx])
            if self.compute_vis:
                vis_states['vis|density_sim_feat'] = (mixed_img, fb["density"].clone(), fb["eroded"].bool())
        else:
            tensors = dict(
                img_src=img, img_src_metas=img_metas, img_trg=mixed_img, img_mixed=mixed_img,
                img_metas_trg=target_img_metas, gt_src=gt_semantic_seg, x_src=src_feats, x_ema=ema_feats,
                x_trg=mixed_feats, logits_src=src_logits, logits_trg=mixed_logits, logits_ema=ema_logits,
                mix_masks=mix_masks, pseudo_weight=pseudo_weight)
            if self.apply_aux:
                aux_losses = self._get_aux_losses(tensors=tensors)
                vis_states.update({k: v for k, v in aux_losses.items() if k.startswith('vis|')})
                for name in vis_states.keys():
                    aux_losses.pop(name)
                aux_loss, aux_log_vars = self._parse_losses(aux_losses)
                log_vars.update(aux_log_vars)
                parts.append(aux_loss); part_w.append(1.0)
            if self.proto_cfg is not None:       # prototypes were accumulated / finalised in group 1
                self.proto_bank = eng.bank
                proto_loss = proto_dist_loss(src_feats, gt_semantic_seg, eng.bank.mu, eng.bank.seen) \
                    * self.proto_cfg.get('weight', 0.1)
                p_loss, p_log_vars = self._parse_losses({'loss_proto_dist': proto_loss})
                log_vars.update(p_log_vars)
                parts.append(p_loss); part_w.append(1.0)

            # ⑩ total = 0 + clean + mix*w + aux (+ proto), one launch
            total_loss = ledger.weighted_total(parts, part_w)
        ledger.end()
        total_loss.backward()

        # ⑪ vis states (pfgst.py:346-352)
        if self.compute_vis:
            vis_pseudo_weight = F.interpolate(pseudo_weight.unsqueeze(1), mixed_lbl.shape[2:])
            vis_mask_mix = torch.where(vis_pseudo_weight > 0.0, mixed_lbl, 255)
            vis_states.update({
                'vis|seg_mask_src': (img, gt_semantic_seg, src_logits.max(dim=1)[1].unsqueeze(1)),
                'vis|seg_mask_mix': (mixed_img, vis_mask_mix, mixed_logits.max(dim=1)[1].unsqueeze(1).float()),
            })

        self.local_iter += 1
        return log_vars, vis_states

    def _get_aux_losses(self, tensors):
        """pfgst.py:358-368."""
        aux_losses = dict()
        for loss_module in self.aux_losses:
            loss_ = loss_module(tensors)
            if loss_ is None:
                continue
            aux_losses.update(loss_)
        return aux_losses
