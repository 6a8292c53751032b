"""Generate the committed golden fixtures from the REFERENCE code itself.

Needs a checkout of the reference named by PFST_REFERENCE: `python tests/golden/make_golden.py`.
Every fixture stores the (small) inputs and the outputs the reference produced for
them, so that tests can pin (a) the oracle and (b) the CUDA path against the
reference on machines where the reference checkout does not exist.

reference_live.npz is the exception: `python tests/golden/make_golden.py reference_live` records
the oracle's outputs on the inputs of the live comparisons in test_oracle_pins.py and
test_host_logic.py, at a commit where each of those comparisons had passed bit for bit against the
reference checkout. Those tests compare against it everywhere, and against the reference itself
when PFST_REFERENCE is set.

  metrics.npz      rsiseg/core/evaluation/metrics.py  eval_metrics / intersect_and_union
  ema.npz          PFGST._init_ema_weights / _update_ema      (pfgst.py:105-127)
  pseudo_mix.npz   pseudo-label block + get_class_masks + strong_transform loop
                   (pfgst.py:259-300, dacs_transforms.py:110-144)
  pfgst_loss.npz   PFGSTLoss.forward + autograd backward      (pfgst_loss.py:44-234)
  pfgst_step.npz   three PFGST.train_step iterations on a tiny segmentor
  weighted_ce.npz  BaseDecodeHead.losses: resize + cross_entropy + accuracy (+ autograd backward)
                   (decode_head.py:249-283, cross_entropy_loss.py:12-65, accuracy.py:6-59)
"""
from __future__ import annotations

import random
import sys
import types
import warnings
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent.parent
sys.path.insert(0, str(ROOT))

from tests.golden import ref_loader as R  # noqa: E402
from tests.fake_segmentor import TinySegmentor  # noqa: E402
from pfst_b200.synthetic import blocky_labels, teacher_logits  # noqa: E402

OUT = Path(__file__).resolve().parent
W6 = {'src_pos': 0.1, 'src_neg': 0.1, 'sim_pos': 0.1, 'sim_neg': 0.1, 'src_pos_std': 0.1, 'src_neg_std': 0.1}
LOSS_KEYS = ("loss_src_pos_mean", "loss_src_neg_mean", "loss_src_pos_std", "loss_src_neg_std",
             "loss_sim_pos", "loss_sim_neg")


def gen_metrics():
    M = R.metrics()
    rs = np.random.RandomState(0)
    C = 19
    pred = rs.randint(0, C, size=(10, 30, 30))
    label = rs.randint(0, C, size=(10, 30, 30))
    label[:, 2, 5:10] = 255                       # the reference test's ignore stripe
    out = {"pred": pred.astype(np.int64), "label": label.astype(np.int64), "C": C}
    ret = M.eval_metrics(pred, label, C, 255, metrics=["mIoU", "mDice", "mFscore"])
    for k, v in ret.items():
        out["all_" + k] = np.asarray(v)
    per = [M.intersect_and_union(pred[i], label[i], C, 255) for i in range(10)]
    out["per_image"] = np.stack([np.stack([a.numpy() for a in p]) for p in per])
    ret = M.pre_eval_to_metrics(per, ["mIoU"])
    out["pre_eval_IoU"] = ret["IoU"]
    # label_map + reduce_zero_label, uint8 labels
    lab8 = rs.randint(0, 8, size=(64, 64)).astype(np.uint8)
    lab8[:4] = 255
    pr = rs.randint(0, 6, size=(64, 64)).astype(np.int64)
    out["lm_pred"], out["lm_label"] = pr, lab8
    a = M.intersect_and_union(pr, lab8.copy(), 6, 255, {7: 0, 6: 255}, True)
    out["lm_areas"] = np.stack([t.numpy() for t in a])
    np.savez_compressed(OUT / "metrics.npz", **out)


def gen_ema():
    M = R.pfgst()
    g = torch.Generator().manual_seed(1234)
    shapes = [(), (1,), (3,), (513,), (4097,), (8, 3, 3, 3)]
    student = [torch.nn.Parameter(0.02 * torch.randn(s, generator=g)) for s in shapes]
    teacher = [torch.nn.Parameter(0.02 * torch.randn(s, generator=g)) for s in shapes]

    class Holder:
        alpha = 0.999

        def get_model(self):
            return types.SimpleNamespace(parameters=lambda: iter(student))

        def get_ema_model(self):
            return types.SimpleNamespace(parameters=lambda: iter(teacher))

    h = Holder()
    out = {f"student_{i}": p.detach().numpy().copy() for i, p in enumerate(student)}
    out.update({f"teacher0_{i}": p.detach().numpy().copy() for i, p in enumerate(teacher)})
    its = [1, 2, 10, 999, 5000]
    out["iters"] = np.array(its)
    for it in its:
        M.PFGST._update_ema(h, it)
        for i, p in enumerate(teacher):
            out[f"teacher_it{it}_{i}"] = p.detach().numpy().copy()
    M.PFGST._init_ema_weights(h)
    for i, p in enumerate(teacher):
        out[f"teacher_init_{i}"] = p.detach().numpy().copy()
    np.savez_compressed(OUT / "ema.npz", **out)


def gen_pseudo_mix():
    """pfgst.py:259-300 executed verbatim through the reference's own functions."""
    D = R.dacs_transforms()
    g = torch.Generator().manual_seed(77)
    B, C, H, W = 2, 6, 64, 64
    logits = teacher_logits(B, C, H, W, g)
    gt = blocky_labels(B, H, W, C, g, min_rect=4, max_rect=32)
    img = torch.randn((B, 3, H, W), generator=g)
    trg = torch.randn((B, 3, H, W), generator=g)
    out = dict(logits=logits.numpy(), gt=gt.numpy().astype(np.uint8), img=img.numpy(), trg=trg.numpy())
    thr, top, bottom = 0.98, 2, 3
    ema_softmax = torch.softmax(logits.detach(), dim=1)
    pseudo_prob, pseudo_label = torch.max(ema_softmax, dim=1)
    ps_large_p = pseudo_prob.ge(thr).long() == 1
    ps_size = np.size(np.array(pseudo_label.cpu()))
    pseudo_weight = torch.sum(ps_large_p).item() / ps_size
    pseudo_weight = pseudo_weight * torch.ones(pseudo_prob.shape)
    pseudo_weight[:, :top, :] = 0
    pseudo_weight[:, -bottom:, :] = 0
    gt_pixel_weight = torch.ones(pseudo_weight.shape)
    np.random.seed(5)
    mix_masks = D.get_class_masks(gt)
    param = dict(mix=None, color_jitter=0.1, color_jitter_s=0.2, color_jitter_p=1.0, blur=0,
                 mean=torch.zeros(1, 3, 1, 1), std=torch.ones(1, 3, 1, 1), denorm_type='mean_std')
    mixed_img, mixed_lbl = [None] * B, [None] * B
    for i in range(B):
        param['mix'] = mix_masks[i]
        mixed_img[i], mixed_lbl[i] = D.strong_transform(param, data=torch.stack((img[i], trg[i])),
                                                        target=torch.stack((gt[i][0], pseudo_label[i])))
        _, pseudo_weight[i] = D.strong_transform(param, target=torch.stack((gt_pixel_weight[i], pseudo_weight[i])))
    out.update(pseudo_label=pseudo_label.numpy().astype(np.uint8), pseudo_prob=pseudo_prob.numpy(),
               large=ps_large_p.numpy(), mixed_img=torch.cat(mixed_img).numpy(),
               mixed_lbl=torch.cat(mixed_lbl).numpy().astype(np.uint8), mixed_weight=pseudo_weight.numpy(),
               mix_masks=torch.cat(mix_masks).numpy().astype(np.uint8), thr=thr, top=top, bottom=bottom, seed=5)
    np.savez_compressed(OUT / "pseudo_mix.npz", **out)


def gen_pfgst_loss():
    L = R.pfgst_loss()
    D = R.dacs_transforms()
    cases = {"a": dict(B=2, C=6, H=128, D=32, dil=2, down=0.5, seed=1),      # identity feature grid
             "b": dict(B=3, C=33, H=48, D=16, dil=2, down=None, seed=2)}     # 2x up-sampled features
    out = {}
    for name, c in cases.items():
        g = torch.Generator().manual_seed(c["seed"])
        B, C, H = c["B"], c["C"], c["H"]
        gt = blocky_labels(B, H, H, C, g, min_rect=4, max_rect=max(8, H // 2))
        logits = 2.0 * torch.randn((B, C, H // 4, H // 4), generator=g)
        x_src = torch.relu(torch.randn((B, c["D"], H // 8, H // 8), generator=g))
        x_ema = torch.relu(torch.randn((B, c["D"], H // 8, H // 8), generator=g))
        np.random.seed(3)
        mix = torch.cat(D.get_class_masks(gt), 0)
        mod = L.PFGSTLoss(top_k=3, dilation=c["dil"], kernel_size=3, weights=W6, sim_type='cosine',
                          feat_level=None, detach_unfold=True, downscale=c["down"])
        lt = logits.clone().requires_grad_(True)
        xs = x_src.clone().requires_grad_(True)
        with R.cpu_cuda_identity():
            res = mod(dict(logits_trg=lt, logits_ema=None, gt_src=gt, x_ema=x_ema, x_src=xs, img_trg=None,
                           mix_masks=mix))
        sum(res[k] for k in LOSS_KEYS).backward()
        out.update({f"{name}_gt": gt.numpy().astype(np.uint8), f"{name}_logits": logits.numpy(),
                    f"{name}_x_src": x_src.numpy(), f"{name}_x_ema": x_ema.numpy(),
                    f"{name}_mix": mix.numpy().astype(np.uint8),
                    f"{name}_losses": np.array([float(res[k]) for k in LOSS_KEYS], dtype=np.float32),
                    f"{name}_grad_x_src": xs.grad.numpy(), f"{name}_grad_logits": lt.grad.numpy(),
                    f"{name}_density": res['vis|density_sim_feat'][1].numpy(),
                    f"{name}_eroded": res['vis|density_sim_feat'][2].numpy(),
                    f"{name}_cfg": np.array([c["dil"], -1 if c["down"] is None else c["down"]], dtype=np.float64)})
    np.savez_compressed(OUT / "pfgst_loss.npz", **out)


LOSS_OPTION_CASES = {
    # name: (geometry case, reference constructor options)
    "gauss": (dict(B=2, C=6, H=128, D=32, dil=2, down=0.5, seed=11), dict(sim_type='gaussian', sigma=3.0,
                                                                          detach_unfold=True)),
    "gauss33": (dict(B=2, C=33, H=48, D=16, dil=2, down=None, seed=12), dict(sim_type='gaussian', sigma=2.0,
                                                                            detach_unfold=True)),
    "ema": (dict(B=2, C=6, H=64, D=16, dil=2, down=None, seed=13), dict(sim_type='cosine', cross_prob_type='ema',
                                                                       detach_unfold=True)),
    "unfold": (dict(B=2, C=6, H=128, D=32, dil=2, down=0.5, seed=14), dict(sim_type='cosine', detach_unfold=False)),
    "unfold33": (dict(B=2, C=33, H=48, D=16, dil=2, down=None, seed=15), dict(sim_type='gaussian', sigma=2.5,
                                                                             detach_unfold=False)),
    "margin": (dict(B=2, C=6, H=128, D=32, dil=2, down=0.5, seed=16), dict(sim_type='cosine', detach_unfold=True,
                                                                          src_loss_type='margin', margin=[0.6, 0.2])),
    "margin2": (dict(B=2, C=33, H=48, D=16, dil=2, down=None, seed=17), dict(sim_type='cosine', detach_unfold=True,
                                                                            src_loss_type='margin2',
                                                                            margin=[0.8, 0.1])),
    "topk_none": (dict(B=2, C=6, H=128, D=32, dil=2, down=0.5, seed=18), dict(sim_type='cosine', detach_unfold=True,
                                                                             top_k=None)),
}


def loss_option_keys(opts):
    if opts.get("src_loss_type", "mean_std") != "mean_std":
        return ("loss_src_pos", "loss_src_neg", "loss_sim_pos", "loss_sim_neg")
    return LOSS_KEYS


def loss_option_inputs(c):
    g = torch.Generator().manual_seed(c["seed"])
    B, C, H = c["B"], c["C"], c["H"]
    gt = blocky_labels(B, H, H, C, g, min_rect=4, max_rect=max(8, H // 2))
    logits = 2.0 * torch.randn((B, C, H // 4, H // 4), generator=g)
    x_src = torch.relu(torch.randn((B, c["D"], H // 8, H // 8), generator=g))
    x_ema = torch.relu(torch.randn((B, c["D"], H // 8, H // 8), generator=g))
    gh = int((H // 4) * c["down"]) if c["down"] is not None else H // 4
    logits_ema = 2.0 * torch.randn((B, C, gh, gh), generator=g)      # already on the loss grid (pfgst_loss.py:175)
    return gt, logits, x_src, x_ema, logits_ema


def gen_pfgst_loss_options():
    """PFGSTLoss options outside the shipped configuration (sim_type='gaussian', cross_prob_type='ema',
    detach_unfold=False), written by the reference module."""
    L = R.pfgst_loss()
    D = R.dacs_transforms()
    out = {}
    for name, (c, opts) in LOSS_OPTION_CASES.items():
        gt, logits, x_src, x_ema, logits_ema = loss_option_inputs(c)
        np.random.seed(3)
        mix = torch.cat(D.get_class_masks(gt), 0)
        kw = dict(top_k=3)
        kw.update(opts)
        mod = L.PFGSTLoss(dilation=c["dil"], kernel_size=3, weights=W6, feat_level=None,
                          downscale=c["down"], **kw)
        lt = logits.clone().requires_grad_(True)
        xs = x_src.clone().requires_grad_(True)
        with R.cpu_cuda_identity():
            res = mod(dict(logits_trg=lt, logits_ema=logits_ema, gt_src=gt, x_ema=x_ema, x_src=xs, img_trg=None,
                           mix_masks=mix))
        keys = loss_option_keys(opts)
        sum(res[k] for k in keys).backward()
        out.update({f"{name}_mix": mix.numpy().astype(np.uint8),
                    f"{name}_losses": np.array([float(res[k]) for k in keys], dtype=np.float32),
                    f"{name}_grad_x_src": xs.grad.numpy(), f"{name}_grad_logits": lt.grad.numpy(),
                    f"{name}_density": res['vis|density_sim_feat'][1].numpy(),
                    f"{name}_eroded": res['vis|density_sim_feat'][2].numpy()})
    np.savez_compressed(OUT / "pfgst_loss_options.npz", **out)


def slide_cases():
    """(name, B, C, H, W, mode, crop, stride, flip, flip_direction, ori_shape, seed)"""
    return [("slide", 2, 6, 24, 40, "slide", (16, 16), (8, 12), False, None, (24, 40), 0),
            ("slide_flip", 2, 6, 24, 40, "slide", (16, 24), (8, 8), True, ["horizontal", "vertical"], (24, 40), 1),
            ("slide_rescale", 1, 3, 20, 28, "slide", (12, 12), (8, 8), True, "horizontal", (31, 45), 2),
            ("big_crop", 1, 33, 10, 14, "slide", (16, 12), (8, 8), False, None, (10, 14), 3),
            ("whole_flip", 2, 6, 18, 22, "whole", None, None, True, "vertical", (27, 33), 4)]


def synthetic_encode_decode(num_classes):
    """A stand-in network pass whose output depends on the crop's content AND on the position inside the
    crop (so overlapping windows disagree), built from single IEEE operations: bit-identical on CPU and GPU."""
    def encode_decode(img, img_meta):
        B, _, h, w = img.shape
        ii = torch.arange(h, device=img.device, dtype=torch.float32).view(1, 1, h, 1)
        jj = torch.arange(w, device=img.device, dtype=torch.float32).view(1, 1, 1, w)
        chans = [img[:, c % 3:c % 3 + 1] * (0.5 + 0.25 * c) + torch.remainder(ii * 3 + jj * 5 + c, 7) * 0.125
                 for c in range(num_classes)]
        return torch.cat(chans, 1), {}
    return encode_decode


def slide_meta(flip, direction, ori_shape, B):
    return [dict(ori_shape=tuple(ori_shape) + (3,), flip=flip, flip_direction=direction) for _ in range(B)]


def gen_slide_inference():
    """EncoderDecoder.slide_inference / inference / simple_test compiled from the reference source."""
    out = {}
    for name, B, C, H, W, mode, crop, stride, flip, direction, ori, seed in slide_cases():
        g = torch.Generator().manual_seed(900 + seed)
        img = torch.randn((B, 3, H, W), generator=g)
        cfg = types.SimpleNamespace(mode=mode, crop_size=crop, stride=stride)
        seg = R.reference_segmentor(synthetic_encode_decode(C), cfg, C)
        meta = slide_meta(flip, direction, ori, B)
        output, _ = seg.inference(img, meta, True)
        seg_pred, _ = seg.simple_test(img, meta, True)
        out[f"{name}_output"] = output.numpy()
        out[f"{name}_pred"] = np.stack(seg_pred).astype(np.uint8)
        if mode == "slide":
            out[f"{name}_slide"] = seg.slide_inference(img, meta, False).numpy()
    np.savez_compressed(OUT / "slide_inference.npz", **out)


def aug_cases():
    """(name, B, C, ori_shape, mode, crop, stride, [(H, W, flip, direction), ...], seed)"""
    return [("whole3", 2, 6, (24, 40), "whole", None, None,
             [(24, 40, False, None), (18, 30, True, "horizontal"), (30, 50, True, "vertical")], 0),
            ("slide2", 1, 33, (20, 28), "slide", (12, 12), (8, 8),
             [(20, 28, False, None), (26, 36, True, ["horizontal", "vertical"])], 1)]


def aug_inputs(case):
    name, B, C, ori, mode, crop, stride, augs, seed = case
    g = torch.Generator().manual_seed(950 + seed)
    imgs = [torch.randn((B, 3, H, W), generator=g) for (H, W, _, _) in augs]
    metas = [slide_meta(flip, direction, ori, B) for (_, _, flip, direction) in augs]
    return imgs, metas


def gen_aug_test():
    """EncoderDecoder.aug_test compiled from the reference source (encoder_decoder.py:355-373)."""
    out = {}
    for case in aug_cases():
        name, B, C, ori, mode, crop, stride, augs, seed = case
        imgs, metas = aug_inputs(case)
        seg = R.reference_segmentor(synthetic_encode_decode(C), types.SimpleNamespace(mode=mode, crop_size=crop,
                                                                                       stride=stride), C)
        pred, _ = seg.aug_test(imgs, metas, True)
        out[f"{name}_pred"] = np.stack(pred).astype(np.uint8)
        acc = None                                   # the averaged soft-max, for the near-tie mask of the tests
        for im, me in zip(imgs, metas):
            o, _ = seg.inference(im, me, True)
            acc = o if acc is None else acc + o
        out[f"{name}_avg"] = (acc / len(imgs)).numpy()
    np.savez_compressed(OUT / "aug_test.npz", **out)


STEP_CFG = dict(max_iters=100, alpha=0.999, pseudo_threshold=0.6, pseudo_weight_ignore_top=2,
                pseudo_weight_ignore_bottom=3, imnet_feature_dist_lambda=0, imnet_feature_dist_classes=None,
                imnet_feature_dist_scale_min_ratio=None, mix='class', blur=False, color_jitter_strength=0.2,
                color_jitter_probability=1.0, print_grad_magnitude=False, trg_loss_weight=1.,
                use_decoded_feats=True, thre_type='all',
                aux_losses=[dict(type='PFGSTLoss', kernel_size=3, dilation=2, top_k=3, weights=W6,
                                 sim_type='cosine', feat_level=None, detach_unfold=True, downscale=0.5)])


def step_batches(n_iters=3, B=2, H=128, C=6):
    g = torch.Generator().manual_seed(0)
    metas = [{'img_norm_cfg': {'mean': [1., 2., 3.], 'std': [1., 1., 1.]}}] * B
    for _ in range(n_iters):
        yield dict(img=torch.randn((B, 3, H, H), generator=g), img_metas=metas,
                   gt_semantic_seg=blocky_labels(B, H, H, C, g, min_rect=4, max_rect=64),
                   target_img=torch.randn((B, 3, H, H), generator=g), target_img_metas=metas,
                   target_img_strong_aug=torch.randn((B, 3, H, H), generator=g))


def gen_pfgst_step():
    M = R.pfgst()
    C = 6
    cfg = dict(STEP_CFG)
    cfg['model'] = {'_instance_factory': lambda: TinySegmentor(C, 16, seed=0), 'train_cfg': {}, 'test_cfg': {},
                    'decode_head': {'num_classes': C}}
    m = M.PFGST(**cfg)
    opt = torch.optim.SGD(m.model.parameters(), lr=0.01)
    random.seed(1); np.random.seed(1); torch.manual_seed(1)
    out = {}
    with R.cpu_cuda_identity():
        for it, batch in enumerate(step_batches()):
            res = m.train_step(batch, opt)
            out[f"log_keys_{it}"] = np.array(list(res['log_vars'].keys()))
            out[f"log_vals_{it}"] = np.array(list(res['log_vars'].values()), dtype=np.float64)
    out["ema_params"] = torch.cat([p.detach().reshape(-1) for p in m.ema_model.parameters()]).numpy()
    out["student_params"] = torch.cat([p.detach().reshape(-1) for p in m.model.parameters()]).numpy()
    np.savez_compressed(OUT / "pfgst_step.npz", **out)


def ce_cases():
    """(name, B, C, lh, lw, scale, use_weight, use_class_weight, loss_weight)"""
    return [("plain", 2, 6, 32, 32, 4, False, False, 1.0), ("weighted", 2, 6, 32, 32, 4, True, False, 1.0),
            ("aux", 1, 6, 16, 24, 4, True, True, 0.4), ("many", 2, 33, 15, 15, 2, True, False, 1.0),
            ("same_res", 1, 3, 20, 12, 1, False, True, 1.0), ("x8", 1, 2, 13, 9, 8, True, False, 1.0)]


def ce_inputs(name, B, C, lh, lw, scale, use_w, use_cw, seed=0):
    g = torch.Generator().manual_seed(seed + sum(map(ord, name)))
    H, W = lh * scale, lw * scale
    logits = 2.0 * torch.randn((B, C, lh, lw), generator=g)
    label = blocky_labels(B, H, W, C, g, min_rect=2, max_rect=max(4, min(H, W) // 2))
    weight = torch.rand((B, H, W), generator=g) if use_w else None
    cw = (0.5 + torch.rand(C, generator=g)) if use_cw else None
    return logits, label, weight, cw


def gen_weighted_ce():
    resize, cross_entropy, accuracy = R.decode_head_loss_fns()
    out = {}
    for name, B, C, lh, lw, scale, use_w, use_cw, lwt in ce_cases():
        logits, label, weight, cw = ce_inputs(name, B, C, lh, lw, scale, use_w, use_cw)
        z = logits.clone().requires_grad_(True)
        up = resize(input=z, size=label.shape[2:], mode='bilinear', align_corners=False)       # decode_head.py:253-257
        lab = label.squeeze(1)
        loss = lwt * cross_entropy(up, lab, weight=weight, class_weight=cw, reduction='mean', avg_factor=None,
                                   ignore_index=255)                                          # CrossEntropyLoss.forward
        acc = accuracy(up, lab, ignore_index=255)
        loss.backward()
        out[f"{name}_loss"] = loss.detach().numpy()
        out[f"{name}_acc"] = acc.detach().numpy()
        out[f"{name}_grad"] = z.grad.numpy()
    np.savez_compressed(OUT / "weighted_ce.npz", **out)
    print("weighted_ce.npz", {k: float(v) for k, v in out.items() if k.endswith("_loss")})


def eval_logits_cases():
    """(name, N, C, H, W, label_map, reduce_zero_label)"""
    return [("isprs", 3, 6, 64, 64, {}, False), ("inria", 2, 2, 48, 80, {}, False),
            ("seasonnet", 2, 33, 30, 30, {}, False), ("remap", 2, 6, 40, 40, {7: 0, 6: 255}, True)]


def eval_logits_inputs(name, N, C, H, W):
    from pfst_b200.synthetic import blocky_labels, teacher_logits
    g = torch.Generator().manual_seed(sum(map(ord, name)))
    logits = teacher_logits(N, C, H, W, g)
    gt = blocky_labels(N, H, W, C + (2 if name == "remap" else 0), g)[:, 0].to(torch.uint8)
    return logits, gt


def gen_eval_logits():
    """The reference's own EncoderDecoder.inference + simple_test (compiled from its source) on
    synthetic logits, then its intersect_and_union per image (dataset.pre_eval, custom.py:644-682)."""
    M = R.metrics()
    out = {}
    for name, N, C, H, W, lm, rz in eval_logits_cases():
        logits, gt = eval_logits_inputs(name, N, C, H, W)
        preds = R.simple_test_on_logits(logits)
        per = [M.intersect_and_union(p, g, C, 255, label_map=dict(lm), reduce_zero_label=rz)
               for p, g in zip(preds, gt.numpy())]
        out[name + "_pred"] = np.stack(preds).astype(np.uint8)
        out[name + "_areas"] = np.stack([np.stack([a.numpy() for a in t]) for t in per])
    np.savez_compressed(OUT / "eval_logits.npz", **out)


def strong_aug_cases():
    """(seed, H, W): image = RandomState(seed).randint(0, 256, (H, W, 3)), draws from np.random.seed(seed + 1000)"""
    return [(s, *[(40, 52), (33, 47), (24, 96), (17, 120), (8, 31), (64, 64)][s % 6]) for s in range(24)]


def strong_aug_image(seed, H, W):
    return np.random.RandomState(seed).randint(0, 256, (H, W, 3)).astype(np.uint8)


def gen_strong_aug():
    """The reference's StrongAugmentation class (compiled from its source, cv2 standing in for
    mmcv.bgr2hsv/hsv2bgr exactly as mmcv defines them) on seeded random uint8 images."""
    aug = R.strong_augmentation_cls()()
    out = {}
    for seed, H, W in strong_aug_cases():
        np.random.seed(seed + 1000)
        res = aug(dict(img=strong_aug_image(seed, H, W), img_fields=['img']))
        out[f"out_{seed}"] = res['img_strong_aug']
        out[f"next_{seed}"] = np.array(np.random.random())        # stream position after the draws
    np.savez_compressed(OUT / "strong_aug.npz", **out)


def offline_label_cases():
    """(name, n_images, C_feat, H, W, dilations, mean_sims, sample_ratio, seed)"""
    return [("a", 3, 16, 16, 16, [1, 2], [0.5, 0.8], 0.5, 0), ("b", 2, 24, 12, 20, [2], [0.6], 1.0, 1)]


def offline_label_feats(n, C, H, W, seed):
    g = torch.Generator().manual_seed(900 + seed)
    return [[torch.relu(torch.randn((C, H, W), generator=g)), torch.relu(torch.randn((C // 2, H // 2, W // 2), generator=g))]
            for _ in range(n)]


def loader_rule_cases():
    """(name, C, H, W, reduce_zero_label, seed)"""
    return [("plain", 6, 24, 20, False, 0), ("rz", 6, 24, 20, True, 1), ("many", 33, 15, 15, False, 2)]


def loader_rule_inputs(C, H, W, seed):
    from pfst_b200.synthetic import teacher_logits
    g = torch.Generator().manual_seed(700 + seed)
    logits = (0.5 * teacher_logits(1, C, H, W, g)[0]).numpy()
    logits[:, 0, 0] = 1.25                       # exact tie: first index
    thres = (0.2 + 1.2 * torch.rand(C, generator=g)).numpy().astype(np.float32)
    thres[C - 1] = 0.0                           # a class the hook never saw
    return logits, thres


def gen_offline_labels():
    """_cal_loc_dis / _cal_sigmas of PseudoLabelingHookV4 and the label rule of
    LoadAnnotationsPseudoLabelsV2.__call__, compiled from the reference sources."""
    import types
    loc, sig = R.hook_sigma_fns()
    out = {}
    for name, n, C, H, W, dils, means, ratio, seed in offline_label_cases():
        me = types.SimpleNamespace(sim_feat_cfg=dict(kernel_size=3, sigmas=None, dilation=dils, mean_sim=means,
                                                     feat_level=[0, 1]))
        with R.cpu_cuda_identity():
            lds = [loc(me, f) for f in offline_label_feats(n, C, H, W, seed)]
        for i, ld in enumerate(lds):
            for k, v in ld.items():
                out[f"{name}_locdis_{i}_{k}"] = v.numpy()
        np.random.seed(40 + seed)
        for k, v in sig(me, lds, ratio).items():
            out[f"{name}_sigma_{k}"] = np.float64(v)
    cls, reg = R.loader_pseudo_labels_cls()
    for name, C, H, W, rz, seed in loader_rule_cases():
        logits, thres = loader_rule_inputs(C, H, W, seed)
        reg['/golden/x.h5'] = {'seg_logits': logits, 'thre@0.5': thres}
        res = cls(pseudo_labels_dir='/golden', pseudo_ratio=0.5, reduce_zero_label=rz)(
            dict(img_info=dict(filename='d/x.png'), seg_fields=[], img_shape=(H, W)))
        out[f"loader_{name}"] = res['gt_semantic_seg']
    np.savez_compressed(OUT / "offline_labels.npz", **out)


def strong_aug_digest(img):
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(img).tobytes()).hexdigest()


def live_eval_logits_inputs(seed, N, C, H, W):
    g = torch.Generator().manual_seed(seed)
    logits = teacher_logits(N, C, H, W, g)
    logits[0, :, 0, 0] = 1.5            # exact tie -> first index
    logits[0, 0, 0, 1] = float("nan")   # NaN -> softmax all NaN -> index 0
    gt = torch.randint(0, C + 1, (N, H, W), generator=g).to(torch.uint8)
    gt[:, :2] = 255
    return logits, gt


LIVE_EVAL_CASES = [(2, 6, 32, 32), (1, 19, 17, 23), (2, 2, 8, 12)]
LIVE_THRESHOLD_CASES = [(2, 6, 32, 32, 0.5), (1, 33, 24, 24, 1.0), (2, 3, 17, 9, 0.3)]
LIVE_FEAT_DIST_SHAPES = [(2, 16, 8, 8), (1, 512, 5, 7), (3, 4, 15, 15)]


def gen_reference_live():
    """What the live comparisons of test_oracle_pins.py / test_host_logic.py check the oracle
    against, on their own inputs (see the module doc-string for where the values come from)."""
    from oracle import class_thresholds as OT, metrics as om, mixing as omix, offline_labels as OLB
    from oracle import pfgst_loss as OL, prototypes as OP, strong_aug as SA
    from pfst_b200.synthetic import WORKLOADS, step_inputs
    out = {}
    # test_class_draw_reproduces_reference_get_class_masks
    g = torch.Generator().manual_seed(0)
    labels = torch.randint(0, 6, (3, 1, 16, 16), generator=g)
    labels[0, 0, :2] = 255
    np.random.seed(42)
    out["class_draw_masks"] = torch.cat(omix.class_masks(labels)).numpy().astype(np.uint8)
    # test_reference_golden_test_retargeted
    o59 = om.eval_metrics(np.array([np.repeat(31, 59)]), np.array([np.arange(59)]), 59, 255, metrics='mIoU')
    out["retargeted_IoU59"] = np.asarray(o59["IoU"])
    # test_oracle_bitwise_equals_reference_live
    inp = step_inputs(WORKLOADS["tiny"], seed=99)
    np.random.seed(11)
    masks = omix.class_masks(inp["gt"])
    out["tiny_mix"] = torch.cat(masks).numpy().astype(np.uint8)
    t = dict(logits_trg=inp['logits_trg'].clone().requires_grad_(True), logits_ema=None, gt_src=inp['gt'],
             x_ema=inp['x_ema'], x_src=inp['x_src'].clone().requires_grad_(True), img_trg=None,
             mix_masks=torch.cat(masks, 0))
    res = OL.pfgst_loss(t, OL.LossCfg())
    sum(res[k] for k in OL.LOSS_KEYS).backward()
    out["tiny_losses"] = np.array([float(res[k].detach()) for k in OL.LOSS_KEYS], dtype=np.float32)
    out["tiny_grad_x_src"] = t['x_src'].grad.numpy()
    out["tiny_grad_logits"] = t['logits_trg'].grad.numpy()
    # test_class_threshold_oracle_equals_reference_live
    for seed, (B, C, H, W, ratio) in enumerate(LIVE_THRESHOLD_CASES):
        logits = teacher_logits(B, C, H, W, torch.Generator().manual_seed(seed))
        thr = OT.cal_threshold(logits, ratio, [0.1, 0.5, 0.9], np.random.RandomState(seed))
        for k, v in thr.items():
            out[f"threshold_{seed}_{k}"] = np.asarray(v, dtype=np.float64)
    # test_masked_feat_dist_equals_reference_live
    g = torch.Generator().manual_seed(21)
    for i, (B, D, h, w) in enumerate(LIVE_FEAT_DIST_SHAPES):
        f1 = torch.randn((B, D, h, w), generator=g).requires_grad_(True)
        f2 = torch.randn((B, D, h, w), generator=g)
        mask = torch.rand((B, 1, h, w), generator=g) > 0.4
        for j, m in enumerate((None, mask)):
            d = OP.masked_feat_dist(f1, f2, m)
            d.backward()
            out[f"feat_dist_{i}_{j}"], out[f"feat_dist_{i}_{j}_grad"] = d.detach().numpy(), f1.grad.numpy().copy()
            f1.grad = None
    # test_offline_labels_oracle_equals_reference_live
    g = torch.Generator().manual_seed(11)
    feats = [[torch.relu(torch.randn((10, 9, 14), generator=g))] for _ in range(2)]
    lds = [OLB.cal_loc_dis(f, 3, [1, 3]) for f in feats]
    for i, ld in enumerate(lds):
        for k, v in ld.items():
            out[f"offline_locdis_{i}_{k}"] = v.numpy()
    for k, v in OLB.cal_sigmas(lds, [0], [1, 3], 0.7, 0.8, np.random.RandomState(5)).items():
        out[f"offline_sigma_{k}"] = np.float64(v)
    logits = (2 * torch.randn((5, 9, 7), generator=g)).numpy()
    logits[1, 2, 3] = np.nan
    thres = np.array([0.5, 1.0, 0.2, 0.0, 0.9], dtype=np.float32)
    for rz in (False, True):
        out[f"offline_loader_{int(rz)}"] = OLB.loader_pseudo_labels(logits, thres, rz)
    # test_eval_logits_oracle_equals_reference_live
    for seed, (N, C, H, W) in enumerate(LIVE_EVAL_CASES):
        logits, gt = live_eval_logits_inputs(seed, N, C, H, W)
        out[f"eval_{seed}_pred"] = om.seg_argmax(logits).numpy().astype(np.uint8)
        out[f"eval_{seed}_areas"] = np.stack([np.stack([a.numpy() for a in t])
                                              for t in om.pre_eval(logits, list(gt.numpy()), C, 255)])
    # test_strong_aug_oracle_equals_reference_class_live: digests keep the 60 images small
    rs = np.random.RandomState(5)
    digests, after = [], []
    for it in range(60):
        H, W = [(64, 64), (33, 47), (120, 120), (16, 100)][it % 4]
        img = rs.randint(0, 256, (H, W, 3)).astype(np.uint8)
        np.random.seed(it)
        ops_ = SA.draw_strong_aug(np.random, 20, (0.7, 1.3), (0.4, 1.6), 10)
        after.append(np.random.random())
        digests.append(strong_aug_digest(SA.apply_strong_aug(img.copy(), ops_)))
    out["strong_aug_sha256"], out["strong_aug_after"] = np.array(digests), np.array(after)
    # test_slide_inference_oracle_equals_reference_live (inputs: the fixture's plus 0.25)
    for case in slide_cases():
        name, B, C, H, W, mode, crop, stride, flip, direction, ori, seed = case
        img = torch.randn((B, 3, H, W), generator=torch.Generator().manual_seed(900 + seed)) + 0.25
        o, _ = om.inference(synthetic_encode_decode(C), img, slide_meta(flip, direction, ori, B), True, mode, crop,
                            stride, C)
        out[f"slide_{name}"] = o.numpy()
    # test_aug_test_oracle_vs_golden_and_reference (inputs: the fixture's, scaled and shifted)
    for case in aug_cases():
        name, B, C, ori, mode, crop, stride, augs, seed = case
        imgs, metas = aug_inputs(case)
        pred, _ = om.aug_test(synthetic_encode_decode(C), [im * 0.5 + 0.1 for im in imgs], metas, True, mode, crop,
                              stride, C)
        out[f"aug_{name}_pred"] = np.stack(pred).astype(np.uint8)
    np.savez_compressed(OUT / "reference_live.npz", **out)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "reference_live":
        warnings.filterwarnings("ignore")
        torch.set_num_threads(1)
        gen_reference_live()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "offline_labels":
        gen_offline_labels()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "strong_aug":
        gen_strong_aug()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "weighted_ce":
        gen_weighted_ce()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "eval_logits":
        gen_eval_logits()
        sys.exit(0)
    warnings.filterwarnings("ignore")
    assert R.available(), "reference checkout not found"
    torch.set_num_threads(1)      # bit-stable reductions
    for fn in (gen_metrics, gen_ema, gen_pseudo_mix, gen_pfgst_loss, gen_pfgst_loss_options, gen_slide_inference, gen_aug_test, gen_pfgst_step, gen_weighted_ce, gen_eval_logits, gen_strong_aug,
               gen_offline_labels):
        fn()
        print("wrote", fn.__name__)
    for p in sorted(OUT.glob("*.npz")):
        print(p.name, p.stat().st_size)
