"""Pins the CPU oracle: (1) against the committed golden fixtures, which were produced by
the REFERENCE code itself (tests/golden/make_golden.py); (2) in the "live reference" tests,
against what the reference computes on their inputs: the committed reference_live.npz and,
when PFST_REFERENCE names a reference checkout, the reference modules loaded by path, live.
Runs without a GPU."""
import random
import warnings
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import ema as oema, metrics as om, mixing as omix, pfgst_loss as OL, pseudo as opl
from tests.golden import ref_loader as R

G = Path(__file__).resolve().parent / "golden"


def load(name):
    return np.load(G / name, allow_pickle=False)


def live():
    return load("reference_live.npz")


def assert_close_to_stored(got, want, rtol):
    """Float results of CPU reductions and resampling: their summation order depends on the host's threads
    and vector width, so the stored vectors are met to `rtol` of the array's largest magnitude (the live
    comparison stays bit-exact)."""
    got = got.detach().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
    assert got.shape == want.shape
    err = np.abs(got.astype(np.float64) - want)
    assert np.array_equal(np.isnan(got), np.isnan(want)) and np.nanmax(err, initial=0) <= rtol * np.nanmax(
        np.abs(want), initial=0) + 1e-12, np.nanmax(err)


# ------------------------------------------------------------------ golden fixtures
def test_metrics_oracle_vs_golden():
    z = load("metrics.npz")
    C = int(z["C"])
    ret = om.eval_metrics(z["pred"], z["label"], C, 255, metrics=["mIoU", "mDice", "mFscore"])
    for k, v in ret.items():
        assert np.array_equal(np.asarray(v), z["all_" + k], equal_nan=True), k
    per = [om.areas(z["pred"][i], z["label"][i], C, 255) for i in range(10)]
    assert np.array_equal(np.stack([np.stack([a.numpy() for a in p]) for p in per]), z["per_image"])
    assert np.array_equal(om.metrics_from_areas(*om.pre_eval_sum(per), ["mIoU"])["IoU"], z["pre_eval_IoU"])
    a = om.areas(z["lm_pred"], z["lm_label"], 6, 255, {7: 0, 6: 255}, True)
    assert np.array_equal(np.stack([t.numpy() for t in a]), z["lm_areas"])
    # and the reference's own golden relation: histc areas == bincount confusion matrix
    tot = sum(om.confusion(z["pred"][i], z["label"][i], C, 255) for i in range(10)).astype(np.float64)
    d = np.diag(tot)
    assert np.allclose(z["all_IoU"], d / (tot.sum(1) + tot.sum(0) - d))
    assert z["all_aAcc"] == d.sum() / tot.sum()


def test_ema_oracle_vs_golden():
    z = load("ema.npz")
    n = 6
    student = [torch.from_numpy(z[f"student_{i}"].copy()) for i in range(n)]
    teacher = [torch.from_numpy(z[f"teacher0_{i}"].copy()) for i in range(n)]
    for it in z["iters"]:
        oema.ema_update(teacher, student, int(it), 0.999)
        for i in range(n):
            assert np.array_equal(teacher[i].numpy(), z[f"teacher_it{it}_{i}"]), (it, i)
    oema.ema_init(teacher, student)
    for i in range(n):
        assert np.array_equal(teacher[i].numpy(), z[f"teacher_init_{i}"])


def test_pseudo_and_mix_oracle_vs_golden():
    z = load("pseudo_mix.npz")
    logits = torch.from_numpy(z["logits"])
    gt = torch.from_numpy(z["gt"]).long()
    img, trg = torch.from_numpy(z["img"]), torch.from_numpy(z["trg"])
    label, prob, large = opl.pseudo_label(logits, float(z["thr"]))
    assert np.array_equal(label.numpy(), z["pseudo_label"])
    assert np.array_equal(prob.numpy(), z["pseudo_prob"])
    assert np.array_equal(large.numpy(), z["large"])
    w = opl.pseudo_weight(large, "all", int(z["top"]), int(z["bottom"]))
    np.random.seed(int(z["seed"]))
    masks = omix.class_masks(gt)
    mi, ml, mw, mm = omix.mix_batch(img, trg, gt, label, w, masks)
    assert np.array_equal(mm.numpy(), z["mix_masks"])
    assert np.array_equal(ml.numpy(), z["mixed_lbl"])
    assert np.array_equal(mi.numpy(), z["mixed_img"])
    assert np.array_equal(mw.numpy(), z["mixed_weight"])


@pytest.mark.parametrize("name", ["a", "b"])
def test_pfgst_loss_oracle_vs_golden(name):
    z = load("pfgst_loss.npz")
    dil, down = z[f"{name}_cfg"]
    lt = torch.from_numpy(z[f"{name}_logits"]).requires_grad_(True)
    xs = torch.from_numpy(z[f"{name}_x_src"]).requires_grad_(True)
    res = OL.pfgst_loss(dict(logits_trg=lt, gt_src=torch.from_numpy(z[f"{name}_gt"]).long(),
                             x_ema=torch.from_numpy(z[f"{name}_x_ema"]), x_src=xs, img_trg=None,
                             mix_masks=torch.from_numpy(z[f"{name}_mix"]).long()),
                        OL.LossCfg(dilation=int(dil), downscale=None if down < 0 else float(down)))
    sum(res[k] for k in OL.LOSS_KEYS).backward()
    got = np.array([float(res[k].detach()) for k in OL.LOSS_KEYS], dtype=np.float32)
    assert np.allclose(got, z[f"{name}_losses"], rtol=2e-6, atol=1e-8)   # thread-count dependent sums
    assert np.allclose(xs.grad.numpy(), z[f"{name}_grad_x_src"], rtol=1e-5, atol=1e-9)
    assert np.allclose(lt.grad.numpy(), z[f"{name}_grad_logits"], rtol=1e-5, atol=1e-9)
    assert np.array_equal(res['vis|density_sim_feat'][2].numpy(), z[f"{name}_eroded"])
    assert np.allclose(res['vis|density_sim_feat'][1].numpy(), z[f"{name}_density"], rtol=0, atol=1e-6)


def _option_cfg(c, opts):
    return OL.LossCfg(dilation=c["dil"], downscale=c["down"], sim_type=opts.get("sim_type", "cosine"),
                      sigma=opts.get("sigma", 30.0), cross_prob_type=opts.get("cross_prob_type", "trg"),
                      detach_unfold=opts.get("detach_unfold", True), top_k=opts.get("top_k", 3),
                      src_loss_type=opts.get("src_loss_type", "mean_std"), margin=tuple(opts.get("margin", (0.5, 0.5))))


@pytest.mark.parametrize("name", ["gauss", "gauss33", "ema", "unfold", "unfold33", "margin", "margin2", "topk_none"])
def test_pfgst_loss_option_oracle_vs_golden(name):
    """sim_type='gaussian', cross_prob_type='ema', detach_unfold=False: the oracle against what the
    reference module wrote (tests/golden/make_golden.py::gen_pfgst_loss_options)."""
    from tests.golden.make_golden import LOSS_OPTION_CASES, loss_option_inputs, loss_option_keys
    z = load("pfgst_loss_options.npz")
    c, opts = LOSS_OPTION_CASES[name]
    keys = loss_option_keys(opts)
    gt, logits, x_src, x_ema, logits_ema = loss_option_inputs(c)
    lt, xs = logits.clone().requires_grad_(True), x_src.clone().requires_grad_(True)
    res = OL.pfgst_loss(dict(logits_trg=lt, logits_ema=logits_ema, gt_src=gt, x_ema=x_ema, x_src=xs, img_trg=None,
                             mix_masks=torch.from_numpy(z[f"{name}_mix"]).long()), _option_cfg(c, opts))
    sum(res[k] for k in keys).backward()
    got = np.array([float(res[k].detach()) for k in keys], dtype=np.float32)
    assert np.allclose(got, z[f"{name}_losses"], rtol=2e-6, atol=1e-8)
    assert np.allclose(xs.grad.numpy(), z[f"{name}_grad_x_src"], rtol=1e-5, atol=1e-9)
    assert np.allclose(lt.grad.numpy(), z[f"{name}_grad_logits"], rtol=1e-5, atol=1e-9)
    assert np.array_equal(res['vis|density_sim_feat'][2].numpy(), z[f"{name}_eroded"])
    assert np.allclose(res['vis|density_sim_feat'][1].numpy(), z[f"{name}_density"], rtol=0, atol=1e-6)


# ------------------------------------------------------------------ live reference
# Each test below checks the oracle against what the reference computes on the test's inputs: the
# vectors the reference wrote (or reference_live.npz, see tests/golden/make_golden.py) everywhere, and
# bit for bit against the reference modules themselves when PFST_REFERENCE names a checkout.
@pytest.mark.parametrize("name", ["gauss", "ema", "unfold33", "margin2", "topk_none"])
def test_pfgst_loss_option_oracle_equals_reference_live(name):
    from tests.golden.make_golden import LOSS_OPTION_CASES, loss_option_inputs, loss_option_keys, W6
    warnings.filterwarnings("ignore")
    c, opts = LOSS_OPTION_CASES[name]
    gt, logits, x_src, x_ema, logits_ema = loss_option_inputs(c)
    np.random.seed(3)
    mix = torch.cat(omix.class_masks(gt), 0)
    keys = loss_option_keys(opts)

    def t():
        return dict(logits_trg=logits.clone().requires_grad_(True), logits_ema=logits_ema, gt_src=gt, x_ema=x_ema,
                    x_src=x_src.clone().requires_grad_(True), img_trg=None, mix_masks=mix)

    t2 = t()
    b = OL.pfgst_loss(t2, _option_cfg(c, opts))
    sum(b[k] for k in keys).backward()
    z = load("pfgst_loss_options.npz")                  # the reference module on the same inputs and masks
    assert np.array_equal(mix.numpy(), z[f"{name}_mix"])
    assert_close_to_stored(torch.stack([b[k].reshape(()) for k in keys]), z[f"{name}_losses"], 2e-6)
    assert_close_to_stored(t2['x_src'].grad, z[f"{name}_grad_x_src"], 1e-5)
    assert_close_to_stored(t2['logits_trg'].grad, z[f"{name}_grad_logits"], 1e-5)
    if not R.available():
        return
    kw = dict(top_k=3)
    kw.update(opts)
    mod = R.pfgst_loss().PFGSTLoss(dilation=c["dil"], kernel_size=3, weights=W6, feat_level=None,
                                   downscale=c["down"], **kw)
    np.random.seed(3)
    assert torch.equal(torch.cat(R.dacs_transforms().get_class_masks(gt), 0), mix)
    t1 = t()
    with R.cpu_cuda_identity():
        a = mod(t1)
    sum(a[k] for k in keys).backward()
    for k in keys:
        assert torch.equal(a[k].reshape(-1), b[k].reshape(-1)), k
    assert torch.equal(t1['x_src'].grad, t2['x_src'].grad)
    assert torch.equal(t1['logits_trg'].grad, t2['logits_trg'].grad)


def test_reference_golden_test_retargeted():
    """The reference's only golden test (tests/test_metrics.py:86-143): eval_metrics must equal
    the bincount confusion-matrix formulas. Checked for the oracle, and for the reference module
    when it is present."""
    rs = np.random.RandomState(123)
    C = 19
    pred, label = rs.randint(0, C, (10, 30, 30)), rs.randint(0, C, (10, 30, 30))
    label[:, 2, 5:10] = 255
    tot = sum(om.confusion(pred[i], label[i], C, 255) for i in range(10)).astype(np.float64)
    d = np.diag(tot)
    impls = (R.metrics().eval_metrics, om.eval_metrics) if R.available() else (om.eval_metrics,)
    for impl in impls:
        ret = impl(pred, label, C, 255, metrics=["mIoU", "mDice"])
        assert ret["aAcc"] == d.sum() / tot.sum()
        assert np.allclose(ret["Acc"], d / tot.sum(1))
        assert np.allclose(ret["IoU"], d / (tot.sum(1) + tot.sum(0) - d))
        assert np.allclose(ret["Dice"], 2 * d / (tot.sum(1) + tot.sum(0)))
    r59 = {"IoU": live()["retargeted_IoU59"]}
    if R.available():
        r59 = R.metrics().eval_metrics(np.array([np.repeat(31, 59)]), np.array([np.arange(59)]), 59, 255,
                                       metrics='mIoU')
    o59 = om.eval_metrics(np.array([np.repeat(31, 59)]), np.array([np.arange(59)]), 59, 255, metrics='mIoU')
    assert not np.any(np.isnan(r59["IoU"])) and np.array_equal(r59["IoU"], o59["IoU"])


def test_oracle_bitwise_equals_reference_live():
    from pfst_b200.synthetic import WORKLOADS, step_inputs
    warnings.filterwarnings("ignore")
    z = live()
    wl = WORKLOADS["tiny"]
    inp = step_inputs(wl, seed=99)
    np.random.seed(11)
    ora_masks = omix.class_masks(inp["gt"])
    mix = torch.cat(ora_masks, 0)
    assert np.array_equal(mix.numpy(), z["tiny_mix"])

    def t():
        return dict(logits_trg=inp['logits_trg'].clone().requires_grad_(True), logits_ema=None, gt_src=inp['gt'],
                    x_ema=inp['x_ema'], x_src=inp['x_src'].clone().requires_grad_(True), img_trg=None, mix_masks=mix)

    t2 = t()
    b = OL.pfgst_loss(t2, OL.LossCfg())
    sum(b[k] for k in OL.LOSS_KEYS).backward()
    assert_close_to_stored(torch.stack([b[k].reshape(()) for k in OL.LOSS_KEYS]), z["tiny_losses"], 2e-6)
    assert_close_to_stored(t2['x_src'].grad, z["tiny_grad_x_src"], 1e-5)
    assert_close_to_stored(t2['logits_trg'].grad, z["tiny_grad_logits"], 1e-5)
    if not R.available():
        return
    D, L = R.dacs_transforms(), R.pfgst_loss()
    np.random.seed(11)
    ref_masks = D.get_class_masks(inp["gt"])
    assert all(torch.equal(a, b) for a, b in zip(ref_masks, ora_masks))
    W6 = {'src_pos': 0.1, 'src_neg': 0.1, 'sim_pos': 0.1, 'sim_neg': 0.1, 'src_pos_std': 0.1, 'src_neg_std': 0.1}
    mod = L.PFGSTLoss(top_k=3, dilation=2, kernel_size=3, weights=W6, sim_type='cosine', feat_level=None,
                      detach_unfold=True, downscale=0.5)
    t1 = t()
    with R.cpu_cuda_identity():
        a = mod(t1)
    sum(a[k] for k in OL.LOSS_KEYS).backward()
    for k in OL.LOSS_KEYS:
        assert torch.equal(a[k].reshape(-1), b[k].reshape(-1)), k
    assert torch.equal(t1['x_src'].grad, t2['x_src'].grad)
    assert torch.equal(t1['logits_trg'].grad, t2['logits_trg'].grad)


def test_weighted_ce_oracle_vs_reference_live_and_golden():
    """Decode-head loss oracle == the reference's resize + cross_entropy + accuracy (loaded by
    path) bit for bit, and == the committed golden vectors."""
    from oracle import weighted_ce as OC
    from tests.golden.make_golden import ce_cases, ce_inputs
    z = np.load(G / "weighted_ce.npz")
    live = R.decode_head_loss_fns() if R.available() else None
    for name, B, C, lh, lw, scale, use_w, use_cw, lwt in ce_cases():
        logits, label, weight, cw = ce_inputs(name, B, C, lh, lw, scale, use_w, use_cw)
        zo = logits.clone().requires_grad_(True)
        lo, ao, _ = OC.decode_head_losses(zo, label, weight, cw, 255, lwt)
        lo.backward()
        assert np.array_equal(lo.detach().numpy(), z[f"{name}_loss"]), name
        assert np.array_equal(ao.numpy(), z[f"{name}_acc"]), name
        assert np.array_equal(zo.grad.numpy(), z[f"{name}_grad"]), name
        if live is not None:
            resize, cross_entropy, accuracy = live
            up = resize(input=logits, size=label.shape[2:], mode='bilinear', align_corners=False)
            lr = lwt * cross_entropy(up, label.squeeze(1), weight=weight, class_weight=cw, ignore_index=255)
            assert torch.equal(lr, lo.detach()) and torch.equal(accuracy(up, label.squeeze(1), ignore_index=255), ao)


def test_class_threshold_oracle_equals_reference_live():
    """oracle.class_thresholds.cal_threshold == PseudoLabelingHookV4._cal_threshold (compiled from the
    reference source), same numpy stream, bit for bit."""
    import types
    from oracle import class_thresholds as OT
    from pfst_b200.synthetic import teacher_logits
    from tests.golden.make_golden import LIVE_THRESHOLD_CASES
    z = live()
    ref = R.cal_threshold_fn() if R.available() else None
    for seed, (B, C, H, W, ratio) in enumerate(LIVE_THRESHOLD_CASES):
        logits = teacher_logits(B, C, H, W, torch.Generator().manual_seed(seed))
        ratios = [0.1, 0.5, 0.9]
        b = OT.cal_threshold(logits, ratio, ratios, np.random.RandomState(seed))
        assert list(b) == [f"thre@{r}" for r in ratios]
        for k in b:
            assert_close_to_stored(np.asarray(b[k], dtype=np.float64), z[f"threshold_{seed}_{k}"], 2e-6)
        if ref is not None:
            np.random.seed(seed)
            a = ref(types.SimpleNamespace(cls_thre_ratios=ratios), logits, ratio)
            assert list(a) == list(b)
            for k in a:
                assert np.array_equal(np.asarray(a[k], dtype=np.float64), np.asarray(b[k], dtype=np.float64)), k


# ------------------------------------------------------------------ G1: the anchor of the prototype loss
def test_masked_feat_dist_equals_reference_live():
    """oracle.prototypes.masked_feat_dist (what proto_dist_loss is built on) == PFGST.masked_feat_dist of
    the reference class (rsiseg/models/uda/pfgst.py:168-177), values and gradients, with and without a
    mask; the drop-in's own method is the same function."""
    from oracle import prototypes as OP
    from tests.golden.make_golden import LIVE_FEAT_DIST_SHAPES
    z = live()
    ref = R.pfgst().PFGST.masked_feat_dist if R.available() else None
    g = torch.Generator().manual_seed(21)
    for i, (B, D, h, w) in enumerate(LIVE_FEAT_DIST_SHAPES):
        f1 = torch.randn((B, D, h, w), generator=g).requires_grad_(True)
        f1b = f1.detach().clone().requires_grad_(True)
        f2 = torch.randn((B, D, h, w), generator=g)
        mask = torch.rand((B, 1, h, w), generator=g) > 0.4
        for j, m in enumerate((None, mask)):
            b = OP.masked_feat_dist(f1b, f2, m)
            b.backward()
            assert_close_to_stored(b, z[f"feat_dist_{i}_{j}"], 2e-6)
            assert_close_to_stored(f1b.grad, z[f"feat_dist_{i}_{j}_grad"], 1e-5)
            if ref is not None:
                a = ref(None, f1, f2, m)
                assert torch.equal(a, b)
                a.backward()
                assert torch.equal(f1.grad, f1b.grad)
            f1.grad = f1b.grad = None


# ------------------------------------------------------------------ offline labels: sigma search, loader rule
def test_offline_labels_oracle_vs_golden():
    """oracle.offline_labels vs the fixture written by PseudoLabelingHookV4._cal_loc_dis/_cal_sigmas and
    LoadAnnotationsPseudoLabelsV2.__call__ (tests/golden/make_golden.py::gen_offline_labels)."""
    from oracle import offline_labels as OL
    from tests.golden.make_golden import (loader_rule_cases, loader_rule_inputs, offline_label_cases,
                                          offline_label_feats)
    z = load("offline_labels.npz")
    for name, n, C, H, W, dils, means, ratio, seed in offline_label_cases():
        lds = [OL.cal_loc_dis(f, 3, dils) for f in offline_label_feats(n, C, H, W, seed)]
        for i, ld in enumerate(lds):
            for k, v in ld.items():
                assert np.array_equal(v.numpy(), z[f"{name}_locdis_{i}_{k}"]), (name, i, k)
        sig = OL.cal_sigmas(lds, [0, 1], dils, means, ratio, np.random.RandomState(40 + seed))
        assert len(sig) == 2 * len(dils) * len(means)
        for k, v in sig.items():
            assert v == float(z[f"{name}_sigma_{k}"]), (name, k)
    for name, C, H, W, rz, seed in loader_rule_cases():
        logits, thres = loader_rule_inputs(C, H, W, seed)
        assert np.array_equal(OL.loader_pseudo_labels(logits, thres, rz), z[f"loader_{name}"]), name


def test_offline_labels_oracle_equals_reference_live():
    import types
    from oracle import offline_labels as OL
    z = live()
    g = torch.Generator().manual_seed(11)
    me = types.SimpleNamespace(sim_feat_cfg=dict(kernel_size=3, sigmas=None, dilation=[1, 3], mean_sim=0.7, feat_level=[0]))
    feats = [[torch.relu(torch.randn((10, 9, 14), generator=g))] for _ in range(2)]
    b = [OL.cal_loc_dis(f, 3, [1, 3]) for f in feats]
    for i, ld in enumerate(b):
        assert len(ld) == sum(k.startswith(f"offline_locdis_{i}_") for k in z.files)
        assert all(np.array_equal(v.numpy(), z[f"offline_locdis_{i}_{k}"]) for k, v in ld.items())
    sigmas = OL.cal_sigmas(b, [0], [1, 3], 0.7, 0.8, np.random.RandomState(5))
    assert len(sigmas) == sum(k.startswith("offline_sigma_") for k in z.files)
    assert all(v == float(z[f"offline_sigma_{k}"]) for k, v in sigmas.items())
    if R.available():
        loc, sig = R.hook_sigma_fns()
        with R.cpu_cuda_identity():
            a = [loc(me, f) for f in feats]
        assert all(torch.equal(x[k], y[k]) for x, y in zip(a, b) for k in x)
        np.random.seed(5)
        assert sig(me, a, 0.8) == sigmas
    logits = (2 * torch.randn((5, 9, 7), generator=g)).numpy()
    logits[1, 2, 3] = np.nan
    thres = np.array([0.5, 1.0, 0.2, 0.0, 0.9], dtype=np.float32)
    for rz in (False, True):
        got = OL.loader_pseudo_labels(logits, thres, rz)
        assert np.array_equal(got, z[f"offline_loader_{int(rz)}"])
        if R.available():
            cls, reg = R.loader_pseudo_labels_cls()
            reg['/p/q.h5'] = {'seg_logits': logits, 'thre@0.3': thres}
            res = cls(pseudo_labels_dir='/p', pseudo_ratio=0.3, reduce_zero_label=rz)(
                dict(img_info=dict(filename='q.tif'), seg_fields=[], img_shape=(9, 7)))
            assert np.array_equal(res['gt_semantic_seg'], got)


# ------------------------------------------------------------------ on-device evaluation path
def test_eval_logits_oracle_vs_golden():
    """oracle simple_test + pre_eval restatement vs the fixture written by the reference's own
    inference/simple_test/intersect_and_union (tests/golden/make_golden.py::gen_eval_logits)."""
    from tests.golden.make_golden import eval_logits_cases, eval_logits_inputs
    z = load("eval_logits.npz")
    for name, N, C, H, W, lm, rz in eval_logits_cases():
        logits, gt = eval_logits_inputs(name, N, C, H, W)
        assert np.array_equal(om.seg_argmax(logits).numpy(), z[name + "_pred"].astype(np.int64)), name
        per = om.pre_eval(logits, list(gt.numpy()), C, 255, lm, rz)
        assert np.array_equal(np.stack([np.stack([a.numpy() for a in t]) for t in per]), z[name + "_areas"]), name


def test_eval_logits_oracle_equals_reference_live():
    from tests.golden.make_golden import LIVE_EVAL_CASES, live_eval_logits_inputs
    z = live()
    for seed, (N, C, H, W) in enumerate(LIVE_EVAL_CASES):
        logits, gt = live_eval_logits_inputs(seed, N, C, H, W)
        pred = om.seg_argmax(logits).numpy()
        got = om.pre_eval(logits, list(gt.numpy()), C, 255)
        assert np.array_equal(pred, z[f"eval_{seed}_pred"].astype(np.int64)), seed
        assert np.array_equal(np.stack([np.stack([a.numpy() for a in t]) for t in got]), z[f"eval_{seed}_areas"]), seed
        if R.available():
            preds = R.simple_test_on_logits(logits)
            assert np.array_equal(np.stack(preds), pred)
            want = [R.metrics().intersect_and_union(p, l, C, 255, label_map=dict(), reduce_zero_label=False)
                    for p, l in zip(preds, gt.numpy())]
            for a, b in zip(got, want):
                assert all(torch.equal(x, y) for x, y in zip(a, b))


# ------------------------------------------------------------------ StrongAugmentation (data pipeline)
def _cv2():
    return pytest.importorskip("cv2")


def test_hsv_restatements_equal_cv2_on_every_colour():
    """mmcv.bgr2hsv / hsv2bgr are cv2.cvtColor on uint8: the oracle's two restatements must equal
    cv2 for ALL 2^24 BGR triples and ALL 180*256*256 HSV triples, in the vectorised body of a row
    (truncating) and in its scalar tail (rounding)."""
    cv2 = _cv2()
    from oracle import strong_aug as SA
    a = np.arange(1 << 24, dtype=np.uint32)
    img = np.stack([a & 255, (a >> 8) & 255, (a >> 16) & 255], -1).astype(np.uint8).reshape(4096, 4096, 3)
    assert np.array_equal(SA.bgr2hsv_u8(img), cv2.cvtColor(img, cv2.COLOR_BGR2HSV))
    del img, a
    H, S, V = np.meshgrid(np.arange(180), np.arange(256), np.arange(256), indexing="ij")
    allhsv = np.stack([H, S, V], -1).astype(np.uint8).reshape(-1, 3)
    for W in (256, 31):                                   # all-SIMD rows, all-tail rows
        pad = (-allhsv.shape[0]) % W
        hsv = np.concatenate([allhsv, np.zeros((pad, 3), np.uint8)]).reshape(-1, W, 3)
        assert np.array_equal(SA.hsv2bgr_u8(hsv), cv2.cvtColor(hsv, cv2.COLOR_HSV2BGR)), W
    rs = np.random.RandomState(0)
    for W in (120, 100, 33, 7):                           # mixed rows: body + tail
        hsv = np.stack([rs.randint(0, 180, (50, W)), rs.randint(0, 256, (50, W)), rs.randint(0, 256, (50, W))],
                       -1).astype(np.uint8)
        assert np.array_equal(SA.hsv2bgr_u8(hsv), cv2.cvtColor(hsv, cv2.COLOR_HSV2BGR)), W


def test_strong_aug_oracle_vs_golden():
    from oracle import strong_aug as SA
    from tests.golden.make_golden import strong_aug_cases, strong_aug_image
    z = load("strong_aug.npz")
    n_ops = 0
    for seed, H, W in strong_aug_cases():
        rs = np.random.RandomState(seed + 1000)
        ops_ = SA.draw_strong_aug(rs)
        n_ops += len(ops_)
        assert rs.random_sample() == float(z[f"next_{seed}"]), seed       # same stream consumption
        assert np.array_equal(SA.apply_strong_aug(strong_aug_image(seed, H, W), ops_), z[f"out_{seed}"]), seed
    assert n_ops >= 30


def test_strong_aug_oracle_equals_reference_class_live():
    from oracle import strong_aug as SA
    from tests.golden.make_golden import strong_aug_digest
    z = live()
    aug = None
    if R.available():
        _cv2()
        aug = R.strong_augmentation_cls()(brightness_delta=20, contrast_range=(0.7, 1.3),
                                          saturation_range=(0.4, 1.6), hue_delta=10)
    rs = np.random.RandomState(5)
    for it in range(60):
        H, W = [(64, 64), (33, 47), (120, 120), (16, 100)][it % 4]
        img = rs.randint(0, 256, (H, W, 3)).astype(np.uint8)
        np.random.seed(it)
        ops_ = SA.draw_strong_aug(np.random, 20, (0.7, 1.3), (0.4, 1.6), 10)
        assert z["strong_aug_after"][it] == np.random.random(), it
        got = SA.apply_strong_aug(img.copy(), ops_)
        assert strong_aug_digest(got) == z["strong_aug_sha256"][it], it
        if aug is not None:
            np.random.seed(it)
            ref = aug(dict(img=img.copy(), img_fields=['img']))['img_strong_aug']
            assert z["strong_aug_after"][it] == np.random.random()
            assert np.array_equal(got, ref), it


# ------------------------------------------------------------------ test-time slide / flip inference
def _slide_case_inputs(case):
    from tests.golden.make_golden import slide_meta, synthetic_encode_decode
    name, B, C, H, W, mode, crop, stride, flip, direction, ori, seed = case
    g = torch.Generator().manual_seed(900 + seed)
    return torch.randn((B, 3, H, W), generator=g), slide_meta(flip, direction, ori, B), synthetic_encode_decode(C)


def test_slide_inference_oracle_vs_golden():
    """oracle.metrics.slide_inference / inference against what the reference methods (compiled from
    encoder_decoder.py:220-353) wrote: bit-exact. The last bit of ATen's CPU soft-max and resampling
    depends on how the work is split over threads; the fixture was written with 8, so the oracle runs
    with 8 here whatever the host's core count."""
    from tests.golden.make_golden import slide_cases
    z = load("slide_inference.npz")
    threads = torch.get_num_threads()
    torch.set_num_threads(8)
    try:
        _check_slide_inference_against(z, slide_cases())
    finally:
        torch.set_num_threads(threads)


def _check_slide_inference_against(z, cases):
    for case in cases:
        name, B, C, H, W, mode, crop, stride = case[:8]
        img, meta, enc = _slide_case_inputs(case)
        out, _ = om.inference(enc, img, meta, True, mode, crop, stride, C)
        assert np.array_equal(out.numpy(), z[f"{name}_output"]), name
        assert np.array_equal(out.argmax(dim=1).numpy().astype(np.uint8), z[f"{name}_pred"]), name
        if mode == "slide":
            raw = om.slide_inference(enc, img, meta, False, crop, stride, C)
            assert np.array_equal(raw.numpy(), z[f"{name}_slide"]), name


def test_slide_inference_oracle_equals_reference_live():
    import types
    from tests.golden.make_golden import slide_cases
    z = live()
    for case in slide_cases():
        name, B, C, H, W, mode, crop, stride = case[:8]
        img, meta, enc = _slide_case_inputs(case)
        img = img + 0.25                                   # not the fixture's input
        got, _ = om.inference(enc, img, meta, True, mode, crop, stride, C)
        assert_close_to_stored(got, z[f"slide_{name}"], 1e-6)
        if R.available():
            seg = R.reference_segmentor(enc, types.SimpleNamespace(mode=mode, crop_size=crop, stride=stride), C)
            want, _ = seg.inference(img, meta, True)
            assert torch.equal(got, want), name


def test_aug_test_oracle_vs_golden_and_reference():
    """oracle.metrics.aug_test against the fixture the reference method wrote and, on other inputs,
    against reference_live.npz and, when the reference is present, the method itself."""
    import types
    from tests.golden.make_golden import aug_cases, aug_inputs, synthetic_encode_decode
    z, zl = load("aug_test.npz"), live()
    for case in aug_cases():
        name, B, C, ori, mode, crop, stride, augs, seed = case
        imgs, metas = aug_inputs(case)
        enc = synthetic_encode_decode(C)
        pred, _ = om.aug_test(enc, imgs, metas, True, mode, crop, stride, C)
        assert np.array_equal(np.stack(pred).astype(np.uint8), z[f"{name}_pred"]), name
        imgs2 = [im * 0.5 + 0.1 for im in imgs]
        got, _ = om.aug_test(enc, imgs2, metas, True, mode, crop, stride, C)
        want = list(zl[f"aug_{name}_pred"])
        if R.available():
            seg = R.reference_segmentor(enc, types.SimpleNamespace(mode=mode, crop_size=crop, stride=stride), C)
            want, _ = seg.aug_test(imgs2, metas, True)
        assert len(got) == len(want) and all(np.array_equal(a, b) for a, b in zip(got, want)), name
