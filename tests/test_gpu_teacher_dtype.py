"""fp16 / bf16 teacher outputs (ema_logits, x_ema) through the training hot path. The rule under test:
converting fp16 / bf16 to fp32 is exact, so a run on a 16-bit teacher tensor `t` gives what the fp32 path
gives on `t.float()` — deterministic outputs bit for bit, float-atomic prototype sums within 1e-6 relative,
and what follows from them (mu, losses, student gradients) within the 1e-5 the step tests allow.
Inputs are drawn in fp32 and rounded to the 16-bit type; the fp32 leg uses `t16.float()`."""
import numpy as np
import pytest
import torch

from pfst_b200 import _lib, ops
from pfst_b200.losses.pfgst_loss import LOSS_KEYS, PFGSTLoss
from pfst_b200.prototypes import PrototypeBank
from pfst_b200.step import SelfTrainingStep
from pfst_b200.synthetic import WORKLOADS, blocky_labels, step_inputs

HALF = [torch.bfloat16, torch.float16]
W6 = {'src_pos': 0.1, 'src_neg': 0.1, 'sim_pos': 0.1, 'sim_neg': 0.1, 'src_pos_std': 0.1, 'src_neg_std': 0.1}


def _loss_module(wl):
    return PFGSTLoss(top_k=3, dilation=wl.dilation, kernel_size=3, weights=W6, sim_type='cosine', feat_level=None,
                     detach_unfold=True, downscale=wl.downscale)


def _close(a, b, rel=1e-5):
    return (a - b).abs().max() <= rel * b.abs().max() + 1e-12


def _view(t, offset):
    """Copy of t at `offset` elements into a fresh buffer (offset > 0: an unaligned view)."""
    flat = torch.empty(t.numel() + offset, dtype=t.dtype, device=t.device)
    v = flat[offset:].view(t.shape)
    v.copy_(t)
    return v


# ------------------------------------------------------------------------------------------ CPU only
def test_float_dtype_tags():
    assert ops.float_dtype_tag(torch.float32) == _lib.DT_F32 == 16
    assert ops.float_dtype_tag(torch.float16) == _lib.DT_F16 == 17
    assert ops.float_dtype_tag(torch.bfloat16) == _lib.DT_BF16 == 18
    assert {_lib.DT_F32, _lib.DT_F16, _lib.DT_BF16}.isdisjoint({_lib.DT_U8, _lib.DT_I32, _lib.DT_I64, 0})
    for dt in (torch.float64, torch.int64, torch.uint8, torch.int32):
        with pytest.raises(TypeError):
            ops.float_dtype_tag(dt, "x")


def test_algorithmic_bytes_teacher_bytes():
    from pfst_b200.step import algorithmic_bytes
    B, C, H, W, D, h, w, n = 8, 6, 512, 512, 256, 64, 64, 1000
    a, b = algorithmic_bytes(B, C, H, W, D, h, w, n), algorithmic_bytes(B, C, H, W, D, h, w, n, teacher_bytes=2)
    P, p = B * H * W, B * h * w
    assert a == algorithmic_bytes(B, C, H, W, D, h, w, n, teacher_bytes=4)
    assert a["pseudo_label"] - b["pseudo_label"] == 2 * C * P
    assert a["neigh_dots"] - b["neigh_dots"] == 2 * D * p
    assert a["proto_accum"] - b["proto_accum"] == 2 * D * p
    for k in ("ema", "class_presence_and_mix", "neigh_grad", "proto_dist_fwd_bwd"):
        assert a[k] == b[k]


# ------------------------------------------------------------------------------------ pseudo labels
def _logits(shape, dt, seed, cuda, specials=False):
    g = torch.Generator().manual_seed(seed)
    x = (3 * torch.randn(shape, generator=g)).to(dt)
    if specials:
        B, C, H, W = shape
        x[0, :, 0, 0] = float("nan")
        x[0, 0, 0, 1] = float("inf")
        x[0, 1 % C, 0, 2] = float("-inf")
        x[0, :, 0, 3] = 1.5                          # ties: every class equal
        if C > 1:
            x[0, 1, 1, :] = x[0, 0, 1, :]            # two-way ties along a row
    return x.to(cuda)


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("C", [2, 6, 33])
@pytest.mark.parametrize("hw", [(64, 64), (5, 7)])
@pytest.mark.parametrize("lab", [torch.int64, torch.uint8])
@pytest.mark.parametrize("rule", ["scalar", "classwise", "entropy"])
def test_pseudo_label_16bit_equals_fp32(cuda, dt, C, hw, lab, rule):
    x = _logits((2, C) + hw, dt, C * 7 + hw[0], cuda, specials=True)
    thr_vec = torch.linspace(0.3, 0.9, C, device=cuda) if rule != "scalar" else None
    kw = dict(thr=0.6, thr_per_class=thr_vec, mode=1 if rule == "entropy" else 0,
              reject_label=255 if rule == "entropy" else -1, want_part_weight=True, label_dtype=lab)
    a = ops.pseudo_label(x.float(), **kw)
    b = ops.pseudo_label(x, **kw)
    c = ops.pseudo_label(_view(x, 1), **kw)               # unaligned view: scalar path
    torch.cuda.synchronize()
    for out in (b, c):
        for u, v in zip(a, out):
            assert torch.equal(u, v) or (u.is_floating_point() and torch.equal(u.isnan(), v.isnan())
                                         and torch.equal(u.nan_to_num(), v.nan_to_num()))


@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("C,hw", [(6, (64, 64)), (33, (8, 8)), (6, (5, 7))])
def test_pseudo_label_16bit_near_ties(cuda, dt, C, hw):
    """Logits of small magnitude with an earlier class a few ulps below the maximum: the re-check of
    torch.max's first-index tie (pl_tie_label) runs on the 16-bit logits."""
    g = torch.Generator().manual_seed(C)
    x = (1e-3 * torch.randn((2, C) + hw, generator=g)).to(dt)
    x[:, 0] = x[:, C - 1]                                    # class 0 ties the last class ...
    x[:, 1] = (x[:, C - 1].float() * (1 - 2 ** -9)).to(dt)   # ... and class 1 sits just below it
    x = x.to(cuda)
    for view in (x, _view(x, 1)):
        a = ops.pseudo_label(x.float(), 0.0, want_part_weight=True)
        b = ops.pseudo_label(view, 0.0, want_part_weight=True)
        torch.cuda.synchronize()
        for u, v in zip(a, b):
            assert torch.equal(u, v)


# ----------------------------------------------------------------------------------- dot maps
@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("shape,dil", [
    ((2, 64, 64, 64), 1), ((2, 64, 64, 64), 2), ((1, 40, 32, 128), 4),   # TMA
    ((4, 64, 15, 15), 1), ((3, 48, 15, 15), 2),                          # small planes (bulk copies)
    ((2, 24, 13, 13), 1),                                                # odd width: generic
    ((2, 20, 24, 12), 2),                                                # 16-bit rows not 16-byte units
])
@pytest.mark.parametrize("offset", [0, 1])
def test_neigh_dots_16bit_equal_fp32(cuda, dt, shape, dil, offset):
    g = torch.Generator().manual_seed(shape[1] + dil)
    x = torch.randn(shape, generator=g).to(dt).to(cuda)
    xv = _view(x, offset)                    # offset 1: an unaligned 16-bit view
    a, ka = ops.neigh_dots_slot(xv.float(), dil, 0)     # the upcast is a fresh, aligned fp32 tensor
    b, kb = ops.neigh_dots_slot(xv, dil, 0)
    torch.cuda.synchronize()
    assert ka == kb and torch.equal(a[:, 0], b[:, 0])   # slot 1 of the (splits, 2, ...) buffer is not written


# ---------------------------------------------------------------------------- prototype accumulation
@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF)
@pytest.mark.parametrize("C,feat,lab,force", [
    (6, (2, 32, 64, 64), 256, None),        # masked
    (6, (2, 32, 64, 64), 256, 0),           # label sort + bulk-copy stream
    (33, (4, 32, 15, 15), 120, None),       # small planes
    (2, (1, 16, 5, 7), 20, None),           # odd plane: small-plane kernel
    (6, (2, 16, 26, 26), 52, 0),            # hw = 676 > 576, hw % 8 = 4: sort + warp-staged planes (no bulk copies)
    (6, (2, 16, 36, 36), 72, None),         # masked, hw % 512 != 0 (bounds-tested chunks)
])
@pytest.mark.parametrize("lab_dt", [torch.int64, torch.uint8])
def test_proto_accum_16bit_close_to_fp32(cuda, monkeypatch, dt, C, feat, lab, force, lab_dt):
    if force is not None:
        monkeypatch.setattr(PrototypeBank, "MASKED_MAX_PIXELS", force)
    g = torch.Generator().manual_seed(C)
    x = torch.randn(feat, generator=g).to(dt).to(cuda)
    labels = blocky_labels(feat[0], lab, lab, C, torch.Generator().manual_seed(8)).to(cuda).to(lab_dt)
    out = []
    for f in (x.float(), x):
        bank = PrototypeBank(C, feat[1], cuda)
        bank.accumulate(f, labels)
        out.append(bank.packed.clone())
        bank.finalize()
        out.append(bank.mu.clone())
    torch.cuda.synchronize()
    pa, mua, pb, mub = out
    CD = C * feat[1]
    assert torch.equal(pa[CD:], pb[CD:])
    assert _close(pb[:CD], pa[:CD], 1e-6) and _close(mub, mua, 1e-6)


# ------------------------------------------------------------------------------------------- errors
@pytest.mark.gpu
def test_teacher_dtype_errors_raise_before_launch(cuda):
    wl = WORKLOADS["tiny"]
    inp = {k: v.to(cuda) for k, v in step_inputs(wl, 5).items()}
    g = torch.Generator().manual_seed(3)
    params = [(0.02 * torch.randn(s, generator=g)).to(cuda) for s in [(64,), (wl.C,)]]
    step = SelfTrainingStep(params, [p.clone() for p in params], wl.C, wl.D, cuda, dilation=wl.dilation,
                            downscale=wl.downscale, max_batch=64)
    base = dict(img=inp["img"], trg_img=inp["target_img_strong_aug"], gt=inp["gt"], ema_logits=inp["ema_logits"],
                logits_trg=inp["logits_trg"], x_src=inp["x_src"], x_ema=inp["x_ema"])
    bad = [("ema_logits", torch.float64), ("ema_logits", torch.int64), ("x_ema", torch.float64),
           ("x_ema", torch.int32), ("x_src", torch.bfloat16), ("logits_trg", torch.bfloat16)]
    packed = step.bank.packed.clone()
    for name, dt in bad:
        np.random.seed(9)
        state = np.random.get_state()[1].copy()
        args = dict(base, **{name: base[name].to(dt)})
        torch.cuda.synchronize()
        with pytest.raises(TypeError):
            step.run(0, **args)
        torch.cuda.synchronize()
        assert np.array_equal(np.random.get_state()[1], state)        # no ClassMix draw
        assert not step._bufs and torch.equal(step.bank.packed, packed)
    for dt in (torch.float64, torch.int64):
        with pytest.raises(TypeError):
            ops.pseudo_label(inp["ema_logits"].to(dt), 0.5)
        with pytest.raises(TypeError):
            ops.neigh_dots_slot(inp["x_ema"].to(dt), 1, 0)
        with pytest.raises(TypeError):
            PrototypeBank(wl.C, wl.D, cuda).accumulate(inp["x_ema"].to(dt), inp["gt"][:, 0])
    loss = _loss_module(wl)
    t = dict(logits_trg=inp["logits_trg"], x_src=inp["x_src"].bfloat16(), x_ema=inp["x_ema"],
             gt_src=inp["gt"], mix_masks=torch.ones_like(inp["gt"]))
    with pytest.raises(TypeError, match="teacher"):
        loss(t)
    # cross_prob_type='ema': a 16-bit logits_ema is refused before the dots kernel is launched
    ema_loss = PFGSTLoss(top_k=3, dilation=wl.dilation, kernel_size=3, weights=W6, sim_type='cosine',
                         feat_level=None, detach_unfold=True, downscale=None, cross_prob_type='ema')
    t = dict(t, x_src=inp["x_src"], logits_ema=inp["logits_trg"].bfloat16())
    calls = []
    real = ops.neigh_dots
    ops.neigh_dots = lambda *a, **k: calls.append(1) or real(*a, **k)
    try:
        with pytest.raises(TypeError, match="logits_ema"):
            ema_loss(t)
    finally:
        ops.neigh_dots = real
    assert not calls


@pytest.mark.gpu
def test_teacher_entry_points_refuse_unknown_tags(cuda):
    B, C, D, h, w = 2, 6, 16, 16, 16
    x = torch.randn((B, C, h, w), device=cuda)
    lab = torch.empty((B, h, w), dtype=torch.int64, device=cuda)
    conf = torch.empty((B, h, w), device=cuda)
    count = torch.zeros(1, dtype=torch.int64, device=cuda)
    feats = torch.randn((B, D, h, w), device=cuda)
    dots = torch.zeros((8, 2, B, 5, h, w), device=cuda)
    packed = torch.zeros(C * D + C, device=cuda)
    ws = torch.zeros(1 << 20, dtype=torch.uint8, device=cuda)
    L = _lib.load()
    s = ops._stream()
    for tag in (0, 1, 2, 15, 19, -1):                        # label tags and neighbours are not float tags
        assert L.pfst_pseudo_label(x.data_ptr(), tag, B, C, h * w, 0.5, None, 0, -1, lab.data_ptr(),
                                   _lib.DT_I64, conf.data_ptr(), None, count.data_ptr(), s) == -2
        assert L.pfst_neigh_dots_slot(feats.data_ptr(), tag, B, D, h, w, 1, 0, 2, dots.data_ptr(), s) == -2
        assert L.pfst_proto_accum(feats.data_ptr(), tag, B, D, h, w, lab.data_ptr(), _lib.DT_I64, h, w, None,
                                  0.0, C, packed.data_ptr(), s) == -2
        assert L.pfst_proto_accum_ordered(feats.data_ptr(), tag, B, D, h, w, C, ws.data_ptr(),
                                          packed.data_ptr(), s) == -2
    # an unknown label tag is refused as well
    assert L.pfst_pseudo_label(x.bfloat16().data_ptr(), _lib.DT_BF16, B, C, h * w, 0.5, None, 0, -1,
                               lab.data_ptr(), 7, conf.data_ptr(), None, count.data_ptr(), s) == -2
    torch.cuda.synchronize()
    assert int(packed.abs().sum()) == 0


# ------------------------------------------------------------------------------------- PFGSTLoss
@pytest.mark.gpu
@pytest.mark.parametrize("dt", HALF)
def test_pfgst_loss_with_16bit_x_ema(cuda, dt):
    wl = WORKLOADS["tiny"]
    inp = {k: v.to(cuda) for k, v in step_inputs(wl, 11).items()}
    x16 = inp["x_ema"].to(dt)
    mix = (torch.rand(inp["gt"].shape, generator=torch.Generator().manual_seed(1)) > 0.5).long().to(cuda)
    res = []
    for xe in (x16.float(), x16):
        loss = _loss_module(wl)
        lt = inp["logits_trg"].clone().requires_grad_(True)
        xs = inp["x_src"].clone().requires_grad_(True)
        out = loss(dict(logits_trg=lt, x_src=xs, x_ema=xe, gt_src=inp["gt"], mix_masks=mix))
        sum(out[k] for k in LOSS_KEYS).backward()
        torch.cuda.synchronize()
        res.append((torch.stack([out[k].detach() for k in LOSS_KEYS]), lt.grad.clone(), xs.grad.clone()))
    (la, ga, xa), (lb, gb, xb) = res
    assert _close(lb, la) and _close(gb, ga) and _close(xb, xa)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["gauss", "topk_none"])
def test_pfgst_loss_options_with_bf16_x_ema(cuda, name):
    from tests.golden.make_golden import LOSS_OPTION_CASES, loss_option_inputs, loss_option_keys
    c, opts = LOSS_OPTION_CASES[name]
    keys = loss_option_keys(opts)
    gt, logits, x_src, x_ema, _ = loss_option_inputs(c)
    x16 = x_ema.bfloat16().to(cuda)
    mix = (torch.rand(gt.shape, generator=torch.Generator().manual_seed(2)) > 0.5).long().to(cuda)
    kw = dict(top_k=3)
    kw.update(opts)
    res = []
    for xe in (x16.float(), x16):
        mod = PFGSTLoss(dilation=c["dil"], kernel_size=3, weights=W6, feat_level=None, downscale=c["down"], **kw)
        lt = logits.clone().to(cuda).requires_grad_(True)
        xs = x_src.clone().to(cuda).requires_grad_(True)
        out = mod(dict(logits_trg=lt, gt_src=gt.to(cuda), x_ema=xe, x_src=xs, img_trg=None, mix_masks=mix))
        sum(out[k] for k in keys).backward()
        torch.cuda.synchronize()
        res.append((torch.stack([out[k].detach() for k in keys]), lt.grad.clone(), xs.grad.clone(),
                    out['vis|density_sim_feat'][2].clone()))
    (la, ga, xa, ea), (lb, gb, xb, eb) = res
    assert torch.equal(ea, eb)                                   # eroded masks
    assert _close(lb, la) and _close(gb, ga) and _close(xb, xa)


# ------------------------------------------------------------------------------- whole step, full size
def _make_step(cuda, wl, graphs):
    g = torch.Generator().manual_seed(3)
    shapes = [(64, 3, 3, 3), (wl.C,), (100003,)]
    student = [(0.02 * torch.randn(s, generator=g)).to(cuda) for s in shapes]
    teacher = [(0.02 * torch.randn(s, generator=g)).to(cuda) for s in shapes]
    down = wl.downscale if wl.downscale != 1.0 else None
    return SelfTrainingStep(teacher, student, wl.C, wl.D, cuda, dilation=wl.dilation, downscale=down,
                            max_batch=max(wl.B, 64), graphs=graphs)


def _run(step, it, inp, ema_logits, x_ema, gt):
    np.random.seed(21 + it)
    out = step.run(it, inp["img"], inp["target_img_strong_aug"], gt, ema_logits, inp["logits_trg"], inp["x_src"],
                   x_ema)
    torch.cuda.synchronize()
    o = {k: v.clone() for k, v in out.items()}
    key = [k for k in step._bufs if k[-2] == ema_logits.dtype and k[-1] == x_ema.dtype and k[4] == gt.dtype][0]
    b, geo = step._bufs[key]
    d = geo.dilation // geo.up
    ref = torch.empty_like(b.dots)
    ops.neigh_dots_slot(x_ema, d, 0, ref)
    ops.neigh_dots_slot(inp["x_src"], d, 1, ref)
    torch.cuda.synchronize()
    o["dots"] = b.dots.clone()
    o["dots_exact"] = torch.equal(b.dots, ref)
    return o


def _compare(a, b, inexact, it):
    for k in ("pseudo_label", "pseudo_conf", "count", "mixed_lbl", "mixed_img", "pseudo_weight", "mix_masks"):
        assert torch.equal(a[k], b[k]), k
    assert _close(b["mu"], a["mu"]) and _close(b["proto_loss"], a["proto_loss"])
    if not (a["dots_exact"] and b["dots_exact"]):
        inexact.append((it, a["dots_exact"], b["dots_exact"]))
        return
    assert torch.equal(a["dots"], b["dots"])
    for k in ("losses", "grad_logits_trg", "grad_x_src"):
        assert _close(b[k], a[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg3", "cfg4"])
@pytest.mark.parametrize("graphs", [False, True])
def test_step_bf16_teacher_equals_fp32_on_upcast(cuda, name, graphs):
    wl = WORKLOADS[name]
    inp = {k: v.to(cuda) for k, v in step_inputs(wl, 1234).items()}
    el16, xe16 = inp["ema_logits"].bfloat16(), inp["x_ema"].bfloat16()
    res = []
    for el, xe in ((el16.float(), xe16.float()), (el16, xe16)):
        step = _make_step(cuda, wl, graphs)
        res.append([_run(step, it, inp, el, xe, inp["gt"]) for it in (0, 1)])
    inexact = []
    for it, (a, b) in enumerate(zip(*res)):
        _compare(a, b, inexact, it)
    if inexact:
        pytest.xfail(f"step dot maps differ from neigh_dots launched alone (DESIGN.md 3.2): {inexact}")


@pytest.mark.gpu
@pytest.mark.parametrize("graphs", [False, True])
def test_step_alternating_teacher_dtypes_and_uint8_labels(cuda, graphs):
    """One step object run fp32 -> bf16 -> fp32 (the graph and buffer keys carry both dtypes), and a
    bf16 teacher with uint8 labels, each against a fresh fp32 step on the upcast tensors."""
    wl = WORKLOADS["cfg2"]
    inp = {k: v.to(cuda) for k, v in step_inputs(wl, 77).items()}
    el16, xe16 = inp["ema_logits"].bfloat16(), inp["x_ema"].bfloat16()
    el32, xe32 = el16.float(), xe16.float()
    mixed = _make_step(cuda, wl, graphs)
    ref = _make_step(cuda, wl, graphs)
    inexact = []
    for it, (el, xe) in enumerate(((el32, xe32), (el16, xe16), (el32, xe32))):
        a = _run(ref, it, inp, el32, xe32, inp["gt"])
        b = _run(mixed, it, inp, el, xe, inp["gt"])
        _compare(a, b, inexact, it)
    gt8 = inp["gt"].to(torch.uint8)
    a = _run(_make_step(cuda, wl, graphs), 0, inp, el32, xe32, gt8)
    b = _run(_make_step(cuda, wl, graphs), 0, inp, el16, xe16, gt8)
    assert b["pseudo_label"].dtype == torch.uint8
    _compare(a, b, inexact, "u8")
    if inexact:
        pytest.xfail(f"step dot maps differ from neigh_dots launched alone (DESIGN.md 3.2): {inexact}")


# ------------------------------------------------------------------------------- autocast reference
@pytest.mark.gpu
def test_reference_teacher_functions_under_autocast_equal_upcast(cuda):
    """The reference's teacher-side arithmetic (softmax / max of ema_logits, pfgst.py:259-266; the unfold
    cosine of x_ema, pfgst_loss.py:181-201) gives under autocast(bf16) what it gives on the upcast
    tensors: softmax and cosine_similarity are on autocast's fp32 list, unfold is exact in any dtype."""
    g = torch.Generator().manual_seed(4)
    el = (3 * torch.randn((2, 6, 32, 32), generator=g)).bfloat16().to(cuda)
    xe = torch.randn((2, 16, 16, 16), generator=g).bfloat16().to(cuda)

    def teacher(el, xe):
        p, lab = torch.max(torch.softmax(el, dim=1), dim=1)
        unf = torch.nn.Unfold(kernel_size=3, dilation=2, padding=2)(xe).view(2, 16, 9, 16, 16)
        sim = torch.nn.functional.cosine_similarity(unf, xe.unsqueeze(2), dim=1)
        return p, lab, sim

    ref = teacher(el.float(), xe.float())
    with torch.autocast("cuda", dtype=torch.bfloat16):
        got = teacher(el, xe)
    for a, b in zip(ref, got):
        assert a.dtype == b.dtype and torch.equal(a, b)


@pytest.mark.gpu
def test_step_bf16_teacher_matches_oracle_cfg2(cuda):
    """The CPU oracle run on the upcast teacher outputs (what the reference computes under autocast)."""
    from oracle import pfgst_loss as OL, step as ostep
    wl = WORKLOADS["cfg2"]
    host = step_inputs(wl, 1234)
    host["ema_logits"] = host["ema_logits"].bfloat16().float()
    host["x_ema"] = host["x_ema"].bfloat16().float()
    g = torch.Generator().manual_seed(3)
    shapes = [(64, 3, 3, 3), (64,), (wl.C, 512, 1, 1), (wl.C,), (100003,)]
    student = [0.02 * torch.randn(s, generator=g) for s in shapes]
    teacher = [0.02 * torch.randn(s, generator=g) for s in shapes]
    d_student, d_teacher = [p.to(cuda) for p in student], [p.to(cuda) for p in teacher]
    inp = {k: v.to(cuda) for k, v in host.items()}
    step = SelfTrainingStep(d_teacher, d_student, wl.C, wl.D, cuda, dilation=wl.dilation, downscale=wl.downscale,
                            max_batch=64, graphs=True)
    it = 7
    np.random.seed(11)
    out = step.run(it, inp["img"], inp["target_img_strong_aug"], inp["gt"], inp["ema_logits"].bfloat16(),
                   inp["logits_trg"], inp["x_src"], inp["x_ema"].bfloat16())
    ref = ostep.hot_path_step(it, teacher, student, host, wl.C, loss_cfg=OL.LossCfg(dilation=wl.dilation,
                              downscale=wl.downscale), rng=np.random.RandomState(11))
    torch.cuda.synchronize()
    for k in ("pseudo_label", "mix_masks", "mixed_lbl", "mixed_img"):
        assert torch.equal(out[k].cpu(), ref[k]), k
    lo, lr = out["losses"].cpu(), ref["losses"]
    assert torch.all((lo - lr).abs() <= 1e-5 * lr.abs() + 1e-9), (lo, lr)
    assert abs(float(out["proto_loss"].cpu()) - float(ref["proto_loss"])) <= 1e-5 * abs(float(ref["proto_loss"]))
    assert (out["mu"].cpu() - ref["mu"]).abs().max() <= 1e-5 * ref["mu"].abs().max()
    for key in ("grad_x_src", "grad_logits_trg"):
        go, gr = out[key].cpu(), ref[key]
        if gr is None:
            gr = torch.zeros_like(go)
        assert (go - gr).abs().max() <= 1e-5 * gr.abs().max() + 1e-12, key


# ------------------------------------------------------------------------------------------ plug-in
def _plugin_run(cuda, mode, fused):
    """Three PFGST.train_steps whose EMA teacher returns its logits and features in bf16 (mode 'bf16') or
    the same bf16-rounded values upcast to fp32 (mode 'upcast')."""
    import random
    from pfst_b200.uda import PFGST
    from tests.fake_segmentor import TinySegmentor
    from tests.golden.make_golden import STEP_CFG, step_batches

    class Teacher16(TinySegmentor):
        out_mode = None                              # set on the EMA copy only

        def encode_decode(self, img, img_metas):
            out, states = super().encode_decode(img, img_metas)
            if self.out_mode is None:
                return out, states
            cast = (lambda t: t.bfloat16()) if self.out_mode == "bf16" else (lambda t: t.bfloat16().float())
            x = cast(states['feats'])
            out = cast(out)
            return out, {'feats': x, 'decoded_features': x, 'seg_logits': out}

    cfg = dict(STEP_CFG)
    cfg['model'] = lambda: Teacher16(6, 16, seed=0)
    if not fused:
        cfg['fused_hot_path'] = False
    m = PFGST(**cfg).to(cuda)
    m.get_ema_model().out_mode = mode
    opt = torch.optim.SGD(m.model.parameters(), lr=0.01)
    random.seed(1); np.random.seed(1); torch.manual_seed(1)
    logs = []
    for batch in step_batches():
        b = {k: (v.to(cuda) if isinstance(v, torch.Tensor) else v) for k, v in batch.items()}
        out = m.train_step(b, opt)
        logs.append(dict(out['log_vars']))
    torch.cuda.synchronize()
    stu = torch.cat([p.detach().reshape(-1) for p in m.model.parameters()])
    ema = torch.cat([p.detach().reshape(-1) for p in m.ema_model.parameters()])
    state = np.random.get_state()
    return dict(logs=logs, stu=stu, ema=ema, rng=(state[1].copy(), state[2]), fused=m.fused)


@pytest.mark.gpu
@pytest.mark.parametrize("fused", [True, False])
def test_plugin_train_steps_bf16_teacher_equal_upcast(cuda, monkeypatch, fused):
    monkeypatch.setattr(torch.backends.cudnn, "deterministic", True)
    monkeypatch.setattr(torch.backends.cudnn, "benchmark", False)
    a = _plugin_run(cuda, "upcast", fused)
    b = _plugin_run(cuda, "bf16", fused)
    assert a["fused"] == b["fused"] == fused
    assert [list(x) for x in a["logs"]] == [list(x) for x in b["logs"]]
    la0, lb0 = a["logs"][0], b["logs"][0]
    if fused:
        assert list(la0.items()) == list(lb0.items())                 # first step: bit-identical
    else:
        # unfused, PFGSTLoss computes the dots of a bf16 x_ema and an fp32 x_src as two slot launches, whose
        # channel splits differ from the one two-tensor launch of two fp32 tensors: 1e-5 on the first step too
        for k in la0:
            assert abs(la0[k] - lb0[k]) <= 1e-5 * abs(la0[k]) + 1e-6, k
    for la, lb in zip(a["logs"][1:], b["logs"][1:]):
        for k in la:
            assert abs(la[k] - lb[k]) <= 1e-5 * abs(la[k]) + 1e-6, k
    assert _close(b["stu"], a["stu"]) and _close(b["ema"], a["ema"])
    assert np.array_equal(a["rng"][0], b["rng"][0]) and a["rng"][1] == b["rng"][1]
