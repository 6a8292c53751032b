"""uint8 label maps through the training hot path: every entry point, the prototype bank, the whole
SelfTrainingStep and the errors. The rule under test: for int64 labels with values in [0, 255], the
run on `x.to(torch.uint8)` gives the same results — deterministic outputs bit for bit, label outputs
equal to the int64 ones cast to uint8, float-atomic sums (prototype sums and what depends on mu)
within the 1e-5 the int64 tests allow."""
import numpy as np
import pytest
import torch

from oracle import pfgst_loss as OL, step as ostep
from pfst_b200 import _lib, ops
from pfst_b200.losses.cross_entropy import upsample_cross_entropy
from pfst_b200.prototypes import PrototypeBank, proto_dist_loss
from pfst_b200.step import SelfTrainingStep
from pfst_b200.synthetic import WORKLOADS, blocky_labels, step_inputs

pytestmark = pytest.mark.gpu

U8 = torch.uint8


def _u8(t, offset=0):
    """uint8 copy of an int64 map; offset > 0 makes it a view at that storage offset (unaligned)."""
    if offset == 0:
        return t.to(U8)
    flat = torch.empty(t.numel() + offset, dtype=U8, device=t.device)
    v = flat[offset:].view(t.shape)
    v.copy_(t.to(U8))
    return v


def _i64(t, offset=0):
    if offset == 0:
        return t.clone()
    flat = torch.empty(t.numel() + offset, dtype=torch.int64, device=t.device)
    v = flat[offset:].view(t.shape)
    v.copy_(t)
    return v


def _labels(B, H, W, C, seed, cuda):
    g = torch.Generator().manual_seed(seed)
    return blocky_labels(B, H, W, C, g).to(cuda)          # int64, with 255 (ignore) pixels


def _close(a, b, rel=1e-5):
    return (a - b).abs().max() <= rel * b.abs().max() + 1e-12


# ------------------------------------------------------------------------------------ pseudo labels
@pytest.mark.parametrize("C", [1, 2, 6, 33])
@pytest.mark.parametrize("hw", [(64, 64), (5, 7), (120, 120)])
@pytest.mark.parametrize("reject", [-1, 255])
def test_pseudo_label_u8_equals_i64(cuda, C, hw, reject):
    g = torch.Generator().manual_seed(C * 31 + hw[0])
    logits = (3 * torch.randn((2, C) + hw, generator=g)).to(cuda)
    thr = 0.6
    a = ops.pseudo_label(logits, thr, reject_label=reject, want_part_weight=True)
    b = ops.pseudo_label(logits, thr, reject_label=reject, want_part_weight=True, label_dtype=U8)
    torch.cuda.synchronize()
    assert b[0].dtype == U8
    assert torch.equal(b[0], a[0].to(U8))
    for x, y in zip(a[1:], b[1:]):
        assert torch.equal(x, y)


# ----------------------------------------------------------------------------------------- ClassMix
@pytest.mark.parametrize("C", [1, 2, 6, 33])
@pytest.mark.parametrize("hw", [(64, 64), (5, 7), (120, 120)])
@pytest.mark.parametrize("offset", [0, 1, 3])
def test_class_presence_and_mix_u8_equal_i64(cuda, C, hw, offset):
    B, (H, W) = 3, hw
    gt = _labels(B, H, W, C, 7 + offset, cuda)
    pl = _labels(B, H, W, C, 9 + offset, cuda)[:, 0]
    g = torch.Generator().manual_seed(5)
    img, trg = torch.randn((B, 3, H, W), generator=g).to(cuda), torch.randn((B, 3, H, W), generator=g).to(cuda)
    pa, pb = ops.class_presence(_i64(gt, offset)), ops.class_presence(_u8(gt, offset))
    torch.cuda.synchronize()
    assert torch.equal(pa, pb)
    chosen = torch.randint(0, 2 ** 31 - 1, (B, 8), generator=g, dtype=torch.int32).to(cuda)
    count = torch.tensor([1234], dtype=torch.int64, device=cuda)
    a = ops.class_mix(_i64(gt, offset), chosen, img, trg, _i64(pl, offset), count=count, ps_size=B * H * W)
    b = ops.class_mix(_u8(gt, offset), chosen, img, trg, _u8(pl, offset), count=count, ps_size=B * H * W)
    torch.cuda.synchronize()
    assert b[1].dtype == U8 and b[3].dtype == U8
    assert torch.equal(a[0], b[0]) and torch.equal(a[2], b[2])
    assert torch.equal(b[1], a[1].to(U8)) and torch.equal(b[3], a[3].to(U8))


# --------------------------------------------------------------------------------------- PFGST loss
_OPTIONS = [
    ("shipped", 0, 3, None),
    ("gaussian", ops.LOSS_SIM_GAUSSIAN, 3, None),
    ("ema", ops.LOSS_CROSS_PROB_EMA, 3, None),
    ("unfold", ops.LOSS_UNFOLD_GRAD, 3, None),
    ("margin", ops.LOSS_SRC_MARGIN, 3, (0.5, -0.1)),
    ("margin2", ops.LOSS_SRC_MARGIN2, 3, (0.5, -0.1)),
    ("top_k_none", 0, 0, None),
]


@pytest.mark.parametrize("name,options,top_k,margin", _OPTIONS)
@pytest.mark.parametrize("shape", [(2, 6, 32, 32, 16, 16, 128), (2, 33, 30, 30, 15, 15, 120)])
def test_pfgst_loss_u8_equals_i64(cuda, name, options, top_k, margin, shape):
    B, C, lh, lw, fh, fw, G = shape
    g = torch.Generator().manual_seed(11)
    logits = torch.randn((B, C, lh, lw), generator=g).to(cuda)
    x_ema, x_src = (torch.randn((B, 16, fh, fw), generator=g).to(cuda) for _ in range(2))
    gt = _labels(B, G, G, C, 3, cuda)
    mix = (torch.rand((B, 1, G, G), generator=g) < 0.5).long().to(cuda)
    geo = ops.LossGeometry(logits.shape, x_src.shape, gt.shape, 0.5, 2)
    dots, ks = ops.neigh_dots(x_ema, x_src, geo.dilation // geo.up)
    q = torch.randn((B, C, geo.gh, geo.gw), generator=g).to(cuda) if options & ops.LOSS_CROSS_PROB_EMA else None
    w6 = (0.1, 0.2, 0.3, 0.4, 0.5, 0.6)
    gl = torch.linspace(0.5, 1.5, 6, device=cuda)
    res = []
    for gt_, mix_ in ((gt, mix), (gt.to(U8), mix.to(U8))):
        losses, st, dens, ero = ops.pfgst_loss_fwd(dots, ks, geo, logits, gt_, mix_, top_k, w6, options=options,
                                                   logits_ema=q, margin=margin)
        coef, glog = ops.pfgst_loss_bwd(dots, ks, geo, logits, gt_, mix_, top_k, w6, st, gl, options=options,
                                        logits_ema=q, margin=margin)
        torch.cuda.synchronize()
        res.append([losses.clone(), dens.clone(), ero.clone(), coef.clone(), glog.clone()])
    for x, y in zip(*res):
        assert torch.equal(x, y), name


# ------------------------------------------------------------------------------------ weighted CE
@pytest.mark.parametrize("C,factor", [(6, 4), (2, 4), (8, 4), (33, 4), (6, 2)])
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("offset", [0, 1])
def test_weighted_ce_u8_equals_i64(cuda, C, factor, weighted, offset):
    B, lh, lw = 2, 30, 32
    H, W = factor * lh, factor * lw
    g = torch.Generator().manual_seed(C + factor)
    logits = torch.randn((B, C, lh, lw), generator=g).to(cuda)
    lab = _labels(B, H, W, C, 4, cuda)[:, 0]
    w = torch.rand((B, H, W), generator=g).to(cuda) if weighted else None
    res = []
    for lab_ in (lab, _u8(lab, offset)):
        x = logits.clone().requires_grad_(True)
        loss, acc = upsample_cross_entropy(x, lab_, w)
        loss.backward()
        torch.cuda.synchronize()
        res.append((loss.detach(), acc, x.grad))
    (la, aa, ga), (lb, ab, gb) = res
    assert torch.equal(aa, ab)                                         # accuracy: integer counts
    # the loss sum and the logits gradient are reduced with float atomics (order-dependent)
    assert _close(lb, la, 1e-6) and _close(gb, ga, 1e-6)


# ------------------------------------------------------------------------------------- prototypes
@pytest.mark.parametrize("C,feat,lab,force", [
    (6, (2, 32, 64, 64), 256, None),        # masked (few classes, 8 k feature pixels)
    (6, (2, 32, 64, 64), 256, 0),           # MASKED_MAX_PIXELS = 0: sort + stream
    (33, (4, 32, 15, 15), 120, None),       # small planes (sorted lists + small-plane stream)
    (6, (2, 32, 64, 64), 255, 10 ** 9),     # masked kept for any batch, unaligned label rows
    (2, (1, 16, 5, 7), 20, None),           # odd plane
])
def test_proto_bank_u8_equals_i64(cuda, monkeypatch, C, feat, lab, force):
    if force is not None:
        monkeypatch.setattr(PrototypeBank, "MASKED_MAX_PIXELS", force)
    g = torch.Generator().manual_seed(C)
    x = torch.randn(feat, generator=g).to(cuda)
    labels = _labels(feat[0], lab, lab, C, 8, cuda)
    out = []
    for lb in (labels, labels.to(U8)):
        bank = PrototypeBank(C, feat[1], cuda)
        bank.accumulate(x, lb)
        packed = bank.packed.clone()
        bank.finalize()
        xs = x.clone().requires_grad_(True)
        loss = proto_dist_loss(xs, lb, bank.mu, bank.seen)
        loss.backward()
        torch.cuda.synchronize()
        out.append((packed, bank.mu.clone(), loss.detach(), xs.grad))
    (pa, mua, la, ga), (pb, mub, lb_, gb) = out
    CD = C * feat[1]
    assert torch.equal(pa[CD:], pb[CD:])                               # counts exact
    assert _close(pb[:CD], pa[:CD]) and _close(mub, mua)               # float-atomic sums
    assert _close(lb_, la) and _close(gb, ga)


def test_neigh_grad_proto_tagged_u8_equals_i64(cuda):
    B, D, h, w, C = 2, 32, 32, 32, 6
    g = torch.Generator().manual_seed(2)
    x = torch.randn((B, D, h, w), generator=g).to(cuda)
    coef = torch.randn((B, 9, h, w), generator=g).to(cuda)
    labels = _labels(B, 128, 128, C, 1, cuda)[:, 0]
    mu = torch.randn((C, D), generator=g).to(cuda)
    seen = torch.ones(C, dtype=U8, device=cuda)
    seen[2] = 0
    out = []
    for lb in (labels, labels.to(U8)):
        dist = torch.empty((B, h, w), device=cuda)
        acc = torch.empty(4, dtype=torch.float64, device=cuda)
        loss = torch.empty(1, device=cuda)
        _lib.call("pfst_proto_dist_fwd", x.data_ptr(), B, D, h, w, lb.data_ptr(), ops._labels(lb, "l"), 128, 128,
                  mu.data_ptr(), seen.data_ptr(), C, dist.data_ptr(), acc.data_ptr(), loss.data_ptr(), ops._stream())
        proto = dict(labels=lb, mu=mu, seen=seen, dist=dist, acc=acc, grad_loss=torch.full((1,), 0.1, device=cuda))
        gx = ops.neigh_grad(x, coef, 2, proto=proto)
        torch.cuda.synchronize()
        out.append((dist, acc, loss, gx))
    (da, aa, la, ga), (db, ab, lb, gb) = out
    assert torch.equal(da, db) and aa[1] == ab[1]                      # distances, number of valid pixels
    assert _close(lb, la, 1e-6) and _close(gb, ga, 1e-6)               # through the atomic distance sum


# ------------------------------------------------------------------------------- whole step, full size
def _step_pair(cuda, name, graphs, its=(0, 1), seed=1234):
    wl = WORKLOADS[name]
    host = step_inputs(wl, seed)
    inp = {k: v.to(cuda) for k, v in host.items()}
    down = wl.downscale if wl.downscale != 1.0 else None
    res = {}
    for dt in (torch.int64, U8):
        g = torch.Generator().manual_seed(3)
        shapes = [(64, 3, 3, 3), (wl.C,), (100003,)]
        student = [(0.02 * torch.randn(s, generator=g)).to(cuda) for s in shapes]
        teacher = [(0.02 * torch.randn(s, generator=g)).to(cuda) for s in shapes]
        step = SelfTrainingStep(teacher, student, wl.C, wl.D, cuda, dilation=wl.dilation, downscale=down,
                                max_batch=max(wl.B, 64), graphs=graphs)
        gt = inp["gt"].to(dt)
        outs = []
        for it in its:
            np.random.seed(21 + it)
            out = step.run(it, inp["img"], inp["target_img_strong_aug"], gt, inp["ema_logits"],
                           inp["logits_trg"], inp["x_src"], inp["x_ema"])
            torch.cuda.synchronize()
            o = {k: v.clone() for k, v in out.items()}
            b, geo = next(iter(step._bufs.values()))
            d = geo.dilation // geo.up
            ref = torch.empty_like(b.dots)
            ops.neigh_dots_slot(inp["x_ema"], d, 0, ref)
            ops.neigh_dots_slot(inp["x_src"], d, 1, ref)
            torch.cuda.synchronize()
            o["dots_exact"] = torch.equal(b.dots, ref)
            outs.append(o)
        res[dt] = (outs, [t.clone() for t in teacher], step)
    return res, host


@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg3", "cfg4"])
@pytest.mark.parametrize("graphs", [False, True])
def test_step_u8_equals_i64(cuda, name, graphs):
    res, _ = _step_pair(cuda, name, graphs)
    (oa, ta, _), (ob, tb, _) = res[torch.int64], res[U8]
    for a, b in zip(ta, tb):
        assert torch.equal(a, b)
    inexact = []
    for it, (a, b) in enumerate(zip(oa, ob)):
        for k in ("pseudo_label", "mixed_lbl", "mix_masks"):
            assert b[k].dtype == U8 and torch.equal(b[k], a[k].to(U8)), k
        for k in ("pseudo_conf", "count", "mixed_img", "pseudo_weight"):
            assert torch.equal(a[k], b[k]), k
        assert _close(b["mu"], a["mu"]) and _close(b["proto_loss"], a["proto_loss"])
        if not (a["dots_exact"] and b["dots_exact"]):
            inexact.append((it, a["dots_exact"], b["dots_exact"]))
            continue
        for k in ("losses", "grad_logits_trg"):
            assert torch.equal(a[k], b[k]), k
        assert _close(b["grad_x_src"], a["grad_x_src"])                # through mu: float-atomic sums
    if inexact:
        # a dots kernel inside the step returned sums that differ from the kernel launched alone: the losses
        # then differ whatever the label dtype (known failure, DESIGN.md §3.2; seen once in an eager cfg1
        # int64 run). (iteration, int64 dots exact, uint8 dots exact):
        pytest.xfail(f"step dot maps differ from neigh_dots launched alone (DESIGN.md 3.2): {inexact}")


def test_step_u8_matches_oracle_cfg2(cuda):
    wl = WORKLOADS["cfg2"]
    host = step_inputs(wl, 1234)
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
    out = step.run(it, inp["img"], inp["target_img_strong_aug"], inp["gt"].to(U8), inp["ema_logits"],
                   inp["logits_trg"], inp["x_src"], inp["x_ema"])
    ref = ostep.hot_path_step(it, teacher, student, host, wl.C, loss_cfg=OL.LossCfg(dilation=wl.dilation,
                              downscale=wl.downscale), rng=np.random.RandomState(11))
    torch.cuda.synchronize()
    for a, b in zip(d_teacher, teacher):
        assert torch.equal(a.cpu(), b)
    assert torch.equal(out["pseudo_label"].cpu(), ref["pseudo_label"].to(U8))
    assert torch.equal(out["mix_masks"].cpu(), ref["mix_masks"].to(U8))
    assert torch.equal(out["mixed_lbl"].cpu(), ref["mixed_lbl"].to(U8))
    assert torch.equal(out["mixed_img"].cpu(), ref["mixed_img"])
    lo, lr = out["losses"].cpu(), ref["losses"]
    assert torch.all((lo - lr).abs() <= 1e-5 * lr.abs() + 1e-9), (lo, lr)
    assert abs(float(out["proto_loss"].cpu()) - float(ref["proto_loss"])) <= 1e-5 * abs(float(ref["proto_loss"]))
    assert (out["mu"].cpu() - ref["mu"]).abs().max() <= 1e-5 * ref["mu"].abs().max()
    for key in ("grad_x_src", "grad_logits_trg"):
        go, gr = out[key].cpu(), ref[key]
        if gr is None:
            gr = torch.zeros_like(go)
        assert (go - gr).abs().max() <= 1e-5 * gr.abs().max() + 1e-12, key


@pytest.mark.parametrize("name", ["cfg2", "cfg3"])
def test_u8_graph_replays_keep_the_dot_maps_exact(cuda, name):
    """The uint8 step keeps the int64 schedule (label sort between the two TMA dots kernels,
    DESIGN.md §3.2): every replay's dot maps equal the kernel launched alone."""
    wl = WORKLOADS[name]
    inp = {k: v.to(cuda) for k, v in step_inputs(wl, 1234).items()}
    down = wl.downscale if wl.downscale != 1.0 else None
    g = torch.Generator().manual_seed(3)
    shapes = [(64, 3, 3, 3), (wl.C,), (100003,)]
    student = [(0.02 * torch.randn(s, generator=g)).to(cuda) for s in shapes]
    teacher = [(0.02 * torch.randn(s, generator=g)).to(cuda) for s in shapes]
    step = SelfTrainingStep(teacher, student, wl.C, wl.D, cuda, dilation=wl.dilation, downscale=down,
                            max_batch=max(wl.B, 64), graphs=True)
    gt = inp["gt"].to(U8)
    for it in range(8):
        np.random.seed(5)
        step.run(it, inp["img"], inp["target_img_strong_aug"], gt, inp["ema_logits"], inp["logits_trg"],
                 inp["x_src"], inp["x_ema"])
        torch.cuda.synchronize()
        b, geo = next(iter(step._bufs.values()))
        d = geo.dilation // geo.up
        ref = torch.empty_like(b.dots)
        ops.neigh_dots_slot(inp["x_ema"], d, 0, ref)
        ops.neigh_dots_slot(inp["x_src"], d, 1, ref)
        torch.cuda.synchronize()
        assert torch.equal(b.dots, ref), (name, it)


# ------------------------------------------------------------------------------------------- errors
def test_label_dtype_errors_raise_before_launch(cuda):
    B, C, H, W = 2, 6, 32, 32
    gt = _labels(B, H, W, C, 1, cuda)
    chosen = torch.zeros((B, 8), dtype=torch.int32, device=cuda)
    img = torch.zeros((B, 3, H, W), device=cuda)
    with pytest.raises(TypeError):                       # uint8 gt, int64 pseudo label
        ops.class_mix(gt.to(U8), chosen, img, img, gt[:, 0].clone(), want_weight=False)
    with pytest.raises(TypeError):                       # int32 labels
        ops.class_presence(gt.to(torch.int32))
    x = torch.randn((B, 16, 8, 8), device=cuda)
    logits = torch.randn((B, C, 16, 16), device=cuda)
    geo = ops.LossGeometry(logits.shape, x.shape, gt.shape, 0.5, 2)
    dots, ks = ops.neigh_dots(x, x, 1)
    with pytest.raises(TypeError):                       # uint8 gt, int64 ClassMix mask
        ops.pfgst_loss_fwd(dots, ks, geo, logits, gt.to(U8), gt.clamp(0, 1), 3, (0.1,) * 6)
    losses, st, _, _ = ops.pfgst_loss_fwd(dots, ks, geo, logits, gt.to(U8), gt.clamp(0, 1).to(U8), 3, (0.1,) * 6)
    with pytest.raises(TypeError):
        ops.pfgst_loss_bwd(dots, ks, geo, logits, gt.to(U8), gt.clamp(0, 1), 3, (0.1,) * 6, st,
                           torch.ones(6, device=cuda))
    with pytest.raises(TypeError):
        upsample_cross_entropy(logits, gt.to(torch.int32))
    with pytest.raises(TypeError):
        ops.pseudo_label(torch.zeros((B, C, H, W), device=cuda), label_dtype=torch.int32)
    with pytest.raises(ValueError):                      # uint8 pseudo labels cannot hold 256 classes
        ops.pseudo_label(torch.zeros((B, 256, 4, 4), device=cuda), label_dtype=U8)
    with pytest.raises(TypeError):
        bank = PrototypeBank(C, 8, cuda)
        bank.accumulate(torch.zeros((B, 8, 8, 8), device=cuda), gt.to(torch.int32))
    wl = WORKLOADS["cfg1"]
    inp = {k: v.to(cuda) for k, v in step_inputs(wl, 1).items()}
    step = SelfTrainingStep([torch.zeros(5, device=cuda)], [torch.zeros(5, device=cuda)], wl.C, wl.D, cuda,
                            dilation=wl.dilation, downscale=wl.downscale)
    with pytest.raises(TypeError):
        step.run(0, inp["img"], inp["target_img_strong_aug"], inp["gt"].to(torch.int32), inp["ema_logits"],
                 inp["logits_trg"], inp["x_src"], inp["x_ema"])
    torch.cuda.synchronize()
    assert step._step_count == 0                         # nothing was enqueued


# --------------------------------------------------------------------------- PFGSTLoss, decode head
def test_pfgst_loss_module_and_decode_head_take_uint8(cuda):
    from pfst_b200.losses import decode_head_losses
    from pfst_b200.losses.pfgst_loss import PFGSTLoss
    B, C, G = 2, 6, 128
    g = torch.Generator().manual_seed(4)
    gt = _labels(B, G, G, C, 6, cuda)
    mix = (torch.rand((B, 1, G, G), generator=g) < 0.5).long().to(cuda)
    logits0 = torch.randn((B, C, 32, 32), generator=g).to(cuda)
    x0 = torch.randn((B, 16, 16, 16), generator=g).to(cuda)
    xe = torch.randn((B, 16, 16, 16), generator=g).to(cuda)
    mod = PFGSTLoss(kernel_size=3, dilation=2, top_k=3, sim_type='cosine', feat_level=None, detach_unfold=True,
                    downscale=0.5, weights=dict(src_pos=0.1, src_neg=0.2, src_pos_std=0.3, src_neg_std=0.4,
                                                sim_pos=0.5, sim_neg=0.6))
    res = []
    for gt_, mix_ in ((gt, mix), (gt.to(U8), mix.to(U8))):
        logits, x = logits0.clone().requires_grad_(True), x0.clone().requires_grad_(True)
        out = mod(dict(logits_trg=logits, gt_src=gt_, x_src=x, x_ema=xe, mix_masks=mix_))
        vals = [v for k, v in out.items() if not k.startswith('vis|')]
        sum(vals).backward()
        ce = decode_head_losses(logits, gt_)
        torch.cuda.synchronize()
        res.append((torch.stack([v.detach() for v in vals]), logits.grad.clone(), x.grad.clone(),
                    ce['loss_ce'].detach(), ce['acc_seg']))
    (la, gla, gxa, cea, aca), (lb, glb, gxb, ceb, acb) = res
    assert torch.equal(la, lb) and torch.equal(gxa, gxb) and torch.equal(aca, acb)
    assert _close(glb, gla, 1e-6) and _close(ceb, cea, 1e-6)      # float-atomic reductions


# ------------------------------------------------------------------------------------------ plug-in

def _plugin_run(cuda, dt, fused):
    import random
    from pfst_b200.uda import PFGST
    from tests.fake_segmentor import TinySegmentor
    from tests.golden.make_golden import STEP_CFG, step_batches

    class Widening(TinySegmentor):
        """Records the dtype of the labels the trainer hands it and widens them: F.cross_entropy takes
        int64 targets only (INTEGRATION.md §2b)."""
        seen = []

        def forward_train(self, img, img_metas, gt_semantic_seg, seg_weight=None, **kw):
            Widening.seen.append(gt_semantic_seg.dtype)
            return super().forward_train(img, img_metas, gt_semantic_seg.long(), seg_weight, **kw)

    Widening.seen = []
    cfg = dict(STEP_CFG)
    cfg['model'] = lambda: Widening(6, 16, seed=0)
    if not fused:
        cfg['fused_hot_path'] = False
    m = PFGST(**cfg).to(cuda)
    opt = torch.optim.SGD(m.model.parameters(), lr=0.01)
    random.seed(1); np.random.seed(1); torch.manual_seed(1)
    d2h0 = m.d2h_bytes()                       # the log ledger is shared per device: count this run only
    logs = []
    for batch in step_batches():
        b = {k: (v.to(cuda) if isinstance(v, torch.Tensor) else v) for k, v in batch.items()}
        b['gt_semantic_seg'] = b['gt_semantic_seg'].to(dt)
        out = m.train_step(b, opt)
        logs.append(dict(out['log_vars']))
    torch.cuda.synchronize()
    stu = torch.cat([p.detach().reshape(-1) for p in m.model.parameters()])
    ema = torch.cat([p.detach().reshape(-1) for p in m.ema_model.parameters()])
    state = np.random.get_state()
    return dict(logs=logs, stu=stu, ema=ema, rng=(state[1].copy(), state[2]), d2h=m.d2h_bytes() - d2h0,
                seen=list(Widening.seen), fused=m.fused)


@pytest.mark.parametrize("fused", [True, False])
def test_plugin_train_steps_u8_equal_i64(cuda, monkeypatch, fused):
    monkeypatch.setattr(torch.backends.cudnn, "deterministic", True)
    monkeypatch.setattr(torch.backends.cudnn, "benchmark", False)
    a = _plugin_run(cuda, torch.int64, fused)
    b = _plugin_run(cuda, U8, fused)
    assert a["fused"] == b["fused"] == fused
    assert a["seen"] == [torch.int64] * 6 and b["seen"] == [U8] * 6       # source and mixed labels, 3 steps
    assert [list(x) for x in a["logs"]] == [list(x) for x in b["logs"]]           # keys and their order
    assert list(a["logs"][0].items()) == list(b["logs"][0].items())              # first step: bit-identical
    # later steps start from the parameters one SGD step produced; the backward sums float gradients with
    # atomics (cuDNN weight gradients, the shared logits of the down-scaled PFGST loss), so two int64 runs
    # already differ in the last bits there: compared within 1e-5
    for la, lb in zip(a["logs"][1:], b["logs"][1:]):
        for k in la:
            assert abs(la[k] - lb[k]) <= 1e-5 * abs(la[k]) + 1e-6, k
    assert _close(b["stu"], a["stu"]) and _close(b["ema"], a["ema"])
    assert np.array_equal(a["rng"][0], b["rng"][0]) and a["rng"][1] == b["rng"][1]
    assert a["d2h"] == b["d2h"] > 0


def test_plugin_refuses_int32_before_any_launch(cuda):
    from pfst_b200.uda import PFGST
    from tests.fake_segmentor import TinySegmentor
    from tests.golden.make_golden import STEP_CFG, step_batches
    cfg = dict(STEP_CFG)
    cfg['model'] = lambda: TinySegmentor(6, 16, seed=0)
    m = PFGST(**cfg).to(cuda)
    b = {k: (v.to(cuda) if isinstance(v, torch.Tensor) else v) for k, v in next(iter(step_batches(1))).items()}
    b['gt_semantic_seg'] = b['gt_semantic_seg'].to(torch.int32)
    state = np.random.get_state()
    d2h0 = m.d2h_bytes()
    with pytest.raises(TypeError):
        m.forward_train(**b)
    assert m.local_iter == 0 and m.d2h_bytes() == d2h0 and m._mix_plan is None
    assert np.array_equal(np.random.get_state()[1], state[1])
