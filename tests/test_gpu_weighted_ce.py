"""Decode-head loss (SURVEY.md §8f rank 1): the fused up-sample + weighted CE + accuracy +
gradient kernel against the CPU oracle and the golden vectors produced by the reference's
own resize / cross_entropy / accuracy (tests/golden/weighted_ce.npz). fp32: 1e-5 relative.
Every kernel the host code can dispatch to is also compared with the oracle evaluated in float64."""
import os
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from oracle import weighted_ce as OC
from pfst_b200 import _lib, ops
from pfst_b200.losses import decode_head_losses, upsample_cross_entropy
from tests.golden.make_golden import ce_cases, ce_inputs

pytestmark = pytest.mark.gpu
G = Path(__file__).resolve().parent / "golden"
TOL = 1e-5


def _close(a, b, what):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    assert (a - b).abs().max() <= TOL * b.abs().max() + 1e-12, (what, float((a - b).abs().max()), float(b.abs().max()))


@pytest.mark.parametrize("case", ce_cases(), ids=[c[0] for c in ce_cases()])
def test_matches_reference_golden_and_oracle(cuda, case):
    name, B, C, lh, lw, scale, use_w, use_cw, lwt = case
    z = np.load(G / "weighted_ce.npz")
    logits, label, weight, cw = ce_inputs(name, B, C, lh, lw, scale, use_w, use_cw)
    zl = logits.to(cuda).requires_grad_(True)
    loss, acc = upsample_cross_entropy(zl, label.to(cuda), None if weight is None else weight.to(cuda),
                                       None if cw is None else cw.to(cuda), 255, lwt)
    loss.backward()
    _close(loss.detach(), z[f"{name}_loss"], "loss vs reference")
    _close(acc, z[f"{name}_acc"], "acc vs reference")
    _close(zl.grad, z[f"{name}_grad"], "grad vs reference")
    zo = logits.clone().requires_grad_(True)
    lo, ao, _ = OC.decode_head_losses(zo, label, weight, cw, 255, lwt)
    lo.backward()
    _close(loss.detach(), lo.detach(), "loss vs oracle")
    _close(acc, ao, "acc vs oracle")
    _close(zl.grad, zo.grad, "grad vs oracle")


def test_full_size_cfg2_and_upstream_gradient(cuda):
    g = torch.Generator().manual_seed(1)
    B, C, lh, H = 8, 6, 128, 512
    logits = 2.0 * torch.randn((B, C, lh, lh), generator=g)
    label = torch.randint(0, C, (B, 1, H, H), generator=g)
    label[:, :, :9] = 255
    weight = torch.rand((B, H, H), generator=g)
    zl = logits.to(cuda).requires_grad_(True)
    out = decode_head_losses(zl, label.to(cuda), weight.to(cuda), loss_weight=0.4)
    (3.0 * out["loss_ce"]).backward()
    zo = logits.clone().requires_grad_(True)
    lo, ao, _ = OC.decode_head_losses(zo, label, weight, None, 255, 0.4)
    (3.0 * lo).backward()
    _close(out["loss_ce"].detach(), lo.detach(), "loss")
    _close(out["acc_seg"], ao, "acc")
    _close(zl.grad, zo.grad, "grad")


def test_all_ignored_and_no_grad(cuda):
    logits = torch.randn((1, 4, 8, 8)).to(cuda)
    label = torch.full((1, 1, 32, 32), 255, dtype=torch.int64).to(cuda)
    loss, acc = upsample_cross_entropy(logits, label)
    lo, ao, _ = OC.decode_head_losses(logits.cpu(), label.cpu())
    assert float(loss) == 0.0 == float(lo)
    _close(acc, ao, "acc of an all-ignored map")


def test_unsupported_resampling_raises(cuda):
    logits = torch.randn((1, 4, 8, 8)).to(cuda)
    with pytest.raises(ops.PfstError):
        upsample_cross_entropy(logits, torch.zeros((1, 1, 30, 32), dtype=torch.int64).to(cuda))
    with pytest.raises(ops.PfstError):
        decode_head_losses(logits, torch.zeros((1, 1, 32, 32), dtype=torch.int64).to(cuda), align_corners=True)


# ---------------------------------------------------------------------------------------------------
# Every kernel the host code can choose, against the oracle evaluated in float64. The dispatch rule
# (csrc/weighted_ce.cu, weighted_ce()): factor 4 with C <= 8 and aligned label / weight maps takes the
# factor-4 kernel (exact instantiations for C = 2 and C = 6, C read at run time up to 8, with or without
# the gradient); everything else up to C = 64 takes the general kernel, which keeps the up-sampled logits
# in registers up to C = 8, sums the gradient in private shared-memory accumulators while they fit and
# scatters it with shared atomics beyond.
LOSS_TOL = 1e-5          # relative, loss vs float64
GRAD_TOL = 1e-5          # of the float64 gradient's largest magnitude
NEAR_TIE = 1e-5          # up-sampled float64 logits this close may legitimately change the fp32 arg-max
UPSTREAM = 0.7           # the gradient that flows into the loss


def _case(B, C, lh, lw, s, *, seed, scale=2.0, weighted=True, class_weight=False, ignore_index=255):
    """float32 CPU inputs: logits, (B,1,H,W) int64 labels with ignored bands crossing every tile,
    pixel weights and class weights (or None)."""
    g = torch.Generator().manual_seed(seed)
    H, W = s * lh, s * lw
    logits = scale * torch.randn((B, C, lh, lw), generator=g)
    label = torch.randint(0, C, (B, 1, H, W), generator=g)
    if ignore_index != 0:                       # with ignore_index 0 the class-0 pixels are the ignored ones
        label[:, :, 3::7] = ignore_index
        label[:, :, :, 5::11] = ignore_index
    weight = torch.rand((B, H, W), generator=g) if weighted else None
    cw = 0.5 + torch.rand(C, generator=g) if class_weight else None
    return logits, label, weight, cw


def _oracle64(logits, label, weight, cw, ignore_index, loss_weight):
    """-> (loss, acc, d(UPSTREAM * loss)/d logits, up-sampled logits), all from float64 copies."""
    z = logits.double().requires_grad_(True)
    loss, acc, up = OC.decode_head_losses(z, label.long(), None if weight is None else weight.double(),
                                          None if cw is None else cw.double(), ignore_index, loss_weight)
    (UPSTREAM * loss).backward()
    return loss.detach(), acc, z.grad, up.detach()


def _check_loss(loss, ref):
    got, want = float(loss), float(ref)
    assert abs(got - want) <= LOSS_TOL * abs(want) + 1e-12, ("loss", got, want)


def _check_acc(acc, ref, up, label, ignore_index):
    """The fp32 kernel may pick another arg-max than float64 only where the top two are within NEAR_TIE."""
    lab = label[:, 0]
    valid = lab != ignore_index
    n_valid = int(valid.sum())
    n_near = 0
    if up.shape[1] > 1:
        top2 = up.topk(2, dim=1).values
        n_near = int(((top2[:, 0] - top2[:, 1] <= NEAR_TIE) & valid).sum())
    got, want = float(acc.reshape(-1)[0]), float(ref.reshape(-1)[0])
    slack = 100.0 * n_near / max(n_valid, 1)
    assert abs(got - want) <= slack + 1e-6 * abs(want) + 1e-6, ("acc", got, want, n_near, n_valid)


def _check_grad(grad, ref):
    got, want = grad.double().cpu(), ref
    err = float((got - want).abs().max())
    assert err <= GRAD_TOL * float(want.abs().max()) + 1e-12, ("grad", err, float(want.abs().max()))


def _run_both(logits, label, weight=None, cw=None, ignore_index=255, loss_weight=1.0, *, cuda,
              dev_label=None, dev_weight=None):
    """Runs the kernel on the GPU copies (or on the given device label / weight views) once with a
    logits gradient and an upstream gradient != 1, once without a gradient, and checks both runs
    against the float64 oracle."""
    lo, ao, go, up = _oracle64(logits, label, weight, cw, ignore_index, loss_weight)
    dl = label.to(cuda) if dev_label is None else dev_label
    dw = (None if weight is None else weight.to(cuda)) if dev_weight is None else dev_weight
    dcw = None if cw is None else cw.to(cuda)
    zl = logits.to(cuda).requires_grad_(True)
    loss, acc = upsample_cross_entropy(zl, dl, dw, dcw, ignore_index, loss_weight)
    (UPSTREAM * loss).backward()
    _check_loss(loss.detach(), lo)
    _check_acc(acc, ao, up, label, ignore_index)
    _check_grad(zl.grad, go)
    loss, acc = upsample_cross_entropy(logits.to(cuda), dl, dw, dcw, ignore_index, loss_weight)
    _check_loss(loss, lo)
    _check_acc(acc, ao, up, label, ignore_index)


# (B, C, lh, lw): the factor-4 kernel's three class-count instantiations, low-res maps with partial
# tiles in both directions (the tile is 16 cells wide and 8 tall), and 1-pixel rows and columns, where
# every high-res pixel reads a clamped tap
_S4_CASES = [(2, 2, 21, 37), (2, 6, 21, 37)] + [(2, C, 21, 37) for C in (1, 3, 4, 5, 7, 8)] + [
    (3, 6, 1, 1), (3, 2, 1, 1), (2, 5, 1, 1), (2, 6, 1, 19), (2, 6, 23, 1), (2, 2, 1, 40), (2, 8, 17, 1),
    (1, 6, 8, 16)]


@pytest.mark.parametrize("B,C,lh,lw", _S4_CASES, ids=[f"B{b}-C{c}-{h}x{w}" for b, c, h, w in _S4_CASES])
def test_factor4_kernel_matches_float64_oracle(cuda, B, C, lh, lw):
    logits, label, weight, cw = _case(B, C, lh, lw, 4, seed=100 * C + lh + lw)
    _run_both(logits, label, weight, cw, cuda=cuda)


# (B, C, lh, lw, factor): C <= 8 at factors other than 4 (odd factors exercise the fp32 source-index
# arithmetic against float64), 9 <= C <= 15 (private accumulators), 16 <= C <= 64 (shared atomics),
# including cfg4's geometry (33 classes, 30x30 -> 120x120, batch 64)
_GENERAL_CASES = [(2, 6, 21, 37, 1), (2, 6, 21, 37, 2), (2, 6, 21, 37, 3), (2, 6, 21, 37, 5), (2, 2, 13, 9, 3),
                  (2, 12, 21, 37, 4), (1, 12, 1, 1, 4), (64, 33, 30, 30, 4), (2, 64, 21, 37, 2)]


@pytest.mark.parametrize("B,C,lh,lw,s", _GENERAL_CASES,
                         ids=[f"B{b}-C{c}-{h}x{w}-x{s}" for b, c, h, w, s in _GENERAL_CASES])
def test_general_kernel_matches_float64_oracle(cuda, B, C, lh, lw, s):
    logits, label, weight, cw = _case(B, C, lh, lw, s, seed=1000 + 10 * C + s)
    _run_both(logits, label, weight, cw, cuda=cuda)


def test_more_than_64_classes_raise(cuda):
    logits, label, _, _ = _case(1, 65, 4, 4, 2, seed=3)
    with pytest.raises(ops.PfstError):
        upsample_cross_entropy(logits.to(cuda), label.to(cuda))


# class weights, a loss weight != 1 and the ignore indices the reference's CrossEntropyLoss users pass,
# on the factor-4 kernel (C = 6, C = 5) and the general kernel (C = 6 at factor 2, C = 12)
_OPTIONS = {"class_weight": dict(class_weight=True), "loss_weight": dict(loss_weight=0.4),
            "ignore0": dict(ignore_index=0), "ignore-100": dict(ignore_index=-100),
            "all": dict(class_weight=True, loss_weight=2.5, ignore_index=-100)}


@pytest.mark.parametrize("C,s", [(6, 4), (5, 4), (6, 2), (12, 4)])
@pytest.mark.parametrize("option,label_dtype", [(o, d) for o in _OPTIONS for d in (torch.int64, torch.uint8)
                                                if d == torch.int64 or _OPTIONS[o].get("ignore_index", 0) >= 0])
def test_options_match_float64_oracle(cuda, C, s, option, label_dtype):
    opt = dict(_OPTIONS[option])
    loss_weight = opt.pop("loss_weight", 1.0)
    logits, label, weight, cw = _case(2, C, 21, 37, s, seed=7 * C + s, **opt)
    _run_both(logits, label, weight, cw, opt.get("ignore_index", 255), loss_weight, cuda=cuda,
              dev_label=label.to(label_dtype).to(cuda))


def _view_at(t, offset, cuda):
    """A contiguous device copy of t that starts `offset` elements into its storage."""
    flat = torch.empty(t.numel() + offset, dtype=t.dtype, device=cuda)
    v = flat[offset:].view(t.shape)
    v.copy_(t)
    return v


# the factor-4 kernel reads label rows with 16-byte (int64) / 2-byte (uint8) loads and weights with
# 8-byte loads: views that are not aligned to that (a contiguous view at an odd storage offset) must take
# the general kernel and give the same results
_LAYOUTS = {"u8": (torch.uint8, 0, 0), "u8_odd": (torch.uint8, 1, 0), "u8_odd3": (torch.uint8, 3, 0),
            "i64": (torch.int64, 0, 0), "i64_odd": (torch.int64, 1, 0), "weight_odd": (torch.int64, 0, 1),
            "u8_weight_odd": (torch.uint8, 0, 1), "i64_weight_odd": (torch.int64, 1, 3)}


@pytest.mark.parametrize("C", [6, 2, 5])
@pytest.mark.parametrize("layout", list(_LAYOUTS))
def test_label_and_weight_layouts_match_float64_oracle(cuda, C, layout):
    dtype, lab_off, w_off = _LAYOUTS[layout]
    logits, label, weight, _ = _case(2, C, 21, 37, 4, seed=50 + C)
    dl = _view_at(label.to(dtype), lab_off, cuda)
    dw = _view_at(weight, w_off, cuda)
    # the factor-4 kernel needs label maps aligned to two elements and weights to 8 bytes
    assert (dl.data_ptr() % (2 * dl.element_size()) != 0) == bool(lab_off % 2)
    assert (dw.data_ptr() % 8 != 0) == bool(w_off % 2)
    _run_both(logits, label, weight, cuda=cuda, dev_label=dl, dev_weight=dw)


def test_full_size_cfg3_matches_float64_oracle(cuda):
    """cfg3's decode-head loss: two classes, 256x256 logits -> 1024x1024 labels, pixel weights."""
    logits, label, weight, _ = _case(4, 2, 256, 256, 4, seed=33)
    label[:, :, :40] = 255                      # a wide ignored band, as the pseudo-label weights leave
    label[:, :, -24:] = 255
    _run_both(logits, label, weight, cuda=cuda)


def test_empty_batch_matches_reference(cuda):
    """B = 0: the reference's loss is the mean of no pixels (NaN) and its accuracy is 0."""
    logits, label, weight, _ = _case(0, 6, 8, 8, 4, seed=1)
    lo, ao, _ = OC.decode_head_losses(logits.double(), label, weight, None, 255, 1.0)
    assert torch.isnan(lo) and float(ao) == 0.0
    zl = logits.to(cuda).requires_grad_(True)
    loss, acc = upsample_cross_entropy(zl, label.to(cuda), weight.to(cuda))
    (UPSTREAM * loss).backward()
    assert torch.isnan(loss).item() and float(acc) == 0.0
    assert zl.grad.shape == logits.shape
    # through the C ABI with real (non-null) buffers: out2 is written, not left as it was
    stats = torch.empty(4, dtype=torch.float64, device=cuda)
    out2 = torch.full((2,), 7.0, device=cuda)
    buf = torch.zeros(64, device=cuda)
    lab = torch.zeros(64, dtype=torch.int64, device=cuda)
    for lwt in (1.0, 0.4):
        out2.fill_(7.0)
        _lib.call("pfst_weighted_ce", buf.data_ptr(), lab.data_ptr(), _lib.DT_I64, buf.data_ptr(), None, 0, 6, 8, 8,
                  32, 32, 255, lwt, buf.data_ptr(), stats.data_ptr(), out2.data_ptr(), ops._stream())
        res = out2.cpu()
        assert torch.isnan(res[0]) and float(res[1]) == 0.0, res
    assert torch.equal(buf.cpu(), torch.zeros(64))          # nothing else is written


# confident predictions: logits ten times the other cases' scale and every valid pixel labelled with the
# arg-max of the up-sampled float64 logits, so that most per-pixel losses are << 1e-2. There even the
# fp32 oracle is off from float64 by more than 1e-5 of many pixels' loss (the soft-max sum 1 + eps
# rounds), so the kernel is held to max(1e-5 relative, 4 x the fp32 oracle's own error)
@pytest.mark.parametrize("C,s", [(2, 4), (6, 4), (5, 4), (6, 2), (12, 4)])
def test_confident_logits_loss_error(cuda, C, s):
    logits, _, weight, _ = _case(2, C, 32, 48, s, seed=90 + C, scale=20.0)
    up64 = torch.nn.functional.interpolate(logits.double(), scale_factor=s, mode="bilinear", align_corners=False)
    label = up64.argmax(1, keepdim=True)
    label[:, :, 3::7] = 255
    lo, ao, go, up = _oracle64(logits, label, weight, None, 255, 1.0)
    l32, _, _ = OC.decode_head_losses(logits, label, weight, None, 255, 1.0)
    err32 = abs(float(l32) - float(lo))
    zl = logits.to(cuda).requires_grad_(True)
    loss, acc = upsample_cross_entropy(zl, label.to(cuda), weight.to(cuda))
    (UPSTREAM * loss).backward()
    err = abs(float(loss.detach()) - float(lo))
    assert err <= max(LOSS_TOL * abs(float(lo)), 4 * err32), (err, err32, float(lo))
    _check_acc(acc, ao, up, label, 255)
    _check_grad(zl.grad, go)


# one representative call per row of the dispatch rule and the kernel it must launch (the shipped
# defaults: fast soft-max, 8-row tiles)
_DISPATCH = [
    ("factor 4, C = 6", dict(C=6), "weighted_ce_s4_kernel<6, true, true, true, 8, long>"),
    ("factor 4, C = 2", dict(C=2), "weighted_ce_s4_kernel<2, true, true, true, 8, long>"),
    ("factor 4, C = 5", dict(C=5), "weighted_ce_s4_kernel<8, false, true, true, 8, long>"),
    ("factor 4, no gradient", dict(C=6, grad=False), "weighted_ce_s4_kernel<6, true, true, false, 8, long>"),
    ("factor 4, C = 2, no gradient", dict(C=2, grad=False),
     "weighted_ce_s4_kernel<2, true, true, false, 8, long>"),
    ("factor 4, C = 3, no gradient", dict(C=3, grad=False),
     "weighted_ce_s4_kernel<8, false, true, false, 8, long>"),
    ("factor 4, uint8", dict(C=6, dtype=torch.uint8),
     "weighted_ce_s4_kernel<6, true, true, true, 8, unsigned char>"),
    ("factor 2, C = 6", dict(C=6, s=2), "weighted_ce_kernel<true, true, long>"),
    ("factor 4, odd uint8 view", dict(C=6, dtype=torch.uint8, lab_off=1),
     "weighted_ce_kernel<true, true, unsigned char>"),
    ("factor 4, 8-byte aligned int64 view", dict(C=6, lab_off=1), "weighted_ce_kernel<true, true, long>"),
    ("factor 4, 4-byte aligned weight view", dict(C=2, w_off=1), "weighted_ce_kernel<true, true, long>"),
    ("C = 12", dict(C=12), "weighted_ce_kernel<false, true, long>"),
    ("C = 33", dict(C=33), "weighted_ce_kernel<false, false, long>"),
    ("C = 64", dict(C=64, s=2), "weighted_ce_kernel<false, false, long>"),
]


def _kernel_name(name):
    """'void pfst::k<(int)6, (bool)1>(...)' or 'void pfst::k<6, true>(...)' -> 'k<6, true>'"""
    name = re.sub(r"\(bool\)1", "true", re.sub(r"\(bool\)0", "false", name))
    name = re.sub(r"\((?:int|long)\)", "", name)
    return name.split("pfst::", 1)[-1].split("(", 1)[0]


@pytest.mark.skipif(any(k.startswith("PFST_CE_") for k in os.environ),
                    reason="a PFST_CE_* switch changes the dispatch")
def test_each_dispatch_row_launches_its_kernel(cuda):
    from torch.profiler import ProfilerActivity, profile
    for what, kw, want in _DISPATCH:
        logits, label, weight, _ = _case(2, kw["C"], 21, 37, kw.get("s", 4), seed=5)
        dl = _view_at(label.to(kw.get("dtype", torch.int64)), kw.get("lab_off", 0), cuda)
        dw = _view_at(weight, kw.get("w_off", 0), cuda)
        z = logits.to(cuda).requires_grad_(kw.get("grad", True))
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            upsample_cross_entropy(z, dl, dw)
            torch.cuda.synchronize()
        names = [_kernel_name(e.name) for e in prof.events() if "weighted_ce" in e.name]
        assert names == [want], (what, names)
    logits, label, _, _ = _case(1, 65, 4, 4, 2, seed=3)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        with pytest.raises(ops.PfstError):          # C > 64: refused before any launch
            upsample_cross_entropy(logits.to(cuda), label.to(cuda))
        torch.cuda.synchronize()
    assert not [e.name for e in prof.events() if "weighted_ce" in e.name]
