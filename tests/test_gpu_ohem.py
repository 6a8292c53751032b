"""OHEM pixel sampler on the device (pfst_ohem_weight, csrc/ohem.cu) and the decode-head loss with a sampler.

Weight maps are compared with oracle/ohem.py run on float64 up-sampled logits: a pixel's weight may differ only
where its float64 key lies within NEAR relative of the float64 threshold (each case prints how many such pixels
it has). The kernel's own keys and order statistic are checked exactly: the returned kth is element k of
torch.sort of its keys over the valid pixels, and the map is exactly what those keys and kth imply, ties at
the top-k boundary going to the lowest flat indices."""
import math
from types import SimpleNamespace

import pytest
import torch
import torch.nn.functional as F

from oracle import ohem as OO, weighted_ce as OC
from pfst_b200 import ops
from pfst_b200._lib import PfstError
from pfst_b200.losses import OHEMPixelSampler, decode_head_losses
from tests.test_gpu_weighted_ce import _kernel_name, _view_at

pytestmark = pytest.mark.gpu
NEAR = 1e-6
THRESH = 0.7
DTYPES = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}


def _inputs(B, C, lh, lw, s, *, seed, ignore_index=255, scale=2.0):
    g = torch.Generator().manual_seed(seed)
    logits = scale * torch.randn((B, C, lh, lw), generator=g)
    label = torch.randint(0, C, (B, 1, s * lh, s * lw), generator=g)
    label[:, :, 3::7] = ignore_index
    label[:, :, :, 5::11] = ignore_index
    return logits, label


def _head(ignore_index=255, loss_weight=1.0, class_weight=None):
    return SimpleNamespace(ignore_index=ignore_index, loss_decode=OO.CrossEntropyLoss(loss_weight, class_weight))


def _keys64(z, label, thresh, ignore_index, loss_weight, cw):
    """float64 keys of every pixel (the sampler's definitions) and the valid mask."""
    up = F.interpolate(z.double(), label.shape[2:], None, "bilinear", False)
    lab = label[:, 0].long()
    valid = lab != ignore_index
    tgt = torch.where(valid, lab, torch.zeros_like(lab))
    if thresh is not None:
        key = torch.softmax(up, 1).gather(1, tgt[:, None])[:, 0]
    else:
        w = None if cw is None else torch.tensor(cw, dtype=torch.float64)
        key = loss_weight * F.cross_entropy(up, lab, weight=w, reduction="none", ignore_index=ignore_index)
    return up, key, valid


def _oracle_map(z, label, thresh, min_kept, ignore_index, loss_weight, cw):
    """-> (float64 oracle map, float64 keys, valid, float64 threshold or None when every valid pixel is kept)."""
    up, key, valid = _keys64(z, label, thresh, ignore_index, loss_weight, cw)
    head = OO.Head(ignore_index, loss_weight, cw)
    want = OO.OHEMPixelSampler(head, thresh=thresh, min_kept=min_kept).sample(up, label.long())
    n, kept = int(valid.sum()), min_kept * z.shape[0]
    srt = key[valid].sort()[0]
    if n == 0:
        thr = None
    elif thresh is not None:
        kth = float(srt[min(kept, n - 1)])
        thr = thresh if thresh > kth else kth
    else:
        thr = float(srt[n - kept]) if kept < n else None
    return want, key, valid, thr


def _check_vs_oracle(w, want, key, thr, what):
    diff = w.cpu().double() != want
    near = torch.zeros_like(diff)
    if thr is not None and math.isnan(thr):               # the boundary is a tie among NaN keys
        near = torch.isnan(key)
    elif thr is not None and math.isfinite(thr):
        near = (key - thr).abs() <= NEAR * abs(thr)
    assert not bool((diff & ~near).any()), (what, int(diff.sum()), int((diff & ~near).sum()))
    print(f"OHEM {what}: pixels {diff.numel()}, within {NEAR:g} of the threshold {int(near.sum())}, "
          f"differing {int(diff.sum())}")


def _ordered(k):
    """int64 order of fp32 keys as the kernel orders them: NaN largest, -0 == +0."""
    k = torch.where(k == 0, torch.zeros_like(k), k)
    u = k.view(torch.int32).to(torch.int64) & 0xffffffff
    o = torch.where(u >= 0x80000000, (~u) & 0xffffffff, u | 0x80000000)
    return torch.where(torch.isnan(k), torch.full_like(o, 0xffffffff), o)


def _check_internal(w, kth, keys, label, thresh, min_kept, ignore_index, what):
    """The map is exactly what the kernel's own keys and kth imply."""
    valid = label[:, 0] != ignore_index
    n, kept = int(valid.sum()), min_kept * label.shape[0]
    kth = kth.cpu()
    if n == 0:
        assert float(kth) == 0.0 and int(w.sum()) == 0, what
        return
    o = _ordered(keys.cpu())
    ov = o[valid.cpu()]
    srt = ov.sort()[0]
    k = min(kept, n - 1) if thresh is not None else max(n - kept, 0)
    assert int(_ordered(kth)[0]) == int(srt[k]), (what, "kth", float(kth), k)
    vm = valid.cpu()
    if thresh is not None:
        t32 = torch.tensor(thresh, dtype=torch.float32)
        th = t32 if bool(t32 > kth[0]) else kth[0]
        want = vm & (keys.cpu() < th)
    else:
        T = int(_ordered(kth)[0])
        gt = vm & (o > T)
        eq = (vm & (o == T)).reshape(-1)
        need = min(kept, n) - int(gt.sum())
        first = eq & (torch.cumsum(eq.to(torch.int64), 0) <= need)
        want = gt | first.reshape(gt.shape)
        assert int(w.sum()) == min(kept, n), (what, int(w.sum()), min(kept, n))
    assert torch.equal(w.cpu(), want.float()), (what, int((w.cpu() != want.float()).sum()))


def _run(cuda, *, mode, s, C, B=2, lh=21, lw=37, label_dtype=torch.int64, dtype="f32", min_kept=None,
         ignore_index=255, loss_weight=1.0, class_weight=False, offset=0, seed=11):
    thresh = THRESH if mode == "thresh" else None
    logits, label = _inputs(B, C, lh, lw, s, seed=seed, ignore_index=ignore_index)
    z16 = logits.to(DTYPES[dtype])
    cw = [0.5 + 0.1 * (c % 7) for c in range(C)] if class_weight else None
    n = int((label != ignore_index).sum())
    mk = min_kept if min_kept is not None else max(2, n // (4 * B))
    what = f"{mode} s={s} C={C} {dtype} {label_dtype} min_kept={mk} n={n} off={offset}"
    zd = _view_at(z16, offset, cuda)
    ld = _view_at(label.to(label_dtype), offset, cuda)
    cwd = None if cw is None else torch.tensor(cw, dtype=torch.float32, device=cuda)
    w, kth, keys = ops.ohem_weight(zd, ld, thresh=thresh, min_kept=mk, ignore_index=ignore_index,
                                   class_weight=cwd, loss_weight=loss_weight, want_keys=True)
    want, key64, valid, thr = _oracle_map(z16.double(), label, thresh, mk, ignore_index, loss_weight, cw)
    _check_vs_oracle(w, want, key64, thr, what)
    _check_internal(w, kth, keys, ld, thresh, mk, ignore_index, what)
    return w


CASES = []
for _mode in ("thresh", "topk"):
    for _s in (1, 2, 4, 8):
        for _C in (2, 6, 33):
            CASES.append(dict(mode=_mode, s=_s, C=_C))
    CASES += [
        dict(mode=_mode, s=4, C=6, label_dtype=torch.uint8),
        dict(mode=_mode, s=1, C=6, label_dtype=torch.uint8, dtype="bf16"),
        dict(mode=_mode, s=4, C=6, dtype="bf16"),
        dict(mode=_mode, s=4, C=33, dtype="f16"),
        dict(mode=_mode, s=8, C=6, dtype="f16", label_dtype=torch.uint8),
        dict(mode=_mode, s=4, C=6, class_weight=True, loss_weight=0.4),
        dict(mode=_mode, s=2, C=6, class_weight=True, loss_weight=2.5, ignore_index=0),
        dict(mode=_mode, s=4, C=6, min_kept=2),                     # thresh wins
        dict(mode=_mode, s=4, C=6, min_kept=100000),                # min_kept above the valid count
        dict(mode=_mode, s=1, C=2, min_kept=100000),
        dict(mode=_mode, s=4, C=6, offset=1),                       # odd-offset views
        dict(mode=_mode, s=4, C=6, offset=3, label_dtype=torch.uint8, dtype="bf16"),
        dict(mode=_mode, s=4, C=6, B=1, lh=1, lw=1),
    ]


@pytest.mark.parametrize("kw", CASES, ids=lambda kw: "-".join(f"{k}={v}" for k, v in kw.items()))
def test_weight_map_matches_float64_oracle(cuda, kw):
    _run(cuda, **kw)


def test_min_threshold_wins_when_min_kept_is_large(cuda):
    """With min_kept above n the k-th key is the largest; when it exceeds thresh it is the threshold, and every
    valid pixel but those with the largest key is kept."""
    logits, label = _inputs(2, 2, 21, 37, 4, seed=4, scale=4.0)     # confident logits: the largest key is > 0.7
    w, kth, keys = ops.ohem_weight(logits.to(cuda), label.to(cuda), thresh=THRESH, min_kept=100000, want_keys=True)
    valid = (label[:, 0] != 255).to(cuda)
    assert float(kth) == float(keys[valid].max()) and float(kth) > THRESH
    assert torch.equal(w, (valid & (keys < kth)).float())


@pytest.mark.parametrize("mode", ["thresh", "topk"])
def test_constant_logits_all_ties_take_lowest_indices(cuda, mode):
    B, C, H, W = 2, 6, 40, 52
    label = torch.randint(0, C, (B, 1, H, W), generator=torch.Generator().manual_seed(1))
    label[:, :, 5::9] = 255
    z = torch.zeros((B, C, H // 4, W // 4), device=cuda)
    thresh = None if mode == "topk" else THRESH
    w, kth, keys = ops.ohem_weight(z, label.to(cuda), thresh=thresh, min_kept=300, want_keys=True)
    valid = (label[:, 0] != 255).reshape(-1)
    if mode == "topk":
        want = valid & (torch.cumsum(valid.long(), 0) <= 600)     # the first 600 valid pixels in flat order
    else:
        want = valid                                               # every key 1/6 < 0.7
    assert torch.equal(w.cpu().reshape(-1), want.float())
    _check_internal(w, kth, keys, label.to(cuda), thresh, 300, 255, mode)


@pytest.mark.parametrize("mode", ["thresh", "topk"])
def test_nan_and_inf_logits_follow_the_oracle(cuda, mode):
    logits, label = _inputs(2, 6, 10, 12, 4, seed=9)
    logits[0, 1, 2, 3] = float("nan")
    logits[1, 2, 4, 5] = float("inf")
    logits[1, 3, 6, 7] = float("-inf")
    logits[0, :, 8, 9] = float("-inf")
    thresh = THRESH if mode == "thresh" else None
    for mk in (5, 400):
        w, kth, keys = ops.ohem_weight(logits.to(cuda), label.to(cuda), thresh=thresh, min_kept=mk, want_keys=True)
        want, key64, valid, thr = _oracle_map(logits.double(), label, thresh, mk, 255, 1.0, None)
        assert torch.equal(torch.isnan(keys.cpu()), torch.isnan(key64.float()))
        _check_internal(w, kth, keys, label.to(cuda), thresh, mk, 255, f"{mode} nan mk={mk}")
        if mode == "topk":          # NaN keys are the largest: they are kept first
            nan = torch.isnan(key64) & valid
            assert int(w.cpu()[nan].sum()) == min(int(nan.sum()), 2 * mk)
        _check_vs_oracle(w, want, key64, thr, f"{mode} nan/inf mk={mk}")


@pytest.mark.parametrize("mode", ["thresh", "topk"])
def test_empty_batch_and_all_ignored_give_zero_maps(cuda, mode):
    thresh = THRESH if mode == "thresh" else None
    w, kth, _ = ops.ohem_weight(torch.zeros((0, 6, 8, 8), device=cuda), torch.zeros((0, 1, 32, 32), dtype=torch.int64,
                                device=cuda), thresh=thresh, min_kept=10)
    assert w.shape == (0, 32, 32) and float(kth) == 0.0
    z, label = _inputs(2, 6, 8, 8, 4, seed=2)
    label[:] = 255
    w, kth, _ = ops.ohem_weight(z.to(cuda), label.to(cuda), thresh=thresh, min_kept=10)
    assert int(w.count_nonzero()) == 0 and float(kth) == 0.0
    want = OO.OHEMPixelSampler(OO.Head(), thresh=thresh, min_kept=10).sample(
        F.interpolate(z, (32, 32), None, "bilinear", False), label)
    assert int(want.count_nonzero()) == 0


def test_unsupported_geometries_raise_before_launch(cuda, monkeypatch):
    from pfst_b200 import _lib
    launched = []
    monkeypatch.setattr(_lib, "call", lambda name, *a: launched.append(name))
    z = torch.randn(2, 6, 10, 10, device=cuda)
    with pytest.raises(PfstError):                               # not an integer factor
        ops.ohem_weight(z, torch.zeros(2, 1, 25, 25, dtype=torch.int64, device=cuda), thresh=0.7)
    with pytest.raises(PfstError):                               # different factors in y and x
        ops.ohem_weight(z, torch.zeros(2, 1, 20, 40, dtype=torch.int64, device=cuda), thresh=0.7)
    with pytest.raises(ValueError):
        ops.ohem_weight(z, torch.zeros(2, 1, 40, 40, dtype=torch.int64, device=cuda), min_kept=1)
    with pytest.raises(TypeError):
        ops.ohem_weight(z.double(), torch.zeros(2, 1, 40, 40, dtype=torch.int64, device=cuda))
    with pytest.raises(TypeError):
        ops.ohem_weight(z, torch.zeros(2, 1, 40, 40, dtype=torch.int32, device=cuda))
    s = OHEMPixelSampler(_head(), thresh=0.7, min_kept=10)
    with pytest.raises(PfstError):
        decode_head_losses(z, torch.zeros(2, 1, 40, 40, dtype=torch.int64, device=cuda), sampler=s,
                           align_corners=True)
    assert launched == []


# ------------------------------------------------------------------------------------------------ composition
def _sampler(mode, loss_weight=1.0, cw=None, min_kept=200):
    return OHEMPixelSampler(_head(255, loss_weight, cw), thresh=THRESH if mode == "thresh" else None, min_kept=min_kept)


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("mode", ["thresh", "topk"])
def test_fused_loss_equals_ce_fed_the_map(cuda, mode, dtype):
    cw = [1.0, 2.0, 0.5, 1.0, 1.5, 0.8]
    S = _sampler(mode, 0.6, cw)
    logits, label = _inputs(2, 6, 32, 48, 4, seed=21)
    z0 = logits.to(DTYPES[dtype]).to(cuda)
    dl = label.to(cuda)
    cwd = torch.tensor(cw, device=cuda)
    W, _, _ = ops.ohem_weight(z0, dl, thresh=S.thresh, min_kept=S.min_kept, class_weight=cwd, loss_weight=0.6)
    res = []
    for kw in (dict(sampler=S, seg_weight=torch.rand(2, 128, 192, device=cuda)), dict(seg_weight=W)):
        z = z0.clone().requires_grad_(True)
        out = decode_head_losses(z, dl, class_weight=cwd, loss_weight=0.6, **kw)
        (0.7 * out["loss_ce"]).backward()
        res.append((out["loss_ce"].detach(), out["acc_seg"], z.grad))
    (l1, a1, g1), (l2, a2, g2) = res
    assert torch.equal(l1, l2) and torch.equal(a1, a2)
    # the gradient tile borders meet in float atomics, whose order varies from launch to launch
    assert g1.dtype == z0.dtype and torch.allclose(g1.float(), g2.float(), rtol=0,
                                                  atol=1e-6 * float(g2.float().abs().max()))
    # the loss against the float64 oracle on the same map
    ref, _, _ = OC.decode_head_losses(z0.double().cpu(), label, W.double().cpu(), cwd.double().cpu(), 255, 0.6)
    assert abs(float(l1) - float(ref)) <= 1e-5 * abs(float(ref))
    # the reference op sequence (float64): its map differs from W only near the threshold
    head = OO.Head(255, 0.6, cw)
    _, _, w64 = OO.decode_head_losses(z0.double().cpu(), label, OO.OHEMPixelSampler(head, S.thresh, S.min_kept),
                                      torch.tensor(cw, dtype=torch.float64), 255, 0.6)
    _, key64, _, thr = _oracle_map(z0.double().cpu(), label, S.thresh, S.min_kept, 255, 0.6, cw)
    _check_vs_oracle(W, w64, key64, thr, f"decode_head_losses {mode} {dtype}")


@pytest.mark.parametrize("mode", ["thresh", "topk"])
def test_sample_on_torch_upsampled_logits_agrees(cuda, mode):
    S = _sampler(mode)
    logits, label = _inputs(2, 6, 32, 48, 4, seed=22)
    z, dl = logits.to(cuda), label.to(cuda)
    W, _, _ = ops.ohem_weight(z, dl, thresh=S.thresh, min_kept=S.min_kept)
    up = F.interpolate(z, dl.shape[2:], None, "bilinear", False)
    got = S.sample(up, dl)
    _, key64, _, thr = _oracle_map(logits.double(), label, S.thresh, S.min_kept, 255, 1.0, None)
    _check_vs_oracle(got, W.cpu().double(), key64, thr, f"sample(up) vs low-res {mode}")


@pytest.mark.parametrize("mode", ["thresh", "topk"])
def test_forward_with_sampler_is_graph_capturable(cuda, mode):
    S = _sampler(mode, 0.5, [1.0, 2.0, 0.5, 1.0, 1.5, 0.8])
    cwd = torch.tensor([1.0, 2.0, 0.5, 1.0, 1.5, 0.8], device=cuda)
    z_s = torch.zeros(2, 6, 32, 48, device=cuda)
    l_s = torch.zeros(2, 1, 128, 192, dtype=torch.int64, device=cuda)
    logits, label = _inputs(2, 6, 32, 48, 4, seed=30)
    z_s.copy_(logits)
    l_s.copy_(label)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        decode_head_losses(z_s, l_s, sampler=S, class_weight=cwd, loss_weight=0.5)    # warm-up
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = decode_head_losses(z_s, l_s, sampler=S, class_weight=cwd, loss_weight=0.5)
    for seed in (31, 32):
        logits, label = _inputs(2, 6, 32, 48, 4, seed=seed)
        z_s.copy_(logits)
        l_s.copy_(label)
        g.replay()
        eager = decode_head_losses(logits.to(cuda), label.to(cuda), sampler=S, class_weight=cwd, loss_weight=0.5)
        torch.cuda.synchronize()
        assert torch.equal(out["loss_ce"], eager["loss_ce"]) and torch.equal(out["acc_seg"], eager["acc_seg"])


_PROFILE_SCRIPT = """
import json, sys
sys.path.insert(0, {root!r})
import torch
from torch.profiler import ProfilerActivity, profile
from tests.test_gpu_ohem import _inputs, _sampler
from pfst_b200.losses import decode_head_losses
cuda = torch.device("cuda:0")
S = _sampler({mode!r})
logits, label = _inputs(2, 6, 32, 48, 4, seed=40)
z, dl = logits.to(cuda), label.to(cuda)
decode_head_losses(z, dl, sampler=S)
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    decode_head_losses(z, dl, sampler=S)
    torch.cuda.synchronize()
print(json.dumps([e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]))
"""


@pytest.mark.parametrize("mode", ["thresh", "topk"])
def test_profiler_lists_only_the_sampler_and_ce_kernels(cuda, mode):
    """Run in a process of its own: a torch.profiler session here left later sessions of the same process without
    the kernels the autograd thread launches."""
    import json
    import subprocess
    import sys
    from pathlib import Path
    root = str(Path(__file__).resolve().parent.parent)
    res = subprocess.run([sys.executable, "-c", _PROFILE_SCRIPT.format(root=root, mode=mode)], capture_output=True,
                         text=True, cwd=root, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    names = [n for n in json.loads(res.stdout.strip().splitlines()[-1]) if "memset" not in n.lower()]
    short = [_kernel_name(n) for n in names]
    assert all("pfst::" in n for n in names), names
    assert not [n for n in names if "sort" in n.lower() or "softmax" in n.lower()]
    want = ["ohem_key_kernel", "ohem_hist_kernel", "ohem_scan_kernel", "ohem_hist_kernel", "ohem_scan_kernel",
            "ohem_hist_kernel", "ohem_scan_kernel"]
    want += ["ohem_tie_count_kernel", "ohem_tie_scan_kernel"] if mode == "topk" else []
    want += ["ohem_weight_kernel", "weighted_ce_s4_kernel"]
    assert [n.split("<")[0] for n in short] == want, short
