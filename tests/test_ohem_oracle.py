"""The OHEM pixel sampler's CPU oracle (oracle/ohem.py) and the checks of the product's sampler that run before
any launch. Runs without a GPU. The oracle is pinned bit for bit against the reference's own OHEMPixelSampler
when PFST_REFERENCE names a checkout."""
import re
from types import SimpleNamespace

import pytest
import torch
import torch.nn as nn

from oracle import ohem as OO
from pfst_b200 import ops
from pfst_b200._lib import PfstError
from pfst_b200.losses import OHEMPixelSampler, decode_head_losses
from pfst_b200.registry import PIXEL_SAMPLERS, build_pixel_sampler
from tests.golden import ref_loader as R

SAMPLER_FILE = "rsiseg/core/seg/sampler/ohem_pixel_sampler.py"


def _inputs(B=2, C=5, H=9, W=11, seed=0):
    g = torch.Generator().manual_seed(seed)
    logit = 2.0 * torch.randn((B, C, H, W), generator=g)
    label = torch.randint(0, C, (B, 1, H, W), generator=g)
    label[:, :, 2] = 255
    return logit, label


def _reference_sampler_module():
    """The reference's OHEMPixelSampler module, loaded by path, or a skip reason."""
    if not R.available():
        return None, "unpinned: PFST_REFERENCE names no reference checkout"
    if not (R.REF_ROOT / SAMPLER_FILE).exists():
        return None, f"unpinned: {SAMPLER_FILE} is not in the reference checkout"

    class _Reg:
        def register_module(self, *a, **k):
            return lambda cls: cls

    R._stub("_pfst_ref_seg")
    R._stub("_pfst_ref_seg.builder", PIXEL_SAMPLERS=_Reg())
    R._stub("_pfst_ref_seg.sampler")
    base = R.REF_ROOT / "rsiseg/core/seg/sampler/base_pixel_sampler.py"
    if base.exists():
        R._load("_pfst_ref_seg.sampler.base_pixel_sampler", "rsiseg/core/seg/sampler/base_pixel_sampler.py")
    else:
        R._stub("_pfst_ref_seg.sampler.base_pixel_sampler", BasePixelSampler=object)
    return R._load("_pfst_ref_seg.sampler.ohem_pixel_sampler", SAMPLER_FILE), None


@pytest.mark.parametrize("thresh,min_kept", [(0.7, 10), (0.7, 100000), (0.3, 4), (None, 10), (None, 100000)])
def test_oracle_equals_reference_sampler(thresh, min_kept):
    mod, why = _reference_sampler_module()
    if mod is None:
        pytest.skip(why)
    logit, label = _inputs()
    head = OO.Head(255, 0.8, [1.0, 2.0, 0.5, 1.0, 1.5])
    want = mod.OHEMPixelSampler(head, thresh=thresh, min_kept=min_kept).sample(logit, label)
    got = OO.OHEMPixelSampler(head, thresh=thresh, min_kept=min_kept).sample(logit, label)
    assert torch.equal(got, want)


def test_reference_decode_head_replaces_seg_weight_with_the_sampler_map():
    if not R.available():
        pytest.skip("unpinned: PFST_REFERENCE names no reference checkout")
    src = (R.REF_ROOT / "rsiseg/models/decode_heads/decode_head.py").read_text()
    assert re.search(r"seg_weight\s*=\s*self\.sampler\.sample\(\s*seg_logit\s*,\s*seg_label\s*\)", src)


def test_oracle_thresh_mode_rule():
    logit, label = _inputs(seed=1)
    head = OO.Head()
    w = OO.OHEMPixelSampler(head, thresh=0.6, min_kept=5).sample(logit, label)
    prob = torch.softmax(logit, 1).gather(1, label.clamp(max=4)).squeeze(1)
    valid = label.squeeze(1) != 255
    kth = prob[valid].sort()[0][min(5 * 2, int(valid.sum()) - 1)]
    thr = max(float(kth), float(torch.tensor(0.6, dtype=torch.float32)))
    assert torch.equal(w, (valid & (prob < thr)).float())


def test_oracle_topk_mode_keeps_min_kept_per_image():
    logit, label = _inputs(seed=2)
    valid = label.squeeze(1) != 255
    for min_kept in (3, 50, 10 ** 6):
        w = OO.OHEMPixelSampler(OO.Head(), min_kept=min_kept).sample(logit, label)
        assert int(w.sum()) == min(2 * min_kept, int(valid.sum()))
        assert not bool((w[~valid] != 0).any())


def test_nan_keys_sort_largest():
    """The rule the kernels follow for NaN keys is the order torch.sort gives: NaN after every number."""
    keys = torch.tensor([0.5, float("nan"), float("inf"), -1.0, 0.0])
    assert torch.isnan(keys.sort()[0][-1]) and torch.isnan(keys.sort(descending=True)[0][0])
    logit, label = _inputs(B=1, C=3, H=4, W=4, seed=3)
    label[:] = 1
    logit[0, :, 0, 0] = float("nan")            # that pixel's loss is NaN: the top-k keeps it first
    w = OO.OHEMPixelSampler(OO.Head(), min_kept=2).sample(logit, label)
    assert w[0, 0, 0] == 1 and int(w.sum()) == 2


def test_registry_builds_the_sampler_with_its_context():
    head = SimpleNamespace(ignore_index=255, loss_decode=OO.CrossEntropyLoss())
    s = build_pixel_sampler(dict(type="OHEMPixelSampler", thresh=0.7, min_kept=100), context=head)
    assert isinstance(s, OHEMPixelSampler) and s.context is head and s.thresh == 0.7 and s.min_kept == 100
    assert PIXEL_SAMPLERS.get("OHEMPixelSampler") is OHEMPixelSampler


def test_errors_raise_before_any_launch():
    """Every check below runs on CPU tensors: a launch would raise PfstError for them instead."""
    head = SimpleNamespace(ignore_index=255, loss_decode=OO.CrossEntropyLoss())
    for mk in (1, 0, -5):
        with pytest.raises(ValueError):
            OHEMPixelSampler(head, min_kept=mk)
        with pytest.raises(ValueError):
            ops.ohem_weight(torch.zeros(1, 2, 4, 4), torch.zeros(1, 4, 4, dtype=torch.int64), min_kept=mk)
    logit, label = _inputs()
    for bad in (nn.ModuleList([OO.CrossEntropyLoss(), OO.CrossEntropyLoss()]), [OO.CrossEntropyLoss()]):
        s = OHEMPixelSampler(SimpleNamespace(ignore_index=255, loss_decode=bad), min_kept=10)
        with pytest.raises(PfstError, match="several"):
            decode_head_losses(logit, label, sampler=s)
    sig = OO.CrossEntropyLoss()
    sig.use_sigmoid = True
    with pytest.raises(PfstError, match="sigmoid"):
        OHEMPixelSampler(SimpleNamespace(ignore_index=255, loss_decode=sig), thresh=0.7).sample(logit, label)
    s = OHEMPixelSampler(head, thresh=0.7, min_kept=10)
    for dt in (torch.float64, torch.int64, torch.int32):
        with pytest.raises(TypeError):
            decode_head_losses(logit.to(dt), label, sampler=s)
    with pytest.raises(PfstError, match="align_corners"):
        decode_head_losses(logit, label, sampler=s, align_corners=True)
    with pytest.raises(ValueError):                       # sample(): logits already at label resolution
        s.sample(logit[:, :, :4, :5], label)
