"""Host-side logic that needs no GPU: the ClassMix class draw (must consume the global numpy
stream exactly like the reference), the EMA coefficient rule (host-only C entry point), the loss
geometry validation, the registry plug-in mechanics and the byte accounting bench.py reports."""
from pathlib import Path

import numpy as np
import pytest
import torch

from pfst_b200 import ops, registry
from pfst_b200._lib import PfstError
from pfst_b200.step import algorithmic_bytes
from pfst_b200.utils.dacs_transforms import _present_classes, draw_class_choice
from tests.golden import ref_loader as R


def _presence_words(values):
    w = np.zeros(9, dtype=np.uint32)
    for v in values:
        w[v >> 5] |= np.uint32(1) << np.uint32(v & 31)
    return w


@pytest.mark.parametrize("seed", range(6))
def test_class_draw_equals_numpy_choice_on_the_same_stream(seed):
    rs = np.random.RandomState(seed)
    classes = np.array(sorted(rs.choice(256, size=rs.randint(1, 40), replace=False)), dtype=np.int64)
    assert np.array_equal(_present_classes(_presence_words(classes.tolist())), classes)
    a, b = np.random.RandomState(seed), np.random.RandomState(seed)
    got = draw_class_choice(classes, 7, a)
    n = len(classes)
    for i in range(7):
        pick = b.choice(n, int((n + n % 2) / 2), replace=False)          # dacs_transforms.py:115-117
        want = _presence_words(classes[pick].tolist())[:8]
        assert np.array_equal(got[i], want)
    assert a.randint(1 << 30) == b.randint(1 << 30)                      # stream left in the same state


@pytest.mark.parametrize("n,batch", [(1, 3), (2, 64), (6, 8), (33, 64), (200, 5), (256, 2)])
def test_class_draw_from_raw_words_leaves_the_global_stream_where_numpy_would(n, batch):
    """The library replays numpy's shuffles from raw MT19937 words (pfst_classmix_draw): same picks as
    `batch` calls of np.random.choice on the GLOBAL stream, and the stream ends in the same state."""
    rs = np.random.RandomState(n * 1000 + batch)
    classes = np.array(sorted(rs.choice(256, size=n, replace=False)), dtype=np.int64)
    np.random.seed(7 + n)
    got = draw_class_choice(classes, batch, np.random)
    after_got = np.random.randint(1 << 30)
    np.random.seed(7 + n)
    for i in range(batch):
        pick = np.random.choice(n, int((n + n % 2) / 2), replace=False)
        assert np.array_equal(got[i], _presence_words(classes[pick].tolist())[:8])
    assert after_got == np.random.randint(1 << 30)


def test_class_draw_reproduces_reference_get_class_masks():
    """Against the masks get_class_masks draws (tests/golden/reference_live.npz) and, with
    PFST_REFERENCE set, against the reference function itself."""
    g = torch.Generator().manual_seed(0)
    labels = torch.randint(0, 6, (3, 1, 16, 16), generator=g)
    labels[0, 0, :2] = 255
    stored = np.load(Path(__file__).resolve().parent / "golden" / "reference_live.npz")["class_draw_masks"]
    want = [torch.from_numpy(m[None]).long() for m in stored]              # list of (1,1,H,W) int64 masks
    if R.available():
        np.random.seed(42)
        live = R.dacs_transforms().get_class_masks(labels)
        assert all(torch.equal(a, b) for a, b in zip(live, want))
    np.random.seed(42)
    classes = torch.unique(labels).numpy()
    chosen = draw_class_choice(classes, 3, np.random)
    for i in range(3):
        members = [v for v in range(256) if (chosen[i, v >> 5] >> np.uint32(v & 31)) & np.uint32(1)]
        mask = torch.isin(labels[i], torch.tensor(members)).long().unsqueeze(0)
        assert torch.equal(mask, want[i])


def test_ema_coefficients_follow_the_reference_rule():
    for it, alpha in [(1, 0.999), (2, 0.999), (10, 0.999), (999, 0.999), (1000, 0.999), (5000, 0.999), (3, 0.5)]:
        a, b = ops.ema_coeffs(it, alpha)                                  # host-only entry point: no GPU needed
        at = min(1 - 1 / (it + 1), alpha)                                 # pfgst.py:117
        assert a == float(np.float32(at)) and b == float(np.float32(1 - at))


def test_loss_geometry_rejects_unsupported_resampling():
    geo = ops.LossGeometry((8, 6, 128, 128), (8, 512, 64, 64), (8, 1, 512, 512), 0.5, 2)
    assert (geo.gh, geo.gw, geo.up, geo.lscale) == (64, 64, 1, 2.0)
    geo = ops.LossGeometry((64, 33, 30, 30), (64, 512, 15, 15), (64, 1, 120, 120), None, 2)
    assert (geo.gh, geo.up) == (30, 2)
    with pytest.raises(PfstError):
        ops.LossGeometry((1, 6, 100, 100), (1, 512, 64, 64), (1, 1, 512, 512), None, 2)     # 100 is not k*64
    with pytest.raises(PfstError):
        ops.LossGeometry((1, 6, 128, 128), (1, 512, 64, 64), (1, 1, 512, 512), None, 3)     # dilation % up


def test_registry_plugs_into_a_foreign_registry():
    import pfst_b200.losses  # noqa: F401  (registers PFGSTLoss)
    import pfst_b200.uda     # noqa: F401  (registers PFGST)

    class Foreign:                       # the slice of mmcv.utils.Registry that register_into uses
        def __init__(self):
            self.modules = {}

        def register_module(self, name=None, force=False, module=None):
            assert force and module is not None
            self.modules[name] = module

    f = Foreign()
    registry.MODELS.register_into(f)
    assert {"PFGST", "PFGSTLoss"} <= set(f.modules)
    assert registry.UDA.get("PFGST") is f.modules["PFGST"]
    with pytest.raises(KeyError):
        registry.LOSSES.build(dict(type="NoSuchLoss"))


def test_algorithmic_bytes_match_the_survey_table():
    ab = algorithmic_bytes(8, 6, 512, 512, 512, 64, 64, 43579868)
    assert ab["ema"] == 522958416                                         # 12 B x 43 579 868 params
    assert ab["pseudo_label"] == (4 * 6 + 12) * 8 * 512 * 512              # 75.5 MB
    assert ab["neigh_dots"] == 2 * 4 * 512 * 8 * 64 * 64                   # 134.2 MB
    assert ab["class_presence_and_mix"] == 84 * 8 * 512 * 512              # 176.2 MB (presence inside 84 P)
    assert ab["proto_dist_fwd_bwd"] == 3 * 4 * 512 * 8 * 64 * 64           # 201 MB for fwd+bwd together
    assert abs(sum(ab.values()) - 1.3115e9) < 1e6                          # SURVEY 8d: 1.31 GB, nothing else


def test_blur_kernel_size_rule_and_sigma_stream():
    """dacs_transforms.py:93-101: kernel edge ~10 % of the image, odd; one uniform(0.15, 1.15) per call.
    The inactive branches must not touch the numpy stream (and need no GPU)."""
    from oracle import strong_aug as osa
    from pfst_b200.utils import dacs_transforms as T
    for n in list(range(1, 300)) + [512, 1000, 1024, 2048]:
        k = ops.blur_kernel_size(n)
        want = int(np.floor(np.ceil(0.1 * n) - 0.5 + np.ceil(0.1 * n) % 2))
        assert k == want == osa.kernel_size(n) and k % 2 == 1 and k // 2 < max(n, 2)
    x = torch.zeros((2, 3, 8, 8))
    np.random.seed(4)
    before = np.random.get_state()[1].copy()
    assert T.gaussian_blur_batch(0.5, x) is x                 # blur <= 0.5: inactive
    assert T.gaussian_blur(0.2, data=x)[0] is x
    assert T.gaussian_blur(0.9, data=torch.zeros((2, 1, 8, 8)))[0].shape[1] == 1    # not an RGB batch
    assert T.gaussian_blur(0.9, data=None, target=x) == (None, x)
    assert np.array_equal(before, np.random.get_state()[1])
    with pytest.raises(PfstError):                            # active branch on a CPU tensor: loud, no fallback
        T.gaussian_blur(0.9, data=x)


def test_eval_logits_argument_validation_needs_no_gpu():
    z = torch.zeros((1, 6, 4, 4))
    with pytest.raises(PfstError):
        ops.argmax_confusion(z, torch.zeros((1, 4, 4), dtype=torch.uint8), 6)      # CPU tensors
    from pfst_b200.evaluation import metrics as M
    with pytest.raises(PfstError):
        M.seg_argmax(z)


def test_strong_augmentation_draws_like_the_reference_and_registers():
    """The drop-in's draws must consume the global numpy stream exactly like
    StrongAugmentation.__call__ (transforms.py:1081-1141); no GPU needed for the draw."""
    from oracle import strong_aug as osa
    from pfst_b200.pipelines import StrongAugmentation
    aug = registry.PIPELINES.build(dict(type="StrongAugmentation", hue_delta=10, contrast_range=(0.8, 1.2)))
    assert isinstance(aug, StrongAugmentation) and "hue_delta=10" in repr(aug)
    for seed in range(40):
        a, b = np.random.RandomState(seed), np.random.RandomState(seed)
        assert aug.draw(a) == osa.draw_strong_aug(b, 32, (0.8, 1.2), (0.5, 1.5), 10)
        assert a.random_sample() == b.random_sample()
    if R.available():
        pytest.importorskip("cv2")
        ref = R.strong_augmentation_cls()(hue_delta=10, contrast_range=(0.8, 1.2))
        img = np.zeros((4, 4, 3), np.uint8)
        for seed in range(20):
            np.random.seed(seed)
            ref(dict(img=img.copy(), img_fields=[]))
            after = np.random.random()
            np.random.seed(seed)
            aug.draw()
            assert after == np.random.random()
    with pytest.raises(PfstError):
        ops.photometric_u8(torch.zeros((1, 4, 4, 3), dtype=torch.uint8), [[]])


def test_colour_jitter_restatement_properties_and_draw_order():
    """Oracle restatement of kornia's ColorJitter (parity unpinned): neutral factors are the identity, the HSV
    pair round-trips, factors land in kornia's ranges, and the host mirror draws exactly like the oracle."""
    from oracle import strong_aug as osa
    from pfst_b200.utils import dacs_transforms as T
    g = torch.Generator().manual_seed(0)
    x = torch.rand((2, 3, 24, 24), generator=g)
    assert float((osa.hsv_to_rgb(osa.rgb_to_hsv(x)) - x).abs().max()) < 2e-6
    neutral = dict(brightness=torch.ones(2), contrast=torch.ones(2), saturation=torch.ones(2), hue=torch.zeros(2),
                   order=torch.tensor([3, 1, 0, 2]))
    assert float((osa.apply_jitter(x, neutral) - x).abs().max()) < 2e-6
    r = osa.jitter_ranges(0.2)
    assert r["brightness"] == (0.8, 1.2) and r["hue"] == (-0.2, 0.2)
    assert osa.jitter_ranges(dict(brightness=1.5, hue=0.7))["brightness"] == (0.0, 2.0)
    assert osa.jitter_ranges(dict(brightness=1.5, hue=0.7))["hue"] == (-0.5, 0.5)
    for seed in range(10):
        torch.manual_seed(seed)
        fac, order = T.draw_color_jitter(0.2)
        torch.manual_seed(seed)
        p = osa.draw_jitter(0.2, 1)
        assert fac == (float(p["brightness"]), float(p["contrast"]), float(p["saturation"]), float(p["hue"]))
        assert order == p["order"].tolist() and sorted(order) == [0, 1, 2, 3]
        assert 0.8 <= fac[0] <= 1.2 and -0.2 <= fac[3] <= 0.2
    # the jitter stays opt-in: default strong_transform refuses it, loudly (no GPU needed for the refusal)
    param = dict(color_jitter=0.9, color_jitter_s=0.2, color_jitter_p=0.2, blur=0, mean=None, std=None)
    with pytest.raises(PfstError):
        T.strong_transform(param, data=x)


def test_softmax_space_argmax_shortcut_holds_on_the_cpu_softmax():
    """csrc/eval_argmax.cu evaluates the soft-max only for pixels with an EARLIER logit within 3e-4 of the
    maximum; everywhere else it returns the first arg-max of the logits (0 when the row holds a NaN after the
    max subtraction). The same statement must hold for torch's own soft-max -> arg-max (encoder_decoder.py:311,332)."""
    g = torch.Generator().manual_seed(0)
    for C in (2, 6, 12, 33):
        x = torch.randn((4, C, 48, 48), generator=g) * 3
        x[1] = 2.0 + 1e-4 * torch.randint(0, 3, (C, 48, 48), generator=g)   # many near and exact ties
        x[0, 1, 0, :8] = float('nan'); x[0, 0, 1, :8] = float('inf'); x[0, C - 1, 2, :8] = float('inf')
        x[0, :, 3, :8] = float('-inf'); x[0, 0, 4, :8] = float('-inf')
        ref = torch.softmax(x, 1).argmax(1)
        m, am = x.max(1)                                                 # first index of the maximum
        first = (x == m.unsqueeze(1)).float().argmax(1)
        d = x - m.unsqueeze(1)
        nan_row = torch.isnan(d).any(1)
        earlier = torch.arange(C).view(1, C, 1, 1) < first.unsqueeze(1)
        near = ((d > -3.0e-4) & earlier).any(1)
        shortcut = torch.where(nan_row, torch.zeros_like(first), first)
        assert torch.equal(shortcut[~near], ref[~near]), C
        assert int(near.sum()) > 0 and int(nan_row.sum()) >= 32


def test_classmix_draw_is_resumable_word_by_word_and_validates_its_arguments():
    """pfst_classmix_draw fed ONE raw word per call (the worst case for its resumable state) gives the same
    masks as a single call with all words, consumes exactly as many words as numpy's shuffles, and rejects
    inconsistent arguments instead of reading out of bounds."""
    import ctypes as C
    from pfst_b200 import _lib
    fn = _lib.load().pfst_classmix_draw
    n, batch = 7, 5
    classes = np.array([0, 3, 31, 32, 100, 200, 255], dtype=np.int64)
    rs = np.random.RandomState(123)
    ref_state = np.random.RandomState(123)
    want = np.zeros((batch, 8), dtype=np.uint32)
    for b in range(batch):
        for c in classes[ref_state.choice(n, int((n + n % 2) / 2), replace=False)]:
            want[b, c >> 5] |= np.uint32(1) << np.uint32(c & 31)
    out = np.zeros((batch, 8), dtype=np.uint32)
    state = np.zeros(258, dtype=np.int32)
    missing = np.zeros(1, dtype=np.int64)
    bg = rs._bit_generator
    used = 0
    rc = fn(None, 0, classes.ctypes.data, n, batch, out.ctypes.data, state.ctypes.data, missing.ctypes.data)
    assert rc == 0 and missing[0] == batch * (n - 1)            # nothing drawn yet: one word per swap at least
    while missing[0]:
        w = bg.random_raw(1)
        used += 1
        assert fn(w.ctypes.data, 1, classes.ctypes.data, n, batch, out.ctypes.data, state.ctypes.data,
                  missing.ctypes.data) == 0
    assert np.array_equal(out, want)
    assert rs.randint(1 << 30) == ref_state.randint(1 << 30)     # both streams advanced by the same words
    assert used >= batch * (n - 1)
    # argument validation (negative return codes, no crash)
    bad_cls = np.array([0, 1, 256], dtype=np.int64)
    state[:] = 0
    assert fn(None, 0, bad_cls.ctypes.data, 3, 1, out.ctypes.data, state.ctypes.data, missing.ctypes.data) < 0
    assert fn(None, 0, classes.ctypes.data, 300, 1, out.ctypes.data, state.ctypes.data, missing.ctypes.data) < 0
    state[0] = 99                                                # resume index beyond the batch
    assert fn(None, 0, classes.ctypes.data, n, batch, out.ctypes.data, state.ctypes.data, missing.ctypes.data) < 0
    state[:] = 0
    w = bg.random_raw(4 * batch * n)                             # more words than the shuffles can consume
    assert fn(w.ctypes.data, w.shape[0], classes.ctypes.data, n, batch, out.ctypes.data, state.ctypes.data,
              missing.ctypes.data) < 0
