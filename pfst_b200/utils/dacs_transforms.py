"""ClassMix utilities — drop-in for rsiseg/models/utils/dacs_transforms.py.

Same function names, argument meaning and return shapes/dtypes as the reference
(`get_class_masks`, `generate_class_mask`, `one_mix`, `strong_transform`,
`get_mean_std`, `denorm`), computed by the sm_100a kernels in csrc/classmix.cu.
`class_mix_batch` is the fused form the PFGST trainer uses instead of the
reference's per-image Python loop (pfgst.py:287-300).

Host RNG: the class draw stays `np.random.choice` on the global numpy stream,
one draw per image in batch order, exactly as dacs_transforms.py:115-117 — the
stream is observable behaviour of the reference.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from .. import _lib, ops
from .._lib import PfstError


def _present_classes(presence_words: np.ndarray) -> np.ndarray:
    """Sorted label values present in the batch (== torch.unique, :113)."""
    if presence_words[8] != 0:
        raise PfstError("gt_semantic_seg holds labels outside [0,255]; the ClassMix kernels "
                        "address classes through a 256-bit mask")
    bits = np.unpackbits(presence_words[:8].view(np.uint8), bitorder="little")
    return np.nonzero(bits)[0].astype(np.int64)




def draw_class_choice(classes: np.ndarray, batch: int, rng=np.random) -> np.ndarray:
    """One `np.random.choice(n, int((n + n % 2) / 2), replace=False)` per image
    (dacs_transforms.py:114-117) -> uint32 (batch, 8) bitmasks of the drawn classes.

    Legacy `RandomState.choice(n, k, replace=False)` IS `permutation(n)[:k]` (numpy
    mtrand: `idx = self.permutation(pop_size)[:size]`), and `permutation` is a Fisher-Yates
    shuffle that consumes successive raw 32-bit outputs of the stream through masked
    rejection. `rng.bytes` hands out exactly those raw words, so the whole batch is replayed
    from them by one host call into the library (`pfst_classmix_draw`): the draws and the
    state the stream is left in are those of `batch` calls of `np.random.choice`
    (tests/test_host_logic.py), at ~10 us per batch instead of ~4 us per image — this draw
    sits on the step's only host round trip. Words are requested in rounds (first one per
    swap, then one per rejection seen so far), never more than the shuffles consume."""
    n = int(classes.shape[0])
    if batch == 0 or n == 0:
        return np.zeros((batch, 8), dtype=np.uint32)
    st = _DrawState.get(batch)
    raw = _raw_words(rng)
    st.cls[:n] = classes
    st.state[:2] = 0
    need = batch * (n - 1)
    while True:
        if need > st.words.shape[0]:
            st.grow(need)
        if need:
            st.words[:need] = raw(need)
        _lib.check(st.fn(st.p_words, need, st.p_cls, n, batch, st.p_out, st.p_state, st.p_missing),
                   "pfst_classmix_draw")
        need = int(st.io[0])
        if need == 0:
            return st.out[:batch].copy()


class _DrawState:
    """Host buffers of draw_class_choice with their addresses (ndarray.ctypes costs ~2 us per access,
    more than the library call itself)."""
    _inst = None

    def __init__(self, batch: int):
        self.fn = _lib.load().pfst_classmix_draw
        self.cls = np.zeros(256, dtype=np.int64)
        self.io = np.zeros(1, dtype=np.int64)                 # words_missing
        self.state = np.zeros(258, dtype=np.int32)            # image, swap index, permutation (resumable)
        self.out = np.zeros((batch, 8), dtype=np.uint32)
        self.words = np.zeros(batch * 255, dtype=np.uint64)
        self._addr()

    def _addr(self):
        self.p_cls, self.p_out, self.p_state = self.cls.ctypes.data, self.out.ctypes.data, self.state.ctypes.data
        self.p_missing, self.p_words = self.io.ctypes.data, self.words.ctypes.data

    def grow(self, words: int):
        self.words = np.zeros(2 * words, dtype=np.uint64)
        self._addr()

    @classmethod
    def get(cls, batch: int):
        st = cls._inst
        if st is None or st.out.shape[0] < batch:
            st = cls._inst = cls(max(batch, 64))
        return st


def _raw_words(rng):
    """-> f(m): the next m raw 32-bit outputs of `rng`'s MT19937 stream as uint64 (the stream advances by
    exactly m words). `rng` is the numpy.random module (global stream) or a RandomState."""
    bg = getattr(rng, "_bit_generator", None)
    if bg is None and rng is np.random:
        bg = np.random.mtrand._rand._bit_generator        # the singleton behind np.random.choice / seed
    if bg is not None and type(bg).__name__ == "MT19937":
        return bg.random_raw
    return lambda m: np.frombuffer(rng.bytes(4 * m), dtype=np.uint32).astype(np.uint64)   # same words, slower


class ClassMixPlan:
    """Two-phase ClassMix: `start(gt)` enqueues the presence kernel and an async D2H of
    its 36-byte result; `choose()` (called later, after other work has been enqueued)
    waits for that copy only, draws the classes on the host and uploads the per-image
    bitmasks. This hides the one unavoidable host round trip (SURVEY.md §7)."""

    SLOTS = 4     # pinned staging slots: the host may run this many steps ahead of the device

    def __init__(self, device: torch.device, max_batch: int = 256):
        self.device = device
        K = self.SLOTS
        self._presence = torch.empty(9, dtype=torch.int32, device=device)
        self._presence_host = torch.empty((K, 9), dtype=torch.int32).pin_memory()
        self._chosen_host = torch.empty((K, max_batch, 8), dtype=torch.int32).pin_memory()
        self._chosen = torch.empty((max_batch, 8), dtype=torch.int32, device=device)
        self._presence_np = self._presence_host.numpy().view(np.uint32)     # views of the pinned buffers
        self._chosen_np = self._chosen_host.numpy()
        self._events = [torch.cuda.Event() for _ in range(K)]               # presence D2H done, per slot
        self._h2d_events = [torch.cuda.Event() for _ in range(K)]           # upload has read the slot
        self._h2d_pending = [False] * K
        self._started, self._chosen_count = 0, 0                            # start() / choose() calls so far
        self._batches = [0] * K
        self._batch = 0

    def start(self, gt: torch.Tensor, stream: Optional[torch.cuda.Stream] = None) -> None:
        """gt: int64 or uint8 label maps of the batch."""
        dt = ops._labels(gt, "gt")              # before any state changes: a refused gt leaves the FIFO aligned
        if self._started - self._chosen_count >= self.SLOTS:
            raise PfstError("ClassMixPlan: more start() calls in flight than staging slots")
        slot = self._started % self.SLOTS
        self._started += 1
        batch = gt.shape[0]
        if batch > self._chosen.shape[0]:
            raise ValueError("batch larger than the plan's capacity")
        self._batches[slot] = batch
        if stream is None:
            stream = torch.cuda.current_stream()
        _lib.call("pfst_class_presence_lbl", gt.data_ptr(), dt, gt.numel(), self._presence.data_ptr(),
                  stream.cuda_stream)
        _lib.call("pfst_copy_async", self._presence_host.data_ptr() + 36 * slot, self._presence.data_ptr(), 36,
                  stream.cuda_stream)
        self._events[slot].record(stream)

    def drop_pending(self) -> int:
        """Forget start() calls that were never matched by choose() (an exception between the two,
        or a prefetch for a batch that was not run): the next start()/choose() pair is aligned
        again. Returns the number of dropped slots."""
        n = self._started - self._chosen_count
        self._chosen_count = self._started
        return n

    def choose(self, rng=np.random) -> torch.Tensor:
        if self._chosen_count >= self._started:
            raise PfstError("ClassMixPlan.choose() without a matching start()")
        slot = self._chosen_count % self.SLOTS
        self._chosen_count += 1
        self._batch = batch = self._batches[slot]
        self._events[slot].synchronize()
        classes = _present_classes(self._presence_np[slot])
        chosen = draw_class_choice(classes, batch, rng)
        if self._h2d_pending[slot]:
            self._h2d_events[slot].synchronize()   # the upload issued SLOTS steps ago has read this slot
        self._chosen_np[slot, :batch] = chosen.view(np.int32)
        dst = self._chosen[:batch]
        _lib.call("pfst_copy_async", dst.data_ptr(), self._chosen_host.data_ptr() + slot * self._chosen_host.stride(0) * 4,
                  32 * batch, ops._stream())
        self._h2d_events[slot].record()
        self._h2d_pending[slot] = True
        return dst


def _chosen_for(labels: torch.Tensor, rng=np.random) -> torch.Tensor:
    plan = ClassMixPlan(labels.device, max_batch=labels.shape[0])
    plan.start(labels)
    return plan.choose(rng)


def get_class_masks(labels: torch.Tensor):
    """dacs_transforms.py:110-119 — list of B masks, each (1,1,H,W) int64."""
    labels = labels.contiguous()
    chosen = _chosen_for(labels)
    _, _, _, mask = ops.class_mix(labels, chosen, None, None, None, want_weight=False)
    return [mask[i:i + 1] for i in range(mask.shape[0])]


def generate_class_mask(label: torch.Tensor, classes: torch.Tensor) -> torch.Tensor:
    """dacs_transforms.py:122-126 — label (1,H,W), classes (K,) -> (1,H,W) int64."""
    vals = classes.detach().cpu().numpy().astype(np.int64)
    if ((vals < 0) | (vals > 255)).any():
        raise PfstError("classes outside [0,255]")
    chosen = np.zeros((1, 8), dtype=np.uint32)
    for v in vals:
        chosen[0, v >> 5] |= np.uint32(1) << np.uint32(v & 31)
    ch = torch.from_numpy(chosen.view(np.int32)).to(label.device)
    H, W = label.shape[-2:]
    _, _, _, mask = ops.class_mix(label.reshape(1, 1, H, W).contiguous(), ch, None, None, None,
                                  want_weight=False)
    return mask.reshape(1, H, W)


def one_mix(mask, data=None, target=None):
    """dacs_transforms.py:129-144 — mask (1,1,H,W); data (2,C,H,W) -> (1,C,H,W);
    target (2,H,W) -> (1,1,H,W)."""
    if mask is None:
        return data, target
    H, W = mask.shape[-2:]
    m = mask.reshape(H * W).contiguous()
    if m.dtype != torch.int64:
        m = m.long()

    def mix(pair, channels, out_shape):
        a, b = pair[0].contiguous(), pair[1].contiguous()
        out = torch.empty(out_shape, dtype=a.dtype, device=a.device)
        if a.dtype == torch.float32:
            dt = 0
        elif a.dtype == torch.int64:
            dt = 2
        else:
            raise TypeError(f"one_mix supports float32/int64 operands, got {a.dtype}")
        from .. import _lib
        _lib.call("pfst_mask_mix", ops._dev(m, "mask", torch.int64), ops._dev(a, "a"), ops._dev(b, "b"),
                  out.data_ptr(), dt, channels, H * W, ops._stream())
        return out

    if data is not None:
        data = mix(data, data.shape[1], (1,) + tuple(data.shape[1:]))
    if target is not None:
        if tuple(target.shape[-2:]) != (H, W):
            raise PfstError("one_mix: target/mask size mismatch (resampling not supported)")
        target = mix(target, 1, (1, 1, H, W))
    return data, target


def gaussian_blur(blur, data=None, target=None, rng=np.random):
    """dacs_transforms.py:88-107. Same host behaviour as the reference: when `blur > 0.5` and data
    has three channels, ONE `np.random.uniform(0.15, 1.15)` is drawn (global numpy stream) and the
    whole `data` batch is blurred with it; the kernel edge is ~10 % of the image (odd). The
    arithmetic is kornia's GaussianBlur2d restated in csrc/blur.cu (third-party, unpinned: see
    oracle/strong_aug.py)."""
    if data is not None and data.shape[1] == 3 and blur > 0.5:
        sigma = rng.uniform(0.15, 1.15)
        data = ops.gaussian_blur(data.contiguous(), [sigma] * data.shape[0])
    return data, target


def gaussian_blur_batch(blur, mixed_img: torch.Tensor, rng=np.random) -> torch.Tensor:
    """The B per-image `gaussian_blur` calls of the mixing loop (pfgst.py:287-300) as ONE launch:
    B sigma draws in image order (exactly the reference's numpy stream), one sigma per image."""
    if mixed_img.shape[1] != 3 or not (blur > 0.5):
        return mixed_img
    sigmas = [rng.uniform(0.15, 1.15) for _ in range(mixed_img.shape[0])]
    return ops.gaussian_blur(mixed_img.contiguous(), sigmas)


def _jitter_ranges(s):
    """kornia `_range_bound` of ColorJitter(brightness=s, contrast=s, saturation=s, hue=s) (or a dict)."""
    if not isinstance(s, dict):
        s = dict(brightness=s, contrast=s, saturation=s, hue=s)
    b, c, sa, h = (float(s.get(k, 0.0)) for k in ("brightness", "contrast", "saturation", "hue"))
    clamp = lambda lo, hi, a, bnd: (min(max(lo, a), bnd), min(max(hi, a), bnd))
    return (clamp(1 - b, 1 + b, 0.0, 2.0), clamp(1 - c, 1 + c, 0.0, float("inf")),
            clamp(1 - sa, 1 + sa, 0.0, float("inf")), clamp(-h, h, -0.5, 0.5))


def draw_color_jitter(s, generator=None):
    """One kornia ColorJitterGenerator draw (0.6 series, restated — see oracle/strong_aug.py): factors in the
    order brightness, contrast, hue, saturation from the torch CPU generator, then randperm(4).
    -> ((brightness, contrast, saturation, hue), order)."""
    rb, rc, rs, rh = _jitter_ranges(s)
    u = lambda r: float(r[0] + (r[1] - r[0]) * torch.rand((1,), generator=generator))
    fb, fc, fh, fs = u(rb), u(rc), u(rh), u(rs)
    return (fb, fc, fs, fh), torch.randperm(4, generator=generator).tolist()


def _host3(x):
    return [float(v) for v in (x.flatten().tolist() if isinstance(x, torch.Tensor) else x)][:3]


def color_jitter(color_jitter, mean, std, data=None, target=None, s=.25, p=.2, denorm_type='mean_std'):
    """dacs_transforms.py:56-85, same signature. The jitter itself is the built-in restatement of
    kornia's ColorJitter (csrc/color_jitter.cu; third-party arithmetic and sampler, PARITY UNPINNED);
    one draw for the whole `data` batch like a kornia module call with same_on_batch=False would make
    per image — the reference always passes one image."""
    if data is not None and data.shape[1] == 3 and color_jitter > p:
        if denorm_type not in ('mean_std', 'none'):
            raise ValueError('No such denorm type!')
        draws = [draw_color_jitter(s) for _ in range(data.shape[0])]
        dn = denorm_type == 'mean_std'
        data = ops.color_jitter(data.contiguous(), [d[0] for d in draws], [d[1] for d in draws],
                                _host3(mean) if dn else None, _host3(std) if dn else None)
    return data, target


def strong_transform(param, data=None, target=None):
    """dacs_transforms.py:12-27: one_mix -> color_jitter -> gaussian_blur. The colour jitter is kornia's
    sampler + arithmetic (third-party, version unpinned, SURVEY.md §8c): by default requesting it raises
    instead of silently skipping; param['kornia_aug'] = 'builtin' runs the built-in restatement."""
    assert (data is not None) or (target is not None)
    if "mix" in param:
        data, target = one_mix(mask=param["mix"], data=data, target=target)
    if data is not None and data.shape[1] == 3 and param.get("color_jitter", 0) > param.get("color_jitter_p", 1.0):
        if param.get("kornia_aug", "error") != "builtin":
            raise PfstError("the kornia ColorJitter branch runs only as the built-in restatement "
                            "(param['kornia_aug']='builtin'); set color_jitter_probability=1.0 to disable it")
        data, target = color_jitter(color_jitter=param["color_jitter"], s=param["color_jitter_s"],
                                    p=param["color_jitter_p"], mean=param["mean"], std=param["std"],
                                    data=data, target=target, denorm_type=param.get("denorm_type", "mean_std"))
    data, target = gaussian_blur(blur=param.get("blur", 0), data=data, target=target)
    return data, target


def get_mean_std(img_metas, dev):
    """dacs_transforms.py:30-41."""
    mean = torch.stack([torch.as_tensor(m["img_norm_cfg"]["mean"], device=dev) for m in img_metas])
    std = torch.stack([torch.as_tensor(m["img_norm_cfg"]["std"], device=dev) for m in img_metas])
    return mean.view(-1, 3, 1, 1), std.view(-1, 3, 1, 1)


def denorm(img, mean, std):
    """dacs_transforms.py:44-45."""
    return img.mul(std).add(mean) / 255.0


def class_mix_batch(img: torch.Tensor, trg_img: torch.Tensor, gt: torch.Tensor, pseudo_lbl: torch.Tensor,
                    chosen: torch.Tensor, count: Optional[torch.Tensor] = None, ps_size: int = 0,
                    weight_in: Optional[torch.Tensor] = None, ignore_top: int = 0, ignore_bottom: int = 0):
    """Fused replacement of pfgst.py:281-300 for the whole batch, one launch.
    -> mixed_img (B,3,H,W), mixed_lbl (B,1,H,W) int64, pseudo_weight (B,H,W), mix_masks (B,1,H,W) int64."""
    return ops.class_mix(gt, chosen, img, trg_img, pseudo_lbl, weight_in=weight_in, count=count,
                         ps_size=ps_size, ignore_top=ignore_top, ignore_bottom=ignore_bottom)
