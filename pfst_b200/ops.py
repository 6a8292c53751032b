"""Tensor-level wrappers over the C ABI (device pointers + current CUDA stream).

PyTorch is used here for device memory and streams only. Every function
requires CUDA tensors and raises on anything else — there is no fallback path.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import torch

from . import _lib
from ._lib import PfstError

_TORCH2DT = {torch.uint8: _lib.DT_U8, torch.int32: _lib.DT_I32, torch.int64: _lib.DT_I64}


def _dev(t: torch.Tensor, name: str, dtype: Optional[torch.dtype] = None) -> int:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name}: expected a torch.Tensor, got {type(t)}")
    if not t.is_cuda:
        raise PfstError(f"{name}: pfst_b200 kernels need CUDA tensors (got {t.device}); "
                        "there is no CPU fallback")
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name}: tensor must be contiguous")
    return t.data_ptr()


def _opt(t: Optional[torch.Tensor], name: str, dtype=None) -> Optional[int]:
    return None if t is None else _dev(t, name, dtype)


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


LABEL_DTYPES = (torch.int64, torch.uint8)


def _labels(t: torch.Tensor, name: str, like: Optional[torch.Tensor] = None) -> int:
    """Checks a label map (int64, the reference dtype, or uint8, the dtype datasets store) and returns
    its PFST_DT_* tag. `like`: another label map of the same call, whose dtype it must share."""
    if isinstance(t, torch.Tensor) and t.dtype not in LABEL_DTYPES:
        raise TypeError(f"{name}: label maps must be torch.int64 or torch.uint8, got {t.dtype}")
    if like is not None and isinstance(t, torch.Tensor) and t.dtype != like.dtype:
        raise TypeError(f"{name}: every label map of one call has one dtype ({like.dtype}), got {t.dtype}")
    _dev(t, name)
    return _TORCH2DT[t.dtype]


# The EMA teacher's outputs (pseudo-label logits, features) may come from a pass run under autocast; the
# kernels that read them take fp32, fp16 or bf16 (converted to fp32 on load, exactly). The student's logits
# and features given to the self-training step and PFGSTLoss stay fp32; only the decode-head loss
# (losses/cross_entropy.py) also takes 16-bit student logits.
TEACHER_DTYPES = (torch.float32, torch.float16, torch.bfloat16)
_FLOAT2DT = {torch.float32: _lib.DT_F32, torch.float16: _lib.DT_F16, torch.bfloat16: _lib.DT_BF16}


def float_dtype_tag(dtype: torch.dtype, name: str = "tensor") -> int:
    """PFST_DT_F32 / F16 / BF16 tag of a teacher-output dtype; TypeError for any other dtype."""
    tag = _FLOAT2DT.get(dtype)
    if tag is None:
        raise TypeError(f"{name}: teacher outputs must be torch.float32, torch.float16 or torch.bfloat16, "
                        f"got {dtype}")
    return tag


def _teacher(t: torch.Tensor, name: str) -> int:
    """Checks a teacher-output tensor and returns its float dtype tag."""
    if isinstance(t, torch.Tensor):
        float_dtype_tag(t.dtype, name)
    _dev(t, name)
    return _FLOAT2DT[t.dtype]


def _stream() -> int:
    # raw cudaStream_t of torch's current stream (also the capturing stream inside torch.cuda.graph);
    # the public torch.cuda.current_stream() builds a Stream object per call (~2 us each, ~10 per step)
    return torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice())


def device_check() -> None:
    _lib.call("pfst_device_check")


# ---------------------------------------------------------------- E1/E2: EMA
def ema_coeffs(it: int, alpha: float) -> tuple[float, float]:
    a, b = C.c_float(), C.c_float()
    _lib.call("pfst_ema_coeffs", int(it), float(alpha), C.byref(a), C.byref(b))
    return a.value, b.value


class EmaTable:
    """Device-resident pointer/chunk tables for a (teacher, student) parameter list.

    Built once per model (the pointers of ``nn.Parameter.data`` are stable while
    the optimiser updates in place); ``update`` is then ONE kernel launch for all
    tensors. ``stale()`` detects re-allocated parameters.
    """

    CHUNK = 4096  # floats per block; must be a multiple of 1024

    def __init__(self, ema_params: Sequence[torch.Tensor], params: Sequence[torch.Tensor]):
        ema_params, params = list(ema_params), list(params)
        if len(ema_params) != len(params):
            raise ValueError("teacher/student parameter lists differ in length")
        self._ema = [p.data for p in ema_params]
        self._src = [p.data for p in params]
        eptr, pptr, numel, ctensor, cbegin = [], [], [], [], []
        device = None
        for i, (e, p) in enumerate(zip(self._ema, self._src)):
            if e.shape != p.shape:
                raise ValueError(f"parameter {i}: shape mismatch {tuple(e.shape)} vs {tuple(p.shape)}")
            eptr.append(_dev(e, f"ema_param[{i}]", torch.float32))
            pptr.append(_dev(p, f"param[{i}]", torch.float32))
            device = e.device
            n = e.numel()
            numel.append(n)
            for start in range(0, n, self.CHUNK):
                ctensor.append(i)
                cbegin.append(start)
        self.device = device
        self.n_tensors = len(numel)
        self.n_chunks = len(ctensor)
        self.total = sum(numel)
        self._key = (tuple(eptr), tuple(pptr))
        if self.n_chunks:
            mk = lambda v, dt: torch.tensor(v, dtype=dt, device=device)
            self._t_eptr = mk(eptr, torch.int64)
            self._t_pptr = mk(pptr, torch.int64)
            self._t_numel = mk(numel, torch.int64)
            self._t_ctensor = mk(ctensor, torch.int32)
            self._t_cbegin = mk(cbegin, torch.int64)
            self._ptrs = (self._t_eptr.data_ptr(), self._t_pptr.data_ptr(), self._t_numel.data_ptr(),
                          self._t_ctensor.data_ptr(), self._t_cbegin.data_ptr())

    def stale(self, ema_params, params) -> bool:
        key = (tuple(p.data.data_ptr() for p in ema_params), tuple(p.data.data_ptr() for p in params))
        return key != self._key

    def update(self, a32: float, b32: float, mode: int = 0, blocks_per_sm: int = 0,
               stream: Optional[int] = None) -> None:
        """blocks_per_sm > 0: bounded persistent grid (lets the update share the SMs with
        kernels of other streams). stream: raw cudaStream_t handle (default: the current
        stream of the table's device)."""
        if not self.n_chunks:
            return
        if stream is None:
            stream = torch.cuda.current_stream(self.device).cuda_stream
        _lib.call("pfst_ema_update_multi", *self._ptrs, self.n_chunks, self.CHUNK, a32, b32, mode,
                  int(blocks_per_sm), stream)


def _ema_update_dev(self, coefs_dev: torch.Tensor, blocks_per_sm: int = 0, stream: Optional[int] = None) -> None:
    """EmaTable.update with {a32, b32} read from a device float[2] (graph-capturable launch)."""
    if not self.n_chunks:
        return
    if stream is None:
        stream = torch.cuda.current_stream(self.device).cuda_stream
    _lib.call("pfst_ema_update_multi_dev", *self._ptrs, self.n_chunks, self.CHUNK,
              _dev(coefs_dev, "coefs_dev", torch.float32), int(blocks_per_sm), stream)


EmaTable.update_dev = _ema_update_dev


def ema_update_flat(ema: torch.Tensor, param: torch.Tensor, a32: float, b32: float, mode: int = 0):
    if ema.shape != param.shape:
        raise ValueError("shape mismatch")
    _lib.call("pfst_ema_update_flat", _dev(ema, "ema", torch.float32), _dev(param, "param", torch.float32),
              ema.numel(), a32, b32, mode, _stream())


# ---------------------------------------------------------- S1/S2: pseudo labels
def pseudo_label(logits: torch.Tensor, thr: float = 0.0, thr_per_class: Optional[torch.Tensor] = None,
                 mode: int = 0, reject_label: int = -1, want_part_weight: bool = False,
                 label_dtype: torch.dtype = torch.int64):
    """-> (label (B,H,W) of label_dtype (int64 or uint8), conf fp32 (B,H,W), count int64[1] on device,
    weight_part|None). logits: fp32, fp16 or bf16 (the outputs equal those of the fp32 logits upcast).
    uint8 labels need C <= 255 and reject_label <= 255 (negative: no rejection)."""
    if logits.dim() != 4:
        raise ValueError("logits must be (B,C,H,W)")
    B, Cc, H, W = logits.shape
    _teacher(logits, "logits")
    if label_dtype not in LABEL_DTYPES:
        raise TypeError(f"label_dtype must be torch.int64 or torch.uint8, got {label_dtype}")
    if label_dtype == torch.uint8 and (Cc > 255 or int(reject_label) > 255):
        raise ValueError(f"uint8 pseudo labels need C <= 255 (got {Cc}) and reject_label <= 255 "
                         f"(got {reject_label}; a negative value means no rejection)")
    label = torch.empty((B, H, W), dtype=label_dtype, device=logits.device)
    conf = torch.empty((B, H, W), dtype=torch.float32, device=logits.device)
    count = torch.empty(1, dtype=torch.int64, device=logits.device)  # written as uint64
    wpart = torch.empty((B, H, W), dtype=torch.float32, device=logits.device) if want_part_weight else None
    if thr_per_class is not None:
        if thr_per_class.numel() != Cc:
            raise ValueError("thr_per_class must have C entries")
        _dev(thr_per_class, "thr_per_class", torch.float32)
    launch_pseudo_label(logits, thr, thr_per_class, mode, reject_label, label, conf, wpart, count, _stream())
    return label, conf, count, wpart


# The launch functions below pass tensors their caller has already validated (and allocated) to one entry
# point, in ABI order, on the raw stream `stream`: no checks, no allocation. The dtype tags, the loss
# weights and the shipped PFGSTLoss options are formed here only.
def launch_pseudo_label(logits, thr, thr_per_class, mode, reject_label, label, conf, wpart, count, stream) -> None:
    B, Cc, H, W = logits.shape
    _lib.call("pfst_pseudo_label", logits.data_ptr(), _FLOAT2DT[logits.dtype], B, Cc, H * W, float(thr),
              _ptr(thr_per_class), int(mode), int(reject_label), label.data_ptr(), _TORCH2DT[label.dtype],
              conf.data_ptr(), _ptr(wpart), count.data_ptr(), stream)


def pseudo_weight_fill(shape, count: torch.Tensor, ps_size: int, ignore_top: int = 0,
                       ignore_bottom: int = 0) -> torch.Tensor:
    B, H, W = shape
    w = torch.empty((B, H, W), dtype=torch.float32, device=count.device)
    _lib.call("pfst_pseudo_weight_fill", _dev(w, "weight"), B, H, W, _dev(count, "count", torch.int64),
              int(ps_size), int(ignore_top), int(ignore_bottom), _stream())
    return w


# ------------------------------------------------------------- M1/M2: ClassMix
def class_presence(gt: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """gt: int64 or uint8. -> int32[9] on device: 256 presence bits + out-of-range flag."""
    dt = _labels(gt, "gt")
    if out is None:
        out = torch.empty(9, dtype=torch.int32, device=gt.device)
    _lib.call("pfst_class_presence", gt.data_ptr(), dt, gt.numel(), _dev(out, "presence", torch.int32),
              _stream())
    return out


def class_mix(gt: torch.Tensor, chosen: torch.Tensor, img: Optional[torch.Tensor],
              trg_img: Optional[torch.Tensor], pseudo_lbl: Optional[torch.Tensor],
              weight_in: Optional[torch.Tensor] = None, count: Optional[torch.Tensor] = None,
              ps_size: int = 0, ignore_top: int = 0, ignore_bottom: int = 0,
              want_weight: bool = True, want_mask: bool = True, weight_out: Optional[torch.Tensor] = None):
    """Fused ClassMix. gt (B,1,H,W) int64 or uint8; chosen int32 (B,8) bitmasks. The pseudo label, the
    mixed label and the mask share gt's dtype.
    -> (mixed_img|None, mixed_lbl|None, mixed_weight|None, mix_mask|None)"""
    _labels(gt, "gt")
    B, H, W = gt.shape[0], gt.shape[-2], gt.shape[-1]
    if gt.numel() != B * H * W:
        raise ValueError("gt must be (B,1,H,W) or (B,H,W)")
    _dev(chosen, "chosen", torch.int32)
    if chosen.numel() != B * 8:
        raise ValueError("chosen must hold 8 words per image")
    dev = gt.device
    mixed_img = mixed_lbl = mixed_w = mask = None
    if img is not None:
        _dev(img, "img", torch.float32)
        _dev(trg_img, "trg_img", torch.float32)
        if img.shape != trg_img.shape or img.shape[0] != B or img.shape[-2:] != gt.shape[-2:]:
            raise ValueError("img/trg_img shape mismatch")
        mixed_img = torch.empty_like(img)
    if pseudo_lbl is not None:
        _labels(pseudo_lbl, "pseudo_label", like=gt)
        if pseudo_lbl.numel() != B * H * W:
            raise ValueError("pseudo_label shape mismatch")
        mixed_lbl = torch.empty((B, 1, H, W), dtype=gt.dtype, device=dev)
    if want_weight:
        if weight_in is not None:
            _dev(weight_in, "weight_in", torch.float32)
        else:
            _dev(count, "count", torch.int64)
        mixed_w = weight_out if weight_out is not None else torch.empty((B, H, W), dtype=torch.float32, device=dev)
        _dev(mixed_w, "weight_out", torch.float32)
    if want_mask:
        mask = torch.empty((B, 1, H, W), dtype=gt.dtype, device=dev)
    launch_class_mix(gt, chosen, img, trg_img, pseudo_lbl, weight_in if want_weight else None, count, ps_size,
                     ignore_top, ignore_bottom, mixed_img, mixed_lbl, mixed_w, mask, _stream())
    return mixed_img, mixed_lbl, mixed_w, mask


def launch_class_mix(gt, chosen, img, trg_img, pseudo_lbl, weight_in, count, ps_size, ignore_top, ignore_bottom,
                     mixed_img, mixed_lbl, mixed_weight, mix_mask, stream) -> None:
    B, H, W = gt.shape[0], gt.shape[-2], gt.shape[-1]
    _lib.call("pfst_class_mix", gt.data_ptr(), chosen.data_ptr(), _ptr(img), _ptr(trg_img), _ptr(pseudo_lbl),
              _ptr(weight_in), _ptr(count), int(ps_size), int(ignore_top), int(ignore_bottom), B,
              0 if img is None else img.shape[1], H, W, _ptr(mixed_img), _ptr(mixed_lbl), _ptr(mixed_weight),
              _ptr(mix_mask), _TORCH2DT[gt.dtype], stream)


# ----------------------------------------------------------- V1/V4: confusion
def confusion_accum(pred: torch.Tensor, label: torch.Tensor, num_classes: int, ignore_index: int = 255,
                    reduce_zero_label: bool = False, lut: Optional[torch.Tensor] = None,
                    per_image: bool = False, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """pred/label: (N,H,W) or (H,W) maps (uint8/int32/int64). -> int64 (slots,C+1,C+1),
    accumulated into ``out`` when given."""
    if pred.shape != label.shape:
        raise ValueError("pred/label shape mismatch")
    if pred.dtype not in _TORCH2DT or label.dtype not in _TORCH2DT:
        raise TypeError("pred/label must be uint8, int32 or int64")
    _dev(pred, "pred")
    _dev(label, "label")
    n_images = pred.shape[0] if pred.dim() >= 3 else 1
    pixels = pred.numel() // max(n_images, 1)
    slots = n_images if per_image else 1
    Cn = int(num_classes)
    if out is None:
        out = torch.zeros((slots, Cn + 1, Cn + 1), dtype=torch.int64, device=pred.device)
    elif out.numel() != slots * (Cn + 1) * (Cn + 1):
        raise ValueError("out has the wrong size")
    _lib.call("pfst_confusion_accum", pred.data_ptr(), _TORCH2DT[pred.dtype], label.data_ptr(),
              _TORCH2DT[label.dtype], n_images, pixels, Cn, int(ignore_index), int(bool(reduce_zero_label)),
              _opt(lut, "lut", torch.uint8), _dev(out, "out", torch.int64), int(per_image), _stream())
    return out


def argmax_confusion(seg_logits: torch.Tensor, label: Optional[torch.Tensor], num_classes: Optional[int] = None,
                     ignore_index: int = 255, reduce_zero_label: bool = False,
                     lut: Optional[torch.Tensor] = None, per_image: bool = False,
                     out: Optional[torch.Tensor] = None, return_pred: Optional[torch.dtype] = None):
    """Fused `softmax(seg_logits,1).argmax(1)` + confusion matrix (encoder_decoder.py:311,329-332 +
    metrics.py:26-86). seg_logits (N,C,H,W) fp32; label (N,H,W) uint8/int32/int64 or None (arg-max
    only, then ``return_pred`` is required). -> (conf int64 (slots,C+1,C+1) or None, pred or None)."""
    _dev(seg_logits, "seg_logits", torch.float32)
    if seg_logits.dim() != 4:
        raise ValueError("seg_logits must be (N,C,H,W)")
    N, Cn, H, W = seg_logits.shape
    if num_classes is not None and int(num_classes) != Cn:
        raise ValueError(f"seg_logits has {Cn} channels, num_classes={num_classes}")
    if return_pred not in (None, torch.uint8, torch.int64):
        raise TypeError("return_pred must be None, torch.uint8 or torch.int64")
    if label is None and return_pred is None:
        raise ValueError("nothing to compute: give a label map and/or return_pred")
    pred = None
    if return_pred is not None:
        pred = torch.empty((N, H, W), dtype=return_pred, device=seg_logits.device)
    conf = None
    ldt = _lib.DT_U8
    if label is not None:
        if label.dtype not in _TORCH2DT:
            raise TypeError("label must be uint8, int32 or int64")
        _dev(label, "label")
        if label.numel() != N * H * W:
            raise ValueError("seg_logits/label shape mismatch")
        ldt = _TORCH2DT[label.dtype]
        slots = N if per_image else 1
        if out is None:
            out = torch.zeros((slots, Cn + 1, Cn + 1), dtype=torch.int64, device=seg_logits.device)
        elif out.numel() != slots * (Cn + 1) * (Cn + 1):
            raise ValueError("out has the wrong size")
        conf = out
    _lib.call("pfst_argmax_confusion", seg_logits.data_ptr(), N, Cn, H * W,
              None if label is None else label.data_ptr(), ldt, int(ignore_index),
              int(bool(reduce_zero_label)), _opt(lut, "lut", torch.uint8),
              None if conf is None else _dev(conf, "out", torch.int64), int(per_image),
              None if pred is None else pred.data_ptr(),
              _lib.DT_I64 if return_pred == torch.int64 else _lib.DT_U8, _stream())
    return conf, pred


# ------------------------------------- strong augmentation: photometric distortion (uint8)
SA_CONVERT, SA_SATURATION, SA_HUE = 1, 2, 3
SA_MAX_OPS = 4


def photometric_u8(imgs: torch.Tensor, op_lists: Sequence[Sequence[tuple]], simd: int = 32,
                   out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """StrongAugmentation's distortions (transforms.py:1075-1141) on uint8 BGR images (N,H,W,3), one
    launch. op_lists[i] = up to four (code, p0, p1) in application order: (SA_CONVERT, alpha, beta),
    (SA_SATURATION, alpha, _), (SA_HUE, integer delta, _). Bit-identical to the reference's
    numpy + cv2 arithmetic (simd = SIMD block width of cv2's HSV->BGR on the reference host)."""
    _dev(imgs, "imgs", torch.uint8)
    if imgs.dim() != 4 or imgs.shape[3] != 3:
        raise ValueError("imgs must be (N,H,W,3) uint8")
    N, H, W, _ = imgs.shape
    if len(op_lists) != N:
        raise ValueError(f"need one op list per image ({N}), got {len(op_lists)}")
    codes = (C.c_int32 * max(N * SA_MAX_OPS, 1))()
    params = (C.c_float * max(2 * N * SA_MAX_OPS, 1))()
    for i, ol in enumerate(op_lists):
        if len(ol) > SA_MAX_OPS:
            raise ValueError("at most four distortions per image")
        for k, (code, p0, p1) in enumerate(ol):
            j = i * SA_MAX_OPS + k
            codes[j] = int(code)
            params[2 * j] = float(p0)      # c_float rounds to float32 exactly like numpy's weak-scalar cast
            params[2 * j + 1] = float(p1)
    if out is None:
        out = torch.empty_like(imgs)
    elif out.shape != imgs.shape:
        raise ValueError("out must have the shape of imgs")
    _lib.call("pfst_photometric_u8", imgs.data_ptr(), _dev(out, "out", torch.uint8), N, H, W, codes, params,
              int(simd), _stream())
    return out


# --------------------------------------------- strong augmentation: colour jitter
def color_jitter(data: torch.Tensor, factors: Sequence[Sequence[float]], orders: Sequence[Sequence[int]],
                 mean: Optional[Sequence[float]] = None, std: Optional[Sequence[float]] = None,
                 out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """kornia ColorJitter arithmetic (0.6 series) on data (N,3,H,W) fp32 with host-drawn parameters:
    factors[i] = (brightness, contrast, saturation, hue), orders[i] = transform indices in application
    order (0 brightness, 1 contrast, 2 saturation, 3 hue). mean/std given: the reference's
    denorm_/renorm_ around it (dacs_transforms.py:48-53); None: data is already in [0,1]."""
    _dev(data, "data", torch.float32)
    if data.dim() != 4 or data.shape[1] != 3:
        raise ValueError("data must be (N,3,H,W)")
    N, _, H, W = data.shape
    if len(factors) != N or len(orders) != N:
        raise ValueError(f"need one (factors, order) per image ({N})")
    fa = (C.c_float * max(4 * N, 1))()
    oa = (C.c_int32 * max(4 * N, 1))()
    for i in range(N):
        if len(factors[i]) != 4 or len(orders[i]) > 4:
            raise ValueError("four factors and at most four transforms per image")
        for k in range(4):
            fa[4 * i + k] = float(factors[i][k])
            oa[4 * i + k] = int(orders[i][k]) if k < len(orders[i]) else -1
    if (mean is None) != (std is None):
        raise ValueError("give both mean and std, or neither")
    m = s = None
    if mean is not None:
        m, s = (C.c_float * 3)(*[float(x) for x in mean]), (C.c_float * 3)(*[float(x) for x in std])
    if out is None:
        out = torch.empty_like(data)
    elif out.shape != data.shape:
        raise ValueError("out must have the shape of data")
    _lib.call("pfst_color_jitter", data.data_ptr(), _dev(out, "out", torch.float32), N, H * W, fa, oa, m, s,
              int(mean is not None), _stream())
    return out


# --------------------------------------------- strong augmentation: Gaussian blur
def blur_kernel_size(n: int) -> int:
    """dacs_transforms.py:94-101: int(floor(ceil(0.1 n) - 0.5 + ceil(0.1 n) % 2)) (always odd)."""
    import math
    c = math.ceil(0.1 * n)
    return int(math.floor(c - 0.5 + c % 2))


def gaussian_blur(data: torch.Tensor, sigmas: Sequence[float], kernel_size: Optional[tuple] = None,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """kornia.filters.GaussianBlur2d(kernel_size, (sigma, sigma)) per image of data (N,C,H,W) fp32 with
    one sigma per image (host floats). kernel_size defaults to the reference's rule (~10 % of the size)."""
    _dev(data, "data", torch.float32)
    if data.dim() != 4:
        raise ValueError("data must be (N,C,H,W)")
    N, Cn, H, W = data.shape
    sig = [float(x) for x in sigmas]
    if len(sig) != N:
        raise ValueError(f"need one sigma per image ({N}), got {len(sig)}")
    ky, kx = kernel_size if kernel_size is not None else (blur_kernel_size(H), blur_kernel_size(W))
    if out is None:
        out = torch.empty_like(data)
    elif out.shape != data.shape or out.data_ptr() == data.data_ptr():
        raise ValueError("out must be a distinct tensor of the same shape")
    arr = (C.c_float * max(N, 1))(*sig)
    _lib.call("pfst_gaussian_blur", data.data_ptr(), _dev(out, "out", torch.float32), N, Cn, H, W,
              int(ky), int(kx), arr, _stream())
    return out


# ------------------------------------------------------- OHEM pixel sampler
def ohem_weight(seg_logit: torch.Tensor, seg_label: torch.Tensor, *, thresh: Optional[float] = None,
                min_kept: int = 100000, ignore_index: int = 255, class_weight: Optional[torch.Tensor] = None,
                loss_weight: float = 1.0, want_keys: bool = False):
    """mmseg OHEMPixelSampler.sample on the bilinear (align_corners=False) up-sampling of seg_logit (B,C,lh,lw;
    fp32, fp16 or bf16) to the size of seg_label ((B,1,H,W) or (B,H,W), int64 or uint8), an integer factor
    H/lh = W/lw >= 1. thresh None: the min_kept * B valid pixels of largest loss_weight * class_weight[label] *
    CE (ties at the boundary: lower flat index first); otherwise the valid pixels whose soft-max probability of
    their label is below max(k-th smallest of those, thresh). -> (weight (B,H,W) fp32 0/1, kth (1,) fp32 on the
    device: the order statistic the threshold came from, keys (B,H,W) fp32 or None)."""
    if int(min_kept) <= 1:
        raise ValueError(f"min_kept must be > 1 (mmseg OHEMPixelSampler), got {min_kept}")
    if isinstance(seg_logit, torch.Tensor) and seg_logit.dtype not in _FLOAT2DT:
        raise TypeError(f"seg_logit: logits must be torch.float32, torch.float16 or torch.bfloat16, "
                        f"got {seg_logit.dtype}")
    _dev(seg_logit, "seg_logit")
    if seg_logit.dim() != 4:
        raise ValueError("seg_logit must be (B,C,lh,lw)")
    if seg_label.dim() == 4:
        if seg_label.shape[1] != 1:
            raise ValueError("seg_label must be (B,1,H,W) or (B,H,W)")
        seg_label = seg_label[:, 0]
    _labels(seg_label, "seg_label")
    B, Cn, lh, lw = seg_logit.shape
    if seg_label.dim() != 3 or seg_label.shape[0] != B:
        raise ValueError("seg_label must hold one (H,W) map per image of seg_logit")
    H, W = seg_label.shape[-2:]
    if lh < 1 or lw < 1 or H % lh or W % lw or H // lh != W // lw:
        raise PfstError(f"ohem_weight: {lh}x{lw} logits -> {H}x{W} labels is not an integer up-sampling factor "
                        "(unsupported resampling)")
    if class_weight is not None:
        _dev(class_weight, "class_weight", torch.float32)
        if class_weight.numel() != Cn:
            raise ValueError("class_weight must have one entry per class")
    dev = seg_logit.device
    weight = torch.empty((B, H, W), dtype=torch.float32, device=dev)
    kth = torch.empty(1, dtype=torch.float32, device=dev)
    keys = torch.empty((B, H, W), dtype=torch.float32, device=dev) if want_keys else None
    ws = torch.empty(max(int(_lib.load().pfst_ohem_ws_bytes(B, H, W)), 16), dtype=torch.uint8, device=dev)
    launch_ohem_weight(seg_logit, seg_label, class_weight, ignore_index, loss_weight, thresh, min_kept, ws, keys, kth,
                       weight, _stream())
    return weight, kth, keys


def launch_ohem_weight(seg_logit, seg_label, class_weight, ignore_index, loss_weight, thresh, min_kept, ws, keys, kth,
                       weight, stream) -> None:
    """seg_label (B,H,W); thresh None selects the top-k mode (a NaN thresh in the C ABI)."""
    B, Cn, lh, lw = seg_logit.shape
    H, W = seg_label.shape[-2:]
    _lib.call("pfst_ohem_weight", seg_logit.data_ptr(), _FLOAT2DT[seg_logit.dtype], seg_label.data_ptr(),
              _TORCH2DT[seg_label.dtype], _ptr(class_weight), B, Cn, lh, lw, H, W, int(ignore_index),
              float(loss_weight), float("nan") if thresh is None else float(thresh), int(min_kept), ws.data_ptr(),
              _ptr(keys), _ptr(kth), weight.data_ptr(), stream)


# ------------------------------------------------------------ L1-L6: PFGST loss
def neigh_dots(x_a: torch.Tensor, x_b: Optional[torch.Tensor], dilation: int):
    """-> (dots float32 (splits, T, B, 5, h, w), splits). x_a / x_b: fp32, fp16 or bf16. Two fp32 tensors
    are one launch; otherwise each tensor is its own slot launch into the same buffer."""
    ta = _teacher(x_a, "x_a")
    B, D, h, w = x_a.shape
    T = 1
    if x_b is not None:
        tb = _teacher(x_b, "x_b")
        if x_b.shape != x_a.shape:
            raise ValueError("x_a / x_b shape mismatch")
        T = 2
        if ta != _lib.DT_F32 or tb != _lib.DT_F32:
            dots, ks = neigh_dots_slot(x_a, dilation, 0)
            neigh_dots_slot(x_b, dilation, 1, dots)
            return dots, ks
    ks = int(_lib.load().pfst_neigh_dots_splits(T, B, D, h, w))
    dots = torch.empty((ks, T, B, 5, h, w), dtype=torch.float32, device=x_a.device)
    _lib.call("pfst_neigh_dots", x_a.data_ptr(), None if x_b is None else x_b.data_ptr(), B, D, h, w,
              int(dilation), dots.data_ptr(), _stream())
    return dots, ks


def neigh_dots_splits(B: int, D: int, h: int, w: int, n_tensors: int = 1) -> int:
    return int(_lib.load().pfst_neigh_dots_splits(n_tensors, B, D, h, w))


def neigh_dots_slot(x: torch.Tensor, dilation: int, slot: int, dots: Optional[torch.Tensor] = None,
                    n_slots: int = 2):
    """One feature tensor into slot `slot` of a (splits, n_slots, B, 5, h, w) dots buffer
    (slot 0 = x_ema, slot 1 = x_src for the loss). x: fp32, fp16 or bf16. -> (dots, splits)."""
    fdt = _teacher(x, "x")
    B, D, h, w = x.shape
    ks = neigh_dots_splits(B, D, h, w)
    if dots is None:
        dots = torch.empty((ks, n_slots, B, 5, h, w), dtype=torch.float32, device=x.device)
    elif dots.numel() != ks * n_slots * B * 5 * h * w:
        raise ValueError("dots buffer has the wrong size")
    _lib.call("pfst_neigh_dots_slot", x.data_ptr(), fdt, B, D, h, w, int(dilation), int(slot), int(n_slots),
              _dev(dots, "dots", torch.float32), _stream())
    return dots, ks


def neigh_grad(x: torch.Tensor, coef: torch.Tensor, dilation: int, out: Optional[torch.Tensor] = None,
               proto: Optional[dict] = None) -> torch.Tensor:
    """grad_x of the neighbourhood-cosine losses; with `proto` (labels (B,H,W) int64 or uint8, mu, seen,
    dist, acc, grad_loss — the saved state of pfst_proto_dist_fwd) the prototype-distance
    gradient is added in the same pass over x."""
    _dev(x, "x", torch.float32)
    _dev(coef, "coef", torch.float32)
    B, _, h, w = x.shape
    if tuple(coef.shape) != (B, 9, h, w):
        raise ValueError("coef must be (B,9,h,w)")
    grad = torch.empty_like(x) if out is None else out
    _dev(grad, "grad_x", torch.float32)
    if proto is None:
        launch_neigh_grad(x, coef, dilation, grad, _stream())
    else:
        lab, mu, seen = proto["labels"], proto["mu"], proto.get("seen")
        _labels(lab, "labels")
        _dev(mu, "mu", torch.float32)
        _opt(seen, "seen", torch.uint8)
        _dev(proto["dist"], "dist", torch.float32)
        _dev(proto["acc"], "acc", torch.float64)
        _dev(proto["grad_loss"], "grad_loss", torch.float32)
        launch_neigh_grad_proto(x, coef, dilation, lab, mu, seen, proto["dist"], proto["acc"], proto["grad_loss"],
                                grad, _stream())
    return grad


def launch_neigh_grad(x, coef, dilation, grad_x, stream) -> None:
    B, D, h, w = x.shape
    _lib.call("pfst_neigh_grad", x.data_ptr(), coef.data_ptr(), B, D, h, w, int(dilation), grad_x.data_ptr(), stream)


def launch_neigh_grad_proto(x, coef, dilation, labels, mu, seen, dist, acc, grad_loss, grad_x, stream) -> None:
    """grad_loss: fp32 tensor whose first element is the upstream gradient of the prototype distance."""
    B, D, h, w = x.shape
    _lib.call("pfst_neigh_grad_proto", x.data_ptr(), coef.data_ptr(), B, D, h, w, int(dilation), labels.data_ptr(),
              _TORCH2DT[labels.dtype], labels.shape[-2], labels.shape[-1], mu.data_ptr(), _ptr(seen), mu.shape[0],
              dist.data_ptr(), acc.data_ptr(), grad_loss.data_ptr(), grad_x.data_ptr(), stream)


def launch_proto_dist_fwd(feats, labels, mu, seen, dist, acc, loss, stream) -> None:
    """mu: (C, D) prototypes; seen: uint8[C] or None."""
    B, D, h, w = feats.shape
    _lib.call("pfst_proto_dist_fwd", feats.data_ptr(), B, D, h, w, labels.data_ptr(), _TORCH2DT[labels.dtype],
              labels.shape[-2], labels.shape[-1], mu.data_ptr(), _ptr(seen), mu.shape[0], dist.data_ptr(),
              acc.data_ptr(), loss.data_ptr(), stream)


class LossGeometry:
    """Shapes / resampling factors of one PFGSTLoss call, derived as the reference does
    (pfgst_loss.py:56-67) and validated against what the kernels support."""

    def __init__(self, logits_shape, feat_shape, gt_shape, downscale, dilation: int):
        B, C, lh, lw = logits_shape
        if downscale is not None:
            gh, gw = int(lh * downscale), int(lw * downscale)   # F.interpolate(scale_factor): floor(in*s)
            ls = 1.0 / downscale
        else:
            gh, gw, ls = lh, lw, 1.0
        fh, fw = feat_shape[2], feat_shape[3]
        if gh < 1 or gw < 1 or gh % fh or gw % fw or gh // fh != gw // fw:
            raise PfstError(f"PFGSTLoss: loss grid {gh}x{gw} is not an integer up-sampling of the "
                            f"{fh}x{fw} feature grid (unsupported resampling)")
        up = gh // fh
        if dilation % up:
            raise PfstError(f"PFGSTLoss: dilation {dilation} is not a multiple of the feature up-sampling {up}")
        self.B, self.C, self.lh, self.lw = B, C, lh, lw
        self.fh, self.fw, self.up = fh, fw, up
        self.gh, self.gw = gh, gw
        self.lscale = ls
        self.gt_h, self.gt_w = gt_shape[-2], gt_shape[-1]
        self.dilation = int(dilation)


LOSS_SIM_GAUSSIAN, LOSS_CROSS_PROB_EMA, LOSS_UNFOLD_GRAD, LOSS_SRC_MARGIN, LOSS_SRC_MARGIN2 = 1, 2, 4, 8, 16   # PFST_LOSS_*


def _loss_options(options: int, logits_ema, geo: LossGeometry):
    if options & LOSS_CROSS_PROB_EMA:
        if logits_ema is None:
            raise PfstError("PFGSTLoss(cross_prob_type='ema') needs tensors['logits_ema']")
        _dev(logits_ema, "logits_ema", torch.float32)
        if tuple(logits_ema.shape) != (geo.B, geo.C, geo.gh, geo.gw):
            # the reference multiplies p (B,C,H,W,k) with unfold(softmax(logits_ema)) element-wise
            # (pfgst_loss.py:175): any other shape fails there too
            raise PfstError(f"PFGSTLoss(cross_prob_type='ema'): logits_ema {tuple(logits_ema.shape)} must have the "
                            f"loss-grid shape {(geo.B, geo.C, geo.gh, geo.gw)} (the reference broadcasts p * q)")
        return logits_ema
    return None


def pfgst_loss_fwd(dots, ks, geo: LossGeometry, logits, gt, mix, top_k, weights6, want_vis=True,
                   options: int = 0, sigma: float = 30.0, logits_ema=None, margin=None):
    """gt / mix: int64 or uint8, one dtype.
    -> (losses float32[6], (stats float64[16], workspace), density|None, eroded|None)."""
    dev = logits.device
    _dev(dots, "dots", torch.float32)
    _dev(logits, "logits", torch.float32)
    _labels(gt, "gt")
    _labels(mix, "mix", like=gt)
    logits_ema = _loss_options(options, logits_ema, geo)
    stats = torch.empty(16, dtype=torch.float64, device=dev)
    ws = torch.empty(pfgst_loss_ws_bytes(geo, options), dtype=torch.uint8, device=dev)
    losses = torch.empty(6, dtype=torch.float32, device=dev)
    density = torch.empty((geo.B, 1, geo.gh, geo.gw), dtype=torch.float32, device=dev) if want_vis else None
    eroded = torch.empty((geo.B, 1, geo.gh, geo.gw), dtype=torch.uint8, device=dev) if want_vis else None
    args = pfgst_loss_args(dots, ks, geo, logits, gt, mix, top_k, weights6, ws, stats)
    launch_pfgst_loss_fwd(args, losses, density, eroded, _stream(), options, sigma, logits_ema, margin)
    return losses, (stats, ws), density, eroded


def pfgst_loss_bwd(dots, ks, geo: LossGeometry, logits, gt, mix, top_k, weights6, stats, grad_losses,
                   want_logits_grad=True, options: int = 0, sigma: float = 30.0, logits_ema=None, margin=None):
    """-> (coef (B,9,fh,fw), grad_logits|None)."""
    dev = logits.device
    _dev(grad_losses, "grad_losses", torch.float32)
    _labels(gt, "gt")
    _labels(mix, "mix", like=gt)
    logits_ema = _loss_options(options, logits_ema, geo)
    stats, ws = stats
    coef = torch.empty((geo.B, 9, geo.fh, geo.fw), dtype=torch.float32, device=dev)
    glog = torch.empty_like(logits) if want_logits_grad else None
    args = pfgst_loss_args(dots, ks, geo, logits, gt, mix, top_k, weights6, ws, stats)
    launch_pfgst_loss_bwd(args, grad_losses, coef, glog, _stream(), options, sigma, logits_ema, margin)
    return coef, glog


def pfgst_loss_ws_bytes(geo: LossGeometry, options: int = 0) -> int:
    """Bytes of the workspace pfgst_loss_fwd leaves for pfgst_loss_bwd."""
    return int(_lib.load().pfst_pfgst_loss_ws_bytes(geo.B, geo.C, geo.fh, geo.fw, geo.up, int(options)))


def pfgst_loss_args(dots, ks, geo: LossGeometry, logits, gt, mix, top_k, weights6, ws, stats) -> tuple:
    """The arguments pfst_pfgst_loss_fwd and _bwd share, marshalled once: addresses, not tensors, so that a
    caller can keep them from the forward to the backward without keeping the inputs alive."""
    w6 = (C.c_float * 6)(*[float(v) for v in weights6])
    return ((dots.data_ptr(), ks, geo.B, geo.fh, geo.fw, geo.up, logits.data_ptr(), geo.C, geo.lh, geo.lw,
             geo.lscale, geo.lscale, gt.data_ptr(), mix.data_ptr(), geo.gt_h, geo.gt_w, geo.dilation, int(top_k), w6,
             ws.data_ptr(), stats.data_ptr()), _TORCH2DT[gt.dtype])


def _margin(margin):
    return None if margin is None else (C.c_float * 2)(float(margin[0]), float(margin[1]))


# options = 0 is the shipped configuration: sigma, logits_ema and margin are then not read
def launch_pfgst_loss_fwd(args, losses, density, eroded, stream, options: int = 0, sigma: float = 0.0,
                          logits_ema=None, margin=None) -> None:
    common, ldt = args
    _lib.call("pfst_pfgst_loss_fwd", *common, losses.data_ptr(), _ptr(density), _ptr(eroded), int(options),
              float(sigma), _ptr(logits_ema), _margin(margin), ldt, stream)


def launch_pfgst_loss_bwd(args, grad_losses, coef, grad_logits, stream, options: int = 0, sigma: float = 0.0,
                          logits_ema=None, margin=None) -> None:
    common, ldt = args
    _lib.call("pfst_pfgst_loss_bwd", *common, grad_losses.data_ptr(), _ptr(coef), _ptr(grad_logits), int(options),
              float(sigma), _ptr(logits_ema), _margin(margin), ldt, stream)
