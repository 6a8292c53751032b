"""Load the reference's hot-path modules BY FILE PATH from a read-only checkout.

Only usable where PFST_REFERENCE names a checkout of the reference. Used by
make_golden.py to produce the committed fixtures and by the `-m "not gpu"` pinning
tests, which then also compare the oracle with the reference live (without it they
compare with the committed fixtures only). Nothing is copied: the files are executed where they lie
with small import stubs for packages that are not installed here (mmcv,
matplotlib, timm, the rsiseg package __init__ that asserts an mmcv version).
SURVEY.md Appendix D is the recipe.
"""
from __future__ import annotations

import importlib.util
import os
import sys
import types
from pathlib import Path

REF_ROOT = Path(os.environ["PFST_REFERENCE"]) if os.environ.get("PFST_REFERENCE") else None


def available() -> bool:
    return REF_ROOT is not None and (REF_ROOT / "rsiseg" / "models" / "uda" / "pfgst.py").exists()


def _load(name: str, rel: str):
    spec = importlib.util.spec_from_file_location(name, REF_ROOT / rel)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def _stub(name: str, **attrs):
    mod = sys.modules.get(name)
    if mod is None:
        mod = types.ModuleType(name)
        mod.__path__ = []  # behaves as a package for submodule imports
        sys.modules[name] = mod
    for k, v in attrs.items():
        setattr(mod, k, v)
    return mod


class _Registry:
    def __init__(self):
        self.modules = {}

    def register_module(self, *a, **k):
        def deco(cls):
            self.modules[cls.__name__] = cls
            return cls
        return deco


_cache: dict = {}


def dacs_transforms():
    # color_jitter / gaussian_blur do `import kornia` before testing whether they are active;
    # an empty stand-in lets the inactive branches (jitter_p=1.0, blur=False) run. Any real
    # use of kornia fails loudly with AttributeError.
    if "kornia" not in sys.modules:
        sys.modules["kornia"] = types.ModuleType("kornia")
    if "dacs" not in _cache:
        _cache["dacs"] = _load("_pfst_ref_dacs_transforms", "rsiseg/models/utils/dacs_transforms.py")
    return _cache["dacs"]


def metrics():
    if "metrics" not in _cache:
        had = "mmcv" in sys.modules
        _stub("mmcv")
        _cache["metrics"] = _load("_pfst_ref_metrics", "rsiseg/core/evaluation/metrics.py")
        if not had:
            sys.modules.pop("mmcv", None)
    return _cache["metrics"]


def pfgst_loss():
    """-> module with class PFGSTLoss (CPU: torch.Tensor.cuda must be patched by the caller
    through `cpu_cuda_identity()` because pfgst_loss.py:225-226 hard-codes .cuda())."""
    if "loss" not in _cache:
        pkg = "_pfst_ref_models"
        _stub(pkg)
        _stub(pkg + ".builder", LOSSES=_Registry())
        _stub(pkg + ".losses")
        _stub(pkg + ".losses.utils", get_class_weight=lambda *a, **k: None,
              weight_reduce_loss=lambda *a, **k: None)
        _cache["loss"] = _load(pkg + ".losses.pfgst_loss", "rsiseg/models/losses/pfgst_loss.py")
    return _cache["loss"]


def decode_head_loss_fns():
    """-> (resize, cross_entropy, accuracy): rsiseg/ops/wrappers.py, rsiseg/models/losses/
    cross_entropy_loss.py (with its real losses/utils.py) and accuracy.py, loaded by path."""
    if "ce" not in _cache:
        had = "mmcv" in sys.modules
        _stub("mmcv")
        pkg = "_pfst_ref_ce"
        _stub(pkg)
        _stub(pkg + ".builder", LOSSES=_Registry())
        _stub(pkg + ".losses")
        _load(pkg + ".losses.utils", "rsiseg/models/losses/utils.py")
        ce = _load(pkg + ".losses.cross_entropy_loss", "rsiseg/models/losses/cross_entropy_loss.py")
        acc = _load(pkg + ".losses.accuracy", "rsiseg/models/losses/accuracy.py")
        wr = _load("_pfst_ref_wrappers", "rsiseg/ops/wrappers.py")
        if not had:
            sys.modules.pop("mmcv", None)
        _cache["ce"] = (wr.resize, ce.cross_entropy, acc.accuracy)
    return _cache["ce"]


def cal_threshold_fn():
    """PseudoLabelingHookV4._cal_threshold compiled straight from the reference source file
    (rsiseg/core/hook/pseudo_labeling_hookv4.py:173-205; its module needs mmcv / h5py)."""
    if "calthr" not in _cache:
        import ast
        import numpy as np
        import torch
        import torch.nn.functional as F
        tree = ast.parse((REF_ROOT / "rsiseg/core/hook/pseudo_labeling_hookv4.py").read_text())
        fn = next(n for n in ast.walk(tree) if isinstance(n, ast.FunctionDef) and n.name == "_cal_threshold")
        ns = {"np": np, "torch": torch, "F": F}
        exec(compile(ast.Module(body=[fn], type_ignores=[]), "ref:pseudo_labeling_hookv4.py:_cal_threshold", "exec"), ns)
        _cache["calthr"] = ns["_cal_threshold"]
    return _cache["calthr"]


def hook_sigma_fns():
    """(PseudoLabelingHookV4._cal_loc_dis, ._cal_sigmas) compiled straight from the reference source
    (rsiseg/core/hook/pseudo_labeling_hookv4.py:208-277); `tqdm.tqdm` is the identity here."""
    if "hooksig" not in _cache:
        import ast
        import numpy as np
        import torch
        tree = ast.parse((REF_ROOT / "rsiseg/core/hook/pseudo_labeling_hookv4.py").read_text())
        fns = [n for n in ast.walk(tree) if isinstance(n, ast.FunctionDef) and n.name in ("_cal_loc_dis", "_cal_sigmas")]
        ns = {"np": np, "torch": torch, "tqdm": types.SimpleNamespace(tqdm=lambda it, *a, **k: it)}
        exec(compile(ast.Module(body=fns, type_ignores=[]), "ref:pseudo_labeling_hookv4.py:_cal_sigmas", "exec"), ns)
        _cache["hooksig"] = (ns["_cal_loc_dis"], ns["_cal_sigmas"])
    return _cache["hooksig"]


class _FakeH5File(dict):
    """Stands in for h5py.File(path, 'r') in the loader: a dict of datasets registered by path."""
    registry: dict = {}

    def __init__(self, path, mode='r'):
        super().__init__(_FakeH5File.registry[path])

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        return False

    def close(self):
        pass


def loader_pseudo_labels_cls():
    """-> (LoadAnnotationsPseudoLabelsV2 compiled from rsiseg/datasets/pipelines/loading.py:391-526,
    the registry dict its fake `h5py.File` reads from: {path: {'seg_logits': ..., 'thre@r': ...}})."""
    if "loadercls" not in _cache:
        import ast
        import os.path as osp
        import numpy as np
        tree = ast.parse((REF_ROOT / "rsiseg/datasets/pipelines/loading.py").read_text())
        cls = next(n for n in ast.walk(tree) if isinstance(n, ast.ClassDef) and n.name == "LoadAnnotationsPseudoLabelsV2")
        cls.decorator_list = []
        ns = {"np": np, "osp": osp, "h5py": types.SimpleNamespace(File=_FakeH5File)}
        exec(compile(ast.Module(body=[cls], type_ignores=[]), "ref:loading.py:LoadAnnotationsPseudoLabelsV2", "exec"), ns)
        _cache["loadercls"] = (ns["LoadAnnotationsPseudoLabelsV2"], _FakeH5File.registry)
    return _cache["loadercls"]


def simple_test_fns():
    """-> (inference, simple_test): EncoderDecoder.inference / simple_test compiled straight from
    the reference source file (rsiseg/models/segmentors/encoder_decoder.py:283-353; its module
    needs mmcv). Usable unbound on a duck-typed object that supplies `test_cfg.mode`,
    `whole_inference` (the network pass, replaced by synthetic logits) and `inference`."""
    if "simple_test" not in _cache:
        import ast
        import torch
        import torch.nn.functional as F

        class DataContainer:  # mmcv.parallel.DataContainer: only used in an isinstance test
            pass

        tree = ast.parse((REF_ROOT / "rsiseg/models/segmentors/encoder_decoder.py").read_text())
        fns = [n for n in ast.walk(tree) if isinstance(n, ast.FunctionDef) and n.name in ("inference", "simple_test")]
        assert len(fns) == 2
        ns = {"torch": torch, "F": F, "DataContainer": DataContainer}
        exec(compile(ast.Module(body=fns, type_ignores=[]), "ref:encoder_decoder.py", "exec"), ns)
        _cache["simple_test"] = (ns["inference"], ns["simple_test"])
    return _cache["simple_test"]


def inference_fns():
    """-> dict of EncoderDecoder.{slide_inference, whole_inference, inference, simple_test, aug_test} compiled
    straight from the reference source (rsiseg/models/segmentors/encoder_decoder.py:220-373); `resize` is
    the reference's own rsiseg/ops/wrappers.py function. Usable unbound on a duck-typed object that
    supplies test_cfg, num_classes, align_corners and encode_decode."""
    if "inference_fns" not in _cache:
        import ast
        import torch
        import torch.nn.functional as F

        class DataContainer:
            pass

        names = ("slide_inference", "whole_inference", "inference", "simple_test", "aug_test")
        tree = ast.parse((REF_ROOT / "rsiseg/models/segmentors/encoder_decoder.py").read_text())
        fns = [n for n in ast.walk(tree) if isinstance(n, ast.FunctionDef) and n.name in names]
        assert len(fns) == len(names)
        ns = {"torch": torch, "F": F, "DataContainer": DataContainer, "resize": decode_head_loss_fns()[0]}
        exec(compile(ast.Module(body=fns, type_ignores=[]), "ref:encoder_decoder.py", "exec"), ns)
        _cache["inference_fns"] = {k: ns[k] for k in names}
    return _cache["inference_fns"]


def reference_segmentor(encode_decode, test_cfg, num_classes, align_corners=False):
    """A duck-typed EncoderDecoder whose four inference methods are the reference's own code and whose
    network pass is `encode_decode(img, img_meta) -> (seg_logit, states)`."""
    import types
    f = inference_fns()
    obj = types.SimpleNamespace(test_cfg=test_cfg, num_classes=num_classes, align_corners=align_corners,
                                encode_decode=encode_decode)
    for k, fn in f.items():
        setattr(obj, k, (lambda fn: lambda *a, **kw: fn(obj, *a, **kw))(fn))
    return obj


def simple_test_on_logits(seg_logits):
    """Run the reference's inference + simple_test on synthetic logits (whole mode, no flip)
    -> list of per-image int64 numpy arg-max maps, as simple_test returns them."""
    import types
    inference, simple_test = simple_test_fns()
    obj = types.SimpleNamespace(test_cfg=types.SimpleNamespace(mode="whole"))
    obj.whole_inference = lambda img, img_meta, rescale: (seg_logits, {})
    obj.inference = lambda img, img_meta, rescale: inference(obj, img, img_meta, rescale)
    meta = [dict(ori_shape=tuple(seg_logits.shape[2:]) + (3,), flip=False)]
    seg_pred, _ = simple_test(obj, None, meta, True)
    return seg_pred


def strong_augmentation_cls():
    """-> the reference's StrongAugmentation class compiled straight from its source
    (rsiseg/datasets/pipelines/transforms.py:1061-1155; the module imports mmcv and skimage).
    `mmcv.bgr2hsv` / `mmcv.hsv2bgr` are what mmcv defines them as: cv2.cvtColor with
    COLOR_BGR2HSV / COLOR_HSV2BGR (mmcv/image/colorspace.py convert_color_factory)."""
    if "strongaug" not in _cache:
        import ast
        import cv2
        import numpy as np
        tree = ast.parse((REF_ROOT / "rsiseg/datasets/pipelines/transforms.py").read_text())
        cls = next(n for n in ast.walk(tree) if isinstance(n, ast.ClassDef) and n.name == "StrongAugmentation")
        cls.decorator_list = []
        mmcv = types.SimpleNamespace(bgr2hsv=lambda img: cv2.cvtColor(img, cv2.COLOR_BGR2HSV),
                                     hsv2bgr=lambda img: cv2.cvtColor(img, cv2.COLOR_HSV2BGR))
        ns = {"np": np, "random": np.random, "mmcv": mmcv}       # transforms.py:4 `from numpy import random`
        exec(compile(ast.Module(body=[cls], type_ignores=[]), "ref:transforms.py:StrongAugmentation", "exec"), ns)
        _cache["strongaug"] = ns["StrongAugmentation"]
    return _cache["strongaug"]


class cpu_cuda_identity:
    """Context manager: make Tensor.cuda() the identity on a CUDA-less host."""

    def __enter__(self):
        import torch
        self._orig = torch.Tensor.cuda
        if not torch.cuda.is_available():
            torch.Tensor.cuda = lambda self, *a, **k: self
        return self

    def __exit__(self, *exc):
        import torch
        torch.Tensor.cuda = self._orig
        return False


def _extract_parse_losses():
    """Compile BaseSegmentor._parse_losses straight from the reference source file
    (rsiseg/models/segmentors/base.py:177-222) without importing its mmcv-bound module."""
    import ast
    from collections import OrderedDict
    import torch
    import torch.distributed as dist
    src = (REF_ROOT / "rsiseg/models/segmentors/base.py").read_text()
    tree = ast.parse(src)
    for node in ast.walk(tree):
        if isinstance(node, ast.FunctionDef) and node.name == "_parse_losses":
            node.decorator_list = []
            mod = ast.Module(body=[node], type_ignores=[])
            ns = {"torch": torch, "dist": dist, "OrderedDict": OrderedDict}
            exec(compile(mod, "ref:base.py:_parse_losses", "exec"), ns)
            return ns["_parse_losses"]
    raise RuntimeError("_parse_losses not found in the reference")


def pfgst():
    """-> module rsiseg/models/uda/pfgst.py with class PFGST (methods usable unbound on a
    duck-typed object; the segmentor passes are supplied by the caller)."""
    if "pfgst" not in _cache:
        import torch.nn as nn

        saved = {k: sys.modules.get(k) for k in (
            "mmcv", "mmcv.parallel", "matplotlib", "matplotlib.pyplot", "timm", "timm.models",
            "timm.models.layers", "rsiseg", "rsiseg.core", "rsiseg.models", "rsiseg.models.uda",
            "rsiseg.models.uda.uda_decorator", "rsiseg.models.utils",
            "rsiseg.models.utils.dacs_transforms")}
        dacs = dacs_transforms()
        mloss = pfgst_loss()

        class _DropPath(nn.Module):
            pass

        class _MMDDP(nn.Module):
            pass

        uda_reg, loss_reg = _Registry(), _Registry()
        _stub("mmcv", print_log=lambda *a, **k: None)
        _stub("mmcv.parallel", MMDistributedDataParallel=_MMDDP)
        _stub("matplotlib")
        _stub("matplotlib.pyplot")
        _stub("timm")
        _stub("timm.models")
        _stub("timm.models.layers", DropPath=_DropPath)

        def add_prefix(inputs, prefix):  # rsiseg/core/utils/misc.py:2-18 (glue)
            return {f"{prefix}.{k}": v for k, v in inputs.items()}

        builder = types.SimpleNamespace(
            build_loss=lambda cfg: mloss.PFGSTLoss(**{k: v for k, v in cfg.items() if k != "type"}))
        _stub("rsiseg")
        _stub("rsiseg.core", add_prefix=add_prefix)
        class BaseSegmentor(nn.Module):
            """stand-in for rsiseg/models/segmentors/base.py (needs mmcv.runner); only
            _parse_losses is used by PFGST and it is compiled from the reference source."""
            _parse_losses = staticmethod(_extract_parse_losses())

            def forward(self, *args, return_loss=True, **kwargs):  # base.py:101-115 (auto_fp16 no-op)
                return self.forward_train(*args, **kwargs)

        _stub("rsiseg.models", UDA=uda_reg, build_segmentor=lambda cfg: cfg["_instance_factory"](),
              builder=builder, BaseSegmentor=BaseSegmentor)
        _stub("rsiseg.models.uda")
        _stub("rsiseg.models.utils")
        sys.modules["rsiseg.models.utils.dacs_transforms"] = dacs
        deco = _load("rsiseg.models.uda.uda_decorator", "rsiseg/models/uda/uda_decorator.py")
        mod = _load("_pfst_ref_pfgst", "rsiseg/models/uda/pfgst.py")
        mod._uda_decorator = deco
        _cache["pfgst"] = mod
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return _cache["pfgst"]
