"""Minimal stand-in for the mmcv Registry the reference plugs into
(rsiseg/models/builder.py:8-17: `UDA = MODELS`, `LOSSES = MODELS`; build via
`Registry.build(cfg)` with cfg['type'] naming the class). When mmcv IS installed,
`register_into(mmcv_registry)` re-registers the B200 classes under the same names
so that `uda.type='PFGST'` / `type='PFGSTLoss'` configs resolve to them
(INTEGRATION.md)."""
from __future__ import annotations


class Registry:
    def __init__(self, name: str):
        self.name = name
        self._modules: dict[str, type] = {}

    def register_module(self, name=None, force=False, module=None):
        def deco(cls):
            key = name or cls.__name__
            if key in self._modules and not force:
                raise KeyError(f"{key} is already registered in {self.name}")
            self._modules[key] = cls
            return cls
        if module is not None:
            return deco(module)
        return deco

    def get(self, key):
        return self._modules.get(key)

    def build(self, cfg, **default_args):
        cfg = dict(cfg)
        typ = cfg.pop("type")
        cls = typ if isinstance(typ, type) else self._modules.get(typ)
        if cls is None:
            raise KeyError(f"{typ} is not in the {self.name} registry")
        for k, v in default_args.items():
            cfg.setdefault(k, v)
        return cls(**cfg)

    def register_into(self, other) -> None:
        for key, cls in self._modules.items():
            other.register_module(name=key, force=True, module=cls)


MODELS = Registry("models")
UDA = MODELS
LOSSES = MODELS
SEGMENTORS = MODELS
PIPELINES = Registry("pipeline")       # rsiseg/datasets/builder.py: PIPELINES = Registry('pipeline')
PIXEL_SAMPLERS = Registry("pixel sampler")   # mmseg/core/builder.py: PIXEL_SAMPLERS = Registry('pixel sampler')


def build_loss(cfg):
    return LOSSES.build(cfg)


def build_pixel_sampler(cfg, **default_args):
    """mmseg's builder: a decode head calls build_pixel_sampler(self.sampler_cfg, context=self)."""
    return PIXEL_SAMPLERS.build(cfg, **default_args)


def build_segmentor(cfg, train_cfg=None, test_cfg=None):
    return SEGMENTORS.build(cfg)
