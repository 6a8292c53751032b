"""ctypes binding of libpfst_sm100.so (see include/pfst_sm100.h).

There is no CPU or PyTorch fallback: if the shared library is missing, or a
compute entry point fails, a :class:`PfstError` is raised.
"""
from __future__ import annotations

import ctypes as C
import threading
from pathlib import Path

import os

# PFST_LIB overrides the library path (A/B experiments with alternative builds only)
LIB_PATH = Path(os.environ.get("PFST_LIB") or (Path(__file__).resolve().parent / "csrc" / "libpfst_sm100.so"))

PFST_OK = 0
DT_U8, DT_I32, DT_I64 = 0, 1, 2
DT_F32, DT_F16, DT_BF16 = 16, 17, 18


class PfstError(RuntimeError):
    pass


_vp, _i32, _i64, _f32, _f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_double

# name -> (restype, argtypes); mirrors include/pfst_sm100.h one to one
SIGNATURES: dict[str, tuple] = {
    "pfst_version": (C.c_char_p, []),
    "pfst_error_string": (C.c_char_p, [C.c_int]),
    "pfst_last_cuda_error": (C.c_char_p, []),
    "pfst_device_check": (C.c_int, []),
    "pfst_copy_async": (C.c_int, [_vp, _vp, _i64, _vp]),
    "pfst_classmix_draw": (C.c_int, [_vp, _i64, _vp, _i32, _i32, _vp, _vp, _vp]),   # host-only (no device work)
    "pfst_ema_coeffs": (C.c_int, [_i64, _f64, C.POINTER(_f32), C.POINTER(_f32)]),
    "pfst_ema_update_multi": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _f32, _f32, _i32, _i32, _vp]),
    "pfst_ema_update_multi_dev": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp, _i32, _vp]),
    "pfst_ema_update_flat": (C.c_int, [_vp, _vp, _i64, _f32, _f32, _i32, _vp]),
    "pfst_pseudo_label": (C.c_int, [_vp, _i32, _i64, _i32, _i64, _f32, _vp, _i32, _i64, _vp, _i32, _vp, _vp, _vp,
                                    _vp]),
    "pfst_selftest_exp": (C.c_int, [_vp, _i64, _vp, _vp]),
    "pfst_pseudo_weight_fill": (C.c_int, [_vp, _i64, _i64, _i64, _vp, _i64, _i32, _i32, _vp]),
    "pfst_class_presence": (C.c_int, [_vp, _i32, _i64, _vp, _vp]),
    "pfst_class_mix": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _i32, _i64, _i32,
                                 _i64, _i64, _vp, _vp, _vp, _vp, _i32, _vp]),
    "pfst_mask_mix": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i64, _i64, _vp]),
    "pfst_neigh_dots_splits": (_i32, [_i64, _i64, _i32, _i32, _i32]),
    "pfst_neigh_dots": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _i32, _i32, _vp, _vp]),
    "pfst_neigh_grad": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _i32, _i32, _vp, _vp]),
    "pfst_neigh_dots_slot": (C.c_int, [_vp, _i32, _i64, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    "pfst_neigh_grad_proto": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _i32, _i32, _vp, _i32, _i32, _i32, _vp, _vp,
                                        _i32, _vp, _vp, _vp, _vp, _vp]),
    "pfst_pfgst_loss_ws_bytes": (_i64, [_i64, _i32, _i32, _i32, _i32, _i32]),
    "pfst_pfgst_loss_fwd": (C.c_int, [_vp, _i32, _i64, _i32, _i32, _i32, _vp, _i32, _i32, _i32, _f32, _f32,
                                      _vp, _vp, _i32, _i32, _i32, _i32, C.POINTER(_f32), _vp, _vp, _vp, _vp, _vp,
                                      _i32, _f32, _vp, C.POINTER(_f32), _i32, _vp]),
    "pfst_pfgst_loss_bwd": (C.c_int, [_vp, _i32, _i64, _i32, _i32, _i32, _vp, _i32, _i32, _i32, _f32, _f32,
                                      _vp, _vp, _i32, _i32, _i32, _i32, C.POINTER(_f32), _vp, _vp, _vp, _vp, _vp,
                                      _i32, _f32, _vp, C.POINTER(_f32), _i32, _vp]),
    "pfst_slide_add": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp]),
    "pfst_slide_finalize": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    "pfst_softmax_accum": (C.c_int, [_vp, _vp, _i64, _i32, _i64, _i32, _vp]),
    "pfst_div_argmax": (C.c_int, [_vp, _i64, _i32, _i64, _f32, _vp, _vp]),
    "pfst_class_quantile_ws_bytes": (_i64, [_i64, _i32, _i32]),
    "pfst_class_quantile": (C.c_int, [_vp, _i64, _i32, _i64, _vp, _i64, _vp, _i32, _vp, _vp, _vp]),
    "pfst_weighted_ce": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _i64, _i32, _i32, _i32, _i32, _i32, _i64, _f32, _vp,
                                   _vp, _vp, _vp]),
    "pfst_weighted_ce_dt": (C.c_int, [_vp, _i32, _vp, _i32, _vp, _vp, _i64, _i32, _i32, _i32, _i32, _i32, _i64,
                                      _f32, _vp, _vp, _vp, _vp]),
    "pfst_scale_cast": (C.c_int, [_vp, _vp, _i64, _vp, _i32, _vp]),
    "pfst_ohem_ws_bytes": (_i64, [_i64, _i32, _i32]),
    "pfst_ohem_weight": (C.c_int, [_vp, _i32, _vp, _i32, _vp, _i64, _i32, _i32, _i32, _i32, _i32, _i64, _f32, _f32,
                                   _i64, _vp, _vp, _vp, _vp, _vp]),
    "pfst_proto_accum_is_masked": (C.c_int, [_i32, _i32, _i32]),
    "pfst_proto_accum": (C.c_int, [_vp, _i32, _i64, _i32, _i32, _i32, _vp, _i32, _i32, _i32, _vp, _f32, _i32, _vp,
                                   _vp]),
    "pfst_proto_order_ws_bytes": (_i64, [_i64, _i32, _i32, _i32]),
    "pfst_proto_order": (C.c_int, [_vp, _i32, _i64, _i32, _i32, _i32, _i32, _vp, _f32, _i32, _vp, _vp, _vp]),
    "pfst_proto_accum_ordered": (C.c_int, [_vp, _i32, _i64, _i32, _i32, _i32, _i32, _vp, _vp, _vp]),
    "pfst_proto_finalize": (C.c_int, [_vp, _i32, _i32, _vp, _vp, _f64, _vp, _vp, _vp, _vp, _i32, _vp]),
    "pfst_feat_dist_fwd": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "pfst_feat_dist_bwd": (C.c_int, [_vp, _vp, _vp, _i64, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pfst_peer_board_bytes": (_i64, [_i32, _i32, _i32, C.POINTER(_i64), C.POINTER(_i64)]),
    "pfst_peer_alloc": (C.c_int, [_i64, C.POINTER(_vp), _vp]),
    "pfst_peer_open": (C.c_int, [_vp, C.POINTER(_vp)]),
    "pfst_peer_close": (C.c_int, [_vp]),
    "pfst_peer_free": (C.c_int, [_vp]),
    "pfst_proto_finalize_peer": (C.c_int, [_vp, _i32, _i32, _vp, _vp, _f64, _vp, _vp, _vp, _vp, _vp, _i32, _i32,
                                           _vp, _i64, _vp]),
    "pfst_loc_dis": (C.c_int, [_vp, _i64, _i32, _i32, _i32, _i32, _vp, _vp]),
    "pfst_gather_rows": (C.c_int, [_vp, _vp, _i64, _i32, _vp, _vp]),
    "pfst_sigma_bisect": (C.c_int, [_vp, _i64, _f32, _f64, _f64, _i32, _vp, _vp]),
    "pfst_loader_pseudo_labels": (C.c_int, [_vp, _i64, _i32, _i64, _vp, _i32, _vp, _vp]),
    "pfst_gather_scalars": (C.c_int, [_vp, _vp, _i32, C.c_uint32, _f32, _vp, _vp, _vp]),
    "pfst_gather_segments": (C.c_int, [_vp, _vp, _vp, _i32, _f32, _vp, _vp, _vp]),
    "pfst_pack_scalars": (C.c_int, [_vp, _vp, _i32, _vp, _vp]),
    "pfst_proto_dist_fwd": (C.c_int, [_vp, _i64, _i32, _i32, _i32, _vp, _i32, _i32, _i32, _vp, _vp, _i32, _vp, _vp,
                                      _vp, _vp]),
    "pfst_proto_dist_bwd": (C.c_int, [_vp, _i64, _i32, _i32, _i32, _vp, _i32, _i32, _i32, _vp, _vp, _i32, _vp, _vp,
                                      _vp, _vp, _i32, _vp]),
    "pfst_proto_dist_all": (C.c_int, [_vp, _i64, _i32, _i32, _i32, _vp, _i32, _vp, _vp]),
    "pfst_confusion_accum": (C.c_int, [_vp, _i32, _vp, _i32, _i64, _i64, _i32, _i64, _i32, _vp, _vp,
                                       _i32, _vp]),
    "pfst_gaussian_blur": (C.c_int, [_vp, _vp, _i64, _i32, _i32, _i32, _i32, _i32, C.POINTER(_f32), _vp]),
    "pfst_photometric_u8": (C.c_int, [_vp, _vp, _i64, _i32, _i32, C.POINTER(_i32), C.POINTER(_f32), _i32, _vp]),
    "pfst_color_jitter": (C.c_int, [_vp, _vp, _i64, _i64, C.POINTER(_f32), C.POINTER(_i32), C.POINTER(_f32),
                                    C.POINTER(_f32), _i32, _vp]),
    "pfst_argmax_confusion": (C.c_int, [_vp, _i64, _i32, _i64, _vp, _i32, _i64, _i32, _vp, _vp, _i32, _vp, _i32,
                                        _vp]),
}

_lock = threading.Lock()
_lib = None


def load() -> C.CDLL:
    """Load the shared library (once). Raises PfstError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not LIB_PATH.exists():
            raise PfstError(
                f"{LIB_PATH} not found: build it with `python -m pfst_b200.build` "
                "(nvcc, sm_100a). pfst_b200 has no CPU/PyTorch fallback.")
        lib = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError here = header/library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(code: int, what: str) -> None:
    if code == PFST_OK:
        return
    lib = load()
    msg = lib.pfst_error_string(code).decode()
    if code == -3:
        msg += ": " + lib.pfst_last_cuda_error().decode()
    raise PfstError(f"{what} failed ({code}): {msg}")


_DEBUG_SYNC = bool(os.environ.get("PFST_DEBUG_SYNC"))


def call(name: str, *args) -> None:
    check(getattr(load(), name)(*args), name)
    if _DEBUG_SYNC:                       # development aid: attribute an asynchronous fault to its launch
        import torch
        try:
            torch.cuda.synchronize()
        except Exception as exc:
            raise PfstError(f"{name}: device fault surfaced after this launch: {exc}") from exc
