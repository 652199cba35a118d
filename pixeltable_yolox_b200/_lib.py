"""ctypes binding of the C-ABI in include/yx_b200.h (libyx_b200.so).

The library is the product: there is NO CPU or PyTorch fallback behind these calls. If the
shared object is missing, `lib()` builds it with nvcc; if that is impossible it raises.
Every wrapper raises ``RuntimeError(yx_last_error())`` on a non-zero status.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path
from typing import Optional

PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("YX_B200_LIB") or PKG / "libyx_b200.so")   # YX_B200_LIB: A/B experiments with a second build

YX_BF16, YX_FP16, YX_FP32, YX_U8 = 0, 1, 2, 3
YX_ACT_NONE, YX_ACT_SILU, YX_ACT_RELU, YX_ACT_LRELU = 0, 1, 2, 3
YX_EPI_STORE, YX_EPI_HEAD = 0, 1
NMS_OFFSET, NMS_PER_CLASS, NMS_AGNOSTIC = 0, 1, 2

ACT_CODES = {"silu": YX_ACT_SILU, "relu": YX_ACT_RELU, "lrelu": YX_ACT_LRELU, None: YX_ACT_NONE, "none": YX_ACT_NONE}


class ConvDesc(C.Structure):
    """Mirror of ``yx_conv_desc`` (include/yx_b200.h)."""

    _fields_ = [
        ("batch", C.c_int32), ("in_h", C.c_int32), ("in_w", C.c_int32), ("in_c", C.c_int32),
        ("out_h", C.c_int32), ("out_w", C.c_int32), ("out_c", C.c_int32),
        ("ksize", C.c_int32), ("stride", C.c_int32),
        ("dtype", C.c_int32), ("act", C.c_int32), ("epilogue", C.c_int32),
        ("in_", C.c_void_p), ("in_ld", C.c_int64),
        ("w", C.c_void_p),
        ("bias", C.c_void_p),
        ("out", C.c_void_p), ("out_ld", C.c_int64),
        ("res", C.c_void_p), ("res_ld", C.c_int64),
        ("ups", C.c_void_p), ("ups_ld", C.c_int64),
        ("head_out", C.c_void_p),
        ("head_anchors", C.c_int32), ("head_anchor_off", C.c_int32), ("head_nc", C.c_int32),
        ("head_decode", C.c_int32),
        ("head_stride", C.c_float),
        ("out2_begin", C.c_int32),
        ("out2", C.c_void_p), ("out2_ld", C.c_int64),
        ("head_cand", C.c_void_p), ("head_keys", C.c_void_p), ("head_counts", C.c_void_p),
        ("head_conf_thre", C.c_float), ("head_xyxy", C.c_int32),
        ("shuffle2_c", C.c_int32),
    ]


class BneckDesc(C.Structure):
    """Mirror of ``yx_bneck_desc`` (include/yx_b200.h)."""

    _fields_ = [
        ("batch", C.c_int32), ("h", C.c_int32), ("w", C.c_int32), ("c", C.c_int32),
        ("dtype", C.c_int32), ("act", C.c_int32), ("use_add", C.c_int32),
        ("x", C.c_void_p), ("x_ld", C.c_int64),
        ("w1", C.c_void_p), ("bias1", C.c_void_p),
        ("w2", C.c_void_p), ("bias2", C.c_void_p),
        ("out", C.c_void_p), ("out_ld", C.c_int64),
    ]


_P, _I32, _I64, _F, _D = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_double

# name -> (restype, argtypes); mirrors include/yx_b200.h one to one
SIGNATURES = {
    "yx_strerror": (C.c_char_p, [C.c_int]),
    "yx_last_error": (C.c_char_p, []),
    "yx_version": (C.c_int, []),
    "yx_device_check": (C.c_int, [C.c_int]),
    "yx_conv_bn_act_fwd": (C.c_int, [C.POINTER(ConvDesc), _P]),
    "yx_conv_bn_act_fwd_simt": (C.c_int, [C.POINTER(ConvDesc), _P]),
    "yx_conv_schedule": (C.c_int, [C.POINTER(ConvDesc), _P, _I32]),
    "yx_bottleneck_fwd": (C.c_int, [C.POINTER(BneckDesc), _P]),
    "yx_bottleneck_supported": (C.c_int, [C.POINTER(BneckDesc)]),
    "yx_dwconv3x3_bn_act_fwd": (C.c_int, [_P, _I64, _P, _P, _P, _I64, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _P]),
    "yx_spp_maxpool": (C.c_int, [_P, _I64, _I32, _I32, _I32, _I32, _I32, _P]),
    "yx_focus_s2d": (C.c_int, [_P, _I32, _P, _I64, _I32, _I32, _I32, _I32, _P]),
    "yx_focus_conv_bn_act_fwd": (C.c_int, [_P, _I32, _P, _P, _P, _I64, _I32, _I32, _I32, _I32, _I32, _I32, _P]),
    "yx_pack_weights": (C.c_int, [_P, _P, _P, _P, _P, _P, _F, _I32, _I32, _I32, _I32, _P, _I32, _I32, _I32, _I32, _P, _I32, _P]),
    "yx_head_decode": (C.c_int, [_P, _I32, _I32, _I32, _P, _P, _I32, _P]),
    "yx_postprocess_workspace_bytes": (_I64, [_I32, _I32]),
    "yx_postprocess": (C.c_int, [_P, _I32, _I32, _I32, _F, _D, _I32, _I32, _P, _P, _P, _I32, _P, _I64, _P]),
    "yx_postprocess_workspace_ptrs": (C.c_int, [_P, _I32, _I32, _P, _P, _P]),
    "yx_postprocess_begin": (C.c_int, [_P, _I32, _I32, _P]),
    "yx_nms_prefiltered": (C.c_int, [_I32, _I32, _D, _I32, _P, _P, _P, _I32, _P, _I64, _P]),
    "yx_score_filter_compact": (C.c_int, [_P, _I32, _I32, _I32, _F, _P, _P, _P, _P, _I64, _P]),
    "yx_batched_nms": (C.c_int, [_P, _P, _P, _P, _I32, _I32, _D, _I32, _P, _P, _P, _I64, _P]),
    "yx_bboxes_iou": (C.c_int, [_P, _I32, _P, _I32, _I32, _P, _P]),
    "yx_simota_workspace_bytes": (_I64, [_I32, _I32, _I32, _I32]),
    "yx_simota_assign": (C.c_int, [_P, _P, _P, _P, _P, _I32, _I32, _I32, _I32, _I32, _P, _P, _P, _P, _P, _P, _P, _P, _I64, _P]),
    "yx_simota_matching": (C.c_int, [_P, _P, _I32, _I32, _I64, _P, _P, _P, _P]),
    "yx_head_losses": (C.c_int, [_P, _P, _I32, _P, _P, _P, _P, _P, _P, _P, _P, _I32, _I32, _I32, _I32, _F, _P, _P, _P, _P]),
    "yx_head_train_decode": (C.c_int, [_P, _P, _P, _I32, _I32, _I32, _I32, _I32, _F, _I32, _I32, _P, _P, _P]),
    "yx_head_train_decode_bwd": (C.c_int, [_P, _P, _P, _I32, _I32, _I32, _I32, _I32, _F, _I32, _I32, _P, _P, _P, _P]),
    "yx_sgd_ema_step": (C.c_int, [_P, _P, _I32, _I32, _F, _F, _I32, _I32, _F, _F, _P, _P]),
    "yx_allreduce_sgd_ema_step": (C.c_int, [_P, _P, _I32, _I32, _F, _I32, _I32, _P, _P, _P, _I64, _I32, _I32, _P, _P]),
    "yx_bn_act_workspace_bytes": (_I64, [_I32, _I32, _I32]),
    "yx_bn_act_train_fwd": (C.c_int, [_P, _I32, _I32, _I32, _I32, _I32, _P, _P, _F, _F, _P, _P, _P, _I32, _P, _P, _P, _P, _I64, _P]),
    "yx_bn_act_train_bwd": (C.c_int, [_P, _P, _I32, _I32, _I32, _I32, _I32, _P, _P, _P, _P, _I32, _P, _P, _P, _P, _P, _I64, _P, _I64, _P]),
    "yx_conv_wgrad_workspace_bytes": (_I64, [_I32] * 9),
    "yx_conv_wgrad": (C.c_int, [_P, _I64, _P, _I64] + [_I32] * 12 + [_P, _I64, _I64, _I64, _I32, _P, _I64, _P]),
    "yx_pack_train_weights": (C.c_int, [_P, _I64, _I64, _I64, _I32, _I32, _I32, _I32, _I32, _P, _P, _I32, _I32, _P]),
    "yx_spp_maxpool_bwd": (C.c_int, [_P, _I64, _P, _I64, _P, _I32, _I32, _I32, _I32, _I32, _P]),
    "yx_pack_train_weights_multi": (C.c_int, [_P, _P, _I32, _I32, _I32, _P]),
    "yx_dilate2": (C.c_int, [_P, _P, _I32, _I32, _I32, _I32, _I32, _I32, _P]),
    "yx_dwconv3x3_train_fwd": (C.c_int, [_P, _I64, _P, _I64, _I64, _P, _I64] + [_I32] * 6 + [_P]),
    "yx_dwconv3x3_dgrad": (C.c_int, [_P, _I64, _P, _I64, _I64, _P, _I64] + [_I32] * 6 + [_P]),
    "yx_dwconv3x3_wgrad_workspace_bytes": (_I64, [_I32] * 5),
    "yx_dwconv3x3_wgrad": (C.c_int, [_P, _I64, _P, _I64] + [_I32] * 6 + [_P, _I64, _I64, _I32, _P, _I64, _P]),
    "yx_letterbox_u8": (C.c_int, [_P, _I32, _I32, _I32, _I32, _P, _I32, _P]),
    "yx_coco_rows": (C.c_int, [_P, _P, _I32, _I32, _P, _P, _P, _I32, _P, _P, _P, _P, _P, _P]),
    "yx_plan_create": (_P, []),
    "yx_plan_destroy": (None, [_P]),
    "yx_plan_add_conv": (C.c_int, [_P, C.POINTER(ConvDesc)]),
    "yx_plan_add_bottleneck": (C.c_int, [_P, C.POINTER(BneckDesc)]),
    "yx_plan_add_dwconv": (C.c_int, [_P, _P, _I64, _P, _P, _P, _I64, _I32, _I32, _I32, _I32, _I32, _I32, _I32]),
    "yx_plan_add_spp": (C.c_int, [_P, _P, _I64, _I32, _I32, _I32, _I32, _I32]),
    "yx_plan_add_focus": (C.c_int, [_P, _P, _I32, _P, _I64, _I32, _I32, _I32, _I32]),
    "yx_plan_add_focus_conv": (C.c_int, [_P, _P, _I32, _P, _P, _P, _I64, _I32, _I32, _I32, _I32, _I32, _I32]),
    "yx_plan_add_postprocess": (C.c_int, [_P, _P, _I32, _I32, _I32, _F, _D, _I32, _I32, _P, _P, _P, _I32, _P, _I64]),
    "yx_plan_add_postprocess_begin": (C.c_int, [_P, _P, _I32, _I32]),
    "yx_plan_add_nms_prefiltered": (C.c_int, [_P, _I32, _I32, _D, _I32, _P, _P, _P, _I32, _P, _I64]),
    "yx_plan_begin_lane": (C.c_int, [_P, _I32, _I32]),
    "yx_plan_end_lane": (C.c_int, [_P]),
    "yx_plan_join_lanes": (C.c_int, [_P]),
    "yx_plan_num_launches": (C.c_int, [_P]),
    "yx_plan_num_ops": (C.c_int, [_P]),
    "yx_plan_profile": (C.c_int, [_P, _P, _P, _P, _I32]),
    "yx_plan_run": (C.c_int, [_P, _P, _I32]),
}

_lib: Optional[C.CDLL] = None


def lib() -> C.CDLL:
    """Load (building first if needed) the CUDA library. Raises if it cannot be had."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists() or os.environ.get("YX_B200_REBUILD"):
        from .build import build_lib

        build_lib()
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} is missing and could not be built: the sm_100a CUDA extension is required "
            "(this package has no CPU or PyTorch fallback)"
        )
    handle = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(handle, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = handle
    return handle


def check(code: int, what: str = "") -> None:
    if code != 0:
        l = lib()
        msg = l.yx_last_error().decode(errors="replace")
        kind = l.yx_strerror(code).decode()
        raise RuntimeError(f"yx_b200 {what}: {kind} ({code}): {msg}")


def dtype_code(torch_dtype) -> int:
    import torch

    table = {torch.bfloat16: YX_BF16, torch.float16: YX_FP16, torch.float32: YX_FP32, torch.uint8: YX_U8}
    if torch_dtype not in table:
        raise TypeError(f"unsupported dtype {torch_dtype}")
    return table[torch_dtype]


def stream_ptr(device=None) -> int:
    import torch

    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(t, what: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(
            f"{what}: tensor is on {t.device}; the B200 path runs hand-written sm_100a CUDA only and has no CPU fallback"
        )
