"""ctypes binding of libhulk_sm100.so (C ABI declared in include/hulk_sm100.h).

There is NO fallback: if the shared library is missing, or a call fails, a RuntimeError is raised.
The library is built in-tree by `python -m hulk_keypoints_b200.build` (or `__graft_entry__.build()`).
"""
from __future__ import annotations

import ctypes as C
import os
import threading

import torch

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# HK_LIB_PATH: another build of the same library (A/B runs of kernel changes on one GPU box)
LIB_PATH = os.environ.get("HK_LIB_PATH") or os.path.join(_PKG_DIR, "libhulk_sm100.so")

# enums of include/hulk_sm100.h
HK_F32, HK_BF16, HK_F64 = 0, 1, 2
HK_CONV_TCGEN05, HK_CONV_FFMA, HK_CONV_TCGEN05_1CTA = 0, 1, 2
ABI_VERSION = 1

EXPORTS = (
    "hk_version", "hk_last_error", "hk_check_device", "hk_pack_conv_weights", "hk_conv_bn_act_fwd",
    "hk_maxpool3x3s2_fwd", "hk_head_fwd", "hk_argmax_workspace_bytes", "hk_argmax_decode",
    "hk_gauss_targets", "hk_bce_workspace_bytes", "hk_bce_fwd_bwd",
    "hk_stem_packed_weight_bytes", "hk_stem_pack_weights", "hk_stem_fwd", "hk_stem_fwd_u8", "hk_adam_step",
    "hk_adam_step_segments",
    # training (SURVEY.md §8 f1)
    "hk_stem_conv_fwd", "hk_bn_workspace_bytes", "hk_bn_train_stats", "hk_bn_apply_fwd", "hk_bn_train_bwd",
    "hk_pack_conv_weights_dgrad", "hk_zero_insert2x", "hk_conv_wgrad_workspace_bytes", "hk_conv_wgrad",
    "hk_stem_wgrad_workspace_bytes", "hk_stem_wgrad", "hk_maxpool3x3s2_bwd", "hk_head_logits_fwd",
    "hk_head_bwd_workspace_bytes", "hk_head_bwd", "hk_sigmoid_fwd", "hk_sigmoid_bwd", "hk_pack_conv_weights_many",
    # round 2
    "hk_soft_argmax_workspace_bytes", "hk_soft_argmax", "hk_l1_normalize_dim1", "hk_stem_pool_fwd", "hk_stem_pool_fwd_u8",
    "hk_conv_ds_fwd", "hk_bn_acc_bytes", "hk_bn_stats_acc", "hk_bn_apply_fwd_acc", "hk_bn_bwd_acc", "hk_conv_bn_stats_fwd", "hk_conv_head_fwd", "hk_head_upsample_fwd", "hk_pack_conv_weights_many_tiled", "hk_maxpool3x3s2_fwd_idx", "hk_maxpool3x3s2_bwd_idx",
    # frozen BatchNorm (eval()-mode BN inside a train()-mode model)
    "hk_bn_fold", "hk_bn_frozen_bwd",
    # training-batch augmentation
    "hk_augment_pick", "hk_augment_images",
    # every keypoint instance: thresholded local-maximum peaks
    "hk_peak_workspace_bytes", "hk_peak_decode",
)


class HkConvDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "batch", "in_h", "in_w", "in_c", "out_h", "out_w", "out_c", "kh", "kw", "stride", "pad", "dil",
        "relu", "in_dtype", "out_dtype", "in_is_nchw", "algo")]


# HkAdamSegment of include/hulk_sm100.h: one row of hk_adam_step_segments' table
ADAM_MAX_SEGMENTS = 256
AUGMENT_MAX_TRIES = 16   # HK_AUGMENT_MAX_TRIES
PEAK_MAX_PEAKS, PEAK_MAX_DISTANCE = 256, 16   # limits of hk_peak_decode


class HkAdamSegment(C.Structure):
    _fields_ = [("begin4", C.c_longlong), ("end4", C.c_longlong)] + [(n, C.c_float) for n in (
        "lr_over_bc1", "inv_sqrt_bc2", "beta1", "beta2", "eps", "weight_decay", "decay")] + [("decoupled", C.c_int)]


_lock = threading.Lock()
_lib = None


def _declare(lib):
    vp, i, f, sz = C.c_void_p, C.c_int, C.c_float, C.c_size_t
    lib.hk_version.restype = i
    lib.hk_version.argtypes = []
    lib.hk_last_error.restype = C.c_char_p
    lib.hk_last_error.argtypes = []
    lib.hk_check_device.restype = i
    lib.hk_check_device.argtypes = []
    lib.hk_pack_conv_weights.restype = i
    lib.hk_pack_conv_weights.argtypes = [vp, vp, vp, vp, vp, f, i, i, i, i, i, vp, vp, vp, vp]
    lib.hk_conv_bn_act_fwd.restype = i
    lib.hk_conv_bn_act_fwd.argtypes = [C.POINTER(HkConvDesc), vp, vp, vp, vp, vp, vp, vp]
    lib.hk_conv_bn_stats_fwd.restype = i
    lib.hk_conv_bn_stats_fwd.argtypes = [C.POINTER(HkConvDesc), vp, vp, vp, vp, vp, vp, vp]
    lib.hk_pack_conv_weights_many_tiled.restype = i
    lib.hk_pack_conv_weights_many_tiled.argtypes = [vp, i, i, C.c_longlong, vp]
    lib.hk_maxpool3x3s2_fwd_idx.restype = i
    lib.hk_maxpool3x3s2_fwd_idx.argtypes = [vp, vp, vp, i, i, i, i, i, i, vp]
    lib.hk_maxpool3x3s2_bwd_idx.restype = i
    lib.hk_maxpool3x3s2_bwd_idx.argtypes = [vp, vp, vp, i, i, i, i, i, i, vp]
    lib.hk_conv_head_fwd.restype = i
    lib.hk_conv_head_fwd.argtypes = [C.POINTER(HkConvDesc), vp, vp, vp, vp, vp, vp, vp, i, vp, vp]
    lib.hk_head_upsample_fwd.restype = i
    lib.hk_head_upsample_fwd.argtypes = [vp, vp, i, i, i, i, i, i, i, vp]
    lib.hk_conv_ds_fwd.restype = i
    lib.hk_conv_ds_fwd.argtypes = [C.POINTER(HkConvDesc), vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.hk_maxpool3x3s2_fwd.restype = i
    lib.hk_maxpool3x3s2_fwd.argtypes = [vp, vp, i, i, i, i, i, i, i, vp]
    lib.hk_head_fwd.restype = i
    lib.hk_head_fwd.argtypes = [vp, i, vp, vp, vp, vp, i, i, i, i, i, i, i, vp]
    lib.hk_argmax_workspace_bytes.restype = sz
    lib.hk_argmax_workspace_bytes.argtypes = [i, i, i, i]
    lib.hk_argmax_decode.restype = i
    lib.hk_argmax_decode.argtypes = [vp, i, i, i, i, vp, vp, vp, sz, vp]
    lib.hk_peak_workspace_bytes.restype = sz
    lib.hk_peak_workspace_bytes.argtypes = [i, i, i, i, i, i]
    lib.hk_peak_decode.restype = i
    lib.hk_peak_decode.argtypes = [vp, i, i, i, i, i, i, f, vp, vp, vp, vp, sz, vp]
    lib.hk_gauss_targets.restype = i
    lib.hk_gauss_targets.argtypes = [vp, i, i, i, i, f, vp, i, vp]
    lib.hk_stem_packed_weight_bytes.restype = sz
    lib.hk_stem_packed_weight_bytes.argtypes = []
    lib.hk_stem_pack_weights.restype = i
    lib.hk_stem_pack_weights.argtypes = [vp, vp, vp]
    lib.hk_stem_fwd.restype = i
    lib.hk_stem_fwd.argtypes = [vp, vp, vp, vp, vp, i, i, i, vp]
    lib.hk_stem_pool_fwd.restype = i
    lib.hk_stem_pool_fwd.argtypes = [vp, vp, vp, vp, vp, i, i, i, vp]
    lib.hk_stem_pool_fwd_u8.restype = i
    lib.hk_stem_pool_fwd_u8.argtypes = [vp, vp, vp, vp, vp, i, i, i, vp]
    lib.hk_adam_step.restype = i
    lib.hk_adam_step.argtypes = [vp, vp, vp, vp, C.c_longlong, f, f, f, f, f, i, vp]
    lib.hk_adam_step_segments.restype = i
    lib.hk_adam_step_segments.argtypes = [vp, vp, vp, vp, C.c_longlong, C.POINTER(HkAdamSegment), i, vp]
    lib.hk_stem_fwd_u8.restype = i
    lib.hk_stem_fwd_u8.argtypes = [vp, vp, vp, vp, vp, i, i, i, vp]
    ll = C.c_longlong
    lib.hk_stem_conv_fwd.restype = i
    lib.hk_stem_conv_fwd.argtypes = [vp, vp, vp, vp, vp, i, i, i, i, vp]
    lib.hk_bn_workspace_bytes.restype = sz
    lib.hk_bn_workspace_bytes.argtypes = [i]
    lib.hk_bn_train_stats.restype = i
    lib.hk_bn_train_stats.argtypes = [vp, ll, i, vp, vp, vp, vp, f, f, vp, vp, vp, vp, vp, sz, vp]
    lib.hk_bn_apply_fwd.restype = i
    lib.hk_bn_apply_fwd.argtypes = [vp, vp, vp, vp, i, vp, vp, ll, i, vp]
    lib.hk_bn_acc_bytes.restype = sz
    lib.hk_bn_acc_bytes.argtypes = [i]
    lib.hk_bn_stats_acc.restype = i
    lib.hk_bn_stats_acc.argtypes = [vp, ll, i, vp, vp]
    lib.hk_bn_apply_fwd_acc.restype = i
    lib.hk_bn_apply_fwd_acc.argtypes = [vp, vp, ll, i, vp, vp, vp, vp, f, f, vp, vp, vp, i, vp, vp, vp]
    lib.hk_bn_bwd_acc.restype = i
    lib.hk_bn_bwd_acc.argtypes = [vp, vp, i, vp, vp, vp, vp, ll, i, vp, vp, vp, i, vp, vp, vp]
    lib.hk_bn_train_bwd.restype = i
    lib.hk_bn_train_bwd.argtypes = [vp, vp, i, vp, vp, vp, vp, ll, i, vp, vp, i, vp, vp, vp, sz, vp]
    lib.hk_bn_fold.restype = i
    lib.hk_bn_fold.argtypes = [vp, i, i, vp]
    lib.hk_bn_frozen_bwd.restype = i
    lib.hk_bn_frozen_bwd.argtypes = [vp, vp, i, vp, vp, vp, vp, ll, i, vp, vp, vp, i, vp, vp, vp]
    lib.hk_pack_conv_weights_dgrad.restype = i
    lib.hk_pack_conv_weights_dgrad.argtypes = [vp, i, i, i, i, vp, vp]
    lib.hk_zero_insert2x.restype = i
    lib.hk_zero_insert2x.argtypes = [vp, vp, i, i, i, i, vp]
    lib.hk_conv_wgrad_workspace_bytes.restype = sz
    lib.hk_conv_wgrad_workspace_bytes.argtypes = [C.POINTER(HkConvDesc)]
    lib.hk_conv_wgrad.restype = i
    lib.hk_conv_wgrad.argtypes = [C.POINTER(HkConvDesc), vp, vp, vp, i, vp, sz, vp]
    lib.hk_stem_wgrad_workspace_bytes.restype = sz
    lib.hk_stem_wgrad_workspace_bytes.argtypes = []
    lib.hk_stem_wgrad.restype = i
    lib.hk_stem_wgrad.argtypes = [vp, vp, vp, i, i, i, i, vp, sz, vp]
    lib.hk_maxpool3x3s2_bwd.restype = i
    lib.hk_maxpool3x3s2_bwd.argtypes = [vp, vp, vp, i, i, i, i, i, i, vp, sz, vp]
    lib.hk_head_logits_fwd.restype = i
    lib.hk_head_logits_fwd.argtypes = [vp, i, vp, vp, vp, vp, i, i, i, i, i, i, i, vp]
    lib.hk_head_bwd_workspace_bytes.restype = sz
    lib.hk_head_bwd_workspace_bytes.argtypes = [i, i, i, i, i]
    lib.hk_head_bwd.restype = i
    lib.hk_head_bwd.argtypes = [vp, vp, vp, vp, vp, vp, vp, i, i, i, i, i, i, i, i, vp, sz, vp]
    lib.hk_pack_conv_weights_many.restype = i
    lib.hk_pack_conv_weights_many.argtypes = [vp, i, ll, vp]
    lib.hk_sigmoid_fwd.restype = i
    lib.hk_sigmoid_fwd.argtypes = [vp, vp, ll, vp]
    lib.hk_sigmoid_bwd.restype = i
    lib.hk_sigmoid_bwd.argtypes = [vp, vp, vp, ll, vp]
    lib.hk_soft_argmax_workspace_bytes.restype = sz
    lib.hk_soft_argmax_workspace_bytes.argtypes = [i, i, i]
    lib.hk_soft_argmax.restype = i
    lib.hk_soft_argmax.argtypes = [vp, i, i, i, vp, vp, vp, sz, vp]
    lib.hk_l1_normalize_dim1.restype = i
    lib.hk_l1_normalize_dim1.argtypes = [vp, i, i, i, vp, vp]
    lib.hk_bce_workspace_bytes.restype = sz
    lib.hk_bce_workspace_bytes.argtypes = [C.c_longlong]
    lib.hk_bce_fwd_bwd.restype = i
    lib.hk_bce_fwd_bwd.argtypes = [vp, i, vp, i, vp, i, i, i, i, f, vp, vp, vp, sz, vp]
    lib.hk_augment_pick.restype = i
    lib.hk_augment_pick.argtypes = [vp, i, i, i, i, i, vp, vp, vp, vp]
    lib.hk_augment_images.restype = i
    lib.hk_augment_images.argtypes = [vp, vp, i, i, i, vp, i, vp, vp, f, C.c_uint64, vp]


def lib():
    """Load (once) and return the ctypes handle.  Raises RuntimeError when the library is absent."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        f"{LIB_PATH} is missing: the CUDA extension has not been built "
                        "(run `python -m hulk_keypoints_b200.build`). There is no CPU or PyTorch fallback.")
                handle = C.CDLL(LIB_PATH)
                _declare(handle)
                v = handle.hk_version()
                if v != ABI_VERSION:
                    raise RuntimeError(f"libhulk_sm100.so ABI version {v} != expected {ABI_VERSION}; rebuild")
                _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().hk_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed with status {rc}: {msg}")


def require_device() -> None:
    """Fail loudly unless the current CUDA device is a B200 (sm_100)."""
    if not torch.cuda.is_available():
        raise RuntimeError("hulk_keypoints_b200 needs a CUDA device (B200, sm_100a); no CPU path exists")
    check(lib().hk_check_device(), "hk_check_device")


# Kernels that write parameters / BatchNorm buffers through raw pointers (hk_adam_step, hk_bn_train_stats, graph replays) do not bump
# torch's tensor `_version`; writers that do not know which model owns the memory (FusedAdam gets bare parameters, like
# torch.optim.Adam in train.py:79) bump this process-wide counter instead and InferenceEngine._weights_key includes it.
_raw_write_generation = 0


def note_raw_parameter_write() -> None:
    global _raw_write_generation
    _raw_write_generation += 1


def raw_write_generation() -> int:
    return _raw_write_generation


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def dtype_code(dt: torch.dtype) -> int:
    if dt == torch.float32:
        return HK_F32
    if dt == torch.bfloat16:
        return HK_BF16
    if dt == torch.float64:
        return HK_F64
    raise ValueError(f"unsupported dtype {dt}")
