"""Tensor-level wrappers over the C ABI (one function per entry point of include/hulk_sm100.h).

torch is used here for device memory and streams only; every computation is a kernel of
libhulk_sm100.so enqueued on torch's current stream.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import HK_BF16, HK_CONV_FFMA, HK_CONV_TCGEN05, HK_F32, HK_F64, HkConvDesc, check, dtype_code, lib, ptr, stream_ptr


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("hulk_keypoints_b200 kernels take CUDA tensors only (no CPU fallback)")


def conv_out_hw(h: int, w: int, k: int, stride: int, pad: int, dil: int) -> Tuple[int, int]:
    eff = dil * (k - 1) + 1
    return (h + 2 * pad - eff) // stride + 1, (w + 2 * pad - eff) // stride + 1


def pack_conv_weights(w_oihw: torch.Tensor, bn: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]],
                      eps: float, w_dtype: torch.dtype):
    """OIHW fp32 (+ BatchNorm vectors) -> ((cout, kh, kw, cin) w_dtype, scale f32, bias f32)."""
    _need_cuda(w_oihw)
    w = w_oihw.detach().contiguous().float()
    cout, cin, kh, kw = w.shape
    w_out = torch.empty((cout, kh, kw, cin), device=w.device, dtype=w_dtype)
    scale = torch.empty(cout, device=w.device, dtype=torch.float32)
    bias = torch.empty(cout, device=w.device, dtype=torch.float32)
    if bn is not None:
        g, b, m, v = (t.detach().contiguous().float() for t in bn)
    else:
        g = b = m = v = None
    check(lib().hk_pack_conv_weights(ptr(w), ptr(g), ptr(b), ptr(m), ptr(v), C.c_float(eps), cout, cin, kh, kw,
                                     dtype_code(w_dtype), ptr(w_out), ptr(scale), ptr(bias), stream_ptr()),
          "hk_pack_conv_weights")
    return w_out, scale, bias


def conv_bn_act(x: torch.Tensor, w_packed: torch.Tensor, scale: torch.Tensor, bias: torch.Tensor, *,
                stride: int, pad: int, dil: int, relu: bool, residual: Optional[torch.Tensor] = None,
                out: Optional[torch.Tensor] = None, out_dtype: Optional[torch.dtype] = None,
                algo: int = HK_CONV_TCGEN05, in_is_nchw: bool = False) -> torch.Tensor:
    """Fused conv + affine (+ residual) (+ ReLU).  x is NHWC (B,H,W,C) unless in_is_nchw (B,C,H,W)."""
    _need_cuda(x, w_packed, scale, bias, residual, out)
    if in_is_nchw:
        B, Cin, H, W = x.shape
    else:
        B, H, W, Cin = x.shape
    cout, kh, kw, cin_w = w_packed.shape
    if cin_w != Cin:
        raise ValueError(f"weight cin {cin_w} != input channels {Cin}")
    Ho, Wo = conv_out_hw(H, W, kh, stride, pad, dil)
    if out is None:
        out = torch.empty((B, Ho, Wo, cout), device=x.device, dtype=out_dtype or (x.dtype if algo == HK_CONV_FFMA else torch.bfloat16))
    elif tuple(out.shape) != (B, Ho, Wo, cout):
        raise ValueError(f"out shape {tuple(out.shape)} != {(B, Ho, Wo, cout)}")
    if residual is not None and (tuple(residual.shape) != tuple(out.shape) or residual.dtype != out.dtype):
        raise ValueError("residual must match the output shape and dtype")
    if not (x.is_contiguous() and w_packed.is_contiguous() and out.is_contiguous() and (residual is None or residual.is_contiguous())):
        raise ValueError("conv_bn_act needs contiguous tensors")
    d = HkConvDesc(B, H, W, Cin, Ho, Wo, cout, kh, kw, stride, pad, dil, int(relu), dtype_code(x.dtype),
                   dtype_code(out.dtype), int(in_is_nchw), algo)
    check(lib().hk_conv_bn_act_fwd(C.byref(d), ptr(x), ptr(w_packed), ptr(scale), ptr(bias), ptr(residual), ptr(out),
                                   stream_ptr()), "hk_conv_bn_act_fwd")
    return out


def conv_ds_supported(x: torch.Tensor, w_packed: torch.Tensor, w_ds_packed: torch.Tensor, stride: int, pad: int, dil: int) -> bool:
    """Shapes hk_conv_ds_fwd takes: bf16 NHWC, odd square kernel with pad = dil*(k/2) (the 1x1 conv is its centre tap), Cout % 128 == 0."""
    cout, kh, kw, cin = w_packed.shape
    return (x.dtype == torch.bfloat16 and w_packed.dtype == torch.bfloat16 and kh == kw and kh % 2 == 1 and pad == dil * (kh // 2)
            and stride in (1, 2) and cout % 128 == 0 and cin % 64 == 0 and tuple(w_ds_packed.shape) == (cout, 1, 1, cin))


def conv_ds(x: torch.Tensor, w_packed: torch.Tensor, scale: torch.Tensor, bias: torch.Tensor,
            w_ds_packed: torch.Tensor, scale_ds: torch.Tensor, bias_ds: torch.Tensor, *, stride: int, pad: int, dil: int,
            relu: bool = True, out: Optional[torch.Tensor] = None, out_ds: Optional[torch.Tensor] = None):
    """Entry of a stride/channel-changing BasicBlock in ONE launch (reference src/resnet.py:56-58 and :64-65 with :184-188):
    out = relu(scale*conv_kxk(x)+bias), out_ds = scale_ds*conv_1x1(x)+bias_ds; the 1x1 conv reads the centre-tap operand of the
    kxk one.  Bit-identical to two conv_bn_act calls.  x NHWC bf16; returns (out, out_ds), both (B,Ho,Wo,Cout) bf16."""
    _need_cuda(x, w_packed, scale, bias, w_ds_packed, scale_ds, bias_ds, out, out_ds)
    if not conv_ds_supported(x, w_packed, w_ds_packed, stride, pad, dil):
        raise ValueError("conv_ds: unsupported shape (needs bf16 NHWC, odd k with pad = dil*(k/2), Cout % 128 == 0, Cin % 64 == 0, 1x1 ds weights)")
    B, H, W, Cin = x.shape
    cout, kh, kw, cin_w = w_packed.shape
    if cin_w != Cin:
        raise ValueError(f"weight cin {cin_w} != input channels {Cin}")
    Ho, Wo = conv_out_hw(H, W, kh, stride, pad, dil)
    outs = []
    for o in (out, out_ds):
        if o is None:
            o = torch.empty((B, Ho, Wo, cout), device=x.device, dtype=torch.bfloat16)
        elif tuple(o.shape) != (B, Ho, Wo, cout) or o.dtype != torch.bfloat16 or not o.is_contiguous():
            raise ValueError(f"conv_ds outputs must be contiguous bf16 {(B, Ho, Wo, cout)} tensors")
        outs.append(o)
    if not (x.is_contiguous() and w_packed.is_contiguous() and w_ds_packed.is_contiguous()):
        raise ValueError("conv_ds needs contiguous tensors")
    d = HkConvDesc(B, H, W, Cin, Ho, Wo, cout, kh, kw, stride, pad, dil, int(relu), dtype_code(x.dtype),
                   dtype_code(torch.bfloat16), 0, HK_CONV_TCGEN05)
    check(lib().hk_conv_ds_fwd(C.byref(d), ptr(x), ptr(w_packed), ptr(scale), ptr(bias), ptr(outs[0]), ptr(w_ds_packed),
                               ptr(scale_ds), ptr(bias_ds), ptr(outs[1]), stream_ptr()), "hk_conv_ds_fwd")
    return outs[0], outs[1]


def stem_pack_weights(w_oihw: torch.Tensor) -> torch.Tensor:
    """conv1.weight (64,3,7,7) fp32 -> the (64,256) bf16 K layout of the tensor-core stem (k = r*32 + s*4 + c)."""
    _need_cuda(w_oihw)
    if tuple(w_oihw.shape) != (64, 3, 7, 7):
        raise ValueError("stem weight must be (64,3,7,7)")
    w = w_oihw.detach().contiguous().float()
    out = torch.empty(int(lib().hk_stem_packed_weight_bytes()) // 2, device=w.device, dtype=torch.bfloat16)
    check(lib().hk_stem_pack_weights(ptr(w), ptr(out), stream_ptr()), "hk_stem_pack_weights")
    return out


def stem(x: torch.Tensor, w_packed: torch.Tensor, scale: torch.Tensor, bias: torch.Tensor,
         out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """conv7x7 s2 + affine + ReLU on tcgen05 -> (B,H/2,W/2,64) bf16 NHWC.
    x: (B,3,H,W) fp32 NCHW (the reference's tensor) or (B,H,W,3) uint8 (cv2 layout; /255 fused into the load)."""
    _need_cuda(x, w_packed, scale, bias, out)
    if not x.is_contiguous() or x.dim() != 4:
        raise ValueError("stem needs a contiguous 4-D input")
    if x.dtype == torch.uint8:
        if x.shape[3] != 3:
            raise ValueError("uint8 input must be (B,H,W,3)")
        B, H, W, _ = x.shape
        fn, name = lib().hk_stem_fwd_u8, "hk_stem_fwd_u8"
    elif x.dtype == torch.float32:
        if x.shape[1] != 3:
            raise ValueError("fp32 input must be (B,3,H,W)")
        B, _, H, W = x.shape
        fn, name = lib().hk_stem_fwd, "hk_stem_fwd"
    else:
        raise ValueError("stem input must be fp32 NCHW or uint8 NHWC")
    Ho, Wo = conv_out_hw(H, W, 7, 2, 3, 1)
    if out is None:
        out = torch.empty((B, Ho, Wo, 64), device=x.device, dtype=torch.bfloat16)
    check(fn(ptr(x), ptr(w_packed), ptr(scale), ptr(bias), ptr(out), B, H, W, stream_ptr()), name)
    return out


def stem_pool_supported(x: torch.Tensor) -> bool:
    """The fused stem + max-pool kernel feeds its input rows by TMA: the row pitch must be a multiple of 16 bytes."""
    if x.dtype == torch.uint8:
        return x.dim() == 4 and x.shape[3] == 3 and (3 * x.shape[2]) % 16 == 0
    return x.dtype == torch.float32 and x.dim() == 4 and x.shape[1] == 3 and x.shape[3] % 4 == 0


def stem_pool(x: torch.Tensor, w_packed: torch.Tensor, scale: torch.Tensor, bias: torch.Tensor,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """conv7x7 s2 + affine + ReLU + MaxPool2d(3,2,1) in one tcgen05 kernel -> (B,Hp,Wp,64) bf16 NHWC (bit-identical to
    maxpool3x3s2(stem(x))).  x: (B,3,H,W) fp32 NCHW or (B,H,W,3) uint8."""
    _need_cuda(x, w_packed, scale, bias, out)
    if not x.is_contiguous() or not stem_pool_supported(x):
        raise ValueError("stem_pool needs a contiguous (B,3,H,W) fp32 input with W % 4 == 0 or (B,H,W,3) uint8 with W % 16 == 0")
    if x.dtype == torch.uint8:
        B, H, W, _ = x.shape
        fn, name = lib().hk_stem_pool_fwd_u8, "hk_stem_pool_fwd_u8"
    else:
        B, _, H, W = x.shape
        fn, name = lib().hk_stem_pool_fwd, "hk_stem_pool_fwd"
    Ho, Wo = conv_out_hw(H, W, 7, 2, 3, 1)
    Hp, Wp = (Ho + 2 - 3) // 2 + 1, (Wo + 2 - 3) // 2 + 1
    if out is None:
        out = torch.empty((B, Hp, Wp, 64), device=x.device, dtype=torch.bfloat16)
    elif tuple(out.shape) != (B, Hp, Wp, 64) or out.dtype != torch.bfloat16 or not out.is_contiguous():
        raise ValueError(f"stem_pool out must be a contiguous bf16 {(B, Hp, Wp, 64)} tensor")
    check(fn(ptr(x), ptr(w_packed), ptr(scale), ptr(bias), ptr(out), B, H, W, stream_ptr()), name)
    return out


def maxpool3x3s2(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _need_cuda(x, out)
    B, H, W, Cc = x.shape
    Ho, Wo = (H + 2 - 3) // 2 + 1, (W + 2 - 3) // 2 + 1
    if out is None:
        out = torch.empty((B, Ho, Wo, Cc), device=x.device, dtype=x.dtype)
    check(lib().hk_maxpool3x3s2_fwd(ptr(x), ptr(out), dtype_code(x.dtype), B, H, W, Cc, Ho, Wo, stream_ptr()),
          "hk_maxpool3x3s2_fwd")
    return out


def head(feat: torch.Tensor, w_fc: torch.Tensor, b_fc: torch.Tensor, H: int, W: int,
         heat: Optional[torch.Tensor] = None, logits_ws: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(B,h,w,C) NHWC features -> (B,K,H,W) fp32 heatmaps.  w_fc (K,C) fp32, b_fc (K) fp32."""
    _need_cuda(feat, w_fc, b_fc, heat, logits_ws)
    B, h, w, Cc = feat.shape
    K = w_fc.shape[0]
    if heat is None:
        heat = torch.empty((B, K, H, W), device=feat.device, dtype=torch.float32)
    if logits_ws is None:
        logits_ws = torch.empty((B, K, h, w), device=feat.device, dtype=torch.float32)
    check(lib().hk_head_fwd(ptr(feat), dtype_code(feat.dtype), ptr(w_fc), ptr(b_fc), ptr(logits_ws), ptr(heat),
                            B, K, Cc, h, w, H, W, stream_ptr()), "hk_head_fwd")
    return heat


HEAD_FUSED_MAX_K = 8


def conv_head_supported(x: torch.Tensor, w_packed: torch.Tensor, w_fc: torch.Tensor, stride: int) -> bool:
    """Shapes hk_conv_head_fwd takes: bf16 NHWC input, 512 output channels, stride 1, at most HEAD_FUSED_MAX_K scoring rows."""
    return (x.dtype == torch.bfloat16 and w_packed.dtype == torch.bfloat16 and w_packed.shape[0] == 512 and w_packed.shape[3] % 64 == 0
            and stride == 1 and 1 <= w_fc.shape[0] <= HEAD_FUSED_MAX_K and w_fc.shape[1] == 512 and w_fc.dtype == torch.float32)


def conv_head(x: torch.Tensor, w_packed: torch.Tensor, scale: torch.Tensor, bias: torch.Tensor, w_fc: torch.Tensor, b_fc: torch.Tensor,
              logits: torch.Tensor, *, stride: int, pad: int, dil: int, relu: bool = True, residual: Optional[torch.Tensor] = None) -> torch.Tensor:
    """The network's last conv (+ BN + shortcut + ReLU) fused with the K live rows of the 1x1 scoring conv: the epilogue adds
    w_fc . row (+ b_fc) into `logits` (B,K,Ho,Wo) fp32, which this call zeroes first; the 512-channel feature map is never written."""
    _need_cuda(x, w_packed, scale, bias, w_fc, b_fc, logits, residual)
    if not conv_head_supported(x, w_packed, w_fc, stride):
        raise ValueError("conv_head: unsupported shape (needs bf16 NHWC, 512 output channels, stride 1, 1..8 fp32 scoring rows)")
    B, H, W, Cin = x.shape
    cout, kh, kw, cin_w = w_packed.shape
    if cin_w != Cin:
        raise ValueError(f"weight cin {cin_w} != input channels {Cin}")
    Ho, Wo = conv_out_hw(H, W, kh, stride, pad, dil)
    K = w_fc.shape[0]
    if tuple(logits.shape) != (B, K, Ho, Wo) or logits.dtype != torch.float32 or not logits.is_contiguous():
        raise ValueError(f"logits must be a contiguous fp32 {(B, K, Ho, Wo)} tensor")
    if residual is not None and (tuple(residual.shape) != (B, Ho, Wo, cout) or residual.dtype != torch.bfloat16 or not residual.is_contiguous()):
        raise ValueError("residual must be a contiguous bf16 tensor of the conv's output shape")
    if not (x.is_contiguous() and w_packed.is_contiguous() and w_fc.is_contiguous() and b_fc.is_contiguous()):
        raise ValueError("conv_head needs contiguous tensors")
    logits.zero_()
    d = HkConvDesc(B, H, W, Cin, Ho, Wo, cout, kh, kw, stride, pad, dil, int(relu), dtype_code(x.dtype), dtype_code(torch.bfloat16), 0,
                   HK_CONV_TCGEN05)
    check(lib().hk_conv_head_fwd(C.byref(d), ptr(x), ptr(w_packed), ptr(scale), ptr(bias), ptr(residual), ptr(w_fc), ptr(b_fc), K, ptr(logits),
                                 stream_ptr()), "hk_conv_head_fwd")
    return logits


def head_upsample(logits: torch.Tensor, H: int, W: int, heat: Optional[torch.Tensor] = None, fast: bool = True) -> torch.Tensor:
    """(B,K,h,w) fp32 logits -> sigmoid(x8 bilinear upsample, align_corners=True) (B,K,H,W) fp32: the second half of head()."""
    _need_cuda(logits, heat)
    B, K, h, w = logits.shape
    if heat is None:
        heat = torch.empty((B, K, H, W), device=logits.device, dtype=torch.float32)
    check(lib().hk_head_upsample_fwd(ptr(logits), ptr(heat), B, K, h, w, H, W, int(fast), stream_ptr()), "hk_head_upsample_fwd")
    return heat


def argmax_workspace_bytes(B: int, K: int, H: int, W: int) -> int:
    return int(lib().hk_argmax_workspace_bytes(B, K, H, W))


def argmax_decode(heat: torch.Tensor, yx: Optional[torch.Tensor] = None, maxval: Optional[torch.Tensor] = None,
                  ws: Optional[torch.Tensor] = None, want_max: bool = False):
    """(B,K,H,W) fp32 -> (B,K,2) int32 (row, col) with numpy's first-index tie-break."""
    _need_cuda(heat, yx, maxval, ws)
    if heat.dtype != torch.float32 or not heat.is_contiguous():
        raise ValueError("argmax_decode needs a contiguous fp32 heatmap")
    B, K, H, W = heat.shape
    if yx is None:
        yx = torch.empty((B, K, 2), device=heat.device, dtype=torch.int32)
    if maxval is None and want_max:
        maxval = torch.empty((B, K), device=heat.device, dtype=torch.float32)
    nbytes = argmax_workspace_bytes(B, K, H, W)
    if ws is None:
        ws = torch.empty(nbytes, device=heat.device, dtype=torch.uint8)
    check(lib().hk_argmax_decode(ptr(heat), B, K, H, W, ptr(yx), ptr(maxval), ptr(ws), ws.numel() * ws.element_size(),
                                 stream_ptr()), "hk_argmax_decode")
    return (yx, maxval) if want_max else yx


def check_peak_args(max_peaks: int, threshold: float, min_distance: int) -> Tuple[int, float, int]:
    """Validate peak_decode's parameters -> (N, the threshold rounded to fp32 as the kernel sees it, r).  Raises ValueError."""
    if isinstance(max_peaks, bool) or int(max_peaks) != max_peaks or not 1 <= max_peaks <= _lib.PEAK_MAX_PEAKS:
        raise ValueError(f"max_peaks must be an integer in [1, {_lib.PEAK_MAX_PEAKS}], got {max_peaks!r}")
    if isinstance(min_distance, bool) or int(min_distance) != min_distance or not 1 <= min_distance <= _lib.PEAK_MAX_DISTANCE:
        raise ValueError(f"min_distance must be an integer in [1, {_lib.PEAK_MAX_DISTANCE}], got {min_distance!r}")
    thr = C.c_float(float(threshold)).value
    if not math.isfinite(thr):
        raise ValueError(f"threshold must be finite in fp32, got {threshold!r}")
    return int(max_peaks), thr, int(min_distance)


def peak_workspace_bytes(B: int, K: int, H: int, W: int, max_peaks: int, min_distance: int) -> int:
    return int(lib().hk_peak_workspace_bytes(B, K, H, W, max_peaks, min_distance))


def peak_decode(heat: torch.Tensor, max_peaks: int, threshold: float, min_distance: int, yx: Optional[torch.Tensor] = None,
                score: Optional[torch.Tensor] = None, count: Optional[torch.Tensor] = None, ws: Optional[torch.Tensor] = None):
    """Every local maximum of each (H, W) map of a (B,K,H,W) fp32 heatmap: pixels >= threshold that are greater than every earlier
    and at least every later pixel of their (2r+1)^2 window (r = min_distance; NaN counts as -inf), the top max_peaks per map by
    value, ties by flat index.  Returns (yx (B,K,N,2) int32 (row, col), score (B,K,N) fp32, count (B,K) int32); unused slots hold
    (-1, -1) and -inf."""
    N, thr, r = check_peak_args(max_peaks, threshold, min_distance)
    _need_cuda(heat, yx, score, count, ws)
    if heat.dtype != torch.float32 or heat.dim() != 4 or not heat.is_contiguous():
        raise ValueError("peak_decode needs a contiguous (B,K,H,W) fp32 heatmap")
    B, K, H, W = heat.shape
    if min(B, K, H, W) < 1 or B * K > 65535 or H * W >= 2 ** 31 - 1:
        raise ValueError(f"peak_decode: unsupported shape {tuple(heat.shape)} (needs B*K <= 65535 and H*W < 2^31)")
    for name, t, shape, dt in (("yx", yx, (B, K, N, 2), torch.int32), ("score", score, (B, K, N), torch.float32),
                               ("count", count, (B, K), torch.int32)):
        if t is not None and (tuple(t.shape) != shape or t.dtype != dt or not t.is_contiguous()):
            raise ValueError(f"peak_decode: {name} must be a contiguous {dt} tensor of shape {shape}")
    if yx is None:
        yx = torch.empty((B, K, N, 2), device=heat.device, dtype=torch.int32)
    if score is None:
        score = torch.empty((B, K, N), device=heat.device, dtype=torch.float32)
    if count is None:
        count = torch.empty((B, K), device=heat.device, dtype=torch.int32)
    nbytes = peak_workspace_bytes(B, K, H, W, N, r)
    if ws is None:
        ws = torch.empty(nbytes, device=heat.device, dtype=torch.uint8)
    elif ws.numel() * ws.element_size() < nbytes:
        raise ValueError(f"peak_decode: workspace of {ws.numel() * ws.element_size()} bytes, needs {nbytes}")
    check(lib().hk_peak_decode(ptr(heat), B, K, H, W, N, r, C.c_float(thr), ptr(yx), ptr(score), ptr(count), ptr(ws),
                               ws.numel() * ws.element_size(), stream_ptr()), "hk_peak_decode")
    return yx, score, count


def soft_argmax(heat: torch.Tensor, want_int: bool = True):
    """Soft-argmax of every (H, W) map of a (..., H, W) fp32 CUDA tensor: Prediction.expectation (reference prediction.py:31-38,
    transposed-ravel quirk included).  Returns (exp_xy fp64 (..., 2) = (E[x'], E[y']), exp_int int32 (..., 2) or None)."""
    _need_cuda(heat)
    if heat.dtype != torch.float32 or not heat.is_contiguous() or heat.dim() < 2:
        raise ValueError("soft_argmax needs a contiguous fp32 tensor of (..., H, W) maps")
    H, W = heat.shape[-2:]
    maps = heat.numel() // (H * W)
    lead = tuple(heat.shape[:-2])
    exp_xy = torch.empty(lead + (2,), device=heat.device, dtype=torch.float64)
    exp_int = torch.empty(lead + (2,), device=heat.device, dtype=torch.int32) if want_int else None
    ws = torch.empty(max(8, int(lib().hk_soft_argmax_workspace_bytes(maps, H, W))), device=heat.device, dtype=torch.uint8)
    check(lib().hk_soft_argmax(ptr(heat), maps, H, W, ptr(exp_xy), ptr(exp_int), ptr(ws), ws.numel(), stream_ptr()), "hk_soft_argmax")
    return exp_xy, exp_int


def l1_normalize_dim1(x: torch.Tensor) -> torch.Tensor:
    """(K,H,W) fp32 -> fp64, L1-normalised over dim 1 (reference dataset.py:33-34, F.normalize(x, p=1))."""
    _need_cuda(x)
    if x.dtype != torch.float32 or x.dim() != 3 or not x.is_contiguous():
        raise ValueError("l1_normalize_dim1 needs a contiguous (K,H,W) fp32 tensor")
    K, H, W = x.shape
    out = torch.empty((K, H, W), device=x.device, dtype=torch.float64)
    check(lib().hk_l1_normalize_dim1(ptr(x), K, H, W, ptr(out), stream_ptr()), "hk_l1_normalize_dim1")
    return out


def gauss_targets(uv: torch.Tensor, H: int, W: int, sigma: float, out_dtype: torch.dtype = torch.float64,
                  out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """uv (B,K,2) = (x, y) -> (B,K,H,W) Gaussian targets (fp32 math, stored as out_dtype)."""
    _need_cuda(uv, out)
    uv32 = uv.detach().to(torch.float32).contiguous()
    B, K, _ = uv32.shape
    if out is None:
        out = torch.empty((B, K, H, W), device=uv.device, dtype=out_dtype)
    check(lib().hk_gauss_targets(ptr(uv32), B, K, H, W, C.c_float(float(sigma)), ptr(out), dtype_code(out.dtype),
                                 stream_ptr()), "hk_gauss_targets")
    return out


def bce_fwd_bwd(pred: torch.Tensor, target: Optional[torch.Tensor] = None, uv: Optional[torch.Tensor] = None,
                sigma: float = 8.0, want_grad: bool = True, pred_is_logits: bool = False):
    """Mean BCE of fp32 heatmaps against fp64/fp32 targets (or Gaussians generated from uv on the fly).

    `pred_is_logits=True`: `pred` holds the upsampled logits and the sigmoid is fused into the kernel.
    Returns (loss f64 0-dim CUDA tensor, grad wrt LOGITS fp32 or None)."""
    _need_cuda(pred, target, uv)
    if pred.dtype != torch.float32 or not pred.is_contiguous() or pred.dim() != 4:
        raise ValueError("bce_fwd_bwd needs a contiguous (B,K,H,W) fp32 prediction")
    B, K, H, W = pred.shape
    n = pred.numel()
    loss = torch.empty((), device=pred.device, dtype=torch.float64)
    grad = torch.empty_like(pred) if want_grad else None
    ws = torch.empty(int(lib().hk_bce_workspace_bytes(n)), device=pred.device, dtype=torch.uint8)
    tcode = 0
    uv32 = None
    if target is not None:
        if tuple(target.shape) != tuple(pred.shape) or not target.is_contiguous():
            raise ValueError("target must be contiguous and shaped like pred")
        tcode = dtype_code(target.dtype)
    else:
        uv32 = uv.detach().to(torch.float32).contiguous()
        if tuple(uv32.shape) != (B, K, 2):
            raise ValueError("uv must be (B,K,2)")
    check(lib().hk_bce_fwd_bwd(ptr(pred), int(pred_is_logits), ptr(target), tcode, ptr(uv32), B, K, H, W, C.c_float(float(sigma)), ptr(loss),
                               ptr(grad), ptr(ws), ws.numel(), stream_ptr()), "hk_bce_fwd_bwd")
    return loss, grad


def _overlap(a: torch.Tensor, b: torch.Tensor) -> bool:
    """Do the memory ranges of two contiguous tensors intersect?"""
    pa, pb = a.data_ptr(), b.data_ptr()
    return pa < pb + b.numel() * b.element_size() and pb < pa + a.numel() * a.element_size()


def _f32_contiguous(name: str, t: torch.Tensor, shape: Tuple[int, ...]) -> None:
    if tuple(t.shape) != shape or t.dtype != torch.float32 or not t.is_contiguous():
        raise ValueError(f"{name} must be a contiguous float32 tensor of shape {shape}, got {tuple(t.shape)} {t.dtype}")


def augment_pick(fwd: torch.Tensor, uv: torch.Tensor, H: int, W: int, uv_out: Optional[torch.Tensor] = None,
                 pick: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Per image the first of `tries` candidate label maps fwd (B,tries,2,3) fp32 that keeps all labels uv (B,K,2) inside
    [0,W-1] x [0,H-1] -> (uv_out (B,K,2) fp32 = the moved labels, pick (B,) int32 = the candidate, -1 = none: identity).
    uv_out must not overlap uv."""
    _need_cuda(fwd, uv, uv_out, pick)
    if uv.dim() != 3 or uv.shape[2] != 2 or fwd.dim() != 4:
        raise ValueError(f"augment_pick: uv must be (B,K,2) and fwd (B,tries,2,3), got {tuple(uv.shape)} and {tuple(fwd.shape)}")
    B, K, _ = uv.shape
    tries = fwd.shape[1]
    if not 1 <= tries <= _lib.AUGMENT_MAX_TRIES:
        raise ValueError(f"augment_pick: tries must be in 1..{_lib.AUGMENT_MAX_TRIES}")
    _f32_contiguous("uv", uv, (B, K, 2))
    _f32_contiguous("fwd", fwd, (B, tries, 2, 3))
    if uv_out is None:
        uv_out = torch.empty_like(uv)
    _f32_contiguous("uv_out", uv_out, (B, K, 2))
    if pick is None:
        pick = torch.empty(B, device=uv.device, dtype=torch.int32)
    elif tuple(pick.shape) != (B,) or pick.dtype != torch.int32 or not pick.is_contiguous():
        raise ValueError("augment_pick: pick must be a contiguous (B,) int32 tensor")
    if _overlap(uv, uv_out):
        raise ValueError("augment_pick: uv_out must not overlap uv (the labels are not moved in place)")
    check(lib().hk_augment_pick(ptr(fwd), B, tries, K, H, W, ptr(uv), ptr(uv_out), ptr(pick), stream_ptr()), "hk_augment_pick")
    return uv_out, pick


def augment_images(img: torch.Tensor, inv: torch.Tensor, pick: torch.Tensor, photo: torch.Tensor, noise_std: float, key: int,
                   out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """img (B,3,H,W) fp32 -> out: bilinear warp by inv[b, pick[b]] (identity for pick -1; zero outside the image), contrast / brightness
    / per-channel gain from photo (B,5) = (c, beta, g0, g1, g2), Gaussian noise of std noise_std (Philox key `key`, 64 bits), clamp to
    [0, 1].  One launch; out must not overlap img."""
    _need_cuda(img, inv, pick, photo, out)
    if img.dim() != 4 or img.shape[1] != 3 or inv.dim() != 4:
        raise ValueError(f"augment_images: img must be (B,3,H,W) and inv (B,tries,2,3), got {tuple(img.shape)} and {tuple(inv.shape)}")
    B, _, H, W = img.shape
    tries = inv.shape[1]
    if not 1 <= tries <= _lib.AUGMENT_MAX_TRIES:
        raise ValueError(f"augment_images: tries must be in 1..{_lib.AUGMENT_MAX_TRIES}")
    _f32_contiguous("img", img, (B, 3, H, W))
    _f32_contiguous("inv", inv, (B, tries, 2, 3))
    _f32_contiguous("photo", photo, (B, 5))
    if tuple(pick.shape) != (B,) or pick.dtype != torch.int32 or not pick.is_contiguous():
        raise ValueError("augment_images: pick must be a contiguous (B,) int32 tensor")
    if not noise_std >= 0.0:
        raise ValueError("augment_images: noise_std must be >= 0")
    if out is None:
        out = torch.empty_like(img)
    _f32_contiguous("out", out, (B, 3, H, W))
    if _overlap(img, out):
        raise ValueError("augment_images: out must not overlap img (no in-place warp)")
    check(lib().hk_augment_images(ptr(img), ptr(out), B, H, W, ptr(inv), tries, ptr(pick), ptr(photo), C.c_float(float(noise_std)),
                                  C.c_uint64(int(key) & 0xFFFFFFFFFFFFFFFF), stream_ptr()), "hk_augment_images")
    return out


# ------------------------------------------------------------------------------------------------ training kernels
def stem_conv(x: torch.Tensor, w_packed: torch.Tensor, scale: torch.Tensor, bias: torch.Tensor, relu: bool,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Stem conv7x7 s2 on tcgen05 with an explicit ReLU switch (relu=False: raw output for train-mode BN)."""
    _need_cuda(x, w_packed, scale, bias, out)
    if x.dtype != torch.float32 or x.dim() != 4 or x.shape[1] != 3 or not x.is_contiguous():
        raise ValueError("stem_conv needs a contiguous (B,3,H,W) fp32 input")
    B, _, H, W = x.shape
    Ho, Wo = conv_out_hw(H, W, 7, 2, 3, 1)
    if out is None:
        out = torch.empty((B, Ho, Wo, 64), device=x.device, dtype=torch.bfloat16)
    check(lib().hk_stem_conv_fwd(ptr(x), ptr(w_packed), ptr(scale), ptr(bias), ptr(out), B, H, W, int(relu), stream_ptr()),
          "hk_stem_conv_fwd")
    return out


def bn_workspace(C_: int, device, extra_coef: bool = True) -> torch.Tensor:
    n = int(lib().hk_bn_workspace_bytes(C_)) + (3 * C_ * 4 if extra_coef else 0)
    return torch.empty(n, device=device, dtype=torch.uint8)


def bn_train_stats(y: torch.Tensor, gamma, beta, running_mean, running_var, momentum: float, eps: float,
                   mean: torch.Tensor, invstd: torch.Tensor, scale: torch.Tensor, shift: torch.Tensor, ws: torch.Tensor) -> None:
    """y (...,C) bf16 NHWC -> batch mean / invstd + fused affine (scale, shift); running stats updated in place."""
    _need_cuda(y, mean, invstd, scale, shift, ws)
    Cc = y.shape[-1]
    P = y.numel() // Cc
    check(lib().hk_bn_train_stats(ptr(y), C.c_longlong(P), Cc, ptr(gamma), ptr(beta), ptr(running_mean), ptr(running_var),
                                  C.c_float(momentum), C.c_float(eps), ptr(mean), ptr(invstd), ptr(scale), ptr(shift), ptr(ws),
                                  ws.numel(), stream_ptr()), "hk_bn_train_stats")


def bn_apply(y: torch.Tensor, scale: torch.Tensor, shift: torch.Tensor, relu: bool, residual: Optional[torch.Tensor] = None,
             out: Optional[torch.Tensor] = None, relu_bits: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out = relu?(y*scale + shift [+ residual]); relu_bits (uint8, numel/8): receives the ReLU mask as one bit per element."""
    _need_cuda(y, scale, shift, residual, out, relu_bits)
    Cc = y.shape[-1]
    P = y.numel() // Cc
    if out is None:
        out = torch.empty_like(y)
    if relu_bits is not None and (relu_bits.dtype != torch.uint8 or relu_bits.numel() < y.numel() // 8):
        raise ValueError("relu_bits must be a uint8 tensor of numel/8 bytes")
    check(lib().hk_bn_apply_fwd(ptr(y), ptr(scale), ptr(shift), ptr(residual), int(relu), ptr(out), ptr(relu_bits), C.c_longlong(P), Cc,
                                stream_ptr()), "hk_bn_apply_fwd")
    return out


def bn_train_bwd(dout: torch.Tensor, out_mask: Optional[torch.Tensor], y: torch.Tensor, mean: torch.Tensor, invstd: torch.Tensor,
                 gamma: Optional[torch.Tensor], dgamma: Optional[torch.Tensor], dbeta: Optional[torch.Tensor], dy: torch.Tensor,
                 ws: torch.Tensor, dmasked: Optional[torch.Tensor] = None, accumulate: bool = False) -> torch.Tensor:
    _need_cuda(dout, out_mask, y, mean, invstd, dy, ws, dmasked)
    Cc = y.shape[-1]
    P = y.numel() // Cc
    bits = out_mask is not None and out_mask.dtype == torch.uint8   # bit array from bn_apply(relu_bits=...) instead of the bf16 output
    check(lib().hk_bn_train_bwd(ptr(dout), ptr(out_mask), int(bits), ptr(y), ptr(mean), ptr(invstd), ptr(gamma), C.c_longlong(P), Cc, ptr(dgamma),
                                ptr(dbeta), int(accumulate), ptr(dy), ptr(dmasked), ptr(ws), ws.numel(), stream_ptr()), "hk_bn_train_bwd")
    return dy


def conv_bn_stats(x: torch.Tensor, w_packed: torch.Tensor, scale: torch.Tensor, bias: torch.Tensor, acc: torch.Tensor, *,
                  stride: int, pad: int, dil: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Raw conv (tcgen05) + the BatchNorm statistics of its output in one launch: acc (zeroed, bn_acc_bytes(cout)) += per-channel
    (sum y, sum y^2) of the stored bf16 values, gathered in the conv epilogue.  x NHWC bf16; scale/bias are the caller's ones/zeros."""
    _need_cuda(x, w_packed, scale, bias, acc, out)
    B, H, W, Cin = x.shape
    cout, kh, kw, cin_w = w_packed.shape
    if cin_w != Cin:
        raise ValueError(f"weight cin {cin_w} != input channels {Cin}")
    Ho, Wo = conv_out_hw(H, W, kh, stride, pad, dil)
    if out is None:
        out = torch.empty((B, Ho, Wo, cout), device=x.device, dtype=torch.bfloat16)
    elif tuple(out.shape) != (B, Ho, Wo, cout) or out.dtype != torch.bfloat16:
        raise ValueError(f"out must be a bf16 {(B, Ho, Wo, cout)} tensor")
    if not (x.is_contiguous() and w_packed.is_contiguous() and out.is_contiguous()) or x.dtype != torch.bfloat16:
        raise ValueError("conv_bn_stats needs contiguous bf16 NHWC tensors")
    if acc.numel() * acc.element_size() < bn_acc_bytes(cout):
        raise ValueError("accumulator buffer too small")
    d = HkConvDesc(B, H, W, Cin, Ho, Wo, cout, kh, kw, stride, pad, dil, 0, dtype_code(x.dtype), dtype_code(out.dtype), 0, HK_CONV_TCGEN05)
    check(lib().hk_conv_bn_stats_fwd(C.byref(d), ptr(x), ptr(w_packed), ptr(scale), ptr(bias), ptr(out), ptr(acc), stream_ptr()),
          "hk_conv_bn_stats_fwd")
    return out


def bn_acc_bytes(C_: int) -> int:
    """Bytes of the 2*C fixed-point accumulators of one BatchNorm reduction (hk_bn_stats_acc / hk_bn_bwd_acc); must be zeroed before use."""
    return int(lib().hk_bn_acc_bytes(C_))


def bn_stats_acc(y: torch.Tensor, acc: torch.Tensor) -> None:
    """acc (zeroed, bn_acc_bytes(C) bytes) += per-channel (sum y, sum y^2) of y (...,C) bf16 NHWC: exact integer accumulation."""
    _need_cuda(y, acc)
    Cc = y.shape[-1]
    if acc.numel() * acc.element_size() < bn_acc_bytes(Cc):
        raise ValueError("accumulator buffer too small")
    check(lib().hk_bn_stats_acc(ptr(y), C.c_longlong(y.numel() // Cc), Cc, ptr(acc), stream_ptr()), "hk_bn_stats_acc")


def bn_apply_acc(y: torch.Tensor, acc: torch.Tensor, gamma, beta, running_mean, running_var, momentum: float, eps: float,
                 mean: torch.Tensor, invstd: torch.Tensor, relu: bool, residual: Optional[torch.Tensor] = None,
                 out: Optional[torch.Tensor] = None, relu_bits: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Train-mode BatchNorm apply straight from the accumulators of bn_stats_acc: batch statistics (saved in mean / invstd), running
    statistics, out = relu?(gamma*xhat + beta [+ residual]) -- no finalize launch in between."""
    _need_cuda(y, acc, mean, invstd, residual, out, relu_bits)
    Cc = y.shape[-1]
    P = y.numel() // Cc
    if out is None:
        out = torch.empty_like(y)
    if relu_bits is not None and (relu_bits.dtype != torch.uint8 or relu_bits.numel() < y.numel() // 8):
        raise ValueError("relu_bits must be a uint8 tensor of numel/8 bytes")
    check(lib().hk_bn_apply_fwd_acc(ptr(y), ptr(acc), C.c_longlong(P), Cc, ptr(gamma), ptr(beta), ptr(running_mean), ptr(running_var),
                                    C.c_float(momentum), C.c_float(eps), ptr(mean), ptr(invstd), ptr(residual), int(relu), ptr(out),
                                    ptr(relu_bits), stream_ptr()), "hk_bn_apply_fwd_acc")
    return out


def bn_bwd_acc(dout: torch.Tensor, out_mask: Optional[torch.Tensor], y: torch.Tensor, mean: torch.Tensor, invstd: torch.Tensor,
               gamma: Optional[torch.Tensor], acc: torch.Tensor, dgamma: Optional[torch.Tensor], dbeta: Optional[torch.Tensor],
               dy: torch.Tensor, dmasked: Optional[torch.Tensor] = None, accumulate: bool = False) -> torch.Tensor:
    """bn_train_bwd through zeroed accumulators (bn_acc_bytes(C)): reduce + apply, two launches."""
    _need_cuda(dout, out_mask, y, mean, invstd, acc, dy, dmasked)
    Cc = y.shape[-1]
    P = y.numel() // Cc
    bits = out_mask is not None and out_mask.dtype == torch.uint8
    check(lib().hk_bn_bwd_acc(ptr(dout), ptr(out_mask), int(bits), ptr(y), ptr(mean), ptr(invstd), ptr(gamma), C.c_longlong(P), Cc, ptr(acc),
                              ptr(dgamma), ptr(dbeta), int(accumulate), ptr(dy), ptr(dmasked), stream_ptr()), "hk_bn_bwd_acc")
    return dy


BN_FOLD_ITEM = None   # numpy dtype of HkBnFoldItem (include/hulk_sm100.h), built on first use


def bn_fold_items(items) -> torch.Tensor:
    """[(gamma, beta, running_mean, running_var, eps, scale_out, shift_out, invstd_out_or_None), ...] -> the HkBnFoldItem array of
    bn_fold as a uint8 CPU tensor (upload it once; the pointers are read by the kernel at every launch)."""
    import numpy as np
    global BN_FOLD_ITEM
    if BN_FOLD_ITEM is None:
        BN_FOLD_ITEM = np.dtype([("g", "<u8"), ("b", "<u8"), ("m", "<u8"), ("v", "<u8"), ("sc", "<u8"), ("sh", "<u8"), ("inv", "<u8"),
                                 ("eps", "<f4"), ("C", "<i4")])
    arr = np.zeros(len(items), dtype=BN_FOLD_ITEM)
    for i, (g, b, m, v, eps, sc, sh, inv) in enumerate(items):
        _need_cuda(g, b, m, v, sc, sh, inv)
        Cc = m.numel()
        if any(t is not None and (t.dtype != torch.float32 or t.numel() != Cc or not t.is_contiguous()) for t in (g, b, m, v, sc, sh, inv)):
            raise ValueError("bn_fold: every tensor of an item must be a contiguous fp32 (C,) tensor")
        arr[i] = tuple(0 if t is None else t.data_ptr() for t in (g, b, m, v, sc, sh, inv)) + (eps, Cc)
    return torch.from_numpy(arr.view(np.uint8).copy())


def bn_fold(items_dev: torch.Tensor, n_items: int, max_c: int) -> None:
    """Frozen BatchNorms in one launch: scale = gamma/sqrt(running_var + eps), shift = beta - running_mean*scale, invstd (items of
    bn_fold_items, on the device)."""
    _need_cuda(items_dev)
    check(lib().hk_bn_fold(ptr(items_dev), n_items, max_c, stream_ptr()), "hk_bn_fold")


def bn_frozen_bwd(dout: torch.Tensor, out_mask: Optional[torch.Tensor], scale: torch.Tensor, dy: Optional[torch.Tensor],
                  dmasked: Optional[torch.Tensor] = None, y: Optional[torch.Tensor] = None, mean: Optional[torch.Tensor] = None,
                  invstd: Optional[torch.Tensor] = None, acc: Optional[torch.Tensor] = None, dgamma: Optional[torch.Tensor] = None,
                  dbeta: Optional[torch.Tensor] = None, accumulate: bool = False) -> Optional[torch.Tensor]:
    """Backward of a BatchNorm in eval() mode (running statistics) + the ReLU after it, one pass: d' = dout*[out>0] (out_mask: the
    bf16 post-ReLU output or the uint8 bit mask of bn_apply; None = no ReLU), dy = scale*d', d' into `dmasked`; with dgamma / dbeta,
    also dbeta = sum d' and dgamma = sum d'*(y - mean)*invstd through `acc` (zeroed, bn_acc_bytes(C)).  mean = running mean."""
    _need_cuda(dout, out_mask, scale, dy, dmasked, y, mean, invstd, acc, dgamma, dbeta)
    Cc = dout.shape[-1]
    P = dout.numel() // Cc
    for t in (out_mask, dy, dmasked, y):
        if t is not None and t.dtype == torch.bfloat16 and t.shape != dout.shape:
            raise ValueError(f"bn_frozen_bwd: shape {tuple(t.shape)} != dout {tuple(dout.shape)}")
    if acc is not None and acc.numel() * acc.element_size() < bn_acc_bytes(Cc):
        raise ValueError("accumulator buffer too small")
    bits = out_mask is not None and out_mask.dtype == torch.uint8
    check(lib().hk_bn_frozen_bwd(ptr(dout), ptr(out_mask), int(bits), ptr(y), ptr(scale), ptr(mean), ptr(invstd), C.c_longlong(P), Cc,
                                 ptr(acc), ptr(dgamma), ptr(dbeta), int(accumulate), ptr(dy), ptr(dmasked), stream_ptr()), "hk_bn_frozen_bwd")
    return dy


def pack_conv_weights_dgrad(w_oihw: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """OIHW fp32 -> (cin, kh, kw, cout) bf16 with flipped taps: the weights of the data-gradient convolution."""
    _need_cuda(w_oihw, out)
    w = w_oihw.detach()
    if w.dtype != torch.float32 or not w.is_contiguous():
        raise ValueError("pack_conv_weights_dgrad needs a contiguous fp32 OIHW weight")
    cout, cin, kh, kw = w.shape
    if out is None:
        out = torch.empty((cin, kh, kw, cout), device=w.device, dtype=torch.bfloat16)
    check(lib().hk_pack_conv_weights_dgrad(ptr(w), cout, cin, kh, kw, ptr(out), stream_ptr()), "hk_pack_conv_weights_dgrad")
    return out


def zero_insert2x(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    _need_cuda(x, out)
    B, h, w, Cc = x.shape
    if out is None:
        out = torch.empty((B, 2 * h, 2 * w, Cc), device=x.device, dtype=x.dtype)
    check(lib().hk_zero_insert2x(ptr(x), ptr(out), B, h, w, Cc, stream_ptr()), "hk_zero_insert2x")
    return out


def _conv_desc(B, H, W, cin, cout, k, stride, pad, dil):
    Ho, Wo = conv_out_hw(H, W, k, stride, pad, dil)
    return HkConvDesc(B, H, W, cin, Ho, Wo, cout, k, k, stride, pad, dil, 0, HK_BF16, HK_BF16, 0, HK_CONV_TCGEN05), Ho, Wo


def conv_wgrad_workspace_bytes(B, H, W, cin, cout, k, stride, pad, dil) -> int:
    d, _, _ = _conv_desc(B, H, W, cin, cout, k, stride, pad, dil)
    return int(lib().hk_conv_wgrad_workspace_bytes(C.byref(d)))


def conv_wgrad(x: torch.Tensor, dy: torch.Tensor, dw: torch.Tensor, *, k: int, stride: int, pad: int, dil: int,
               ws: Optional[torch.Tensor] = None, accumulate: bool = False) -> torch.Tensor:
    """dw (cout,cin,k,k) fp32 (+)= conv weight gradient from x (B,H,W,cin) bf16 and dy (B,Ho,Wo,cout) bf16 (tcgen05)."""
    _need_cuda(x, dy, dw, ws)
    B, H, W, cin = x.shape
    cout = dy.shape[3]
    d, Ho, Wo = _conv_desc(B, H, W, cin, cout, k, stride, pad, dil)
    if tuple(dy.shape) != (B, Ho, Wo, cout) or tuple(dw.shape) != (cout, cin, k, k):
        raise ValueError(f"conv_wgrad shape mismatch: dy {tuple(dy.shape)} dw {tuple(dw.shape)}")
    if not (x.is_contiguous() and dy.is_contiguous() and dw.is_contiguous()) or dw.dtype != torch.float32:
        raise ValueError("conv_wgrad needs contiguous tensors and an fp32 gradient")
    nbytes = int(lib().hk_conv_wgrad_workspace_bytes(C.byref(d)))
    if ws is None:
        ws = torch.empty(nbytes, device=x.device, dtype=torch.uint8)
    check(lib().hk_conv_wgrad(C.byref(d), ptr(x), ptr(dy), ptr(dw), int(accumulate), ptr(ws), ws.numel(), stream_ptr()), "hk_conv_wgrad")
    return dw


def stem_wgrad(x_nchw: torch.Tensor, dy: torch.Tensor, dw: torch.Tensor, ws: Optional[torch.Tensor] = None,
               accumulate: bool = False) -> torch.Tensor:
    _need_cuda(x_nchw, dy, dw, ws)
    B, _, H, W = x_nchw.shape
    if ws is None:
        ws = torch.empty(int(lib().hk_stem_wgrad_workspace_bytes()), device=dy.device, dtype=torch.uint8)
    check(lib().hk_stem_wgrad(ptr(x_nchw), ptr(dy), ptr(dw), int(accumulate), B, H, W, ptr(ws), ws.numel(), stream_ptr()), "hk_stem_wgrad")
    return dw


def maxpool3x3s2_bwd(dout: torch.Tensor, x: torch.Tensor, dx: Optional[torch.Tensor] = None,
                     idx_ws: Optional[torch.Tensor] = None) -> torch.Tensor:
    _need_cuda(dout, x, dx, idx_ws)
    B, H, W, Cc = x.shape
    Ho, Wo = dout.shape[1], dout.shape[2]
    if dx is None:
        dx = torch.empty_like(x)
    if idx_ws is None:
        idx_ws = torch.empty(B * Ho * Wo * Cc, device=x.device, dtype=torch.uint8)
    check(lib().hk_maxpool3x3s2_bwd(ptr(dout), ptr(x), ptr(dx), B, H, W, Cc, Ho, Wo, ptr(idx_ws), idx_ws.numel(), stream_ptr()),
          "hk_maxpool3x3s2_bwd")
    return dx


def maxpool3x3s2_fwd_idx(x: torch.Tensor, out: Optional[torch.Tensor] = None, idx: Optional[torch.Tensor] = None):
    """MaxPool2d(3,2,1) forward on bf16 NHWC that also records the winning tap of every window (uint8, B*Ho*Wo*C) -> (out, idx)."""
    _need_cuda(x, out, idx)
    B, H, W, Cc = x.shape
    Ho, Wo = (H + 2 - 3) // 2 + 1, (W + 2 - 3) // 2 + 1
    if x.dtype != torch.bfloat16 or not x.is_contiguous():
        raise ValueError("maxpool3x3s2_fwd_idx needs a contiguous bf16 NHWC tensor")
    if out is None:
        out = torch.empty((B, Ho, Wo, Cc), device=x.device, dtype=torch.bfloat16)
    if idx is None:
        idx = torch.empty(B * Ho * Wo * Cc, device=x.device, dtype=torch.uint8)
    if tuple(out.shape) != (B, Ho, Wo, Cc) or idx.numel() < B * Ho * Wo * Cc or idx.dtype != torch.uint8:
        raise ValueError("maxpool3x3s2_fwd_idx: bad out / idx buffer")
    check(lib().hk_maxpool3x3s2_fwd_idx(ptr(x), ptr(out), ptr(idx), B, H, W, Cc, Ho, Wo, stream_ptr()), "hk_maxpool3x3s2_fwd_idx")
    return out, idx


def maxpool3x3s2_bwd_idx(dout: torch.Tensor, idx: torch.Tensor, H: int, W: int, dx: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Backward of maxpool3x3s2_fwd_idx: dout (B,Ho,Wo,C) bf16 routed through the recorded indices -> dx (B,H,W,C) bf16."""
    _need_cuda(dout, idx, dx)
    B, Ho, Wo, Cc = dout.shape
    if dx is None:
        dx = torch.empty((B, H, W, Cc), device=dout.device, dtype=torch.bfloat16)
    check(lib().hk_maxpool3x3s2_bwd_idx(ptr(dout), ptr(idx), ptr(dx), B, H, W, Cc, Ho, Wo, stream_ptr()), "hk_maxpool3x3s2_bwd_idx")
    return dx


def head_logits(feat: torch.Tensor, w_fc: torch.Tensor, b_fc: torch.Tensor, H: int, W: int, out: Optional[torch.Tensor] = None,
                logits_ws: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(B,h,w,C) features -> (B,K,H,W) fp32 upsampled LOGITS (no sigmoid): the training-side head."""
    _need_cuda(feat, w_fc, b_fc, out, logits_ws)
    B, h, w, Cc = feat.shape
    K = w_fc.shape[0]
    if out is None:
        out = torch.empty((B, K, H, W), device=feat.device, dtype=torch.float32)
    if logits_ws is None:
        logits_ws = torch.empty((B, K, h, w), device=feat.device, dtype=torch.float32)
    check(lib().hk_head_logits_fwd(ptr(feat), dtype_code(feat.dtype), ptr(w_fc), ptr(b_fc), ptr(logits_ws), ptr(out), B, K, Cc, h, w,
                                   H, W, stream_ptr()), "hk_head_logits_fwd")
    return out


def head_bwd(g_up: torch.Tensor, feat: torch.Tensor, w_fc: torch.Tensor, dfeat: Optional[torch.Tensor], dw_fc: Optional[torch.Tensor],
             db_fc: Optional[torch.Tensor], dlogits_ws: Optional[torch.Tensor] = None, ws: Optional[torch.Tensor] = None,
             accumulate: bool = False):
    """Backward of head_logits: g_up (B,K,H,W) fp32 -> dfeat (B,h,w,C) bf16, dw_fc (K,C) fp32, db_fc (K) fp32 (each may be None:
    not computed)."""
    _need_cuda(g_up, feat, w_fc, dfeat, dw_fc, db_fc, dlogits_ws, ws)
    B, K, H, W = g_up.shape
    _, h, w, Cc = feat.shape
    if dlogits_ws is None:
        dlogits_ws = torch.empty((B, K, h, w), device=feat.device, dtype=torch.float32)
    nbytes = int(lib().hk_head_bwd_workspace_bytes(B, K, Cc, h, w))
    if ws is None:
        ws = torch.empty(nbytes, device=feat.device, dtype=torch.uint8)
    check(lib().hk_head_bwd(ptr(g_up), ptr(feat), ptr(w_fc), ptr(dlogits_ws), ptr(dfeat), ptr(dw_fc), ptr(db_fc), int(accumulate), B, K,
                            Cc, h, w, H, W, ptr(ws), ws.numel(), stream_ptr()), "hk_head_bwd")
    return dfeat, dw_fc, db_fc
