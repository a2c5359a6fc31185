"""ctypes binding of the C-ABI library ``librehrseg_b200.so`` (see include/rehrseg_b200.h).

The library is the product: there is NO CPU / PyTorch fallback.  Importing this module never touches a GPU
(so the CPU test-suite can check that the library loads and exports every declared symbol), but every
compute entry point raises if the shared object is missing or a call returns a non-zero ``rehr_status``.
"""
from __future__ import annotations

import ctypes as C
import os
import re
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librehrseg_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "rehrseg_b200.h")


class RehrTensor(C.Structure):
    """Mirror of ``rehr_tensor``: channels-last activation with a voxel pitch."""

    _fields_ = [("ptr", C.c_void_p), ("n", C.c_int), ("d", C.c_int), ("h", C.c_int), ("w", C.c_int),
                ("c", C.c_int), ("ld", C.c_longlong), ("dtype", C.c_int)]


BF16, F16 = 0, 1   # rehr_dtype


class RehrConvDesc(C.Structure):
    _fields_ = [(k, C.c_int) for k in ("kd", "kh", "kw", "sd", "sh", "sw", "pd", "ph", "pw")]


ACT_NONE, ACT_RELU, ACT_LRELU = 0, 1, 2

_lib: Optional[C.CDLL] = None


class RehrError(RuntimeError):
    pass


def declared_symbols() -> list[str]:
    """Every ``rehr_*`` function include/rehrseg_b200.h declares (used by the CPU ABI test)."""
    with open(HEADER_PATH) as f:
        text = f.read()
    return sorted(set(re.findall(r"\b(rehr_[a-z0-9_]+)\s*\(", text)))


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RehrError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU or PyTorch fallback for the hot path)")
        _lib = C.CDLL(LIB_PATH)
        _declare(_lib)
    return _lib


def _declare(L: C.CDLL) -> None:
    T, D = C.POINTER(RehrTensor), C.POINTER(RehrConvDesc)
    vp, i, f, ll, sz = C.c_void_p, C.c_int, C.c_float, C.c_longlong, C.c_size_t
    sig = {
        "rehr_strerror": (C.c_char_p, [i]),
        "rehr_last_cuda_error": (i, []),
        "rehr_version": (i, []),
        "rehr_device_sm_count": (i, []),
        "rehr_pack_weight": (i, [vp, vp, i, i, i, ll, ll, ll, i, vp]),
        "rehr_conv3d_fwd": (i, [D, T, vp, vp, T, i, i, f, vp, vp]),
        "rehr_conv3d_stats_tiles": (i, [T]),
        "rehr_conv3d_dgrad": (i, [D, T, vp, vp, T, i, i, f, vp]),
        "rehr_conv3d_splitk_workspace": (sz, [D, T, vp, T, i]),
        "rehr_conv3d_fwd_ws": (i, [D, T, vp, vp, T, i, i, f, vp, vp, sz, vp]),
        "rehr_conv3d_dgrad_ws": (i, [D, T, vp, vp, T, i, i, f, vp, sz, vp]),
        "rehr_conv3d_wgrad_workspace": (sz, [D, T, T]),
        "rehr_conv3d_wgrad": (i, [D, T, T, vp, i, vp, sz, vp]),
        "rehr_convtranspose3d_fwd": (i, [D, T, vp, vp, T, i, f, vp]),
        "rehr_convtranspose3d_fused_supported": (i, [D, i, i]),
        "rehr_convtranspose3d_fused_fwd": (i, [D, T, vp, vp, T, i, f, vp]),
        "rehr_convtranspose3d_fused_fwd2": (i, [D, T, vp, vp, T, T, i, f, vp]),
        "rehr_convtranspose3d_dgrad": (i, [D, T, vp, T, vp]),
        "rehr_convtranspose3d_wgrad_workspace": (sz, [D, T, T]),
        "rehr_convtranspose3d_wgrad": (i, [D, T, T, vp, i, vp, sz, vp]),
        "rehr_conv3d_march_supported": (i, [D, i, i]),
        "rehr_conv3d_march_weight_bytes": (sz, [i, i, i]),
        "rehr_pack_weight_march": (i, [vp, vp, i, i, i, ll, ll, i, i, vp]),
        "rehr_conv3d_march_stats_tiles": (i, [T, T, i]),
        "rehr_conv3d_march_fwd": (i, [T, vp, vp, T, i, i, i, f, vp, vp]),
        "rehr_conv3d_march_s2dgrad_supported": (i, [D, i, i]),
        "rehr_conv3d_march_s2dgrad_weight_bytes": (sz, [D, i, i]),
        "rehr_pack_weight_march_s2dgrad": (i, [D, vp, vp, i, i, vp]),
        "rehr_pack_batch_begin": (i, []),
        "rehr_pack_batch_launch": (i, [vp]),
        "rehr_pack_batch_abort": (i, []),
        "rehr_conv3d_march_s2dgrad": (i, [D, T, vp, T, vp]),
        "rehr_conv3d_wgrad_march_supported": (i, [D, T, T]),
        "rehr_conv3d_wgrad_march_workspace": (sz, [T, T, i]),
        "rehr_conv3d_wgrad_march": (i, [T, T, i, i, vp, i, vp, sz, vp]),
        "rehr_conv3d_wgrad_march_s2_supported": (i, [D, T, T]),
        "rehr_conv3d_wgrad_march_s2_workspace": (sz, [D, T, T]),
        "rehr_conv3d_wgrad_march_s2": (i, [D, T, T, vp, i, vp, sz, vp]),
        "rehr_conv3d_smallcin_fwd": (i, [D, vp, i, i, i, i, i, vp, vp, T, i, f, vp, vp]),
        "rehr_conv3d_smallcin_wgrad": (i, [D, vp, i, i, i, i, i, T, vp, i, vp, sz, vp]),
        "rehr_conv3d_smallcin_wgrad_workspace": (sz, [D, i, T]),
        "rehr_conv3d_smallcin_dgrad": (i, [D, T, vp, vp, i, i, i, i, i, vp]),
        "rehr_instnorm_stats_tiles": (i, [T]),
        "rehr_instnorm_stats": (i, [T, vp, vp]),
        "rehr_instnorm_finalize": (i, [vp, i, i, i, ll, f, vp, vp, vp]),
        "rehr_instnorm_lrelu_apply": (i, [T, vp, vp, vp, vp, f, T, T, vp]),
        "rehr_convert16": (i, [T, T, vp]),
        "rehr_instnorm_lrelu_bwd_reduce": (i, [T, T, T, vp, vp, vp, vp, f, vp, vp]),
        "rehr_instnorm_lrelu_bwd_finalize": (i, [vp, i, i, i, vp, vp, vp, vp, i, vp]),
        "rehr_instnorm_lrelu_bwd_apply": (i, [T, T, T, vp, vp, vp, vp, f, vp, T, vp]),
        "rehr_pointwise_fwd": (i, [T, vp, vp, vp, i, vp]),
        "rehr_pointwise_bwd": (i, [T, vp, vp, i, T, vp, vp, i, vp, sz, vp]),
        "rehr_pointwise_bwd_workspace": (sz, [T, i]),
        "rehr_channel_sum": (i, [T, vp, i, vp, sz, vp]),
        "rehr_channel_sum_workspace": (sz, [T]),
        "rehr_upsample_linear_d": (i, [T, T, vp]),
        "rehr_upsample_linear_d_bwd": (i, [T, T, vp]),
        "rehr_ncdhw_f32_to_ndhwc_bf16": (i, [vp, T, vp]),
        "rehr_ndhwc_bf16_to_ncdhw_f32": (i, [T, vp, vp]),
        "rehr_segate_scale_add_act": (i, [T, vp, T, i, f, T, vp]),
        "rehr_segate_bwd_reduce": (i, [T, T, T, i, f, vp, vp]),
        "rehr_segate_bwd_apply": (i, [T, T, i, f, vp, vp, T, T, vp]),
        "rehr_act_bwd": (i, [T, T, i, f, T, vp]),
        "rehr_sw_accumulate": (i, [vp, vp, vp, i, vp] + [i] * 10 + [vp]),
        "rehr_sw_finalize": (i, [vp, vp, i, ll, vp, vp]),
        "rehr_blur1d": (i, [vp, vp, i, vp, ll, i, i, vp]),
        "rehr_uasr_mixture_blocks": (i, [ll, i]),
        "rehr_uasr_mixture_fwd": (i, [vp, vp, vp, vp, vp, vp, ll, ll, i, i, vp]),
        "rehr_uasr_mixture_bwd": (i, [vp, vp, vp, vp, vp, vp, vp, vp, vp, ll, ll, i, i, vp]),
        "rehr_resample_axis": (i, [vp, vp, ll, i, i, ll, f, i, vp]),
        "rehr_bspline_prefilter_axis": (i, [vp, ll, i, ll, vp]),
        "rehr_affine_sample2d": (i, [vp, vp, vp, i, i, i, i, i, i, i, f, vp, i, vp]),
        "rehr_intensity_moment_doubles": (i, []),
        "rehr_intensity_moments": (i, [vp, vp, i, i, ll, vp, vp]),
        "rehr_intensity_pointwise": (i, [vp, vp, i, ll, i, vp, vp, vp]),
        "rehr_intensity_blur_axis": (i, [vp, i, vp, i, vp, i, i, i, i, i, vp]),
        "rehr_intensity_gamma": (i, [vp, vp, i, ll, vp, vp, i, vp]),
        "rehr_intensity_lowres_gather": (i, [vp, vp, vp, i, i, i, i, ll, vp]),
        "rehr_intensity_lowres_prefilter": (i, [vp, vp, i, i, i, ll, vp]),
        "rehr_intensity_lowres_upsample": (i, [vp, vp, vp, i, i, i, i, vp, vp]),
        "rehr_rot90": (i, [vp, vp, i, i, ll, i, vp]),
        "rehr_fba_combine": (i, [vp, i, f, vp, ll, vp]),
        "rehr_mean_stack": (i, [vp, i, vp, ll, vp]),
        "rehr_loss_blocks": (i, [ll]),
        "rehr_seg_loss_sums": (i, [vp, vp, vp, i, i, ll, vp, vp]),
        "rehr_seg_loss_bwd": (i, [vp, vp, vp, i, i, ll, vp, vp, vp, vp, vp]),
        "rehr_cosine_sums": (i, [vp, vp, i, i, ll, vp, vp]),
        "rehr_cosine_sums_bwd": (i, [vp, vp, i, i, ll, vp, vp, vp, vp]),
        "rehr_plane_maxpool": (i, [vp, i, i, i, i, i, i, i, vp, vp, vp]),
        "rehr_plane_maxpool_bwd": (i, [vp, vp, i, i, i, i, i, i, i, vp, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    L._rehr_signatures = sig  # noqa: SLF001  (kept for the ABI test)


def check(status: int, what: str = "") -> None:
    if status != 0:
        L = lib()
        msg = L.rehr_strerror(status).decode()
        extra = f" (cudaError {L.rehr_last_cuda_error()})" if status == -4 else ""
        raise RehrError(f"{what or 'rehrseg_b200 call'} failed: {msg}{extra}")


def stream_ptr(device: Optional[torch.device] = None) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def ptr(t: Optional[torch.Tensor]) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


def cl_strides_ok(t: torch.Tensor) -> bool:
    """True if `t` ([N,D,H,W,C]) is channels-last dense except for a voxel pitch >= C (a channel slice)."""
    if t.dim() != 5 or t.stride(4) != 1:
        return False
    n, d, h, w, c = t.shape
    ld = t.stride(3) if w > 1 else (t.stride(2) if h > 1 else (t.stride(1) if d > 1 else c))
    if ld < c:
        return False
    exp = (d * h * w * ld, h * w * ld, w * ld, ld, 1)
    return all(t.shape[k] == 1 or t.stride(k) == exp[k] for k in range(5))


def check_device(t: torch.Tensor) -> None:
    """The library launches on the CURRENT device and stream (tensor maps, streams, kernel attributes are per device): a tensor
    that lives on another GPU must not reach it.  Model-level entry points switch to their input's device (device_of)."""
    if t.device.index != torch.cuda.current_device():
        raise RehrError(f"tensor on {t.device} but the current CUDA device is cuda:{torch.cuda.current_device()}: wrap the call in "
                        "`with torch.cuda.device(tensor.device):` (the module-level forwards of rehrseg_b200 do)")


def device_of(t: torch.Tensor):
    """Context manager making `t`'s GPU the current device for the engine calls inside."""
    if not t.is_cuda:
        raise RehrError("rehrseg_b200 runs on CUDA (sm_100a) only; there is no CPU path")
    return torch.cuda.device(t.device)


def as_cl(t: torch.Tensor) -> torch.Tensor:
    """Return a channels-last ([N,D,H,W,C], pitch-strided) bf16 CUDA view/copy of `t` that the ABI accepts."""
    if not t.is_cuda:
        raise RehrError("rehrseg_b200 ops need CUDA tensors (no CPU fallback)")
    check_device(t)
    if t.dtype != torch.bfloat16:
        t = t.to(torch.bfloat16)
    if not cl_strides_ok(t) or (t.data_ptr() % 16) != 0 or (_pitch(t) % 8) != 0:
        t = t.contiguous()
    return t


def _pitch(t: torch.Tensor) -> int:
    n, d, h, w, c = t.shape
    if w > 1:
        return t.stride(3)
    if h > 1:
        return t.stride(2)
    if d > 1:
        return t.stride(1)
    if n > 1:
        return t.stride(0)
    return c


def rt(t: torch.Tensor, f16: bool = False) -> RehrTensor:
    """rehr_tensor descriptor of a channels-last [N,D,H,W,C] tensor (see as_cl).  `f16`: the 16-bit payload is fp16 (the
    forward activations of the SegModel path, see functional.is_h), not the tensor's nominal bf16."""
    n, d, h, w, c = t.shape
    return RehrTensor(t.data_ptr(), n, d, h, w, c, _pitch(t), F16 if f16 else BF16)


def conv_desc(kernel, stride, padding) -> RehrConvDesc:
    return RehrConvDesc(*[int(v) for v in (*kernel, *stride, *padding)])
