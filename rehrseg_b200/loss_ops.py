"""Fused CUDA reductions for the stage-2 losses (csrc/loss_ops.cu) as autograd Functions, and the loss modules built on them.

Opt-in counterparts of the plain-PyTorch mirrors in `train_step.py` (same constructors, same values):
  * `FusedDCAndWeightedCELoss` <- `DC_and_weighted_CE_loss` as `_build_loss` configures it (utils/seg_utils.py:305-372)
  * `FusedDistiller`           <- `Distiller` (models/seg_model.py:115-151)
  * `FusedSRLoss`              <- the SR-stage loss statements of `sr_train_step` with `nn.L1Loss()` and `BCEDiceLoss(alpha, beta)`
                                  (train_all.py:124-133, incl. the UASR terms)
Each kernel makes one pass over the fp32 NCDHW tensor and returns per-(sample, class/channel) SUMS; the handful of scalar
operations that turn sums into the loss stay ordinary autograd ops on tiny tensors, and the backward kernels consume the
gradients of the sums.  CUDA only: like every engine op they raise `RehrError` on a CPU tensor or a missing library.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch
import torch.nn.functional as F
from torch import nn

from . import _lib as L
from ._lib import check, lib, ptr, stream_ptr


def _f32c(t: torch.Tensor, what: str) -> torch.Tensor:
    if not t.is_cuda:
        raise L.RehrError(f"{what}: expected a CUDA tensor (rehrseg_b200 has no CPU path)")
    t = t if t.dtype == torch.float32 else t.float()
    return t if t.is_contiguous() else t.contiguous()


class SegLossSums(torch.autograd.Function):
    """(logits [B,C,*], target [B,1,*] class indices, weight [*] or None) ->
    ce_sum [B] = sum_v weight*CE, inter [B,C] = sum p*[y=c], pred [B,C] = sum p, count [B,C] = sum [y=c]   (p = softmax)."""

    @staticmethod
    def forward(ctx, logits, target, weight):
        lg = _f32c(logits.detach(), "seg_loss_sums")
        tg = _f32c(target.detach(), "seg_loss_sums")
        wt = _f32c(weight.detach(), "seg_loss_sums") if weight is not None else None
        b, c = lg.shape[0], lg.shape[1]
        v = lg[0, 0].numel()
        if tg.numel() != b * v or (wt is not None and wt.numel() != v):
            raise L.RehrError("seg_loss_sums: target must be [B,1,*] and weight [*] matching the logits")
        blocks = lib().rehr_loss_blocks(v)
        k = 1 + 3 * c
        partial = torch.empty((b, blocks, k), dtype=torch.float32, device=lg.device)
        check(lib().rehr_seg_loss_sums(ptr(lg), ptr(tg), ptr(wt), b, c, v, ptr(partial), stream_ptr()), "seg_loss_sums")
        sums = partial.sum(1)
        ctx.save_for_backward(lg, tg, wt)
        per = sums[:, 1:].reshape(b, c, 3)
        count = per[:, :, 2]
        ctx.mark_non_differentiable(count)
        return sums[:, 0], per[:, :, 0], per[:, :, 1], count

    @staticmethod
    def backward(ctx, g_ce, g_int, g_pred, _g_cnt):
        lg, tg, wt = ctx.saved_tensors
        b, c = lg.shape[0], lg.shape[1]
        v = lg[0, 0].numel()
        dl = torch.empty_like(lg)
        z = lambda g, shape: (g if g is not None else torch.zeros(shape, device=lg.device)).float().contiguous()  # noqa: E731
        check(lib().rehr_seg_loss_bwd(ptr(lg), ptr(tg), ptr(wt), b, c, v, ptr(z(g_ce, (b,))), ptr(z(g_int, (b, c))),
                                      ptr(z(g_pred, (b, c))), ptr(dl), stream_ptr()), "seg_loss_bwd")
        return dl, None, None


class CosineSums(torch.autograd.Function):
    """(a [B,C,*], b [B,C,*]) -> (sum_v ahat*bhat, sum_v ahat^2, sum_v bhat^2), each [B,C]; xhat = F.normalize(x, dim=1).
    Gradient flows to `a` only (the teacher map is detached in the reference)."""

    @staticmethod
    def forward(ctx, a, b):
        a32, b32 = _f32c(a.detach(), "cosine_sums"), _f32c(b.detach(), "cosine_sums")
        if a32.shape != b32.shape:
            raise L.RehrError("cosine_sums: shape mismatch")
        n, c = a32.shape[0], a32.shape[1]
        v = a32[0, 0].numel()
        blocks = lib().rehr_loss_blocks(v)
        partial = torch.empty((n, blocks, 3, c), dtype=torch.float32, device=a32.device)
        check(lib().rehr_cosine_sums(ptr(a32), ptr(b32), n, c, v, ptr(partial), stream_ptr()), "cosine_sums")
        s = partial.sum(1)
        ctx.save_for_backward(a32, b32)
        ctx.adtype = a.dtype
        return s[:, 0], s[:, 1], s[:, 2]

    @staticmethod
    def backward(ctx, g_ab, g_aa, _g_bb):
        a32, b32 = ctx.saved_tensors
        n, c = a32.shape[0], a32.shape[1]
        v = a32[0, 0].numel()
        z = lambda g: (g if g is not None else torch.zeros((n, c), device=a32.device)).float().contiguous()  # noqa: E731
        da = torch.empty_like(a32)
        check(lib().rehr_cosine_sums_bwd(ptr(a32), ptr(b32), n, c, v, ptr(z(g_ab)), ptr(z(g_aa)), ptr(da), stream_ptr()),
              "cosine_sums_bwd")
        return da.to(ctx.adtype), None


class PlaneMaxPool(torch.autograd.Function):
    """x [N,C,S,H,W] -> [(N S), C, OH, OW]: per slice, max over non-overlapping ph x pw windows, ceil mode -- the
    `rearrange 'b c s h w -> (b s) c h w'` + `nn.MaxPool2d(k, stride=k, ceil_mode=True)` of models/seg_model.py:103-110."""

    @staticmethod
    def forward(ctx, x, ph, pw):
        x32 = _f32c(x.detach(), "plane_maxpool")
        n, c, s, h, w = x32.shape
        oh, ow = -(-h // ph), -(-w // pw)
        out = torch.empty((n * s, c, oh, ow), dtype=torch.float32, device=x32.device)
        idx = torch.empty((n * s, c, oh, ow), dtype=torch.int32, device=x32.device)
        check(lib().rehr_plane_maxpool(ptr(x32), n, c, s, h, w, int(ph), int(pw), ptr(out), ptr(idx), stream_ptr()), "plane_maxpool")
        ctx.save_for_backward(idx)
        ctx.cfg = (n, c, s, h, w, int(ph), int(pw), x.dtype)
        return out

    @staticmethod
    def backward(ctx, g):
        (idx,) = ctx.saved_tensors
        n, c, s, h, w, ph, pw, dt = ctx.cfg
        dx = torch.zeros((n, c, s, h, w), dtype=torch.float32, device=g.device)
        check(lib().rehr_plane_maxpool_bwd(ptr(g.float().contiguous()), ptr(idx), n, c, s, h, w, ph, pw, ptr(dx), stream_ptr()),
              "plane_maxpool_bwd")
        return dx.to(dt), None, None


def _plane_strides(t: torch.Tensor, what: str) -> tuple:
    """(batch, channel, depth) element strides of a [B,C,S,H,W] CUDA tensor whose H*W planes are contiguous."""
    if not t.is_cuda:
        raise L.RehrError(f"{what}: expected a CUDA tensor (rehrseg_b200 has no CPU path)")
    h, w = t.shape[3], t.shape[4]
    if (w > 1 and t.stride(4) != 1) or (h > 1 and t.stride(3) != w):
        raise L.RehrError(f"{what}: the H*W planes must be contiguous (strides {tuple(t.stride())})")
    return t.stride(0), t.stride(1), t.stride(2)


class SRLossSums(torch.autograd.Function):
    """(hat [B,C,S,H,W], target [B,C,S,H,W] with contiguous H*W planes, u [B,1,S,H,W] or None) -> sums [3 + 4 (C-1)]:
    sum |e|, sum |e|/u + log u, sum |u - |e||, then per segmentation channel c = 1..C-1: sum bce(hat_c, t_c), sum p*t_c,
    sum p^2, sum t_c^2, where e = hat_0 - t_0 and p = sigmoid(hat_c) (the u terms are 0 without u).  The target is read in
    place (a depth window of patches_hr needs no copy); gradients flow to `hat` and `u` only."""

    @staticmethod
    def forward(ctx, hat, target, u):
        from . import functional as F_
        h32 = _f32c(hat.detach(), "sr_loss_sums")
        u32 = _f32c(u.detach(), "sr_loss_sums") if u is not None else None
        if h32.dim() != 5 or target.shape != h32.shape or h32.shape[1] < 2:
            raise L.RehrError(f"sr_loss_sums: hat and target must be equal [B,C>=2,S,H,W] shapes, got {tuple(h32.shape)} and "
                              f"{tuple(target.shape)}")
        tg = target.detach() if target.dtype == torch.float32 else target.detach().float()
        strides = _plane_strides(tg, "sr_loss_sums target")
        b, c, s, hh, ww = h32.shape
        if u32 is not None and u32.shape != (b, 1, s, hh, ww):
            raise L.RehrError(f"sr_loss_sums: uncertainty must be [B,1,S,H,W] = {(b, 1, s, hh, ww)}, got {tuple(u32.shape)}")
        if tg.device != h32.device or (u32 is not None and u32.device != h32.device):
            raise L.RehrError("sr_loss_sums: hat, target and uncertainty must be on one device")
        with L.device_of(h32):
            blocks = lib().rehr_loss_blocks(b * s * hh * ww)
            partial = torch.empty((blocks, 3 + 4 * (c - 1)), dtype=torch.float32, device=h32.device)
            check(lib().rehr_sr_loss_sums(ptr(h32), ptr(tg), ptr(u32), b, c, s, hh * ww, *strides, ptr(partial), stream_ptr()),
                  "sr_loss_sums")
            F_._count()
            sums = partial.sum(0)
        ctx.save_for_backward(h32, tg, u32)
        ctx.meta = (strides, hat.dtype, None if u is None else u.dtype)
        return sums

    @staticmethod
    def backward(ctx, g):
        from . import functional as F_
        h32, tg, u32 = ctx.saved_tensors
        strides, hdt, udt = ctx.meta
        b, c, s, hh, ww = h32.shape
        d_hat = torch.empty_like(h32)
        d_u = torch.empty_like(u32) if u32 is not None else None
        with L.device_of(h32):
            check(lib().rehr_sr_loss_bwd(ptr(h32), ptr(tg), ptr(u32), b, c, s, hh * ww, *strides, ptr(g.float().contiguous()),
                                         ptr(d_hat), ptr(d_u), stream_ptr()), "sr_loss_bwd")
            F_._count()
        return d_hat.to(hdt), None, (d_u.to(udt) if d_u is not None else None)


# ---------------------------------------------------------------------------------------------------------------
# loss modules
# ---------------------------------------------------------------------------------------------------------------
class FusedDCAndWeightedCELoss(nn.Module):
    """`train_step.DCAndWeightedCELoss` on the fused sums.  The reference multiplies the CE map [B,D,H,W] by the uncertainty
    [B,1,D,H,W] (utils/seg_utils.py:299-301,349), which broadcasts over the batch: mean over [B,B,V] of ce[b']*unc[b] equals
    the mean over [B,V] of ce[b'] * mean_b unc[b] -- the per-voxel weight handed to the kernel."""

    def __init__(self, weight_ce: float = 1, weight_dice: float = 1, smooth: float = 1e-5):
        super().__init__()
        self.weight_ce, self.weight_dice, self.smooth = weight_ce, weight_dice, smooth

    def forward(self, net_output: torch.Tensor, target: torch.Tensor, uncertainty: Optional[torch.Tensor] = None):
        assert target.shape[1] == 1, "target must be [B,1,...] label indices"
        b = net_output.shape[0]
        v = net_output[0, 0].numel()
        w = uncertainty.float().mean(0)[0] if (uncertainty is not None and self.weight_ce != 0) else None
        ce_sum, inter, pred, count = SegLossSums.apply(net_output, target, w)
        total = 0
        if self.weight_dice != 0:
            dc = (2 * inter[:, 1:] + self.smooth) / torch.clip(count[:, 1:] + pred[:, 1:] + self.smooth, 1e-8)
            total = total + self.weight_dice * (-dc.mean())
        if self.weight_ce != 0:
            total = total + self.weight_ce * ce_sum.sum() / (b * v)
        return total


def fused_cosine_distance_loss(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """models/seg_model.py:60-78 on the fused sums."""
    ab, aa, bb = CosineSums.apply(a, b)
    cos = ab / (aa.sqrt().clamp_min(1e-8) * bb.sqrt().clamp_min(1e-8))
    return (1 - cos).mean()


def fused_structure_loss(student: torch.Tensor, teacher: torch.Tensor, scale: float = 0.5) -> torch.Tensor:
    """models/seg_model.py:80-113 with the two max-pools on the fused kernel; the 4x4 Gram matrices stay PyTorch."""
    from .train_step import _gram
    _, _, s, th, tw = student.shape
    ph, pw = int(th * scale), int(tw * scale)
    ps = PlaneMaxPool.apply(student, ph, pw)
    pt = PlaneMaxPool.apply(teacher.detach(), ph, pw)
    err = (_gram(pt) - _gram(ps)).pow(2) / float((pt.shape[-1] * pt.shape[-2]) ** 2) / pt.shape[0]
    return err.sum() / s


class FusedDistiller(nn.Module):
    """`train_step.Distiller` (same constructor / state_dict) with the cosine and structure terms on the fused kernels."""

    def __init__(self, student_dim, teacher_dim, lambda_l1=0.0, lambda_cosine=0.0, lambda_structure=0.0):
        super().__init__()
        self.lambda_l1, self.lambda_cosine, self.lambda_structure = lambda_l1, lambda_cosine, lambda_structure
        self.distill = nn.Conv3d(student_dim, teacher_dim, kernel_size=1, stride=1, padding=0)

    def forward(self, feature_student, feature_teacher):
        loss = 0
        if self.lambda_structure > 0:
            loss = loss + self.lambda_structure * fused_structure_loss(feature_student, feature_teacher, 0.5)
        projected = self.distill(feature_student)
        if self.lambda_l1 > 0:
            loss = loss + self.lambda_l1 * F.smooth_l1_loss(projected, feature_teacher)
        if self.lambda_cosine > 0:
            loss = loss + self.lambda_cosine * fused_cosine_distance_loss(projected, feature_teacher)
        return loss


class FusedSRLoss(nn.Module):
    """The SR-stage loss of `train_step.sr_train_step` (train_all.py:124-133) on one fused reduction per direction:
    `L1Loss` on channel 0, with the UASR head `mean(|e| / u + log u) + L1Loss(u, |e|.detach())`, plus
    `BCEDiceLoss(alpha, beta)` on channels 1..C-1.  `forward(hat, target, uncertainty)` takes the network output, the target
    window (a strided view is read in place) and, exactly when `enable_uncertainty`, the uncertainty map."""

    def __init__(self, alpha: float = 1.0, beta: float = 1.0, enable_uncertainty: bool = False):
        super().__init__()
        self.alpha, self.beta, self.enable_uncertainty = alpha, beta, enable_uncertainty

    def forward(self, hat: torch.Tensor, target: torch.Tensor, uncertainty: Optional[torch.Tensor] = None) -> torch.Tensor:
        if (uncertainty is not None) != self.enable_uncertainty:
            raise L.RehrError(f"FusedSRLoss(enable_uncertainty={self.enable_uncertainty}) called "
                              f"{'without' if uncertainty is None else 'with'} an uncertainty map")
        sums = SRLossSums.apply(hat, target, uncertainty)
        n = hat[:, 0].numel()
        k = hat.shape[1] - 1
        loss = sums[0] / n
        if uncertainty is not None:
            loss = loss + (sums[1] + sums[2]) / n
        per = sums[3:].view(k, 4)
        dice = 2 * per[:, 1] / (per[:, 2] + per[:, 3]).clamp(min=1e-6)
        return loss + (self.alpha * per[:, 0].sum() / (n * k) + self.beta * (1.0 - dice.mean()))


def build_fused_loss(enable_deep_supervision: bool = False, weight_dice: float = 1) -> nn.Module:
    """`_build_loss` (utils/seg_utils.py:355-372) on the fused kernels; deep supervision is off (train_all.py:471)."""
    if enable_deep_supervision:
        raise NotImplementedError("train_all.py:471 fixes enable_deep_supervision=False")
    return FusedDCAndWeightedCELoss(weight_ce=1, weight_dice=weight_dice, smooth=1e-5)
