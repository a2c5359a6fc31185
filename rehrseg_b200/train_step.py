"""Stage-2 joint SR + segmentation training step (BASELINE config 4) on the B200 engine: the caller-side pieces of
`train_all.py:494-558` that sit either side of the conv hot path, with the reference's names and argument meaning.

  * `Distiller`            <- models/seg_model.py:115-151 (+ helpers :60-113): 1x1x1 projection of the student's stage-1
                              skip, cosine distance to the teacher feature over the spatial axis, optional smooth-L1, and the
                              pair-wise structure loss on per-slice max-pooled (kernel = half plane, ceil mode) feature maps.
                              Same constructor, same `state_dict` keys (`distill.weight`, `distill.bias`).
  * `build_loss`           <- `_build_loss`, utils/seg_utils.py:355-372 with `DC_and_weighted_CE_loss` :305-353 and
                              `RobustCrossEntropyLoss` :289-303 (deep supervision off, as train_all.py:471 hard-codes).
  * `joint_train_step`     <- the loop body train_all.py:519-558: teacher sweep under no_grad, student forward with
                              `return_inetermediate_feature=True`, LR loss (uncertainty-weighted CE), HR loss (CE + Dice),
                              distillation on `features_seg[1]` / `features_sr[1]`, zero_grad / backward / step.
  * `BCEDiceLoss`, `sr_train_step` <- the SR-stage loss `BCEDiceLoss(alpha, beta)` (utils/seg_utils.py:786-886) and the loop body
                              of `train_sr`, train_all.py:118-139, incl. the UASR terms :125-130 (L1 + |err|/u + log u + L1(u, |err|)).
  * `GraphedSRStep`        <- the same SR-stage iteration replayed from one CUDA graph (as `GraphedJointStep` for stage 2).
  * `allreduce_gradients`  <- what DistributedDataParallel would do for the reference: one flat bucket, mean over ranks
                              (NCCL over NVLink; InstanceNorm is per sample, so no other cross-rank traffic exists).

The network forwards/backwards inside run on the CUDA engine (rehrseg_b200.seg_model / rehrseg_b200.flavr); the loss
arithmetic here is a handful of full-tensor reductions on [B,2,D,H,W] logits and stays PyTorch, as SURVEY.md 8(a) rows
a9/a10 specify.  File:line citations are relative to /root/reference.
"""
from __future__ import annotations

from typing import Iterable, Optional, Sequence

import torch
import torch.nn.functional as F
from torch import nn

from . import flavr as _flavr


# ---------------------------------------------------------------------------------------------------------------
# Distillation
# ---------------------------------------------------------------------------------------------------------------
def cosine_distance_loss(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """models/seg_model.py:60-78: channel-normalise both maps, then 1 - cos over the flattened spatial axis, mean over
    (batch, channel)."""
    a = F.normalize(a, p=2, dim=1).flatten(2)
    b = F.normalize(b, p=2, dim=1).flatten(2)
    return (1 - torch.cosine_similarity(a, b, dim=2)).mean()


def _gram(feat: torch.Tensor) -> torch.Tensor:
    """models/seg_model.py:80-88: [N,C,h,w] -> channel-L2-normalised (norm detached, +1e-8) -> [N, h*w, h*w] Gram matrix."""
    feat = feat.float()
    norm = (feat.pow(2).sum(dim=1, keepdim=True).sqrt() + 1e-8).detach()
    f = (feat / norm).flatten(2)
    return torch.bmm(f.transpose(1, 2), f)


def structure_loss(student: torch.Tensor, teacher: torch.Tensor, scale: float = 0.5) -> torch.Tensor:
    """`CriterionPairWiseforWholeFeatAfterPool(scale)` + `sim_dis_compute`, models/seg_model.py:90-113.  [B,C,S,H,W]
    maps are pooled slice by slice with a max-pool whose kernel = stride = int(scale * plane) (ceil mode), the 4x4 Gram
    matrices of student and teacher are compared squared, divided by (pooled h*w)^2, by B*S, and once more by S."""
    b, c, s, th, tw = student.shape
    fs = student.permute(0, 2, 1, 3, 4).reshape(b * s, c, th, tw)
    ft = teacher.permute(0, 2, 1, 3, 4).reshape(b * s, teacher.shape[1], th, tw)
    k = (int(th * scale), int(tw * scale))
    ps = F.max_pool2d(fs, k, k, 0, ceil_mode=True)
    pt = F.max_pool2d(ft, k, k, 0, ceil_mode=True)
    err = (_gram(pt) - _gram(ps)).pow(2) / float((pt.shape[-1] * pt.shape[-2]) ** 2) / pt.shape[0]
    return err.sum() / s


class Distiller(nn.Module):
    """Drop-in for `models.seg_model.Distiller` (models/seg_model.py:115-151)."""

    def __init__(self, student_dim, teacher_dim, lambda_l1=0.0, lambda_cosine=0.0, lambda_structure=0.0):
        super().__init__()
        self.lambda_l1, self.lambda_cosine, self.lambda_structure = lambda_l1, lambda_cosine, lambda_structure
        self.distill = nn.Conv3d(student_dim, teacher_dim, kernel_size=1, stride=1, padding=0)

    def forward(self, feature_student, feature_teacher):
        loss = 0
        if self.lambda_structure > 0:
            loss = loss + self.lambda_structure * structure_loss(feature_student, feature_teacher, 0.5)
        projected = self.distill(feature_student)
        if self.lambda_l1 > 0:
            loss = loss + self.lambda_l1 * F.smooth_l1_loss(projected, feature_teacher)
        if self.lambda_cosine > 0:
            loss = loss + self.lambda_cosine * cosine_distance_loss(projected, feature_teacher)
        return loss


# ---------------------------------------------------------------------------------------------------------------
# Segmentation loss
# ---------------------------------------------------------------------------------------------------------------
class DCAndWeightedCELoss(nn.Module):
    """`DC_and_weighted_CE_loss` as `_build_loss` configures it (utils/seg_utils.py:305-353,355-358): per-voxel
    cross-entropy (optionally multiplied by an uncertainty map) averaged, plus the nnU-Net memory-efficient soft Dice
    (softmax, foreground classes only, per sample, smooth 1e-5) negated.

    Reference quirk kept on purpose: the CE map is [B,D,H,W] and the uncertainty map is [B,1,D,H,W]
    (utils/seg_utils.py:299-301 with the call at :349), so their product broadcasts to [B,B,D,H,W] before the mean --
    every sample's CE is weighted by every sample's uncertainty."""

    def __init__(self, weight_ce: float = 1, weight_dice: float = 1, smooth: float = 1e-5):
        super().__init__()
        self.weight_ce, self.weight_dice, self.smooth = weight_ce, weight_dice, smooth

    def forward(self, net_output: torch.Tensor, target: torch.Tensor, uncertainty: Optional[torch.Tensor] = None):
        assert target.shape[1] == 1, "target must be [B,1,...] label indices"
        labels = target[:, 0].long()
        total = 0
        if self.weight_dice != 0:
            prob = torch.softmax(net_output, 1)[:, 1:]
            axes = tuple(range(2, net_output.ndim))
            with torch.no_grad():
                onehot = torch.stack([labels == c for c in range(1, net_output.shape[1])], dim=1)
                sum_gt = onehot.sum(axes)
            intersect = (prob * onehot).sum(axes)
            dc = (2 * intersect + self.smooth) / torch.clip(sum_gt + prob.sum(axes) + self.smooth, 1e-8)
            total = total + self.weight_dice * (-dc.mean())
        if self.weight_ce != 0:
            ce = F.cross_entropy(net_output, labels, reduction="none")
            if uncertainty is not None:
                ce = ce * uncertainty          # [B,D,H,W] * [B,1,D,H,W] -> [B,B,D,H,W], see the class docstring
            total = total + self.weight_ce * ce.mean()
        return total


def build_loss(enable_deep_supervision: bool = False, weight_dice: float = 1) -> nn.Module:
    """`_build_loss` (utils/seg_utils.py:355-372).  Deep supervision is hard-wired off by the caller (train_all.py:471)."""
    if enable_deep_supervision:
        raise NotImplementedError("train_all.py:471 fixes enable_deep_supervision=False; the wrapper is not mirrored")
    return DCAndWeightedCELoss(weight_ce=1, weight_dice=weight_dice, smooth=1e-5)


# ---------------------------------------------------------------------------------------------------------------
# Data-parallel gradient mean
# ---------------------------------------------------------------------------------------------------------------
def allreduce_gradients(params: Iterable[torch.nn.Parameter], group=None) -> int:
    """Mean of every existing `.grad` over the ranks of `group` through ONE flat bucket (gather -> all-reduce ->
    scatter).  Returns the number of bucket elements (0 when torch.distributed is not initialised / world size 1)."""
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return 0
    grads = [p.grad for p in params if p.grad is not None]
    if not grads:
        return 0
    flat = torch.cat([g.reshape(-1) for g in grads])
    if dist.get_backend(group) == "nccl":
        dist.all_reduce(flat, op=dist.ReduceOp.AVG, group=group)
    else:                                      # gloo (CPU tests) has no AVG
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        flat /= dist.get_world_size(group)
    off, views = 0, []
    for g in grads:
        views.append(flat[off:off + g.numel()].view_as(g))
        off += g.numel()
    torch._foreach_copy_(grads, views)
    return flat.numel()


# ---------------------------------------------------------------------------------------------------------------
# The step
# ---------------------------------------------------------------------------------------------------------------
def joint_train_step(model_seg: nn.Module, batch: Sequence[torch.Tensor], loss_obj_lr_seg: nn.Module, loss_obj_hr_seg: nn.Module,
                     opt: Optional[torch.optim.Optimizer] = None, model_sr: Optional[nn.Module] = None,
                     distiller: Optional[nn.Module] = None, enable_uncertainty: bool = True, group=None, device=None,
                     teacher_keys: Optional[Sequence[int]] = None) -> dict:
    """One iteration of the stage-2 loop, train_all.py:519-558.  `batch` = (img, label_lr, label, uncertainty_lr) exactly
    as the reference DataLoader yields them; `model_sr` + `distiller` switch distillation on (train_all.py:494-495,
    530-533, 547-552).  With an initialised process group the gradients are averaged over ranks before `opt.step()`.
    `teacher_keys` (opt-in): passed to `get_intermediate_features(keys=...)`; the loop reads only `features_sr[1]` (:550), so
    `(1,)` lets an engine teacher stop after layer1 -- same losses and gradients, none of the discarded maps computed.  Default
    None = the reference's workload (all five maps).  Returns the detached loss terms."""
    img, label_lr, label, uncertainty_lr = batch
    device = device if device is not None else next(model_seg.parameters()).device
    model_seg.train()
    pseudo_img_lr = img.to(device, non_blocking=True)
    pseudo_label_lr = label_lr.to(device, non_blocking=True)
    label_sr = label.to(device, non_blocking=True)
    distill = model_sr is not None and distiller is not None
    if distill:
        with torch.no_grad():
            # the reference's zscore_normalization mutates `pseudo_img_lr` in place (utils/seg_utils.py:137-148), so the
            # student below sees the normalised image as well -- preserved
            features_sr = _flavr.get_intermediate_features(model_sr, pseudo_img_lr, pseudo_label_lr, device,
                                                           normalize=_flavr.zscore_normalization, keys=teacher_keys)
        pseudo_seg_lr, seg_sr, features_seg = model_seg(pseudo_img_lr, return_inetermediate_feature=True)
    else:
        pseudo_seg_lr, seg_sr = model_seg(pseudo_img_lr)
    if enable_uncertainty:
        loss_lr_seg = loss_obj_lr_seg(pseudo_seg_lr, pseudo_label_lr, uncertainty_lr.to(device, non_blocking=True))
        loss_hr_seg = loss_obj_hr_seg(seg_sr, label_sr, None)
    else:
        loss_lr_seg = loss_obj_lr_seg(pseudo_seg_lr, pseudo_label_lr)
        loss_hr_seg = loss_obj_hr_seg(seg_sr, label_sr)
    loss = loss_lr_seg + loss_hr_seg
    out = {"loss_lr_seg": loss_lr_seg.detach(), "loss_hr_seg": loss_hr_seg.detach()}
    if distill:
        distill_loss = distiller(features_seg[1], features_sr[1])
        loss = loss + distill_loss
        out["distill_loss"] = distill_loss.detach()
    params = list(model_seg.parameters()) + (list(distiller.parameters()) if distill else [])
    if opt is not None:
        opt.zero_grad()
    else:
        for p in params:
            p.grad = None
    loss.backward()
    allreduce_gradients(params, group)
    if opt is not None:
        opt.step()
    out["loss"] = loss.detach()
    return out


class _JointGraphModule(nn.Module):
    """What graphs.GraphedTrainStep needs of a "model" for the stage-2 step: the trainable parameters (student + distiller) and a
    forward on the first static input.  The frozen teacher is deliberately NOT a sub-module (its parameters get no gradients)."""

    def __init__(self, model_seg: nn.Module, distiller: Optional[nn.Module], model_sr: Optional[nn.Module]):
        super().__init__()
        self.model_seg = model_seg
        self.distiller = distiller
        self._teacher = [model_sr]

    def forward(self, img: torch.Tensor):
        model_sr = self._teacher[0]
        if model_sr is not None and self.distiller is not None:
            return ("distill", img)
        return ("plain", img)


class GraphedJointStep:
    """The stage-2 iteration (train_all.py:519-558: teacher window sweep, student forward, uncertainty-weighted CE + CE/Dice,
    structural distillation, backward) captured into ONE CUDA graph and replayed; the optimiser step stays outside.

        step = GraphedJointStep(model_seg, batch0, loss_lr, loss_hr, model_sr, distiller)
        for batch in loader:                      # host (pinned) or device tensors of the captured shapes
            out = step(batch)                     # copies the batch into the static inputs, replays; out = static loss terms
            opt.step()                            # .grad tensors are static, re-attached after every replay

    Same arithmetic as `joint_train_step` (tests/test_joint_gpu.py compares the two); inside the graph the weight gradients stay
    on their side stream until the end of the step and the 16-bit weight copies are re-packed in a few batched launches."""

    def __init__(self, model_seg: nn.Module, example_batch: Sequence[torch.Tensor], loss_obj_lr_seg: nn.Module,
                 loss_obj_hr_seg: nn.Module, model_sr: Optional[nn.Module] = None, distiller: Optional[nn.Module] = None,
                 enable_uncertainty: bool = True, dp_group=None, teacher_keys: Optional[Sequence[int]] = None,
                 range_check: bool = False):
        from .graphs import GraphedTrainStep
        device = next(model_seg.parameters()).device
        model_seg.train()
        self.terms: dict = {}
        distill = model_sr is not None and distiller is not None
        terms = self.terms

        def loss_fn(tagged, pseudo_label_lr, label_sr, uncertainty_lr):
            _, pseudo_img_lr = tagged
            if distill:
                with torch.no_grad():
                    features_sr = _flavr.get_intermediate_features(model_sr, pseudo_img_lr, pseudo_label_lr, device,
                                                                   normalize=_flavr.zscore_normalization, keys=teacher_keys)
                pseudo_seg_lr, seg_sr, features_seg = model_seg(pseudo_img_lr, return_inetermediate_feature=True)
            else:
                pseudo_seg_lr, seg_sr = model_seg(pseudo_img_lr)
            if enable_uncertainty:
                loss_lr_seg = loss_obj_lr_seg(pseudo_seg_lr, pseudo_label_lr, uncertainty_lr)
                loss_hr_seg = loss_obj_hr_seg(seg_sr, label_sr, None)
            else:
                loss_lr_seg = loss_obj_lr_seg(pseudo_seg_lr, pseudo_label_lr)
                loss_hr_seg = loss_obj_hr_seg(seg_sr, label_sr)
            loss = loss_lr_seg + loss_hr_seg
            terms["loss_lr_seg"], terms["loss_hr_seg"] = loss_lr_seg.detach(), loss_hr_seg.detach()
            if distill:
                distill_loss = distiller(features_seg[1], features_sr[1])
                loss = loss + distill_loss
                terms["distill_loss"] = distill_loss.detach()
            return loss

        self.module = _JointGraphModule(model_seg, distiller if distill else None, model_sr if distill else None)
        self.step = GraphedTrainStep(self.module, loss_fn, tuple(example_batch), dp_group=dp_group, range_check=range_check)

    def range_report(self):
        """fp16 saturation of the last replay's student forward (`range_check=True`; names are prefixed `model_seg.`)."""
        return self.step.range_report()

    def __call__(self, batch: Sequence[torch.Tensor]) -> dict:
        self.step.load(*batch)
        loss = self.step.replay()
        out = dict(self.terms)
        out["loss"] = loss
        return out

    def close(self) -> None:
        self.step.close()


# ---------------------------------------------------------------------------------------------------------------
# SR stage (BASELINE config 2's training step): train_all.py:114-152
# ---------------------------------------------------------------------------------------------------------------
class BCEDiceLoss(nn.Module):
    """`BCEDiceLoss(alpha, beta)` = alpha * BCEWithLogits + beta * (1 - mean per-channel Dice of sigmoid(input)), the Dice with the
    V-Net denominator sum(p^2) + sum(t^2) clamped at 1e-6 (utils/seg_utils.py:821-886; channel axis first, batch flattened in)."""

    def __init__(self, alpha: float, beta: float):
        super().__init__()
        self.alpha, self.beta = alpha, beta
        self.bce = nn.BCEWithLogitsLoss()

    def forward(self, input: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
        prob = torch.sigmoid(input)
        c = prob.size(1)
        p = prob.transpose(0, 1).reshape(c, -1)
        t = target.transpose(0, 1).reshape(c, -1).float()
        dice = 2 * ((p * t).sum(-1) / ((p * p).sum(-1) + (t * t).sum(-1)).clamp(min=1e-6))
        return self.alpha * self.bce(input, target) + self.beta * (1.0 - dice.mean())


def _sr_loss(out, patches_hr: torch.Tensor, loss_obj: Optional[nn.Module], loss_seg: Optional[nn.Module], slice_separation: int,
             num_slices: int, enable_uncertainty: bool, fused_loss: Optional[nn.Module]) -> torch.Tensor:
    """The loss of train_all.py:122-133 from the model output `out` ((prediction, uncertainty) with the UASR head) and the full
    HR batch: the target window, then the plain statements or, when given, `fused_loss` (loss_ops.FusedSRLoss)."""
    if num_slices > 1:
        patches_hr = patches_hr[:, :, int(slice_separation) * (num_slices // 2 - 1):int(slice_separation) * (num_slices // 2), ...]
    patches_hr_hat, uncertainty = out if enable_uncertainty else (out, None)
    if fused_loss is not None:
        return fused_loss(patches_hr_hat, patches_hr, uncertainty)
    if enable_uncertainty:
        loss = loss_obj(patches_hr_hat[:, 0:1, ...], patches_hr[:, 0:1, ...])
        loss = loss + torch.mean(torch.div(torch.abs(patches_hr_hat[:, 0:1, ...] - patches_hr[:, 0:1, ...]), uncertainty)
                                 + torch.log(uncertainty))
        error_map = torch.abs(patches_hr_hat[:, 0:1, ...].detach() - patches_hr[:, 0:1, ...])
        loss = loss + loss_obj(uncertainty, error_map)
    else:
        loss = loss_obj(patches_hr_hat[:, 0:1, ...], patches_hr[:, 0:1, ...])
    return loss + loss_seg(patches_hr_hat[:, 1:, ...], patches_hr[:, 1:, ...]) * 1.0


def sr_train_step(model: nn.Module, batch: Sequence[torch.Tensor], loss_obj: nn.Module, loss_seg: nn.Module,
                  opt: Optional[torch.optim.Optimizer] = None, scheduler=None, slice_separation: int = 4, num_slices: int = 4,
                  enable_uncertainty: bool = False, group=None, device=None, fused_loss: Optional[nn.Module] = None) -> dict:
    """One iteration of `train_sr` (train_all.py:118-139).  `batch` = (patches_lr [B,2,num_slices,H,W], patches_hr [B,2,S,H,W]) as the
    DataLoader yields them; with `num_slices > 1` the target is the `slice_separation` HR slices between the two central LR slices
    (:122-123).  `enable_uncertainty` adds the UASR terms :125-130 on the model's (prediction, uncertainty) pair.  The reference
    calls `model(patches_lr)`, whose forward subtracts the channel-0 mean IN PLACE from the batch (FLAVR_arch.py:180-181) --
    preserved: `patches_lr` on the device is mutated.  Gradients are averaged over `group` before the optimiser step.
    `fused_loss` (opt-in, a `loss_ops.FusedSRLoss` built with the same alpha, beta and enable_uncertainty) replaces the loss
    statements with one fused CUDA reduction per direction; `loss_obj` / `loss_seg` are then unused."""
    patches_lr, patches_hr = batch
    device = device if device is not None else next(model.parameters()).device
    patches_hr = patches_hr.to(device, non_blocking=True)
    patches_lr = patches_lr.to(device, non_blocking=True)
    loss = _sr_loss(model(patches_lr), patches_hr, loss_obj, loss_seg, slice_separation, num_slices, enable_uncertainty, fused_loss)
    params = list(model.parameters())
    if opt is not None:
        opt.zero_grad()
    else:
        for p in params:
            p.grad = None
    loss.backward()
    allreduce_gradients(params, group)
    if opt is not None:
        opt.step()
    if scheduler is not None:
        scheduler.step()
    return {"loss": loss.detach()}


class GraphedSRStep:
    """The SR-stage iteration (train_all.py:118-138: forward, target window, L1 / UASR / BCE-Dice loss, backward) captured into ONE
    CUDA graph and replayed; the optimiser and scheduler steps stay outside.  Same loss as `sr_train_step` with the same
    arguments: the plain `loss_obj` / `loss_seg` statements, or `fused_loss` (loss_ops.FusedSRLoss) when given.

        step = GraphedSRStep(model, batch0, fused_loss=loss_ops.FusedSRLoss(1, 1, enable_uncertainty=True), enable_uncertainty=True)
        for batch in loader:                      # (patches_lr, patches_hr), host (pinned) or device tensors of the captured shapes
            out = step(batch)                     # copies the batch into the static inputs, replays; out["loss"] is static
            opt.step(); scheduler.step()          # .grad tensors are static, re-attached after every replay

    One difference from `sr_train_step`: the model's forward subtracts the channel-0 mean in place from the STATIC copy of
    `patches_lr` on every replay; the caller's `patches_lr` is left unchanged.  `dp_group` is passed to `graphs.GraphedTrainStep`
    (the gradient mean over ranks is then part of the captured step)."""

    def __init__(self, model: nn.Module, example_batch: Sequence[torch.Tensor], loss_obj: Optional[nn.Module] = None,
                 loss_seg: Optional[nn.Module] = None, slice_separation: int = 4, num_slices: int = 4, enable_uncertainty: bool = False,
                 fused_loss: Optional[nn.Module] = None, dp_group=None, range_check: bool = False):
        from .graphs import GraphedTrainStep
        if fused_loss is None and (loss_obj is None or loss_seg is None):
            raise ValueError("GraphedSRStep needs either fused_loss or both loss_obj and loss_seg")

        def loss_fn(out, patches_hr):
            return _sr_loss(out, patches_hr, loss_obj, loss_seg, slice_separation, num_slices, enable_uncertainty, fused_loss)

        self.step = GraphedTrainStep(model, loss_fn, tuple(example_batch), dp_group=dp_group, range_check=range_check)

    def range_report(self):
        """fp16 saturation records of the last replay (`range_check=True`).  The FLAVR network stores its activations in bf16,
        so its report is empty."""
        return self.step.range_report()

    def __call__(self, batch: Sequence[torch.Tensor]) -> dict:
        self.step.load(*batch)
        return {"loss": self.step.replay()}

    def close(self) -> None:
        self.step.close()
