"""GPU-side spatial augmentation of the stage-2 data pipeline (SURVEY.md section 8(f) row 2).

The reference rotates / scales every training patch on the CPU: `MySpatialTransform` -> `augment_spatial`
(utils/seg_utils.py:378-631) -> batchgenerators `interpolate_img` -> `scipy.ndimage.map_coordinates`, order-3 splines for the image
and the uncertainty map, order-1 per-label interpolation for the two segmentations, in 4 DataLoader worker processes
(train_all.py:502-509).  In the configuration `get_training_transforms` builds (utils/seg_utils.py:652-676: dummy-2D, no elastic
deformation, rotation about x and isotropic scaling with p = 0.2 each, no random crop) the coordinate field of a sample is AFFINE,
so the whole transform is two kernels: scipy's cubic B-spline prefilter along both image axes (`rehr_bspline_prefilter_axis`) and
one gather per output pixel (`rehr_affine_sample2d`).  The random decisions are drawn from `np.random` in the reference's order.
The intensity transforms that follow the spatial part (utils/seg_utils.py:677-689) are rehrseg_b200/intensity.py; `Stage2Sampler`
runs them when given an `IntensityAugment`.

Parity: tests/test_augment_gpu.py against tests/golden/spatial_aug.npz (the reference's OWN `augment_spatial` with scipy's real
map_coordinates) and against oracle/augment.py on other shapes."""
from __future__ import annotations

import ctypes as C
import math
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import functional as F_
from ._lib import RehrError, check, lib, ptr, stream_ptr
from .intensity import IntensityAugment, IntensityPlan


def draw_affine_2d(rng=np.random, do_rotation=True, angle_x=(-math.pi, math.pi), do_scale=True, scale=(0.7, 1.4),
                   p_scale_per_sample=0.2, p_rot_per_sample=0.2, p_rot_per_axis=1.0):
    """The random decisions of one sample, in the order of utils/seg_utils.py:409-446 (dim == 2, no elastic deformation, one scale
    for both axes): (rotation angle or None, scale or None)."""
    a_x = None
    if do_rotation and rng.uniform() < p_rot_per_sample:
        a_x = rng.uniform(angle_x[0], angle_x[1]) if rng.uniform() <= p_rot_per_axis else 0
    sc = None
    if do_scale and rng.uniform() < p_scale_per_sample:
        if rng.random() < 0.5 and scale[0] < 1:
            sc = rng.uniform(scale[0], 1)
        else:
            sc = rng.uniform(max(scale[0], 1), scale[1])
    return a_x, sc


def _affine_rows(params, X: int, Y: int) -> torch.Tensor:
    """[(angle, scale)] -> f32 [samples][6]: source position = A (i - (PX-1)/2, j - (PY-1)/2) + c with A = s R^T (rotate_coords_2d
    multiplies the row vectors by R = [[cos, -sin], [sin, cos]]), c = image centre (random_crop=False, utils/seg_utils.py:453)."""
    rows = []
    for a_x, sc in params:
        cs, sn = (math.cos(a_x), math.sin(a_x)) if a_x is not None else (1.0, 0.0)
        s = 1.0 if sc is None else float(sc)
        rows.append([s * cs, s * sn, -s * sn, s * cs, X / 2.0 - 0.5, Y / 2.0 - 0.5])
    return torch.tensor(rows, dtype=torch.float32)


def _sample(img: torch.Tensor, affine_dev: torch.Tensor, patch: Tuple[int, int], order: int, cval: float,
            labels: Optional[Sequence[float]] = None) -> torch.Tensor:
    b, c, X, Y = img.shape
    out = torch.empty((b, c, patch[0], patch[1]), dtype=torch.float32, device=img.device)
    if order == 3:
        src = img.float().clone()                      # the prefilter works in place
        check(lib().rehr_bspline_prefilter_axis(ptr(src), b * c, X, Y, stream_ptr()), "bspline_prefilter")
        check(lib().rehr_bspline_prefilter_axis(ptr(src), b * c * X, Y, 1, stream_ptr()), "bspline_prefilter")
        F_._count(2)
        lab_arr, nlab = None, 0
    else:
        src = img.float().contiguous()
        if labels is None:
            labels = torch.unique(src).tolist()        # np.unique(img) of interpolate_img (host read: the label set is data)
        if len(labels) > 8:
            raise RehrError("augment: more than 8 distinct labels in a segmentation are not implemented")
        lab_arr = (C.c_float * len(labels))(*[float(v) for v in sorted(labels)])
        nlab = len(labels)
    check(lib().rehr_affine_sample2d(ptr(src), ptr(out), ptr(affine_dev), b * c, X, Y, patch[0], patch[1], c, order, float(cval),
                                     lab_arr, nlab, stream_ptr()), "affine_sample2d")
    F_._count()
    return out


def augment_spatial(data: torch.Tensor, seg_list: Optional[List[torch.Tensor]], patch_size: Sequence[int], do_rotation=True,
                    angle_x=(-math.pi, math.pi), do_scale=True, scale=(0.7, 1.4), border_cval_data=0.0, order_data=3,
                    border_cval_seg=-1.0, order_seg=1, p_scale_per_sample=0.2, p_rot_per_sample=0.2, p_rot_per_axis=1.0,
                    enable_uncertainty=False, rng=np.random, seg_labels: Optional[Sequence[float]] = None):
    """`augment_spatial` (utils/seg_utils.py:378-458) for 2-D batches `data` [b, c, x, y] on the GPU with the stage-2 settings
    (border modes "constant", no elastic deformation, no random crop).  Returns (data_result, seg_result) as fp32 CUDA tensors of
    shape [b, c_k, *patch_size]; the LAST entry of `seg_list` is interpolated like the image when `enable_uncertainty`."""
    if data.dim() != 4 or len(patch_size) != 2:
        raise RehrError("augment_spatial: 2-D batches [b, c, x, y] (the dummy-2D configuration of the stage-2 pipeline)")
    if not data.is_cuda:
        raise RehrError("rehrseg_b200 ops need CUDA tensors (no CPU fallback)")
    if order_data != 3 or order_seg != 1:
        raise RehrError("augment_spatial: order 3 (data) / order 1 (segmentations) are implemented")
    b, _, X, Y = data.shape
    params = [draw_affine_2d(rng, do_rotation, angle_x, do_scale, scale, p_scale_per_sample, p_rot_per_sample, p_rot_per_axis)
              for _ in range(b)]
    affine = _affine_rows(params, X, Y).to(data.device)
    patch = (int(patch_size[0]), int(patch_size[1]))
    data_result = _sample(data, affine, patch, 3, border_cval_data)
    seg_result = None
    if seg_list is not None:
        seg_result = []
        for i, seg in enumerate(seg_list):
            if i == len(seg_list) - 1 and enable_uncertainty:
                seg_result.append(_sample(seg, affine, patch, 3, border_cval_data))
            else:
                seg_result.append(_sample(seg, affine, patch, 1, border_cval_seg, seg_labels))
    return data_result, seg_result


def spatial_transform_dummy_2d(data_dict: dict, patch_size_zxy: Sequence[int], keys=("seg", "seg_sr", "uncertainty"),
                               enable_uncertainty=True, rng=np.random, seg_labels: Optional[Sequence[float]] = None, **aug_kw) -> dict:
    """Convert3DTo2DTransform -> MySpatialTransform(patch_size[1:]) -> Convert2DTo3DTransform (utils/seg_utils.py:652-676) on CUDA
    tensors {'data', *keys} of shape [b, c, z, x, y]: the slices of a patch become channels and share the sample's affine map."""
    shapes, flat = {}, {}
    for k in ("data", *keys):
        t = data_dict[k]
        shapes[k] = t.shape
        flat[k] = t.reshape(t.shape[0], t.shape[1] * t.shape[2], t.shape[3], t.shape[4])
    d, segs = augment_spatial(flat["data"], [flat[k] for k in keys], tuple(patch_size_zxy[1:]), enable_uncertainty=enable_uncertainty,
                              rng=rng, seg_labels=seg_labels, **aug_kw)
    out = {"data": d.reshape(shapes["data"][0], shapes["data"][1], shapes["data"][2], d.shape[-2], d.shape[-1])}
    for k, s in zip(keys, segs):
        out[k] = s.reshape(shapes[k][0], shapes[k][1], shapes[k][2], s.shape[-2], s.shape[-1])
    return out


class Stage2Sampler:
    """`TrainSetMultipleSegSREfficient` (utils/train_set.py:21-159) with the subjects resident on the GPU: `sample(i)` is
    `__getitem__` -- z-score of the volume, random crop (Python `random`, the reference's order), constant padding, flips, slice
    decimation, the [1, 1, z, y, x] layout, the uncertainty rescaling -- followed by the SPATIAL part of `self.train_transform`
    (`spatial_transform_dummy_2d`, `np.random`) and, when `intensity` is given, by the intensity transforms `get_training_transforms`
    appends after it (`rehrseg_b200.intensity.IntensityAugment`, drawn right after the sample's spatial decisions); `batch` stacks
    samples like the DataLoader's collate and runs the intensity transforms of all its samples in one pass."""

    def __init__(self, patch_size: Sequence[int], separation: int, norm: bool = True, random_flip: bool = True,
                 uncertainty: bool = True, device=None, p_rot_per_sample: float = 0.2, p_scale_per_sample: float = 0.2,
                 intensity: Optional["IntensityAugment"] = None):
        self.patch_size = list(patch_size)            # (x, y, z_lr) as in the reference's patch_size_ori
        self.separation = int(separation)
        self.norm, self.random_flip, self.uncertainty = bool(norm), bool(random_flip), bool(uncertainty)
        self.p_rot, self.p_scale = float(p_rot_per_sample), float(p_scale_per_sample)
        self.intensity = intensity
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.imgs: List[torch.Tensor] = []
        self.labels: List[torch.Tensor] = []
        self.uncertainties: List[Optional[torch.Tensor]] = []

    def __len__(self) -> int:
        return len(self.imgs)

    def add_subject(self, img, label, uncertainty=None) -> None:
        """[X, Y, Z] volumes.  The reference z-scores the volume it has just read on every `__getitem__` (utils/train_set.py:106-107,
        utils/seg_utils.py:149-155); the volume is constant, so it is normalised once here."""
        im = torch.as_tensor(img).to(self.device, torch.float32).clone()
        if self.norm:
            mean, std = im.mean(), im.std(unbiased=False)
            im = (im - mean) / torch.clamp(std, min=1e-8)
        self.imgs.append(im)
        self.labels.append(torch.as_tensor(label).to(self.device))
        self.uncertainties.append(None if uncertainty is None else torch.as_tensor(uncertainty).to(self.device))

    @staticmethod
    def _pad(t: torch.Tensor, target) -> torch.Tensor:
        from .volume_ops import get_pads
        flat = []
        for b, a in reversed([get_pads(tt, d) for tt, d in zip(target, t.shape)]):
            flat += [b, a]
        return torch.nn.functional.pad(t, flat) if any(flat) else t

    def sample(self, i: int, rng_py=None, rng_np=np.random, seg_labels: Optional[Sequence[float]] = None):
        out, plan = self._sample(i, rng_py, rng_np, seg_labels)
        if plan is not None:
            self.intensity.apply(out[0][None], plan)
        return out

    def _sample(self, i: int, rng_py, rng_np, seg_labels):
        """One sample before its intensity transforms: (outputs of `sample`, the drawn IntensityPlan or None)."""
        import random as _random
        rng = rng_py or _random
        img, label = self.imgs[i], self.labels[i]
        ps, sep = self.patch_size, self.separation
        x_0 = rng.randint(0, max(img.shape[0] - ps[0], 0))
        y_0 = rng.randint(0, max(img.shape[1] - ps[1], 0))
        z_0 = rng.randint(0, max(img.shape[2] - ps[2] * sep, 0))
        sl = (slice(x_0, x_0 + ps[0]), slice(y_0, y_0 + ps[1]), slice(z_0, z_0 + ps[2] * sep))
        img = img[sl]
        target = [max(s, p) for s, p in zip(img.shape, (ps[0], ps[1], ps[2] * sep))]
        img = self._pad(img, target)
        label = self._pad(label[sl], target)
        unc = self._pad(self.uncertainties[i][sl], target) if self.uncertainty else None
        if self.random_flip:
            for axis in (0, 1, 2):
                if rng.random() < 0.5:
                    img, label = img.flip(axis), label.flip(axis)
                    unc = unc.flip(axis) if unc is not None else None
        img = img[:, :, ::sep]
        label_lr = label[:, :, ::sep]
        dd = {"data": img.permute(2, 1, 0)[None, None].float(), "seg": label_lr.permute(2, 1, 0)[None, None].float(),
              "seg_sr": label.permute(2, 1, 0)[None, None].float()}
        keys = ["seg", "seg_sr"]
        if self.uncertainty:
            unc_lr = unc[:, :, ::sep].permute(2, 1, 0)[None, None]
            dd["uncertainty"] = 1 - unc_lr.double() / 255. * 0.99        # numpy promotes the uint8 map to float64 here
            dd["uncertainty"] = dd["uncertainty"].float()
            keys.append("uncertainty")
        patch_zyx = (ps[2], ps[1], ps[0])                                  # target_patch_size[::-1], utils/train_set.py:77
        out = spatial_transform_dummy_2d({k: v.contiguous() for k, v in dd.items()}, patch_zyx, keys=tuple(keys),
                                         enable_uncertainty=self.uncertainty, rng=rng_np, seg_labels=seg_labels,
                                         p_rot_per_sample=self.p_rot, p_scale_per_sample=self.p_scale)
        plan = None
        if self.intensity is not None:
            plan = self.intensity.draw(1, 1, out["data"].shape[2:], rng, rng_np)
        unc_out = out["uncertainty"].squeeze(0) if self.uncertainty else 0
        return (out["data"].squeeze(0), out["seg"].squeeze(0), out["seg_sr"].squeeze(0), unc_out), plan

    def batch(self, indices: Sequence[int], rng_py=None, rng_np=np.random, seg_labels: Optional[Sequence[float]] = None):
        drawn = [self._sample(i, rng_py, rng_np, seg_labels) for i in indices]
        out = tuple(torch.stack([r[k] for r, _ in drawn]) for k in range(4 if self.uncertainty else 3))
        if self.intensity is not None:
            self.intensity.apply(out[0], IntensityPlan.concat([p for _, p in drawn]))
        return out
