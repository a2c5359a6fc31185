"""GPU intensity augmentation of the stage-2 data pipeline: the seven transforms `get_training_transforms` appends after the spatial
part (utils/seg_utils.py:677-689) -- Gaussian noise, Gaussian blur, multiplicative brightness, contrast, simulated low resolution,
gamma on the inverted image, gamma -- on `data` [b, c, z, x, y] fp32 after Convert2DTo3DTransform.

Parity unpinned: batchgenerators is not installed where this was written, so the semantics are batchgenerators 0.25's as published
and scikit-image's `resize(mode='edge', anti_aliasing=False)` as scipy.ndimage.map_coordinates (restated in oracle/intensity.py),
and the default parameters are nnU-Net v2's `get_training_transforms` values for the same seven classes.  Every parameter is a
keyword argument, so checking them against the reference's lines means changing defaults, not kernels.

None of the random decisions depends on the data, so `draw` makes all of them on the host in the reference's order (`rng_np` for
np.random, `rng_py` for Python's random), including the noise field, which only `rng_np.normal` can produce without disturbing every
later draw; it goes to pinned memory and reaches the GPU with an asynchronous copy.  `apply` then runs every transform that fired
anywhere in the batch with a fixed number of launches over the (sample, channel) rows it fired on (csrc/intensity.cu)."""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Optional, Sequence

import numpy as np
import torch

from . import functional as F_
from ._lib import RehrError, check, check_device, lib, ptr, stream_ptr

NOISE = dict(noise_variance=(0.0, 0.1), p_per_sample=0.1, p_per_channel=1.0, per_channel=False)
BLUR = dict(blur_sigma=(0.5, 1.0), different_sigma_per_channel=True, different_sigma_per_axis=False, p_isotropic=0.0,
            p_per_channel=0.5, p_per_sample=0.2)
BRIGHTNESS = dict(multiplier_range=(0.75, 1.25), per_channel=True, p_per_sample=0.15)
CONTRAST = dict(contrast_range=(0.75, 1.25), preserve_range=True, per_channel=True, p_per_channel=1.0, p_per_sample=0.15)
LOWRES = dict(zoom_range=(0.5, 1.0), per_channel=True, p_per_channel=0.5, order_downsample=0, order_upsample=3, ignore_axes=(0,),
              p_per_sample=0.25)
GAMMA_INV = dict(gamma_range=(0.7, 1.5), invert_image=True, per_channel=True, retain_stats=True, p_per_sample=0.1)
GAMMA = dict(gamma_range=(0.7, 1.5), invert_image=False, per_channel=True, retain_stats=True, p_per_sample=0.3)
# (keyword, defaults) in list order
TRANSFORMS = (("noise", NOISE), ("blur", BLUR), ("brightness", BRIGHTNESS), ("contrast", CONTRAST), ("lowres", LOWRES),
              ("gamma_inv", GAMMA_INV), ("gamma", GAMMA))
NAMES = tuple(k for k, _ in TRANSFORMS)

_PAD = 12               # scipy's pre-padding of an order-3 spline in mode 'nearest' (csrc/intensity.cu kLowresPad)
_MAX_BLUR_RADIUS = 63   # csrc/intensity.cu kMaxBlurRadius
# mirror of rehr_irow (include/rehrseg_b200.h)
IROW = np.dtype([("off", "<i8"), ("aux", "<i8"), ("len", "<i8"), ("n", "<i4", (4,)), ("p", "<f8", (4,))], align=True)
assert IROW.itemsize == 72


def _range_val(rng_py, r):
    """batchgenerators `get_range_val` for a (lo, hi) pair."""
    return r[0] if r[0] == r[1] else rng_py.uniform(r[0], r[1])


def _split_uniform(rng_np, r):
    """`U(lo, 1) if R() < 0.5 and lo < 1 else U(max(lo, 1), hi)` (contrast factor, gamma)."""
    if rng_np.random() < 0.5 and r[0] < 1:
        return rng_np.uniform(r[0], 1)
    return rng_np.uniform(max(r[0], 1), r[1])


class IntensityPlan:
    """The host-drawn decisions for a batch [b, c, *shape]: per transform, the rows (sample, channel, parameters...) it fired on,
    and the noise fields (fp32 host tensors, pinned when CUDA is available) in the order of the noise rows."""

    def __init__(self, b: int, c: int, shape: Sequence[int]):
        self.b, self.c, self.shape = int(b), int(c), tuple(int(s) for s in shape)
        self.rows: Dict[str, List[tuple]] = {k: [] for k in NAMES}
        self.noise: List[torch.Tensor] = []

    def fired(self) -> List[str]:
        return [k for k in NAMES if self.rows[k]]

    @staticmethod
    def concat(plans: Sequence["IntensityPlan"]) -> "IntensityPlan":
        """The plan of the samples of `plans` stacked along the batch."""
        if not plans or any(p.c != plans[0].c or p.shape != plans[0].shape for p in plans):
            raise RehrError("IntensityPlan.concat: plans of the same channel count and spatial shape")
        out = IntensityPlan(sum(p.b for p in plans), plans[0].c, plans[0].shape)
        b0 = 0
        for p in plans:
            for k in NAMES:
                out.rows[k] += [(r[0] + b0,) + tuple(r[1:]) for r in p.rows[k]]
            out.noise += p.noise
            b0 += p.b
        return out


class IntensityAugment:
    """The seven intensity transforms in list order.  Keywords `noise`, `blur`, `brightness`, `contrast`, `lowres`, `gamma_inv`,
    `gamma` take dicts that override that transform's defaults (the module constants), e.g. noise={"p_per_sample": 1.0}.

    `draw(b, c, spatial_shape, rng_py, rng_np)` makes every random decision on the host, consuming both streams exactly as the
    batchgenerators transforms do; `apply(data, plan)` runs the plan in place on a CUDA fp32 [b, c, z, x, y] tensor; calling the
    object does both."""

    def __init__(self, **overrides):
        unknown = set(overrides) - set(NAMES)
        if unknown:
            raise TypeError(f"IntensityAugment: unknown transforms {sorted(unknown)}")
        self.params = {k: {**d, **(overrides.get(k) or {})} for k, d in TRANSFORMS}
        for k, d in TRANSFORMS:
            extra = set(self.params[k]) - set(d)
            if extra:
                raise TypeError(f"IntensityAugment: unknown {k} parameters {sorted(extra)}")
        P = self.params
        for k in ("contrast", "lowres", "gamma_inv", "gamma"):
            if not P[k]["per_channel"]:
                raise RehrError(f"IntensityAugment: {k} with per_channel=False is not implemented")
        lr = P["lowres"]
        if lr["order_downsample"] != 0 or lr["order_upsample"] != 3 or 0 not in tuple(lr["ignore_axes"] or ()):
            raise RehrError("IntensityAugment: low resolution is implemented for order 0 down / order 3 up with z (axis 0) kept")

    # ---- host: the random decisions ------------------------------------------------------------------------------------------------
    def draw(self, b: int, c: int, spatial_shape: Sequence[int], rng_py, rng_np) -> IntensityPlan:
        shape = tuple(int(s) for s in spatial_shape)
        if len(shape) != 3:
            raise RehrError("IntensityAugment: spatial shape (z, x, y)")
        plan = IntensityPlan(b, c, shape)
        P, R = self.params, plan.rows
        V = int(np.prod(shape))
        pin = torch.cuda.is_available()

        q = P["noise"]
        for bi in range(b):
            if rng_np.uniform() < q["p_per_sample"]:
                v = None if q["per_channel"] else rng_py.uniform(q["noise_variance"][0], q["noise_variance"][1])
                for ci in range(c):
                    if rng_np.uniform() < q["p_per_channel"]:
                        vh = v if v is not None else _range_val(rng_py, q["noise_variance"])
                        field = torch.empty(V, dtype=torch.float32, pin_memory=pin)
                        field.numpy()[:] = rng_np.normal(0.0, vh, size=shape).reshape(-1)
                        R["noise"].append((bi, ci))
                        plan.noise.append(field)

        q = P["blur"]

        def sig():
            if (not q["different_sigma_per_axis"]) or (rng_np.uniform() < q["p_isotropic"]):
                return (_range_val(rng_py, q["blur_sigma"]),) * 3
            return tuple(_range_val(rng_py, q["blur_sigma"]) for _ in range(3))

        for bi in range(b):
            if rng_np.uniform() < q["p_per_sample"]:
                s = None if q["different_sigma_per_channel"] else sig()
                for ci in range(c):
                    if rng_np.uniform() <= q["p_per_channel"]:
                        if q["different_sigma_per_channel"]:
                            s = sig()
                        R["blur"].append((bi, ci, tuple(float(v) for v in s)))

        q = P["brightness"]
        for bi in range(b):
            if rng_np.uniform() < q["p_per_sample"]:
                m = rng_np.uniform(q["multiplier_range"][0], q["multiplier_range"][1])
                for ci in range(c):
                    if q["per_channel"]:
                        m = rng_np.uniform(q["multiplier_range"][0], q["multiplier_range"][1])
                    R["brightness"].append((bi, ci, float(m)))

        q = P["contrast"]
        for bi in range(b):
            if rng_np.uniform() < q["p_per_sample"]:
                for ci in range(c):
                    if rng_np.uniform() < q["p_per_channel"]:
                        R["contrast"].append((bi, ci, float(_split_uniform(rng_np, q["contrast_range"])), bool(q["preserve_range"])))

        q = P["lowres"]
        shp = np.array(shape)
        for bi in range(b):
            if rng_np.uniform() < q["p_per_sample"]:
                for ci in range(c):
                    if rng_np.uniform() < q["p_per_channel"]:
                        zm = rng_np.uniform(q["zoom_range"][0], q["zoom_range"][1])
                        t = np.round(shp * zm).astype(int)
                        for i in q["ignore_axes"]:
                            t[i] = shp[i]
                        if (t <= 0).any():
                            raise RehrError(f"IntensityAugment: low-resolution target shape {t.tolist()} (zoom {zm}) is empty")
                        R["lowres"].append((bi, ci, int(t[1]), int(t[2])))

        for k in ("gamma_inv", "gamma"):
            q = P[k]
            sign = -1.0 if q["invert_image"] else 1.0
            for bi in range(b):
                if rng_np.uniform() < q["p_per_sample"]:
                    for ci in range(c):
                        R[k].append((bi, ci, float(_split_uniform(rng_np, q["gamma_range"])), sign, bool(q["retain_stats"])))

        for row in R["blur"]:
            if max(int(4.0 * s + 0.5) for s in row[2]) > _MAX_BLUR_RADIUS:
                raise RehrError(f"IntensityAugment: blur sigma {row[2]} needs more than {2 * _MAX_BLUR_RADIUS + 1} taps")
        return plan

    # ---- device: the kernels ----------------------------------------------------------------------------------------------------------
    def apply(self, data: torch.Tensor, plan: IntensityPlan) -> torch.Tensor:
        """Run `plan` in place on `data` (CUDA, fp32, contiguous [b, c, z, x, y]); returns `data`."""
        _check_data(data)
        if (data.shape[0], data.shape[1], tuple(data.shape[2:])) != (plan.b, plan.c, plan.shape):
            raise RehrError(f"IntensityAugment.apply: data {tuple(data.shape)} but the plan is for "
                            f"{(plan.b, plan.c) + plan.shape}")
        fired = plan.fired()
        if not fired:
            return data
        Z, X, Y = plan.shape
        V = Z * X * Y
        dev = data.device

        # one row table per transform, all in one buffer: a single host-to-device copy
        tables, aux_len = {}, {}
        for k in fired:
            rows = plan.rows[k]
            t = np.zeros(len(rows), IROW)
            t["off"] = [(r[0] * plan.c + r[1]) * V for r in rows]
            t["len"] = V
            t["aux"] = np.arange(len(rows), dtype=np.int64) * V
            if k == "blur":
                t["p"][:, :3] = [r[2] for r in rows]
                t["n"][:, :3] = [[int(4.0 * s + 0.5) for s in r[2]] for r in rows]      # scipy: radius = int(truncate * sigma + 0.5)
            elif k == "brightness":
                t["p"][:, 0] = [r[2] for r in rows]
            elif k == "contrast":
                t["p"][:, 0] = [r[2] for r in rows]
                t["n"][:, 0] = [int(r[3]) for r in rows]
            elif k == "lowres":
                t["n"][:, 0] = [r[2] for r in rows]
                t["n"][:, 1] = [r[3] for r in rows]
                t["len"] = [Z * (r[2] + 2 * _PAD) * (r[3] + 2 * _PAD) for r in rows]
                t["aux"] = np.concatenate([[0], np.cumsum(t["len"])[:-1]])
                aux_len[k] = int(t["len"].sum())
            elif k in ("gamma_inv", "gamma"):
                t["p"][:, 0] = [r[2] for r in rows]
                t["p"][:, 1] = [r[3] for r in rows]
                t["n"][:, 0] = [int(r[4]) for r in rows]
            tables[k] = t
        blob = np.concatenate([tables[k].view(np.uint8) for k in fired])
        dev_blob = torch.from_numpy(blob).pin_memory().to(dev, non_blocking=True)
        addr, o = {}, 0
        for k in fired:
            addr[k] = C.c_void_p(dev_blob.data_ptr() + o)
            o += tables[k].nbytes

        L, s = lib(), stream_ptr()
        md = L.rehr_intensity_moment_doubles()
        x = ptr(data)
        f32 = dict(dtype=torch.float32, device=dev)

        def moments(base, k, from_aux, max_len):
            m = torch.empty(len(plan.rows[k]) * md, dtype=torch.float64, device=dev)
            check(L.rehr_intensity_moments(ptr(base), addr[k], len(plan.rows[k]), from_aux, max_len, ptr(m), s), "intensity_moments")
            return m

        for k in fired:
            n, tab = len(plan.rows[k]), addr[k]
            if k == "noise":
                nz = torch.empty(n * V, **f32)
                for r, field in enumerate(plan.noise):
                    nz[r * V:(r + 1) * V].copy_(field, non_blocking=True)
                check(L.rehr_intensity_pointwise(x, tab, n, V, 0, ptr(nz), None, s), "intensity_noise")
                F_._count(1)
            elif k == "blur":
                t1, t2 = torch.empty(n * V, **f32), torch.empty(n * V, **f32)
                for src, sa, dst, da, axis in ((data, 0, t1, 1, 0), (t1, 1, t2, 1, 1), (t2, 1, data, 0, 2)):
                    check(L.rehr_intensity_blur_axis(ptr(src), sa, ptr(dst), da, tab, n, Z, X, Y, axis, s), "intensity_blur")
                F_._count(3)
            elif k == "brightness":
                check(L.rehr_intensity_pointwise(x, tab, n, V, 1, None, None, s), "intensity_brightness")
                F_._count(1)
            elif k == "contrast":
                m = moments(data, k, 0, V)
                check(L.rehr_intensity_pointwise(x, tab, n, V, 2, None, ptr(m), s), "intensity_contrast")
                F_._count(2)
            elif k == "lowres":
                rows = plan.rows[k]
                pad = torch.empty(aux_len[k], **f32)
                max_len = int(tables[k]["len"].max())
                check(L.rehr_intensity_lowres_gather(x, ptr(pad), tab, n, Z, X, Y, max_len, s), "intensity_lowres_gather")
                m = moments(pad, k, 1, max_len)
                check(L.rehr_intensity_lowres_prefilter(ptr(pad), tab, n, Z, 1, max(Z * (r[3] + 2 * _PAD) for r in rows), s),
                      "intensity_lowres_prefilter")
                check(L.rehr_intensity_lowres_prefilter(ptr(pad), tab, n, Z, 2, max(Z * (r[2] + 2 * _PAD) for r in rows), s),
                      "intensity_lowres_prefilter")
                check(L.rehr_intensity_lowres_upsample(x, ptr(pad), tab, n, Z, X, Y, ptr(m), s), "intensity_lowres_upsample")
                F_._count(5)
            else:
                m = moments(data, k, 0, V)
                pw = torch.empty(n * md, dtype=torch.float64, device=dev)
                check(L.rehr_intensity_gamma(x, tab, n, V, ptr(m), ptr(pw), 0, s), "intensity_gamma")
                check(L.rehr_intensity_gamma(x, tab, n, V, ptr(m), ptr(pw), 1, s), "intensity_gamma")
                F_._count(3)
        return data

    def __call__(self, data: torch.Tensor, rng_py=None, rng_np=np.random) -> torch.Tensor:
        import random as _random
        _check_data(data)
        plan = self.draw(data.shape[0], data.shape[1], data.shape[2:], rng_py or _random, rng_np)
        return self.apply(data, plan)


def _check_data(data: torch.Tensor) -> None:
    if not data.is_cuda:
        raise RehrError("rehrseg_b200 ops need CUDA tensors (no CPU fallback)")
    check_device(data)
    if data.dim() != 5 or data.dtype != torch.float32 or not data.is_contiguous():
        raise RehrError("IntensityAugment: contiguous fp32 [b, c, z, x, y] data")
