"""CPU oracle of the stage-2 intensity augmentations: the seven transforms `get_training_transforms` appends after the spatial part
(utils/seg_utils.py:677-689) -- Gaussian noise, Gaussian blur, multiplicative brightness, contrast, simulated low resolution, gamma
on the inverted image, gamma -- acting on `data` [b, c, z, x, y] float32 after Convert2DTo3DTransform.
TEST INFRASTRUCTURE: imported only by tests/ and tools/.

Parity unpinned: batchgenerators is not installed here, so the per-sample semantics are restated from batchgenerators 0.25 as
published (`augment_gaussian_noise`, `augment_gaussian_blur`, `augment_brightness_multiplicative`, `augment_contrast`,
`augment_linear_downsampling_scipy`, `augment_gamma` and the p_per_sample loops of their Transform classes), scikit-image's
`resize(mode='edge', anti_aliasing=False)` is restated as `scipy.ndimage.map_coordinates` at (i + 0.5) * n_in / n_out - 0.5 with
mode 'nearest' plus the clip to the input's range, and the parameters are nnU-Net v2's `get_training_transforms` values for the same
seven classes.  Every parameter is a keyword argument, so a correction against the reference's lines is a change of default.

Random streams: `rng_np` stands for `np.random` (every `np.random.uniform / random / normal` of batchgenerators), `rng_py` for
Python's `random` (batchgenerators' `get_range_val` and the noise variance).  Each transform loops over the samples inside itself,
so with b > 1 the draw order is transform-major."""
from __future__ import annotations

import numpy as np
from scipy.ndimage import gaussian_filter, map_coordinates

# nnU-Net v2 get_training_transforms values (see the module docstring: unpinned against utils/seg_utils.py:677-689)
NOISE = dict(noise_variance=(0.0, 0.1), p_per_sample=0.1, p_per_channel=1.0, per_channel=False)
BLUR = dict(blur_sigma=(0.5, 1.0), different_sigma_per_channel=True, different_sigma_per_axis=False, p_isotropic=0.0,
            p_per_channel=0.5, p_per_sample=0.2)
BRIGHTNESS = dict(multiplier_range=(0.75, 1.25), per_channel=True, p_per_sample=0.15)
CONTRAST = dict(contrast_range=(0.75, 1.25), preserve_range=True, per_channel=True, p_per_channel=1.0, p_per_sample=0.15)
LOWRES = dict(zoom_range=(0.5, 1.0), per_channel=True, p_per_channel=0.5, order_downsample=0, order_upsample=3, ignore_axes=(0,),
              p_per_sample=0.25)
GAMMA_INV = dict(gamma_range=(0.7, 1.5), invert_image=True, per_channel=True, retain_stats=True, p_per_sample=0.1)
GAMMA = dict(gamma_range=(0.7, 1.5), invert_image=False, per_channel=True, retain_stats=True, p_per_sample=0.3)


def _range_val(rng_py, r):
    """batchgenerators `get_range_val` for a (lo, hi) pair."""
    return r[0] if r[0] == r[1] else rng_py.uniform(r[0], r[1])


def _split_uniform(rng_np, r):
    """`U(lo, 1) if R() < 0.5 and lo < 1 else U(max(lo, 1), hi)` (contrast factor, gamma)."""
    if rng_np.random() < 0.5 and r[0] < 1:
        return rng_np.uniform(r[0], 1)
    return rng_np.uniform(max(r[0], 1), r[1])


def gaussian_noise(data, rng_np, rng_py, noise_variance=(0.0, 0.1), p_per_sample=0.1, p_per_channel=1.0, per_channel=False):
    """GaussianNoiseTransform: the drawn "variance" is used as the standard deviation; the float64 sum is stored as float32."""
    for b in range(data.shape[0]):
        if rng_np.uniform() < p_per_sample:
            v = None if per_channel else rng_py.uniform(noise_variance[0], noise_variance[1])
            for c in range(data.shape[1]):
                if rng_np.uniform() < p_per_channel:
                    vh = v if v is not None else _range_val(rng_py, noise_variance)
                    data[b, c] = data[b, c] + rng_np.normal(0.0, vh, size=data[b, c].shape)
    return data


def gaussian_blur(data, rng_np, rng_py, blur_sigma=(0.5, 1.0), different_sigma_per_channel=True, different_sigma_per_axis=False,
                  p_isotropic=0.0, p_per_channel=0.5, p_per_sample=0.2):
    """GaussianBlurTransform: scipy.ndimage.gaussian_filter over every axis of the channel (z included), mode 'reflect'."""
    nd = data.ndim - 2

    def sig():
        if (not different_sigma_per_axis) or (rng_np.uniform() < p_isotropic):
            return _range_val(rng_py, blur_sigma)
        return [_range_val(rng_py, blur_sigma) for _ in range(nd)]

    for b in range(data.shape[0]):
        if rng_np.uniform() < p_per_sample:
            s = None if different_sigma_per_channel else sig()
            for c in range(data.shape[1]):
                if rng_np.uniform() <= p_per_channel:
                    if different_sigma_per_channel:
                        s = sig()
                    data[b, c] = gaussian_filter(data[b, c], s, order=0)
    return data


def brightness_multiplicative(data, rng_np, multiplier_range=(0.75, 1.25), per_channel=True, p_per_sample=0.15):
    """BrightnessMultiplicativeTransform: one multiplier is drawn (and, per channel, discarded) before the per-channel ones."""
    for b in range(data.shape[0]):
        if rng_np.uniform() < p_per_sample:
            m = rng_np.uniform(multiplier_range[0], multiplier_range[1])
            if not per_channel:
                data[b] *= m
            else:
                for c in range(data.shape[1]):
                    data[b, c] *= rng_np.uniform(multiplier_range[0], multiplier_range[1])
    return data


def contrast_augmentation(data, rng_np, contrast_range=(0.75, 1.25), preserve_range=True, per_channel=True, p_per_channel=1.0,
                          p_per_sample=0.15):
    """ContrastAugmentationTransform, per channel: (x - mean) * f + mean, clipped to the channel's former [min, max]."""
    if not per_channel:
        raise NotImplementedError("contrast: per_channel=False")
    for b in range(data.shape[0]):
        if rng_np.uniform() < p_per_sample:
            for c in range(data.shape[1]):
                if rng_np.uniform() < p_per_channel:
                    f = _split_uniform(rng_np, contrast_range)
                    x = data[b, c]
                    mn = x.mean()
                    lo, hi = x.min(), x.max()
                    x = (x - mn) * f + mn
                    if preserve_range:
                        x[x < lo] = lo
                        x[x > hi] = hi
                    data[b, c] = x
    return data


def resize_edge(img, shape, order):
    """scikit-image `resize(img, shape, order, mode='edge', anti_aliasing=False)`: map_coordinates at (i + 0.5) * n_in / n_out - 0.5
    per axis, mode 'nearest', then clipped to the input's [min, max]."""
    axes = [(np.arange(n_out) + 0.5) * (n_in / n_out) - 0.5 for n_in, n_out in zip(img.shape, shape)]
    coords = np.array(np.meshgrid(*axes, indexing="ij"))
    out = map_coordinates(img, coords, order=order, mode="nearest")
    return np.clip(out, img.min(), img.max())


def simulate_low_resolution(data, rng_np, zoom_range=(0.5, 1.0), per_channel=True, p_per_channel=0.5, order_downsample=0,
                            order_upsample=3, ignore_axes=(0,), p_per_sample=0.25):
    """SimulateLowResolutionTransform: nearest downsampling to round(shape * zoom) (z kept), cubic upsampling back."""
    if not per_channel:
        raise NotImplementedError("simulate_low_resolution: per_channel=False")
    shp = np.array(data.shape[2:])
    for b in range(data.shape[0]):
        if rng_np.uniform() < p_per_sample:
            for c in range(data.shape[1]):
                if rng_np.uniform() < p_per_channel:
                    zm = rng_np.uniform(zoom_range[0], zoom_range[1])
                    t = np.round(shp * zm).astype(int)
                    for i in ignore_axes or ():
                        t[i] = shp[i]
                    if (t <= 0).any():
                        raise ValueError(f"simulate_low_resolution: target shape {t.tolist()}")
                    down = resize_edge(data[b, c].astype(float), t, order_downsample)
                    data[b, c] = resize_edge(down, shp, order_upsample)
    return data


def augment_gamma(data, rng_np, gamma_range=(0.7, 1.5), invert_image=False, per_channel=True, retain_stats=True, p_per_sample=0.3,
          epsilon=1e-7):
    """GammaTransform (augment_gamma, per channel, epsilon 1e-7): ((x - min) / (range + eps)) ** g * (range + eps) + min, mean and
    std (ddof 0) restored afterwards; on the negated sample when `invert_image`."""
    if not per_channel:
        raise NotImplementedError("gamma: per_channel=False")
    for b in range(data.shape[0]):
        if rng_np.uniform() < p_per_sample:
            x = -data[b] if invert_image else data[b].copy()
            for c in range(x.shape[0]):
                if retain_stats:
                    mn, sd = x[c].mean(), x[c].std()
                g = _split_uniform(rng_np, gamma_range)
                lo = x[c].min()
                r = x[c].max() - lo
                x[c] = np.power((x[c] - lo) / float(r + epsilon), g) * float(r + epsilon) + lo
                if retain_stats:
                    x[c] = x[c] - x[c].mean()
                    x[c] = x[c] / (x[c].std() + 1e-8) * sd
                    x[c] = x[c] + mn
            data[b] = -x if invert_image else x
    return data


# (keyword, defaults) of the seven transforms in list order
TRANSFORMS = (("noise", NOISE), ("blur", BLUR), ("brightness", BRIGHTNESS), ("contrast", CONTRAST), ("lowres", LOWRES),
              ("gamma_inv", GAMMA_INV), ("gamma", GAMMA))


def intensity_transform(data, rng_np, rng_py, **overrides):
    """The seven transforms in list order on a float32 [b, c, z, x, y] array, in place.  `overrides[name]` (a dict, name one of
    TRANSFORMS' keywords) replaces some of that transform's defaults, e.g. noise={"p_per_sample": 1.0}."""
    unknown = set(overrides) - {k for k, _ in TRANSFORMS}
    if unknown:
        raise TypeError(f"intensity_transform: unknown transforms {sorted(unknown)}")
    kw = {k: {**d, **(overrides.get(k) or {})} for k, d in TRANSFORMS}
    gaussian_noise(data, rng_np, rng_py, **kw["noise"])
    gaussian_blur(data, rng_np, rng_py, **kw["blur"])
    brightness_multiplicative(data, rng_np, **kw["brightness"])
    contrast_augmentation(data, rng_np, **kw["contrast"])
    simulate_low_resolution(data, rng_np, **kw["lowres"])
    augment_gamma(data, rng_np, **kw["gamma_inv"])
    augment_gamma(data, rng_np, **kw["gamma"])
    return data


def training_transform(patch_size_zyx, enable_uncertainty=True, rng=np.random, rng_py=None, intensity_kw=None, **aug_kw):
    """`get_training_transforms` (utils/seg_utils.py:632-689) as far as this project restates it: the spatial part
    (`oracle.augment.spatial_transform_dummy_2d`), then the seven intensity transforms on `data`, then NumpyToTensor('float').
    Usable as the `transform` of `oracle.augment.stage2_sample`."""
    import random as _random
    import torch
    from .augment import spatial_transform_dummy_2d
    keys = ("seg", "seg_sr", "uncertainty") if enable_uncertainty else ("seg", "seg_sr")
    rpy = rng_py or _random

    def run(**dd):
        out = spatial_transform_dummy_2d(dd, patch_size_zyx, keys=keys, enable_uncertainty=enable_uncertainty, rng=rng, **aug_kw)
        out["data"] = intensity_transform(np.ascontiguousarray(out["data"], dtype=np.float32), rng, rpy, **(intensity_kw or {}))
        return {k: torch.from_numpy(np.ascontiguousarray(v)).float() for k, v in out.items()}

    return run
