"""CPU oracle of the opt-in device noise of the stage-2 intensity augmentation (`IntensityAugment(noise_rng="philox")`,
rehrseg_b200/intensity.py).  TEST INFRASTRUCTURE: imported only by tests/ and tools/.

The chain is oracle/intensity.py's with one change in the Gaussian noise: where batchgenerators calls `np.random.normal` for a noised
(sample, channel) row, this mode draws `key = rng_np.randint(0, 2**64, size=2, dtype=np.uint64)`, and the row's field is
Box-Muller over the words of `np.random.Philox(key=key).random_raw` (numpy's own Philox4x64-10; `philox4x64_10` below restates one
block so that the tests can pin the counter convention).  Every other draw, and every other transform, is oracle/intensity.py's."""
from __future__ import annotations

import numpy as np

from . import intensity as oi

_M64 = (1 << 64) - 1


def philox4x64_10(counter, key):
    """One Philox4x64-10 block (Random123's multipliers and Weyl constants) as Python integers: 4 words of 64 bits."""
    c, (k0, k1) = [int(v) for v in counter], (int(key[0]), int(key[1]))
    for r in range(10):
        if r:
            k0, k1 = (k0 + 0x9E3779B97F4A7C15) & _M64, (k1 + 0xBB67AE8584CAA73B) & _M64
        p0, p1 = 0xD2E7470EE14C6C93 * c[0], 0xCA5A826395121157 * c[2]
        c = [(p1 >> 64) ^ c[1] ^ k0, p1 & _M64, (p0 >> 64) ^ c[3] ^ k1, p0 & _M64]
    return c


def philox_normals(key, n):
    """n standard normals of one row: element e takes word e % 4 of block e // 4 = philox(counter (e // 4 + 1, 0, 0, 0), key), i.e.
    word e of np.random.Philox(key=key).random_raw; Box-Muller in float64 over the word pairs (2j, 2j + 1) with
    u1 = ((w >> 11) + 1) 2^-53 in (0, 1], u2 = (w' >> 11) 2^-53: z_2j = r cos(2 pi u2), z_2j+1 = r sin(2 pi u2), r = sqrt(-2 ln u1).
    An odd n uses only the cosine of its last pair."""
    w = np.random.Philox(key=np.asarray(key, dtype=np.uint64)).random_raw(n + (n & 1))
    u1 = ((w[0::2] >> np.uint64(11)) + np.uint64(1)).astype(np.float64) * 2.0 ** -53
    u2 = (w[1::2] >> np.uint64(11)).astype(np.float64) * 2.0 ** -53
    r, t = np.sqrt(-2.0 * np.log(u1)), 2.0 * np.pi * u2
    z = np.empty(w.size)
    z[0::2], z[1::2] = r * np.cos(t), r * np.sin(t)
    return z[:n]


def gaussian_noise(data, rng_np, rng_py, noise_variance=(0.0, 0.1), p_per_sample=0.1, p_per_channel=1.0, per_channel=False):
    """oracle.intensity.gaussian_noise with the field of a drawn key: `philox_normals` scaled by the drawn standard deviation and
    rounded to float32, then added in float64 and stored as float32 (the engine's arithmetic)."""
    for b in range(data.shape[0]):
        if rng_np.uniform() < p_per_sample:
            v = None if per_channel else rng_py.uniform(noise_variance[0], noise_variance[1])
            for c in range(data.shape[1]):
                if rng_np.uniform() < p_per_channel:
                    vh = v if v is not None else oi._range_val(rng_py, noise_variance)
                    key = rng_np.randint(0, 2 ** 64, size=2, dtype=np.uint64)
                    field = (vh * philox_normals(key, data[b, c].size)).astype(np.float32).reshape(data[b, c].shape)
                    data[b, c] = data[b, c] + field.astype(np.float64)
    return data


def intensity_transform(data, rng_np, rng_py, **overrides):
    """oracle.intensity.intensity_transform with this module's `gaussian_noise`: the seven transforms in list order on a float32
    [b, c, z, x, y] array, in place, with the same `overrides`."""
    unknown = set(overrides) - {k for k, _ in oi.TRANSFORMS}
    if unknown:
        raise TypeError(f"intensity_transform: unknown transforms {sorted(unknown)}")
    kw = {k: {**d, **(overrides.get(k) or {})} for k, d in oi.TRANSFORMS}
    gaussian_noise(data, rng_np, rng_py, **kw["noise"])
    oi.gaussian_blur(data, rng_np, rng_py, **kw["blur"])
    oi.brightness_multiplicative(data, rng_np, **kw["brightness"])
    oi.contrast_augmentation(data, rng_np, **kw["contrast"])
    oi.simulate_low_resolution(data, rng_np, **kw["lowres"])
    oi.augment_gamma(data, rng_np, **kw["gamma_inv"])
    oi.augment_gamma(data, rng_np, **kw["gamma"])
    return data


def training_transform(patch_size_zyx, enable_uncertainty=True, rng=np.random, rng_py=None, intensity_kw=None, **aug_kw):
    """oracle.intensity.training_transform with this module's `intensity_transform`: the spatial part, the seven intensity transforms
    with the Philox noise, then NumpyToTensor('float').  Usable as the `transform` of `oracle.augment.stage2_sample`."""
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
