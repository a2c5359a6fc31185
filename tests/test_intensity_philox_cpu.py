"""CPU: the opt-in device noise of the stage-2 intensity augmentation (`IntensityAugment(noise_rng="philox")`) -- the oracle's
Philox4x64-10 restatement against numpy's own generator (which pins the counter convention the kernel uses), the oracle's
Box-Muller field against a scalar restatement, the random streams `draw` leaves behind against the oracle's philox chain, and the
refusals."""
import math
import random

import numpy as np
import pytest

from oracle import intensity_philox as op
from rehrseg_b200._lib import RehrError
from rehrseg_b200.intensity import NAMES, IntensityAugment, IntensityPlan

FORCED = {"noise": {"p_per_sample": 1.0}, "blur": {"p_per_sample": 1.0, "p_per_channel": 1.0},
          "brightness": {"p_per_sample": 1.0}, "contrast": {"p_per_sample": 1.0}, "lowres": {"p_per_sample": 1.0, "p_per_channel": 1.0},
          "gamma_inv": {"p_per_sample": 1.0}, "gamma": {"p_per_sample": 1.0}}
KEYS = [(0, 0), (1, 2), (2 ** 64 - 1, 12345), (0x0123456789ABCDEF, 0xFEDCBA9876543210)]


@pytest.mark.parametrize("key", KEYS)
def test_philox_restatement_is_numpys_philox_from_counter_one(key):
    raw = np.random.Philox(key=np.array(key, dtype=np.uint64)).random_raw(4 * 5)
    mine = [w for g in range(5) for w in op.philox4x64_10((g + 1, 0, 0, 0), key)]
    assert [int(w) for w in raw] == mine
    # numpy's first block is counter 1, not counter 0
    assert op.philox4x64_10((0, 0, 0, 0), key) != mine[:4]


@pytest.mark.parametrize("n", [1, 2, 7, 8, 13])
def test_philox_normals_are_box_muller_over_word_pairs(n):
    key = (0xDEADBEEF, 42)
    words = [w for g in range((n + 3) // 4) for w in op.philox4x64_10((g + 1, 0, 0, 0), key)]
    want = []
    for j in range(0, n, 2):
        u1 = ((words[j] >> 11) + 1) * 2.0 ** -53
        u2 = (words[j + 1] >> 11) * 2.0 ** -53
        r = math.sqrt(-2.0 * math.log(u1))
        want += [r * math.cos(2.0 * math.pi * u2), r * math.sin(2.0 * math.pi * u2)]
    got = op.philox_normals(np.array(key, dtype=np.uint64), n)
    assert got.shape == (n,)
    np.testing.assert_allclose(got, want[:n], rtol=1e-15, atol=1e-15)


def _states_after(b, seed, overrides, draw):
    rng_np, rng_py = np.random.RandomState(seed), random.Random(seed)
    shape = (b, 2, 3, 9, 8)
    if draw:
        plan = IntensityAugment(noise_rng="philox", **overrides).draw(b, shape[1], shape[2:], rng_py, rng_np)
    else:
        data = np.random.RandomState(1000 + seed).randn(*shape).astype(np.float32)
        op.intensity_transform(data, rng_np, rng_py, **overrides)
        plan = None
    return rng_np.get_state(), rng_py.getstate(), plan


@pytest.mark.parametrize("b", [1, 3])
@pytest.mark.parametrize("forced", [False, True])
def test_philox_draw_consumes_both_streams_like_the_oracle(b, forced):
    overrides = FORCED if forced else {}
    noised = 0
    for seed in range(50):
        np_e, py_e, plan = _states_after(b, seed, overrides, draw=True)
        np_o, py_o, _ = _states_after(b, seed, overrides, draw=False)
        assert py_e == py_o, seed
        assert np_e[0] == np_o[0] and np.array_equal(np_e[1], np_o[1]) and np_e[2:] == np_o[2:], seed
        assert plan.noise == [] and plan.noise_keys.dtype == np.uint64
        assert plan.noise_keys.shape == (len(plan.rows["noise"]), 2)
        noised += len(plan.rows["noise"])
    if forced:
        assert noised == 50 * b * 2
    else:
        assert noised > 0


def test_philox_keys_replace_the_normal_draw_in_place():
    """Same draws as the numpy mode up to the first noised row; its key is the next randint of the stream."""
    aug = IntensityAugment(noise_rng="philox", **{**{k: {"p_per_sample": 0.0} for k in NAMES}, "noise": {"p_per_sample": 1.0}})
    rn = np.random.RandomState(3)
    plan = aug.draw(1, 1, (2, 4, 4), random.Random(3), rn)
    want = np.random.RandomState(3)
    want.uniform(), want.uniform()          # p_per_sample, p_per_channel
    assert np.array_equal(plan.noise_keys[0], want.randint(0, 2 ** 64, size=2, dtype=np.uint64))


@pytest.mark.parametrize("bad", ["", "Philox", "mt19937", None, 1])
def test_bad_noise_rng_raises(bad):
    with pytest.raises(RehrError):
        IntensityAugment(noise_rng=bad)


def test_noise_rng_is_not_a_noise_parameter():
    with pytest.raises(TypeError):
        IntensityAugment(noise={"noise_rng": "philox"})


def test_philox_plans_concatenate_with_their_keys():
    aug = IntensityAugment(noise_rng="philox", **FORCED)
    p0 = aug.draw(1, 2, (3, 9, 8), random.Random(0), np.random.RandomState(0))
    p1 = aug.draw(2, 2, (3, 9, 8), random.Random(1), np.random.RandomState(1))
    cat = IntensityPlan.concat([p0, p1])
    assert cat.noise_rng == "philox" and cat.b == 3
    assert [r[:2] for r in cat.rows["noise"]] == [(0, 0), (0, 1), (1, 0), (1, 1), (2, 0), (2, 1)]
    assert np.array_equal(cat.noise_keys, np.concatenate([p0.noise_keys, p1.noise_keys]))


def test_plans_of_mixed_noise_rng_do_not_concatenate():
    shape = (3, 9, 8)
    pn = IntensityAugment(**FORCED).draw(1, 1, shape, random.Random(0), np.random.RandomState(0))
    pp = IntensityAugment(noise_rng="philox", **FORCED).draw(1, 1, shape, random.Random(0), np.random.RandomState(0))
    with pytest.raises(RehrError):
        IntensityPlan.concat([pn, pp])
    with pytest.raises(RehrError):
        IntensityPlan.concat([pp, pn])
