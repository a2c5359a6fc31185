"""CPU: the host half of the stage-2 intensity augmentation (rehrseg_b200/intensity.py) -- `IntensityAugment.draw` consumes
np.random and Python's random exactly as the oracle chain (oracle/intensity.py) does -- and its refusals."""
import random

import numpy as np
import pytest
import torch

from oracle import intensity as oi
from rehrseg_b200._lib import RehrError
from rehrseg_b200.intensity import NAMES, IntensityAugment, IntensityPlan

FORCED = {"noise": {"p_per_sample": 1.0}, "blur": {"p_per_sample": 1.0, "p_per_channel": 1.0},
          "brightness": {"p_per_sample": 1.0}, "contrast": {"p_per_sample": 1.0}, "lowres": {"p_per_sample": 1.0, "p_per_channel": 1.0},
          "gamma_inv": {"p_per_sample": 1.0}, "gamma": {"p_per_sample": 1.0}}


def _states_after(b, seed, overrides, draw):
    rng_np, rng_py = np.random.RandomState(seed), random.Random(seed)
    shape = (b, 2, 3, 9, 8)
    if draw:
        plan = IntensityAugment(**overrides).draw(b, shape[1], shape[2:], rng_py, rng_np)
    else:
        data = np.random.RandomState(1000 + seed).randn(*shape).astype(np.float32)
        oi.intensity_transform(data, rng_np, rng_py, **overrides)
        plan = None
    return rng_np.get_state(), rng_py.getstate(), plan


@pytest.mark.parametrize("b", [1, 3])
@pytest.mark.parametrize("forced", [False, True])
def test_draw_consumes_both_streams_like_the_oracle(b, forced):
    overrides = FORCED if forced else {}
    fired = set()
    for seed in range(50):
        np_e, py_e, plan = _states_after(b, seed, overrides, draw=True)
        np_o, py_o, _ = _states_after(b, seed, overrides, draw=False)
        assert py_e == py_o, seed
        assert np_e[0] == np_o[0] and np.array_equal(np_e[1], np_o[1]) and np_e[2:] == np_o[2:], seed
        fired |= set(plan.fired())
    if forced:
        assert fired == set(NAMES)
        assert len(plan.rows["gamma"]) == b * 2 and len(plan.noise) == b * 2


def test_plans_concatenate_along_the_batch():
    aug = IntensityAugment(**FORCED)
    p0 = aug.draw(1, 2, (3, 9, 8), random.Random(0), np.random.RandomState(0))
    p1 = aug.draw(2, 2, (3, 9, 8), random.Random(1), np.random.RandomState(1))
    cat = IntensityPlan.concat([p0, p1])
    assert cat.b == 3
    assert [r[0] for r in cat.rows["brightness"]] == [0, 0, 1, 1, 2, 2]
    assert cat.rows["gamma"][2:] == [(r[0] + 1,) + r[1:] for r in p1.rows["gamma"]]
    assert len(cat.noise) == 6


def test_cpu_tensor_raises():
    aug = IntensityAugment()
    with pytest.raises(RehrError):
        aug(torch.zeros(1, 1, 2, 4, 4))
    plan = IntensityAugment(**FORCED).draw(1, 1, (2, 4, 4), random.Random(0), np.random.RandomState(0))
    with pytest.raises(RehrError):
        aug.apply(torch.zeros(1, 1, 2, 4, 4), plan)


def test_empty_low_resolution_target_raises():
    aug = IntensityAugment(lowres={"p_per_sample": 1.0, "p_per_channel": 1.0, "zoom_range": (0.1, 0.2)})
    with pytest.raises(RehrError):
        aug.draw(1, 1, (4, 2, 40), random.Random(0), np.random.RandomState(0))


def test_unknown_parameters_and_unimplemented_options_are_refused():
    with pytest.raises(TypeError):
        IntensityAugment(sharpen={})
    with pytest.raises(TypeError):
        IntensityAugment(noise={"p": 1.0})
    with pytest.raises(RehrError):
        IntensityAugment(lowres={"ignore_axes": None})
