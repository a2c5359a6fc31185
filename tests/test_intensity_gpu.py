"""GPU: stage-2 intensity augmentation (rehrseg_b200/intensity.py, csrc/intensity.cu) against the numpy / scipy oracle
(oracle/intensity.py) under the same np.random / random seeds: each transform alone, the default chain, the Stage2Sampler
integration, batch = stacked samples bit for bit, and the launch count."""
import random

import numpy as np
import pytest
import torch

from oracle import intensity as oi
from rehrseg_b200.intensity import NAMES, IntensityAugment

pytestmark = pytest.mark.gpu

FORCED = {"noise": {"p_per_sample": 1.0}, "blur": {"p_per_sample": 1.0, "p_per_channel": 1.0},
          "brightness": {"p_per_sample": 1.0}, "contrast": {"p_per_sample": 1.0}, "lowres": {"p_per_sample": 1.0, "p_per_channel": 1.0},
          "gamma_inv": {"p_per_sample": 1.0}, "gamma": {"p_per_sample": 1.0}}
OFF = {k: {"p_per_sample": 0.0} for k in NAMES}
TOL = {"noise": 1e-5, "blur": 1e-5, "brightness": 1e-5, "contrast": 1e-5, "lowres": 1e-4, "gamma_inv": 1e-4, "gamma": 1e-4}
SHAPES = [(1, 1, 16, 64, 48), (3, 2, 5, 33, 31), (2, 1, 1, 40, 40), (2, 1, 2, 17, 23)]


def _err(got, want):
    want = np.asarray(want, dtype=np.float64)
    return float(np.abs(got.cpu().double().numpy() - want).max()) / max(1.0, float(np.abs(want).max()))


def _run_both(data, overrides, seed):
    """(engine result, oracle result, engine rng states, oracle rng states, plan) from the same seeds."""
    rn, rp = np.random.RandomState(seed), random.Random(seed)
    aug = IntensityAugment(**overrides)
    x = torch.from_numpy(data).cuda()
    plan = aug.draw(x.shape[0], x.shape[1], x.shape[2:], rp, rn)
    aug.apply(x, plan)
    torch.cuda.synchronize()
    on, op = np.random.RandomState(seed), random.Random(seed)
    want = oi.intensity_transform(data.copy(), on, op, **overrides)
    return x, want, (rn.get_state(), rp.getstate()), (on.get_state(), op.getstate()), plan


def _same_states(a, b):
    return a[1] == b[1] and a[0][0] == b[0][0] and np.array_equal(a[0][1], b[0][1]) and a[0][2:] == b[0][2:]


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("shape", SHAPES + ["constant"])
def test_each_transform_alone(name, shape):
    overrides = {**OFF, name: FORCED[name]}
    if shape == "constant":
        shape = (2, 2, 5, 33, 31)
        data = np.random.RandomState(3).randn(*shape).astype(np.float32)
        data[0, 1] = 0.7
    else:
        data = np.random.RandomState(sum(shape)).randn(*shape).astype(np.float32) * 1.5 + 0.25
    for seed in range(3):
        got, want, st_e, st_o, plan = _run_both(data, overrides, seed)
        assert plan.fired() == [name]
        assert np.isfinite(got.cpu().numpy()).all()
        err = _err(got, want)
        assert err <= TOL[name], (name, shape, seed, err)
        assert _same_states(st_e, st_o), (name, shape, seed)


def test_default_chain_over_60_seeds():
    data = np.random.RandomState(7).randn(1, 1, 16, 128, 96).astype(np.float32)
    fired = set()
    for seed in range(60):
        got, want, st_e, st_o, plan = _run_both(data, {}, seed)
        fired |= set(plan.fired())
        assert _err(got, want) <= 1e-4, (seed, plan.fired())
        assert _same_states(st_e, st_o), seed
    assert fired == set(NAMES), fired


def _subject():
    rng = np.random.RandomState(8)                 # the subject of oracle/make_golden.py stage2_sample_fixture
    X, Y, Z = 36, 30, 20
    return ((rng.rand(X, Y, Z) * 300).astype(np.float32), (rng.rand(X, Y, Z) > 0.6).astype(np.uint8),
            (rng.rand(X, Y, Z) * 255).astype(np.uint8))


@pytest.mark.parametrize("overrides", [{}, FORCED], ids=["defaults", "forced"])
def test_stage2_sampler_matches_the_oracle_getitem(overrides):
    from oracle import augment as oa
    from rehrseg_b200 import augment
    img, lab, unc = _subject()
    ps, sep = (32, 24, 3), 4
    ds = augment.Stage2Sampler(ps, sep, p_rot_per_sample=1.0, p_scale_per_sample=1.0, intensity=IntensityAugment(**overrides))
    ds.add_subject(img, lab, unc)
    for seed in range(8):
        random.seed(seed)
        np.random.seed(seed)
        got = ds.sample(0)
        st_e = (np.random.get_state(), random.getstate())
        random.seed(seed)
        np.random.seed(seed)
        tr = oi.training_transform((ps[2], ps[1], ps[0]), rng=np.random, rng_py=random, p_rot_per_sample=1.0, p_scale_per_sample=1.0,
                                   intensity_kw=overrides)
        want = oa.stage2_sample(img, lab, unc, ps, sep, transform=tr)
        assert _same_states(st_e, (np.random.get_state(), random.getstate())), seed
        for name, g, w in zip(("img", "label_lr", "label", "uncertainty_lr"), got, want):
            w = w.numpy()
            assert tuple(g.shape) == w.shape, (seed, name)
            if name in ("img", "uncertainty_lr"):
                assert _err(g, w) <= 3e-4, (seed, name, _err(g, w))
            else:
                assert float((g.cpu().numpy() == w).mean()) >= 0.999, (seed, name)


def test_batch_is_bit_identical_to_stacked_samples():
    from rehrseg_b200 import augment
    img, lab, unc = _subject()
    ds = augment.Stage2Sampler((32, 24, 3), 4, intensity=IntensityAugment(**FORCED))
    ds.add_subject(img, lab, unc)
    random.seed(5)
    np.random.seed(5)
    got = ds.batch([0, 0, 0, 0])
    random.seed(5)
    np.random.seed(5)
    rows = [ds.sample(0) for _ in range(4)]
    for k in range(4):
        assert torch.equal(got[k], torch.stack([r[k] for r in rows])), k


def _launches(b, overrides):
    from rehrseg_b200 import functional as F_
    aug = IntensityAugment(**overrides)
    x = torch.randn(b, 1, 4, 32, 24, device="cuda")
    plan = aug.draw(b, 1, x.shape[2:], random.Random(0), np.random.RandomState(0))
    l0 = F_.launches()
    aug.apply(x, plan)
    return F_.launches() - l0, plan


def test_launch_count_does_not_grow_with_the_batch():
    n1, p1 = _launches(1, FORCED)
    n8, p8 = _launches(8, FORCED)
    assert p1.fired() == list(NAMES) and p8.fired() == list(NAMES)
    assert n1 == n8 == 1 + 3 + 1 + 2 + 5 + 3 + 3


def test_nothing_fires_nothing_launches():
    n, plan = _launches(8, OFF)
    assert plan.fired() == [] and n == 0
