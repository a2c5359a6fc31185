"""GPU: the opt-in device noise of the stage-2 intensity augmentation (`IntensityAugment(noise_rng="philox")`,
csrc/intensity.cu intensity_noise_philox_kernel) against the oracle's philox chain (oracle/intensity_philox.py) under the same
seeds: noise alone, the default chain, the Stage2Sampler integration, batch = stacked samples bit for bit, the launch count, the
distribution of the generated field, and the default numpy mode left as it was."""
import random

import numpy as np
import pytest
import torch

from oracle import intensity as oi
from oracle import intensity_philox as op
from rehrseg_b200.intensity import NAMES, IntensityAugment

pytestmark = pytest.mark.gpu

FORCED = {"noise": {"p_per_sample": 1.0}, "blur": {"p_per_sample": 1.0, "p_per_channel": 1.0},
          "brightness": {"p_per_sample": 1.0}, "contrast": {"p_per_sample": 1.0}, "lowres": {"p_per_sample": 1.0, "p_per_channel": 1.0},
          "gamma_inv": {"p_per_sample": 1.0}, "gamma": {"p_per_sample": 1.0}}
OFF = {k: {"p_per_sample": 0.0} for k in NAMES}
NOISE_ONLY = {**OFF, "noise": FORCED["noise"]}
SHAPES = [(1, 1, 16, 64, 48), (3, 2, 5, 33, 31), (2, 1, 1, 40, 40), (2, 1, 2, 17, 23)]


def _err(got, want):
    want = np.asarray(want, dtype=np.float64)
    return float(np.abs(got.cpu().double().numpy() - want).max()) / max(1.0, float(np.abs(want).max()))


def _run_both(data, overrides, seed, noise_rng="philox"):
    """(engine result, oracle result, engine rng states, oracle rng states, plan) from the same seeds."""
    rn, rp = np.random.RandomState(seed), random.Random(seed)
    aug = IntensityAugment(noise_rng=noise_rng, **overrides)
    x = torch.from_numpy(data).cuda()
    plan = aug.draw(x.shape[0], x.shape[1], x.shape[2:], rp, rn)
    aug.apply(x, plan)
    torch.cuda.synchronize()
    on, opy = np.random.RandomState(seed), random.Random(seed)
    chain = op.intensity_transform if noise_rng == "philox" else oi.intensity_transform
    want = chain(data.copy(), on, opy, **overrides)
    return x, want, (rn.get_state(), rp.getstate()), (on.get_state(), opy.getstate()), plan


def _same_states(a, b):
    return a[1] == b[1] and a[0][0] == b[0][0] and np.array_equal(a[0][1], b[0][1]) and a[0][2:] == b[0][2:]


@pytest.mark.parametrize("shape", SHAPES)
def test_noise_alone_matches_the_oracle(shape):
    data = np.random.RandomState(sum(shape)).randn(*shape).astype(np.float32) * 1.5 + 0.25
    for seed in range(3):
        got, want, st_e, st_o, plan = _run_both(data, NOISE_ONLY, seed)
        assert plan.fired() == ["noise"] and len(plan.rows["noise"]) == shape[0] * shape[1]
        assert not np.array_equal(got.cpu().numpy(), data)
        # host and device f64 log / sincos may differ in the last ulp: at most one f32 ulp of the result
        err = _err(got, want)
        assert err <= 1e-6, (shape, seed, err)
        assert _same_states(st_e, st_o), (shape, seed)


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
    rng = np.random.RandomState(8)
    X, Y, Z = 36, 30, 20
    return ((rng.rand(X, Y, Z) * 300).astype(np.float32), (rng.rand(X, Y, Z) > 0.6).astype(np.uint8),
            (rng.rand(X, Y, Z) * 255).astype(np.uint8))


@pytest.mark.parametrize("overrides", [{}, FORCED], ids=["defaults", "forced"])
def test_stage2_sampler_matches_the_oracle_getitem(overrides):
    from oracle import augment as oa
    from rehrseg_b200 import augment
    img, lab, unc = _subject()
    ps, sep = (32, 24, 3), 4
    ds = augment.Stage2Sampler(ps, sep, p_rot_per_sample=1.0, p_scale_per_sample=1.0,
                               intensity=IntensityAugment(noise_rng="philox", **overrides))
    ds.add_subject(img, lab, unc)
    for seed in range(8):
        random.seed(seed)
        np.random.seed(seed)
        got = ds.sample(0)
        st_e = (np.random.get_state(), random.getstate())
        random.seed(seed)
        np.random.seed(seed)
        tr = op.training_transform((ps[2], ps[1], ps[0]), rng=np.random, rng_py=random, p_rot_per_sample=1.0, p_scale_per_sample=1.0,
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
    ds = augment.Stage2Sampler((32, 24, 3), 4, intensity=IntensityAugment(noise_rng="philox", **FORCED))
    ds.add_subject(img, lab, unc)
    random.seed(5)
    np.random.seed(5)
    got = ds.batch([0, 0, 0, 0])
    random.seed(5)
    np.random.seed(5)
    rows = [ds.sample(0) for _ in range(4)]
    for k in range(4):
        assert torch.equal(got[k], torch.stack([r[k] for r in rows])), k


def _launches(b, noise_rng):
    from rehrseg_b200 import functional as F_
    aug = IntensityAugment(noise_rng=noise_rng, **FORCED)
    x = torch.randn(b, 1, 4, 32, 24, device="cuda")
    plan = aug.draw(b, 1, x.shape[2:], random.Random(0), np.random.RandomState(0))
    l0 = F_.launches()
    aug.apply(x, plan)
    return F_.launches() - l0, plan


@pytest.mark.parametrize("b", [1, 8])
def test_launch_count_is_the_numpy_modes(b):
    n_philox, p = _launches(b, "philox")
    n_numpy, _ = _launches(b, "numpy")
    assert p.fired() == list(NAMES)
    assert n_philox == n_numpy == 1 + 3 + 1 + 2 + 5 + 3 + 3


def test_generated_field_is_standard_normal():
    """One [8,1,16,256,256] batch of zeros with the noise forced: x = field exactly.  Fixed seeds, so the check is deterministic."""
    from scipy import stats
    b, shape = 8, (16, 256, 256)
    aug = IntensityAugment(noise_rng="philox", **NOISE_ONLY)
    plan = aug.draw(b, 1, shape, random.Random(11), np.random.RandomState(11))
    x = torch.zeros(b, 1, *shape, device="cuda")
    aug.apply(x, plan)
    f = x.reshape(b, -1).double().cpu().numpy()
    N = f.shape[1]
    vh = np.array([r[2] for r in plan.rows["noise"]])
    assert len(vh) == b and (vh > 1e-3).all(), vh
    z = f / vh[:, None]
    bound = 5.0 / np.sqrt(N)
    for r in range(b):
        assert abs(z[r].mean()) < bound, (r, z[r].mean())
        assert abs(z[r].std() - 1.0) < 5.0 / np.sqrt(2 * N), (r, z[r].std())
        p = stats.kstest(z[r], "norm").pvalue
        assert p > 1e-4, (r, p)
        assert abs(np.corrcoef(z[r, :-1], z[r, 1:])[0, 1]) < bound, r
    cross = np.corrcoef(z)[np.triu_indices(b, 1)]
    assert np.abs(cross).max() < bound, cross
    assert len({tuple(k) for k in plan.noise_keys.tolist()}) == b


def test_numpy_mode_is_the_default():
    data = np.random.RandomState(4).randn(3, 2, 5, 33, 31).astype(np.float32)
    outs = []
    for kw in ({}, {"noise_rng": "numpy"}):
        rn, rp = np.random.RandomState(2), random.Random(2)
        aug = IntensityAugment(**kw, **NOISE_ONLY)
        x = torch.from_numpy(data).cuda()
        plan = aug.draw(*x.shape[:2], x.shape[2:], rp, rn)
        assert plan.noise_rng == "numpy" and len(plan.noise) == 6 and plan.noise_keys.shape == (0, 2)
        aug.apply(x, plan)
        outs.append(x.cpu())
    assert torch.equal(outs[0], outs[1])
    want = oi.intensity_transform(data.copy(), np.random.RandomState(2), random.Random(2), **NOISE_ONLY)
    assert _err(outs[0], want) <= 1e-5
