"""GPU: the fused SR-stage loss (loss_ops.SRLossSums / FusedSRLoss, csrc/loss_ops.cu sr_loss_sums / sr_loss_bwd) against the loss
statements of train_step.sr_train_step (nn.L1Loss, the UASR terms, train_step.BCEDiceLoss) evaluated in float64: values,
gradients w.r.t. the prediction and the uncertainty, ties, saturated logits, a clamped Dice denominator, determinism, launches."""
import pytest
import torch

pytestmark = pytest.mark.gpu

SHAPES = [(1, 2, 4, 32, 32), (2, 2, 4, 64, 48), (3, 3, 1, 17, 29), (8, 2, 4, 256, 256)]


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _inputs(shape, unc, seed):
    """hat [B,C,S,H,W] (image channel in [0,1], logits), the HR batch [B,C,16,H,W] (binary label channels) and u."""
    b, c, s, h, w = shape
    g = torch.Generator(device="cuda").manual_seed(seed)
    hat = torch.randn(shape, generator=g, device="cuda") * 3
    hat[:, 0] = torch.rand((b, s, h, w), generator=g, device="cuda")
    hr = torch.rand((b, c, 16, h, w), generator=g, device="cuda")
    hr[:, 1:] = (hr[:, 1:] > 0.8).float()
    u = torch.rand((b, 1, s, h, w), generator=g, device="cuda") * 0.9 + 0.05 if unc else None
    return hat, hr, u


def _window(hr, s):
    """The target window sr_train_step reads with slice_separation = s, num_slices = 4: depth s .. 2s."""
    return hr[:, :, s:2 * s]


def _reference(hat, target, u, alpha=1.0, beta=1.0):
    """sr_train_step's loss statements in float64 (num_slices = 1: `target` is already the window)."""
    from rehrseg_b200 import train_step as ts
    h64 = hat.detach().double().requires_grad_(True)
    u64 = u.detach().double().requires_grad_(True) if u is not None else None
    out = (h64, u64) if u is not None else h64
    loss = ts._sr_loss(out, target.double(), torch.nn.L1Loss(), ts.BCEDiceLoss(alpha, beta), 4, 1, u is not None, None)
    loss.backward()
    return loss.detach(), h64.grad, (u64.grad if u is not None else None)


def _fused(hat, target, u, alpha=1.0, beta=1.0):
    from rehrseg_b200 import loss_ops
    h = hat.detach().clone().requires_grad_(True)
    uu = u.detach().clone().requires_grad_(True) if u is not None else None
    loss = loss_ops.FusedSRLoss(alpha, beta, enable_uncertainty=u is not None)(h, target, uu)
    loss.backward()
    torch.cuda.synchronize()
    return loss.detach(), h.grad, (uu.grad if u is not None else None)


def _check(hat, target, u, alpha=1.0, beta=1.0, tol=1e-5):
    lf, gh, gu = _fused(hat, target, u, alpha, beta)
    lr_, rh, ru = _reference(hat, target, u, alpha, beta)
    assert abs(float(lf) - float(lr_)) <= tol * abs(float(lr_)), (float(lf), float(lr_))
    assert rel(gh, rh) <= tol, rel(gh, rh)
    if u is not None:
        assert rel(gu, ru) <= tol, rel(gu, ru)
    return lf, gh, gu


@pytest.mark.parametrize("unc", [False, True])
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("windowed", [True, False])
def test_sr_loss_matches_float64_statements(shape, unc, windowed):
    hat, hr, u = _inputs(shape, unc, seed=sum(shape) + unc)
    target = _window(hr, shape[2]) if windowed else _window(hr, shape[2]).contiguous()
    assert target.is_contiguous() != windowed
    _check(hat, target, u, alpha=0.7, beta=1.3)


@pytest.mark.parametrize("unc", [False, True])
def test_sr_loss_ties_follow_torch_sign(unc):
    """hat_0 == t_0 at chosen voxels and u == |e| at others (dyadic values: the float32 and float64 differences are exact)."""
    shape = (2, 2, 4, 32, 40)
    hat, hr, u = _inputs(shape, unc, seed=21)
    g = torch.Generator(device="cuda").manual_seed(22)
    target = _window(hr, 4)
    t0 = torch.randint(0, 64, target[:, 0].shape, generator=g, device="cuda").float() / 64
    target[:, 0] = t0
    h0 = torch.randint(0, 64, t0.shape, generator=g, device="cuda").float() / 64
    tie = torch.rand(t0.shape, generator=g, device="cuda") < 0.2
    h0 = torch.where(tie, t0, h0)
    hat[:, 0] = h0
    assert int(tie.sum()) > 100 and int((h0 == t0).sum()) >= int(tie.sum())
    if unc:
        ae = (h0 - t0).abs()
        u_tie = (torch.rand(t0.shape, generator=g, device="cuda") < 0.3) & (ae > 0)
        u[:, 0] = torch.where(u_tie, ae, u[:, 0])
        assert int(u_tie.sum()) > 100
    _check(hat, target, u)


@pytest.mark.parametrize("unc", [False, True])
def test_sr_loss_saturated_logits(unc):
    hat, hr, u = _inputs((2, 2, 4, 32, 32), unc, seed=31)
    sign = (torch.rand(hat[:, 1:].shape, generator=torch.Generator(device="cuda").manual_seed(32), device="cuda") > 0.5).float()
    hat[:, 1:] = 60 * (2 * sign - 1)
    _check(hat, _window(hr, 4), u)


def test_sr_loss_tiny_uncertainty():
    hat, hr, u = _inputs((2, 2, 4, 32, 32), True, seed=41)
    u.fill_(1e-6)
    _check(hat, _window(hr, 4), u)


@pytest.mark.parametrize("unc", [False, True])
def test_sr_loss_clamped_dice_denominator(unc):
    """An all-zero label channel under logits of -30: sum p^2 + sum y^2 < 1e-6, so the Dice denominator is clamped and passes no
    gradient (clamp's backward)."""
    hat, hr, u = _inputs((2, 3, 4, 32, 32), unc, seed=51)
    target = _window(hr, 4)
    target[:, 1] = 0
    hat[:, 1] = -30
    p = torch.sigmoid(hat[:, 1].double())
    assert float((p * p).sum()) < 1e-6
    _check(hat, target, u)


@pytest.mark.parametrize("unc", [False, True])
def test_sr_loss_is_deterministic_and_one_launch_per_direction(unc):
    from rehrseg_b200 import functional as F_, loss_ops
    hat, hr, u = _inputs((8, 2, 4, 256, 256), unc, seed=61)
    target = _window(hr, 4)
    runs = []
    for _ in range(2):
        h = hat.clone().requires_grad_(True)
        uu = u.clone().requires_grad_(True) if unc else None
        l0 = F_.launches()
        loss = loss_ops.FusedSRLoss(1.0, 1.0, enable_uncertainty=unc)(h, target, uu)
        assert F_.launches() - l0 == 1
        loss.backward()
        assert F_.launches() - l0 == 2
        torch.cuda.synchronize()
        runs.append((loss.detach(), h.grad, uu.grad if unc else None))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    if unc:
        assert torch.equal(runs[0][2], runs[1][2])


def test_sr_loss_refusals():
    from rehrseg_b200 import loss_ops
    from rehrseg_b200._lib import RehrError
    hat, hr, u = _inputs((2, 2, 4, 32, 32), True, seed=71)
    target = _window(hr, 4)
    with pytest.raises(RehrError):
        loss_ops.SRLossSums.apply(hat.cpu(), target.cpu(), u.cpu())
    with pytest.raises(RehrError):
        loss_ops.SRLossSums.apply(hat, target.cpu(), u)
    with pytest.raises(RehrError):
        loss_ops.SRLossSums.apply(hat, hr[:, :, 4:9], u)                    # shape mismatch
    with pytest.raises(RehrError):
        loss_ops.SRLossSums.apply(hat, target, u[:, :, :3])
    with pytest.raises(RehrError):
        loss_ops.SRLossSums.apply(hat, target.transpose(3, 4), u)          # planes not contiguous (H == W keeps the shape)
    with pytest.raises(RehrError):
        loss_ops.FusedSRLoss(enable_uncertainty=False)(hat, target, u)      # head and module disagree
