"""GPU: the SR-stage training iteration (train_sr, train_all.py:118-139) replayed from one CUDA graph (train_step.GraphedSRStep),
with the plain loss statements and with the fused loss (loss_ops.FusedSRLoss): against the oracle's fp32 CPU step, against the
Python-launched sr_train_step over consecutive batches, fused against plain, and what each leaves of the caller's batch."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _flavr(unc, seed):
    from rehrseg_b200 import flavr
    torch.manual_seed(seed)
    return flavr.UNet_3D_3D(2, "unet_18", 4, 4, False, "concat", "transpose", use_uncertainty=unc).cuda().train()


def _batch(seed):
    g = torch.Generator().manual_seed(seed)
    lr = torch.rand((2, 2, 4, 64, 64), generator=g)
    lr[:, 1] = (lr[:, 1] > 0.8).float()
    hr = torch.rand((2, 2, 16, 64, 64), generator=g)
    hr[:, 1] = (hr[:, 1] > 0.8).float()
    return lr, hr


def _losses(unc, fused):
    from rehrseg_b200 import loss_ops, train_step as ts
    if fused:
        return {"fused_loss": loss_ops.FusedSRLoss(1.0, 1.0, enable_uncertainty=unc)}
    return {"loss_obj": torch.nn.L1Loss(), "loss_seg": ts.BCEDiceLoss(1, 1)}


def _graphed(model, batch, unc, fused):
    from rehrseg_b200 import train_step as ts
    return ts.GraphedSRStep(model, tuple(t.clone().cuda() for t in batch), slice_separation=4, num_slices=4, enable_uncertainty=unc,
                            **_losses(unc, fused))


def _grads(model):
    return [None if p.grad is None else p.grad.clone() for p in model.parameters()]


@pytest.mark.parametrize("unc", [False, True])
def test_graphed_fused_sr_step_vs_oracle(unc):
    """Same weights, batch and bounds as test_flavr_gpu.py::test_sr_train_step_on_the_engine_vs_oracle."""
    from oracle import flavr as of, joint as oj
    from rehrseg_b200 import flavr
    ref = of.build(unc, seed=9).train()
    torch.manual_seed(9)
    mine = flavr.UNet_3D_3D(2, "unet_18", 4, 4, False, "concat", "transpose", use_uncertainty=unc)
    assert all(torch.equal(a, b) for a, b in zip(ref.state_dict().values(), mine.state_dict().values()))
    mine = mine.cuda().train()
    g = torch.Generator().manual_seed(13)
    lr = torch.rand((2, 2, 4, 64, 64), generator=g)
    lr[:, 1] = (lr[:, 1] > 0.8).float()
    hr = torch.rand((2, 2, 16, 64, 64), generator=g)
    hr[:, 1] = (hr[:, 1] > 0.8).float()
    want = float(oj.ref_sr_step(ref, lr.clone(), hr.clone(), torch.nn.L1Loss(), oj.RefBCEDiceLoss(1, 1), 4, 4, unc))
    step = _graphed(mine, (lr, hr), unc, fused=True)
    got = float(step((lr.clone().cuda(), hr.clone().cuda()))["loss"])
    torch.cuda.synchronize()
    assert abs(got - want) <= 1e-2 * abs(want), (got, want)
    pr = dict(ref.named_parameters())
    num = den = 0.0
    for name, p in mine.named_parameters():
        assert (p.grad is None) == (pr[name].grad is None), name
        if p.grad is None:
            continue
        a, b = p.grad.double().cpu(), pr[name].grad.double()
        num += float((a - b).pow(2).sum()); den += float(b.pow(2).sum())
    print("graphed fused sr step", "uasr" if unc else "plain", "loss", got, want, "grads global", (num / den) ** 0.5)
    assert (num / den) ** 0.5 <= 8e-2
    step.close()


@pytest.mark.parametrize("fused", [False, True])
@pytest.mark.parametrize("unc", [False, True])
def test_graphed_sr_step_matches_the_python_launched_one(unc, fused):
    """Three different batches replayed in a row each match a fresh eager sr_train_step with the same loss objects: the static
    input is re-loaded before every replay, so the in-place mean subtraction of the forward never accumulates."""
    from rehrseg_b200 import train_step as ts
    model = _flavr(unc, seed=17)
    batches = [_batch(s) for s in (1, 2, 3)]
    losses = _losses(unc, fused)
    want = []
    for lr, hr in batches:
        out = ts.sr_train_step(model, (lr.clone().cuda(), hr.clone().cuda()), losses.get("loss_obj"), losses.get("loss_seg"), None, None,
                               4, 4, unc, fused_loss=losses.get("fused_loss"))
        torch.cuda.synchronize()
        want.append((float(out["loss"]), _grads(model)))
    assert len({w[0] for w in want}) == 3
    step = ts.GraphedSRStep(model, tuple(t.clone().cuda() for t in batches[0]), slice_separation=4, num_slices=4,
                            enable_uncertainty=unc, **losses)
    for (lr, hr), (loss, grads) in zip(batches, want):
        got = float(step((lr.clone().cuda(), hr.clone().cuda()))["loss"])
        torch.cuda.synchronize()
        assert abs(got - loss) <= 1e-4 * max(1.0, abs(loss)), (got, loss)
        for p, g in zip(model.parameters(), grads):
            assert (p.grad is None) == (g is None)
            if g is not None:
                assert rel(p.grad, g) <= 2e-3, rel(p.grad, g)
    step.close()


@pytest.mark.parametrize("unc", [False, True])
def test_graphed_fused_sr_step_matches_graphed_plain(unc):
    plain_model, fused_model = _flavr(unc, seed=23), _flavr(unc, seed=23)
    batch = _batch(5)
    plain = _graphed(plain_model, batch, unc, fused=False)
    fused = _graphed(fused_model, batch, unc, fused=True)
    lp = float(plain((batch[0].clone().cuda(), batch[1].clone().cuda()))["loss"])
    lf = float(fused((batch[0].clone().cuda(), batch[1].clone().cuda()))["loss"])
    torch.cuda.synchronize()
    assert abs(lf - lp) <= 1e-5 * abs(lp), (lf, lp)
    # The two losses round differently in the last fp32 bit; the bf16 backward turns that into element noise of ~1e-3 that grows
    # through the layers; some tensors of the UASR network have gradients of ~1e-10: the whole gradient is held to 2e-3, each tensor to 1e-2.
    num = den = 0.0
    for (name, a), b in zip(fused_model.named_parameters(), plain_model.parameters()):
        assert (a.grad is None) == (b.grad is None)
        if b.grad is not None:
            assert rel(a.grad, b.grad) <= 1e-2, (name, rel(a.grad, b.grad))
            num += float((a.grad.double() - b.grad.double()).pow(2).sum()); den += float(b.grad.double().pow(2).sum())
    assert (num / den) ** 0.5 <= 2e-3, (num / den) ** 0.5
    assert fused.step.engine_launches == plain.step.engine_launches + 2, (fused.step.engine_launches, plain.step.engine_launches)
    plain.close()
    fused.close()


@pytest.mark.parametrize("unc", [False, True])
def test_what_each_sr_step_leaves_of_the_callers_batch(unc):
    """GraphedSRStep subtracts the channel-0 mean from its static copy only; sr_train_step(..., fused_loss=...) still mutates the
    caller's device batch in place, as the reference does."""
    from rehrseg_b200 import loss_ops, train_step as ts
    model = _flavr(unc, seed=29)
    lr, hr = _batch(7)
    step = _graphed(model, (lr, hr), unc, fused=True)
    lr_dev, hr_dev = lr.clone().cuda(), hr.clone().cuda()
    step((lr_dev, hr_dev))
    torch.cuda.synchronize()
    assert torch.equal(lr_dev.cpu(), lr) and torch.equal(hr_dev.cpu(), hr)
    step.close()
    lr_dev = lr.clone().cuda()
    ts.sr_train_step(model, (lr_dev, hr.clone().cuda()), None, None, None, None, 4, 4, unc,
                     fused_loss=loss_ops.FusedSRLoss(1.0, 1.0, enable_uncertainty=unc))
    torch.cuda.synchronize()
    assert rel(lr_dev[:, 0], lr[:, 0] - lr[:, 0:1].mean((2, 3, 4), keepdim=True)[:, 0]) <= 1e-5
    assert torch.equal(lr_dev[:, 1].cpu(), lr[:, 1])
