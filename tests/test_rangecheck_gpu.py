"""The opt-in fp16 saturation check (rehrseg_b200.rangecheck) on the B200: clean inputs report nothing and change no result,
unnormalised inputs flag exactly the stem's pre-norm output with the count an fp32 conv gives, one scaled layer flags its own
slot first on every store route, graph replays report themselves only, and with no check in scope the launches are those of an
unchecked run."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as TF

from oracle import seg_model as ref_seg
from rehrseg_b200 import _lib, functional as F_, seg_model as sm
from rehrseg_b200.graphs import GraphedForward, GraphedTrainStep
from rehrseg_b200.rangecheck import RangeCheck

pytestmark = pytest.mark.gpu

THRESH = 65520.0
SCALE = 1e5      # an input that was not z-scored: the stem's outputs reach ~6e4 (std) at the default init


def _near(ref):
    """Reference values too close to the threshold to decide: within 1e-3 relative.  The 1-channel stem computes in
    split bf16 pairs (about 16 mantissa bits), so its sums may differ from the float64 ones in the fifth digit."""
    return int(((ref - THRESH).abs() <= THRESH * 1e-3).sum())


def _model(plan="tiny", input_channels=1, seed=0):
    torch.manual_seed(seed)
    kw = ref_seg.plan_kwargs(plan)
    kw["input_channels"] = input_channels
    return sm.SegModel(**kw).cuda()


def _x(shape, seed=1, scale=1.0):
    return (torch.randn(shape, generator=torch.Generator().manual_seed(seed)) * scale).cuda()


def _loss(out, tgt):
    lo, hr = out
    return (lo.float() * tgt).mean() + hr.float().square().mean()


def _fwd_bwd(model, x, tgt):
    for p in model.parameters():
        p.grad = None
    out = model(x)
    _loss(out, tgt).backward()
    torch.cuda.synchronize()
    return [out[0].detach().clone(), out[1].detach().clone()] + [p.grad.clone() for p in model.parameters() if p.grad is not None]


def _same(on, off, off2, exact):
    """The first `exact` tensors (the forward's results) are bit-identical with the check on and off.  The gradients are not
    bit-reproducible from one unchecked run to the next (split-K and weight-gradient reductions finish in arrival order), so
    they are held to a few times that run-to-run spread, floored at a few fp32 ulps of their scale."""
    assert len(on) == len(off) == len(off2)
    for i, (a, b, c) in enumerate(zip(on, off, off2)):
        if i < exact:
            assert torch.equal(b, c) and torch.equal(a, b), i
        else:
            noise = max(float((c - b).abs().max()), 2.0 ** -20 * float(b.abs().max()))
            assert float((a - b).abs().max()) <= 4 * noise, i


def _first(rec):
    return (rec[0].name, rec[0].kind) if rec else None


@pytest.mark.parametrize("plan,shape", [("tiny", (2, 1, 16, 32, 32)), ("3d_fullres", (2, 1, 64, 64, 64))])
def test_clean_input_reports_nothing_and_changes_no_bit(plan, shape):
    model = _model(plan)
    x = _x(shape)
    tgt = _x((shape[0], 2) + shape[2:], seed=2)
    off = _fwd_bwd(model, x, tgt)
    with RangeCheck(model) as rc:
        on = _fwd_bwd(model, x, tgt)
    assert rc.report() == []
    assert len(rc.labels) > 0 and ("sr_head", "sr_up") in rc.labels
    off2 = _fwd_bwd(model, x, tgt)
    _same(on, off, off2, exact=2)


def test_clean_c1_graphed_train_step_bit_identical():
    """The benchmarked C1 shape (2 x 1 x 128^3, PlainConvUNet 3d_fullres) through GraphedTrainStep, check off and on."""
    torch.manual_seed(0)
    model = sm.plainconv_unet_3d_fullres().cuda()
    x = _x((2, 1, 128, 128, 128))
    tgt = _x((2, 2, 128, 128, 128), seed=2)

    def loss_fn(out, t):
        return (out.float() * t).mean()

    def run(step):
        loss = step(x, tgt).clone()
        torch.cuda.synchronize()
        return [loss] + [g.clone() for g in step.grads if g is not None]

    plain = GraphedTrainStep(model, loss_fn, (x, tgt))
    checked = GraphedTrainStep(model, loss_fn, (x, tgt), range_check=True)
    assert checked.engine_launches == plain.engine_launches
    off = run(plain)
    on = run(checked)
    assert checked.range_report() == []
    off2 = run(plain)
    _same(on, off, off2, exact=1)


def test_unnormalised_input_flags_exactly_the_stem_with_the_fp32_count():
    model = _model("3d_fullres")
    x = _x((2, 1, 64, 64, 64), scale=SCALE)
    with torch.no_grad(), RangeCheck(model) as rc:
        model(x)
    rec = rc.report()
    stem = "encoder.stages.0.0.convs.0"
    assert [(r.name, r.kind) for r in rec] == [(stem, "y")], rec
    w = model.encoder.stages[0][0].convs[0].conv.weight.detach()
    ref = TF.conv3d(x.double(), w.double(), None, padding=1).abs()    # the engine adds no bias in front of InstanceNorm
    want = int((ref >= THRESH).sum())
    near = _near(ref)
    assert want > 1000 and abs(rec[0].count - want) <= near, (rec[0].count, want, near)
    assert rec[0].max_abs == pytest.approx(float(ref.max()), rel=1e-3)


def _scaled_first_flag(model, x, param, factor, want):
    with torch.no_grad():
        param.mul_(factor)
    try:
        with torch.no_grad(), RangeCheck(model) as rc:
            model(x)
        rec = rc.report()
    finally:
        with torch.no_grad():
            param.div_(factor)
    assert rec and _first(rec) == want, rec      # records come in slot (forward) order: no earlier slot saturated
    return rec


@pytest.mark.parametrize("route", ["march", "tapped_s2", "tapped_256", "tconv_scatter", "in_apply", "sr_feed"])
def test_one_scaled_layer_is_flagged_first(route):
    model = _model("3d_fullres")
    model.eval()
    x = _x((1, 1, 64, 64, 64))
    enc, dec = model.encoder.stages, model.decoder
    if route == "march":          # 32 -> 32, k3 s1: the marching kernel
        blk = enc[0][0].convs[1]
        _scaled_first_flag(model, x, blk.conv.weight, 1e6, ("encoder.stages.0.0.convs.1", "y"))
    elif route == "tapped_s2":    # 32 -> 64, stride-2 stage entry: the tapped GEMM
        blk = enc[1][0].convs[0]
        _scaled_first_flag(model, x, blk.conv.weight, 1e6, ("encoder.stages.1.0.convs.0", "y"))
    elif route == "tapped_256":   # 256 -> 256: the tapped GEMM with 256 input channels
        blk = enc[3][0].convs[1]
        _scaled_first_flag(model, x, blk.conv.weight, 1e6, ("encoder.stages.3.0.convs.1", "y"))
    elif route == "tconv_scatter":  # transposed conv scattered into the [up | skip] buffer
        _scaled_first_flag(model, x, dec.transpconvs[2].weight, 1e6, ("decoder.transpconvs.2", "up"))
    elif route == "in_apply":     # a large gamma saturates the normalised output, not the conv output before it
        blk = enc[2][0].convs[0]
        _scaled_first_flag(model, x, blk.norm.weight, 1e6, ("encoder.stages.2.0.convs.0", "a"))
    else:                         # the activation the sr_head up-sampling reads: flagged where it is stored in fp16
        blk = dec.stages[-1].convs[-1]
        name = f"decoder.stages.{len(dec.stages) - 1}.convs.{len(dec.stages[-1].convs) - 1}"
        rec = _scaled_first_flag(model, x, blk.norm.weight, 1e6, (name, "a"))
        assert ("sr_head", "sr_up") not in [(r.name, r.kind) for r in rec]     # the up-sampled copy is bf16


def test_small_cin_stem_is_flagged():
    model = _model("tiny", input_channels=2)
    x = _x((2, 2, 16, 32, 32), scale=SCALE)
    with torch.no_grad(), RangeCheck(model) as rc:
        model(x)
    rec = rc.report()
    assert [(r.name, r.kind) for r in rec] == [("encoder.stages.0.0.convs.0", "y")], rec
    w = model.encoder.stages[0][0].convs[0].conv.weight.detach()
    ref = TF.conv3d(x.double(), w.double(), None, padding=1).abs()
    want = int((ref >= THRESH).sum())
    assert want > 100 and abs(rec[0].count - want) <= _near(ref), (rec[0].count, want)


def test_upsample_and_convert16_kernels_count_their_fp16_stores():
    """The two elementwise fp16 store sites reached directly through the C ABI (the SegModel's up-sampled sr_head input is bf16):
    bf16 values of 1e5 stored as fp16 saturate, all of them; the stored bits are those of an unchecked call."""
    L = _lib.lib()
    slots = torch.zeros((2, 2), dtype=torch.int64, device="cuda")
    x = torch.full((1, 4, 3, 5, 16), 1e5, dtype=torch.bfloat16, device="cuda")
    x[..., :8] = 1.0
    y_off = torch.empty((1, 8, 3, 5, 16), dtype=torch.bfloat16, device="cuda")
    y_on = torch.empty_like(y_off)
    c_off, c_on = torch.empty_like(x), torch.empty_like(x)
    xt = _lib.rt(x)
    _lib.check(L.rehr_upsample_linear_d(C.byref(xt), C.byref(_lib.rt(y_off, True)), _lib.stream_ptr()))
    _lib.check(L.rehr_convert16(C.byref(xt), C.byref(_lib.rt(c_off, True)), _lib.stream_ptr()))
    _lib.check(L.rehr_range_sink(_lib.ptr(slots), 0))
    try:
        _lib.check(L.rehr_upsample_linear_d(C.byref(xt), C.byref(_lib.rt(y_on, True)), _lib.stream_ptr()))
        _lib.check(L.rehr_range_sink(_lib.ptr(slots), 1))
        _lib.check(L.rehr_convert16(C.byref(xt), C.byref(_lib.rt(c_on, True)), _lib.stream_ptr()))
    finally:
        L.rehr_range_sink(None, 0)
    h = slots.cpu()
    assert int(h[0, 0]) == y_on.numel() // 2 and int(h[1, 0]) == x.numel() // 2
    big = float(x.float().max())
    max_abs = torch.tensor([int(h[0, 1]), int(h[1, 1])], dtype=torch.int32).view(torch.float32)
    assert float(max_abs[0]) == pytest.approx(big, rel=1e-6) and float(max_abs[1]) == big
    assert torch.equal(y_on, y_off) and torch.equal(c_on, c_off)


def test_graph_replays_report_themselves_only():
    model = _model("tiny")
    clean = _x((2, 1, 16, 32, 32))
    hot = clean * SCALE
    tgt = _x((2, 2, 16, 32, 32), seed=2)
    with RangeCheck(model) as rc:
        _fwd_bwd(model, hot, tgt)
    eager = rc.report()
    assert eager and _first(eager) == ("encoder.stages.0.0.convs.0", "y")

    step = GraphedTrainStep(model, _loss, (clean, tgt), range_check=True)
    step(hot, tgt)
    assert step.range_report() == eager
    step(clean, tgt)
    assert step.range_report() == []

    model.eval()
    with torch.no_grad(), RangeCheck(model) as rc:
        model(hot)
    eager_fwd = rc.report()
    g = GraphedForward(model, clean, range_check=True)
    g(hot)
    assert g.range_report() == eager_fwd == eager
    g(clean)
    assert g.range_report() == []


def test_check_off_launches_as_unchecked():
    model = _model("tiny")
    x = _x((2, 1, 16, 32, 32))
    tgt = _x((2, 2, 16, 32, 32), seed=2)
    with torch.no_grad():
        model(x)                                  # packs and kernel attributes outside the counted runs
    l0 = F_.launches()
    with torch.no_grad():
        model(x)
    plain = F_.launches() - l0
    with RangeCheck(model):
        pass
    l0 = F_.launches()
    with torch.no_grad():
        model(x)
    assert F_.launches() - l0 == plain
    l0 = F_.launches()
    with torch.no_grad(), RangeCheck(model):
        model(x)
    assert F_.launches() - l0 == plain           # the check adds no engine launch, only arguments
    a = GraphedTrainStep(model, _loss, (x, tgt))
    b = GraphedTrainStep(model, _loss, (x, tgt), range_check=True)
    c = GraphedTrainStep(model, _loss, (x, tgt))
    assert a.engine_launches == b.engine_launches == c.engine_launches
    assert a.range is None and c.range is None
