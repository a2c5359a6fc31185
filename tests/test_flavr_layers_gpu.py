"""GPU: every engine layer call of the FLAVR SR network (`UNet_3D_3D`, both heads) at the shapes the benchmarked C2 step
([8, 2, 4, 256, 256]) and `train_sr` ([32, 2, 4, 96, 96]) run, each against a float64 reference of the same operation.

* `LAYERS_C2` / `LAYERS_TRAIN` list one row per distinct engine call of the forward.  `test_layer_table_is_what_the_network_runs`
  records the calls of a real forward + backward and checks the table against them, so a FLAVR change that adds or reshapes a
  layer fails there instead of leaving the table behind.
* The same recording notes, per call, the conv kernel families its forward and backward launch (under `kernel_timer`), the
  engine launches, the side-stream forks of the weight gradient and the channel pitch of the cotangent it receives.
  `kernel_timer` turns the side-stream weight gradient off, so the families come from a second, timed pass and the numerics
  below never run under it.
* `test_layer_vs_float64` runs each row alone with random operands and checks every output and gradient tensor against a
  float64 reference, and that the isolated call takes the route the row took inside the network.

Reference arithmetic.  Operands are rounded to bf16 wherever the engine stores bf16, so the reference sees the values the
engine computed with.  Reductions (SE pool and gate gradient, attention dW / db, bias sums, the uncertainty-layer sums of the
mixture) are float64.  Convolutions run in fp32 with TF32 off (float64 convolutions at these sizes, up to 0.6 TFLOP per
layer, are too slow): an fp32 dot product of length K has a relative error of about sqrt(K) * 2^-24 <= 1e-5 for K <= 13824,
far below one bf16 ulp (2^-8) and 10x below the 1e-4 bound of the fp32 outputs.  Activation masks of the reference backward
come from the engine's own stored forward output (the engine evaluates act' from it), so a sign flip at |z| ~ 0 between the
engine's and the reference's forward is not counted as a backward error.

Bounds, per tensor:
* bf16 outputs and input gradients: rel-L2 <= 4e-3 and every element within 3 bf16 ulps of max|ref| (test_conv_gpu's rules);
* fp32 outputs: rel-L2 <= 1e-4;
* weight and bias gradients (conv, attention layer, uncertainty layer): rel-L2 <= 1e-3, fp32 sums of exact bf16 products.
"""
import collections
import inspect
import math
import zlib

import pytest
import torch
import torch.nn.functional as F

from test_conv_gpu import TOL, bf16r, max_abs_ok, rel_l2

pytestmark = pytest.mark.gpu

SHAPES = {"C2": (8, 2, 4, 256, 256), "TRAIN": (32, 2, 4, 96, 96), "SMALL": (2, 2, 4, 64, 64)}   # SMALL: the whole-network tests' size
FAMILIES = ("conv_march_kernel", "conv_tapped_gemm_kernel", "wgrad_march_kernel", "conv_wgrad_kernel")
ACTS = {0: "none", 1: "relu", 2: "lrelu"}
ACT_IDS = {v: k for k, v in ACTS.items()}

Row = collections.namedtuple("Row", "fn x w k s p act slope want_pool out_f32 residual pool bias",
                             defaults=(None, None, None, "none", 0.0, False, False, False, False, True))
Row.__doc__ = """One engine call: `x` = input shape (channels-last [N, D, H, W, C]; NCDHW for smallcin_conv_act; the fp32
feature_fuse1 output [B, 1, H, W, 32 n_out] for uasr_mixture), `w` = weight shape (uncertainty_out's for uasr_mixture),
`residual` / `pool` / `bias` = whether a residual / a precomputed SE pool / a conv bias is passed."""

K3, S1, P1 = (3, 3, 3), (1, 1, 1), (1, 1, 1)
K1, P0 = (1, 1, 1), (0, 0, 0)
KUP, SUP = (3, 4, 4), (1, 2, 2)
K2D, P2D = (1, 3, 3), (0, 1, 1)


LAYERS_C2 = [
    # encoder: stem, layer1 (64), layer2 (128, s(1,2,2)), layer3 (256, s(1,2,2)), layer4 (512)
    Row("smallcin_conv_act", (8, 2, 4, 256, 256), (64, 2, 3, 7, 7), (3, 7, 7), (1, 2, 2), (1, 3, 3), "relu"),
    Row("conv_act", (8, 4, 128, 128, 64), (64, 64, 3, 3, 3), K3, S1, P1, "relu"),
    Row("conv_act", (8, 4, 128, 128, 64), (64, 64, 3, 3, 3), K3, S1, P1, want_pool=True),
    Row("se_gate", (8, 4, 128, 128, 64), (64, 64, 1, 1, 1), act="relu", residual=True, pool=True),
    Row("conv_act", (8, 4, 128, 128, 64), (128, 64, 3, 3, 3), K3, SUP, P1, "relu"),
    Row("conv_act", (8, 4, 64, 64, 128), (128, 128, 3, 3, 3), K3, S1, P1, want_pool=True),
    Row("conv_act", (8, 4, 128, 128, 64), (128, 64, 1, 1, 1), K1, SUP, P0, bias=False),
    Row("se_gate", (8, 4, 64, 64, 128), (128, 128, 1, 1, 1), act="relu", residual=True, pool=True),
    Row("conv_act", (8, 4, 64, 64, 128), (128, 128, 3, 3, 3), K3, S1, P1, "relu"),
    Row("conv_act", (8, 4, 64, 64, 128), (256, 128, 3, 3, 3), K3, SUP, P1, "relu"),
    Row("conv_act", (8, 4, 32, 32, 256), (256, 256, 3, 3, 3), K3, S1, P1, want_pool=True),
    Row("conv_act", (8, 4, 64, 64, 128), (256, 128, 1, 1, 1), K1, SUP, P0, bias=False),
    Row("se_gate", (8, 4, 32, 32, 256), (256, 256, 1, 1, 1), act="relu", residual=True, pool=True),
    Row("conv_act", (8, 4, 32, 32, 256), (256, 256, 3, 3, 3), K3, S1, P1, "relu"),
    Row("conv_act", (8, 4, 32, 32, 256), (512, 256, 3, 3, 3), K3, S1, P1, "relu"),
    Row("conv_act", (8, 4, 32, 32, 512), (512, 512, 3, 3, 3), K3, S1, P1, want_pool=True),
    Row("conv_act", (8, 4, 32, 32, 256), (512, 256, 1, 1, 1), K1, S1, P0, bias=False),
    Row("se_gate", (8, 4, 32, 32, 512), (512, 512, 1, 1, 1), act="relu", residual=True, pool=True),
    Row("conv_act", (8, 4, 32, 32, 512), (512, 512, 3, 3, 3), K3, S1, P1, "relu"),
    # decoder: Conv_3d 512->256, upConv3D 512->128, 256->64, Conv_3d 128->64, upConv3D 128->64 (each + SE + LeakyReLU 0.2)
    Row("conv_act", (8, 4, 32, 32, 512), (256, 512, 3, 3, 3), K3, S1, P1, want_pool=True),
    Row("se_gate", (8, 4, 32, 32, 256), (256, 256, 1, 1, 1), act="lrelu", slope=0.2, pool=True),
    Row("conv_transpose", (8, 4, 32, 32, 512), (512, 128, 3, 4, 4), KUP, SUP, P1),
    Row("se_gate", (8, 4, 64, 64, 128), (128, 128, 1, 1, 1), act="lrelu", slope=0.2),
    Row("conv_transpose", (8, 4, 64, 64, 256), (256, 64, 3, 4, 4), KUP, SUP, P1),
    Row("se_gate", (8, 4, 128, 128, 64), (64, 64, 1, 1, 1), act="lrelu", slope=0.2),
    Row("conv_act", (8, 4, 128, 128, 128), (64, 128, 3, 3, 3), K3, S1, P1, want_pool=True),
    Row("se_gate", (8, 4, 128, 128, 64), (64, 64, 1, 1, 1), act="lrelu", slope=0.2, pool=True),
    Row("conv_transpose", (8, 4, 128, 128, 128), (128, 64, 3, 4, 4), KUP, SUP, P1),
    Row("se_gate", (8, 4, 256, 256, 64), (64, 64, 1, 1, 1), act="lrelu", slope=0.2),
    # plain head: feature_fuse 256->64 k(3,3) + LeakyReLU 0.2, outconv 64->8 k(7,7) on the reflection-padded map, fp32 out
    Row("conv_act", (8, 1, 256, 256, 256), (64, 256, 1, 3, 3), K2D, S1, P2D, "lrelu", 0.2),
    Row("conv_act", (8, 1, 262, 262, 64), (8, 64, 1, 7, 7), (1, 7, 7), S1, P0, out_f32=True),
    # UASR head: feature_fuse 256->256, feature_fuse1 256->128 and uncertainty_early 256->64 (1x1, fp32 out), the mixture
    Row("conv_act", (8, 1, 256, 256, 256), (256, 256, 1, 3, 3), K2D, S1, P2D, "lrelu", 0.2),
    Row("conv_act", (8, 1, 256, 256, 256), (128, 256, 1, 1, 1), K1, S1, P0, out_f32=True),
    Row("conv_act", (8, 1, 256, 256, 256), (64, 256, 1, 1, 1), K1, S1, P0, out_f32=True),
    Row("uasr_mixture", (8, 1, 256, 256, 128), (1, 16, 1, 1, 1)),
]

LAYERS_TRAIN = [
    Row("smallcin_conv_act", (32, 2, 4, 96, 96), (64, 2, 3, 7, 7), (3, 7, 7), (1, 2, 2), (1, 3, 3), "relu"),
    Row("conv_act", (32, 4, 48, 48, 64), (64, 64, 3, 3, 3), K3, S1, P1, "relu"),
    Row("conv_act", (32, 4, 48, 48, 64), (64, 64, 3, 3, 3), K3, S1, P1, want_pool=True),
    Row("se_gate", (32, 4, 48, 48, 64), (64, 64, 1, 1, 1), act="relu", residual=True, pool=True),
    Row("conv_act", (32, 4, 48, 48, 64), (128, 64, 3, 3, 3), K3, SUP, P1, "relu"),
    Row("conv_act", (32, 4, 24, 24, 128), (128, 128, 3, 3, 3), K3, S1, P1, want_pool=True),
    Row("conv_act", (32, 4, 48, 48, 64), (128, 64, 1, 1, 1), K1, SUP, P0, bias=False),
    Row("se_gate", (32, 4, 24, 24, 128), (128, 128, 1, 1, 1), act="relu", residual=True, pool=True),
    Row("conv_act", (32, 4, 24, 24, 128), (128, 128, 3, 3, 3), K3, S1, P1, "relu"),
    Row("conv_act", (32, 4, 24, 24, 128), (256, 128, 3, 3, 3), K3, SUP, P1, "relu"),
    Row("conv_act", (32, 4, 12, 12, 256), (256, 256, 3, 3, 3), K3, S1, P1, want_pool=True),
    Row("conv_act", (32, 4, 24, 24, 128), (256, 128, 1, 1, 1), K1, SUP, P0, bias=False),
    Row("se_gate", (32, 4, 12, 12, 256), (256, 256, 1, 1, 1), act="relu", residual=True, pool=True),
    Row("conv_act", (32, 4, 12, 12, 256), (256, 256, 3, 3, 3), K3, S1, P1, "relu"),
    Row("conv_act", (32, 4, 12, 12, 256), (512, 256, 3, 3, 3), K3, S1, P1, "relu"),
    Row("conv_act", (32, 4, 12, 12, 512), (512, 512, 3, 3, 3), K3, S1, P1, want_pool=True),
    Row("conv_act", (32, 4, 12, 12, 256), (512, 256, 1, 1, 1), K1, S1, P0, bias=False),
    Row("se_gate", (32, 4, 12, 12, 512), (512, 512, 1, 1, 1), act="relu", residual=True, pool=True),
    Row("conv_act", (32, 4, 12, 12, 512), (512, 512, 3, 3, 3), K3, S1, P1, "relu"),
    Row("conv_act", (32, 4, 12, 12, 512), (256, 512, 3, 3, 3), K3, S1, P1, want_pool=True),
    Row("se_gate", (32, 4, 12, 12, 256), (256, 256, 1, 1, 1), act="lrelu", slope=0.2, pool=True),
    Row("conv_transpose", (32, 4, 12, 12, 512), (512, 128, 3, 4, 4), KUP, SUP, P1),
    Row("se_gate", (32, 4, 24, 24, 128), (128, 128, 1, 1, 1), act="lrelu", slope=0.2),
    Row("conv_transpose", (32, 4, 24, 24, 256), (256, 64, 3, 4, 4), KUP, SUP, P1),
    Row("se_gate", (32, 4, 48, 48, 64), (64, 64, 1, 1, 1), act="lrelu", slope=0.2),
    Row("conv_act", (32, 4, 48, 48, 128), (64, 128, 3, 3, 3), K3, S1, P1, want_pool=True),
    Row("se_gate", (32, 4, 48, 48, 64), (64, 64, 1, 1, 1), act="lrelu", slope=0.2, pool=True),
    Row("conv_transpose", (32, 4, 48, 48, 128), (128, 64, 3, 4, 4), KUP, SUP, P1),
    Row("se_gate", (32, 4, 96, 96, 64), (64, 64, 1, 1, 1), act="lrelu", slope=0.2),
    Row("conv_act", (32, 1, 96, 96, 256), (64, 256, 1, 3, 3), K2D, S1, P2D, "lrelu", 0.2),
    Row("conv_act", (32, 1, 102, 102, 64), (8, 64, 1, 7, 7), (1, 7, 7), S1, P0, out_f32=True),
    Row("conv_act", (32, 1, 96, 96, 256), (256, 256, 1, 3, 3), K2D, S1, P2D, "lrelu", 0.2),
    Row("conv_act", (32, 1, 96, 96, 256), (128, 256, 1, 1, 1), K1, S1, P0, out_f32=True),
    Row("conv_act", (32, 1, 96, 96, 256), (64, 256, 1, 1, 1), K1, S1, P0, out_f32=True),
    Row("uasr_mixture", (32, 1, 96, 96, 128), (1, 16, 1, 1, 1)),
]

TABLES = {"C2": LAYERS_C2, "TRAIN": LAYERS_TRAIN}


@pytest.fixture(autouse=True)
def _fp32_reference():
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


# ----------------------------------------------------------------------------------------------------------------------
# recording the calls of the network
# ----------------------------------------------------------------------------------------------------------------------
def _t(v):
    return None if v is None else tuple(int(i) for i in v)


def row_of(fn: str, a: dict) -> Row:
    """The table row of one call, from its bound arguments (names as in rehrseg_b200.functional / flavr)."""
    if fn == "uasr_mixture":
        out, ue = a["out_cl"], a["ue_cl"]
        assert tuple(ue.shape) == (*out.shape[:4], out.shape[4] // 2)
        return Row(fn, _t(out.shape), _t(a["uncertainty_out"].weight.shape))
    if fn == "se_gate":
        return Row(fn, _t(a["x"].shape), _t(a["attn_w"].shape), act=ACTS[int(a["act"])], slope=float(a["slope"]),
                   residual=a["residual"] is not None, pool=a["pool"] is not None)
    common = dict(k=_t(a["kernel"]), s=_t(a["stride"]), p=_t(a["padding"]), act=ACTS[int(a["act"])], slope=float(a["slope"]),
                  bias=a["bias"] is not None)
    if fn == "conv_act":
        return Row(fn, _t(a["x"].shape), _t(a["weight"].shape), want_pool=bool(a["want_pool"]), out_f32=bool(a["out_f32"]), **common)
    return Row(fn, _t(a["x"].shape), _t(a["weight"].shape), **common)


class _Counters:
    """Engine launches, kernel_timer records and weight-gradient side-stream forks so far."""

    def __init__(self, Fn, monkeypatch):
        self.Fn, self.kt, self.forks = Fn, None, 0
        counters, real_fork = self, Fn._fork

        class CountingFork(real_fork):
            def __init__(self, *a, **k):
                counters.forks += 1
                super().__init__(*a, **k)

        monkeypatch.setattr(Fn, "_fork", CountingFork)

    def now(self):
        return (self.Fn.launches(), len(self.kt.records) if self.kt is not None else 0, self.forks)

    def families(self, a, b):
        return tuple(r[0] for r in self.kt.records[a:b] if r[0] in FAMILIES) if self.kt is not None else ()


def _record_pass(monkeypatch, model, x, timed):
    """One engine forward + backward of `model` on a copy of `x`; [(row, info)] in call order.  info: engine launches, side-stream
    forks and conv kernel families (timed pass only) of the call's forward and of its backward, and the channel pitch of the
    cotangent its backward receives (0: compact, or re-laid-out before use).  A call's backward is the stretch from the moment
    its output's gradient is complete (a tensor hook, which runs right before the call's autograd node) to the next such moment."""
    from rehrseg_b200 import flavr, functional as Fn
    calls, starts = [], []
    cnt = _Counters(Fn, monkeypatch)

    def wrap(mod, name):
        orig = getattr(mod, name)
        sig = inspect.signature(orig)

        def wrapper(*args, **kwargs):
            bound = sig.bind(*args, **kwargs)
            bound.apply_defaults()
            row = row_of(name, bound.arguments)
            c0 = cnt.now()
            out = orig(*args, **kwargs)
            c1 = cnt.now()
            idx = len(calls)
            calls.append((row, {"fwd": (c1[0] - c0[0], c1[2] - c0[2], cnt.families(c0[1], c1[1])), "gpitch": 0}))
            y = out[0] if isinstance(out, tuple) else out

            def hook(g, idx=idx):
                if g.dim() == 5 and g.stride(4) == 1 and g.stride(3) > g.shape[4] and not g.is_contiguous():
                    calls[idx][1]["gpitch"] = int(g.stride(3))
                starts.append((idx, cnt.now()))
            y.register_hook(hook)
            return out
        monkeypatch.setattr(mod, name, wrapper)

    for name in ("smallcin_conv_act", "conv_act", "se_gate", "conv_transpose"):
        wrap(Fn, name)
    wrap(flavr, "uasr_mixture")
    for p_ in model.parameters():
        p_.grad = None
    if timed:
        cnt.kt = Fn.kernel_timer().__enter__()
    try:
        outs = model(x.clone())
        outs = outs if isinstance(outs, tuple) else (outs,)
        loss = sum((o.float() * torch.randn(o.shape, device="cuda", generator=_gen(i))).mean() for i, o in enumerate(outs))
        loss.backward()
        torch.cuda.synchronize()
        end = cnt.now()
    finally:
        if timed:
            cnt.kt.__exit__(None, None, None)
        monkeypatch.undo()
    for j, (idx, c0) in enumerate(starts):
        c1 = starts[j + 1][1] if j + 1 < len(starts) else end
        calls[idx][1]["bwd"] = (c1[0] - c0[0], c1[2] - c0[2], cnt.families(c0[1], c1[1]))
    return calls


_recorded: dict = {}


def record_network(monkeypatch, shape_key, unc):
    """[(row, route)] in call order for one (shape, head): route = {launches: (fwd, bwd) of the timed pass (weights already
    packed), forks: (fwd, bwd) of the untimed pass, families: (fwd, bwd) of the timed pass, gpitch}."""
    key = (shape_key, unc)
    if key not in _recorded:
        from rehrseg_b200 import flavr
        torch.manual_seed(5)
        model = flavr.UNet_3D_3D(2, "unet_18", 4, 4, False, "concat", "transpose", use_uncertainty=unc).cuda().train()
        x = torch.rand(SHAPES[shape_key], device="cuda", generator=_gen(1))
        x[:, 1] = (x[:, 1] > 0.8).float()
        plain = _record_pass(monkeypatch, model, x, timed=False)
        timed = _record_pass(monkeypatch, model, x, timed=True)
        assert [r for r, _ in plain] == [r for r, _ in timed]
        _recorded[key] = [(row, {"launches": (b["fwd"][0], b["bwd"][0]), "forks": (a["fwd"][1], a["bwd"][1]),
                                 "families": (b["fwd"][2], b["bwd"][2]), "gpitch": a["gpitch"]})
                          for (row, a), (_, b) in zip(plain, timed)]
        del model, x
        torch.cuda.empty_cache()
    return _recorded[key]


def network_routes(monkeypatch, shape_key, unc) -> dict:
    """{row: route}; every repeat of a row inside the network must have taken the same route."""
    merged = {}
    for row, route in record_network(monkeypatch, shape_key, unc):
        assert merged.setdefault(row, route) == route, (row, merged[row], route)
    return merged


def _heads_of(row):
    """The heads whose forward makes this call: the 2-D layers (D = 1) and the mixture belong to one head."""
    if row.fn != "uasr_mixture" and row.x[1] != 1:
        return (False, True)
    return (False,) if row.w in ((64, 256, 1, 3, 3), (8, 64, 1, 7, 7)) else (True,)


@pytest.mark.parametrize("shape_key", ["C2", "TRAIN"])
@pytest.mark.parametrize("unc", [False, True], ids=["plain", "uasr"])
def test_layer_table_is_what_the_network_runs(monkeypatch, shape_key, unc):
    """The set of engine calls of one FLAVR forward equals the table rows of that head.  Also prints each call's route and
    the calls whose route differs from the same call at the 64 x 64, batch-2 size of the whole-network tests."""
    calls = record_network(monkeypatch, shape_key, unc)
    want = {r for r in TABLES[shape_key] if unc in _heads_of(r)}
    got = {r for r, _ in calls}
    assert got == want, {"missing from the table": sorted(got - want), "not run by the network": sorted(want - got)}
    routes = network_routes(monkeypatch, shape_key, unc)
    small = record_network(monkeypatch, "SMALL", unc)
    assert len(small) == len(calls)
    print(f"\n{shape_key} {'uasr' if unc else 'plain'}: {len(calls)} calls, {len(got)} distinct rows")
    for row in TABLES[shape_key]:
        if row in routes:
            i = routes[row]
            print(f"  {_row_id(row)}: launches {i['launches']} forks {i['forks']} gpitch {i['gpitch']} families {i['families']}")
    print("  differs from the 64x64 batch-2 route of the same call:")
    for (row, r), (srow, s) in zip(calls, small):
        if (r["launches"], r["forks"], r["families"], r["gpitch"] > 0) != (s["launches"], s["forks"], s["families"], s["gpitch"] > 0):
            print(f"    {_row_id(row)}: {r['launches']} {r['forks']} {r['families']} | 64x64: {s['launches']} {s['forks']} {s['families']}")


# ----------------------------------------------------------------------------------------------------------------------
# each row against float64
# ----------------------------------------------------------------------------------------------------------------------
def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _bf16_cotangent(shape, g, pitch=0, like=None):
    """Random bf16 cotangent of the channels-last `shape`.  `pitch` > C: a channel slice [..., :C] of a wider buffer, the way the
    gradient of a tensor concatenated with a skip (torch.cat(..., dim=4)) arrives.  `like`: 0.5 * like is added."""
    c = shape[-1]
    buf = torch.randn((*shape[:-1], max(pitch, c)), device="cuda", generator=g)
    if like is not None:
        buf[..., :c] += 0.5 * like.float()
    return buf.to(torch.bfloat16)[..., :c]


def _ncdhw(t):
    return t.permute(0, 4, 1, 2, 3)


def _mask(y_engine, act, slope):
    """act'(z) as the engine evaluates it, from its stored output: 1 where y > 0, else the slope (0 for ReLU); None: no act."""
    if act == "none":
        return None
    return torch.where(y_engine.detach().float() > 0, 1.0, 0.0 if act == "relu" else slope)


def _act(z, act, slope):
    return F.relu(z) if act == "relu" else (F.leaky_relu(z, slope) if act == "lrelu" else z)


def _where(err):
    """Worst element, worst channel and per-sample worst error: a localised pattern (one channel block, one sample, one tile)
    points to a kernel bug rather than rounding noise."""
    i, idx = int(err.argmax()), []
    for s in reversed(err.shape):
        idx.append(i % s)
        i //= s
    return {"argmax": tuple(reversed(idx)), "worst channel": int(err.flatten(0, -2).max(0).values.argmax()),
            "per-sample max": [round(v, 6) for v in err.flatten(1).max(1).values.tolist()[:8]]}


def _check16(name, got, ref):
    """bf16 result: rel-L2 <= 4e-3 and every element within 3 bf16 ulps of max|ref|."""
    r = rel_l2(got, ref)
    err = (got.double() - ref.double()).abs()
    assert r <= TOL and max_abs_ok(got, ref), (name, r, float(err.max()), float(ref.abs().max()), _where(err))


def _check(name, got, ref, bound):
    r = rel_l2(got, ref)
    assert r <= bound, (name, r, _where((got.double() - ref.double()).abs()) if got.dim() > 1 else None)


def _conv_act(row, gpitch, seed, Fn):
    g = _gen(seed)
    cin, k = row.x[4], row.k
    two_d = row.x[1] == 1 and k[0] == 1
    x = torch.randn(row.x, device="cuda", generator=g).to(torch.bfloat16)
    w = torch.randn(row.w, device="cuda", generator=g) / math.sqrt(cin * k[0] * k[1] * k[2])
    b = torch.randn((row.w[0],), device="cuda", generator=g)
    # a Conv2d layer (FLAVR's fuse convs and outconv) hands the engine a fresh 5-D view of its 4-D weight on every call
    xe = x.clone().requires_grad_(True)
    be = b.clone().requires_grad_(True) if row.bias else None
    we = (w.squeeze(2) if two_d else w).clone().requires_grad_(True)
    out_shape = (row.x[0], *[(i + 2 * p - kk) // s + 1 for i, kk, s, p in zip(row.x[1:4], k, row.s, row.p)], row.w[0])
    if row.out_f32:
        gy = torch.randn(out_shape, device="cuda", generator=g).to(torch.bfloat16).float()
    else:
        gy = _bf16_cotangent(out_shape, g, gpitch)

    def engine():
        out = Fn.conv_act(xe, we.unsqueeze(2) if two_d else we, be, k, row.s, row.p, act=ACT_IDS[row.act], slope=row.slope,
                          out_f32=row.out_f32, want_pool=row.want_pool)
        y, pool = out if row.want_pool else (out, None)
        grads = torch.autograd.grad(y, (xe, we, be) if row.bias else (xe, we), gy)
        return (y, pool) + grads + ((None,) if not row.bias else ())

    y, pool, dx, dw, db = engine()
    torch.cuda.synchronize()
    # reference: fp32 conv (TF32 off) on the same bf16 operands
    xr = _ncdhw(x.float()).requires_grad_(True)
    wr = bf16r(w).requires_grad_(True)
    z = F.conv3d(xr, wr, b if row.bias else None, stride=row.s, padding=row.p)
    yg = _ncdhw(y.detach().float())
    if row.out_f32:
        _check("y", yg, _act(z.detach(), row.act, row.slope), 1e-4)
    else:
        _check16("y", yg, _act(z.detach(), row.act, row.slope))
    if pool is not None:
        # the engine's pool is the mean of the fp32 accumulators (epilogue sums per tile, then over tiles); each fp32 partial
        # sum errs by at most ~sqrt(terms) * 2^-24 of its |terms|, so the mean stays within 1e-5 of mean|z| up to 2^20 voxels
        pref = z.detach().double().mean((2, 3, 4))
        err = float((pool.double() - pref).abs().max())
        assert err <= 1e-5 * float(z.detach().abs().double().mean()), ("pool", err)
    m = _mask(y, row.act, row.slope)
    dz = _ncdhw((gy.float() if m is None else gy.float() * m).to(torch.bfloat16).float())   # the engine stores dz in bf16
    del z, yg
    rdx, rdw = torch.autograd.grad(F.conv3d(xr, wr, None, stride=row.s, padding=row.p), (xr, wr), dz)
    _check16("dx", _ncdhw(dx.float()), rdx)
    _check("dw", dw.unsqueeze(2) if two_d else dw, rdw, 1e-3)
    if row.bias:
        _check("db", db, dz.double().sum((0, 2, 3, 4)), 1e-3)
    return engine


def _smallcin(row, gpitch, seed, Fn):
    g = _gen(seed)
    cin, k = row.x[1], row.k
    x = torch.randn(row.x, device="cuda", generator=g)           # the caller's NCDHW fp32 image: read as fp32, not rounded
    w = torch.randn(row.w, device="cuda", generator=g) / math.sqrt(cin * k[0] * k[1] * k[2])
    b = torch.randn((row.w[0],), device="cuda", generator=g)
    we, be = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    gys = []

    def engine():
        y = Fn.smallcin_conv_act(x, we, be, k, row.s, row.p, act=ACT_IDS[row.act], slope=row.slope)
        if not gys:
            gys.append(_bf16_cotangent(tuple(y.shape), g, gpitch))
        return (y,) + torch.autograd.grad(y, (we, be), gys[0])   # the network's images need no gradient

    y, dw, db = engine()
    torch.cuda.synchronize()
    wr = w.clone().requires_grad_(True)
    z = F.conv3d(x, wr, b, stride=row.s, padding=row.p)
    _check16("y", _ncdhw(y.detach().float()), _act(z.detach(), row.act, row.slope))
    dz = _ncdhw((gys[0].float() * _mask(y, row.act, row.slope)).to(torch.bfloat16).float())
    (rdw,) = torch.autograd.grad(z, (wr,), dz)
    _check("dw", dw, rdw, 1e-3)
    _check("db", db, dz.double().sum((0, 2, 3, 4)), 1e-3)
    return engine


def _conv_transpose(row, gpitch, seed, Fn):
    g = _gen(seed)
    cin, k = row.x[4], row.k
    x = torch.randn(row.x, device="cuda", generator=g).to(torch.bfloat16)
    w = torch.randn(row.w, device="cuda", generator=g) / math.sqrt(cin * k[0] * k[1] * k[2])
    b = torch.randn((row.w[1],), device="cuda", generator=g)
    xe, we, be = x.clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    gys = []

    def engine():
        y = Fn.conv_transpose(xe, we, be, k, row.s, row.p)
        if not gys:
            gys.append(_bf16_cotangent(tuple(y.shape), g, gpitch))
        return (y,) + torch.autograd.grad(y, (xe, we, be), gys[0])

    y, dx, dw, db = engine()
    torch.cuda.synchronize()
    xr = _ncdhw(x.float()).requires_grad_(True)
    wr = bf16r(w).requires_grad_(True)
    z = F.conv_transpose3d(xr, wr, b, stride=row.s, padding=row.p)
    _check16("y", _ncdhw(y.detach().float()), z.detach())
    dz = _ncdhw(gys[0].float())
    rdx, rdw = torch.autograd.grad(z, (xr, wr), dz)
    _check16("dx", _ncdhw(dx.float()), rdx)
    _check("dw", dw, rdw, 1e-3)
    _check("db", db, dz.double().sum((0, 2, 3, 4)), 1e-3)
    return engine


def _se_gate(row, gpitch, seed, Fn):
    """The cotangent is correlated with x (0.5 x + noise).  With an independent one, the gradient through the average pool (the
    per-channel `shift` of SEGate.backward) is O(1/sqrt(voxels)) of dx, under the bf16 bound; correlated, the gate gradient, a
    sum over V voxels, grows like V, and the pool term is O(1) of dx, so dx checks it."""
    g = _gen(seed)
    c = row.x[4]
    vox = row.x[1] * row.x[2] * row.x[3]
    x = torch.randn(row.x, device="cuda", generator=g).to(torch.bfloat16)
    w = torch.randn(row.w, device="cuda", generator=g) / math.sqrt(c)
    b = torch.randn((c,), device="cuda", generator=g)
    res = torch.randn(row.x, device="cuda", generator=g).to(torch.bfloat16) if row.residual else None
    pool = x.double().mean((1, 2, 3)).float() if row.pool else None
    xe, we, be = x.clone().requires_grad_(True), w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    re = res.clone().requires_grad_(True) if res is not None else None
    gy = _bf16_cotangent(row.x, g, gpitch, like=x)

    def engine():
        y = Fn.se_gate(xe, we, be, residual=re, act=ACT_IDS[row.act], slope=row.slope, pool=pool)
        return (y,) + torch.autograd.grad(y, (xe, we, be) + ((re,) if re is not None else ()), gy)

    y, *grads = engine()
    torch.cuda.synchronize()
    xd = x.double()
    pd = pool.double() if pool is not None else xd.mean((1, 2, 3))
    w2 = w.double().reshape(c, c)
    gate = torch.sigmoid(pd @ w2.t() + b.double())                            # [n, c]
    z = xd * gate[:, None, None, None, :]
    if res is not None:
        z = z + res.double()
    _check16("y", y.detach(), _act(z, row.act, row.slope))
    del z
    m = _mask(y, row.act, row.slope)
    dz = gy.double() * (m.double() if m is not None else 1.0)
    dgate = (xd * dz).sum((1, 2, 3))                                          # [n, c]
    dzg = dgate * gate * (1 - gate)
    shift = dzg @ w2 / vox
    _check16("dx", grads[0], dz * gate[:, None, None, None, :] + shift[:, None, None, None, :])
    _check("dW", grads[1].reshape(c, c), dzg.t() @ pd, 1e-3)
    _check("db", grads[2], dzg.sum(0), 1e-3)
    if res is not None:
        _check16("dres", grads[3], dz)
    return engine


def _uasr_ref(out_cl, ue_cl, w, b, n_out):
    """FLAVR_arch.py:203-227,244-246 on the channels-last conv outputs (channel = output * experts + expert)."""
    bsz, _, h, wd, c = out_cl.shape
    o = out_cl[:, 0].reshape(bsz, h, wd, n_out, c // n_out)
    usm = torch.softmax(ue_cl[:, 0].reshape(bsz, h, wd, n_out, -1), dim=-1)
    img = ((torch.tanh(o[..., 0::2]) + 1) / 2 * usm).sum(-1)
    seg = (o[..., 1::2] * usm).sum(-1)
    res = torch.stack([img, seg], 1).permute(0, 1, 4, 2, 3)                   # [B, 2, n_out, H, W]
    unc = torch.sigmoid((usm * w.reshape(-1)).sum(-1) + b.reshape(())).unsqueeze(1).permute(0, 1, 4, 2, 3)
    return res, unc


def _uasr(row, gpitch, seed, Fn):
    """Outputs and conv-output gradients are element-wise fp32 arithmetic (softmax over 16 experts, tanh, sigmoid: some 50
    roundings of 2^-24 each, plus the kernel's fast exp / tanh at a few ulps), so 1e-4 rel-L2 holds for them as for the fp32 conv
    outputs.  The uncertainty layer's dW / db are per-block fp32 partials summed in double: 1e-3, like every weight gradient."""
    from rehrseg_b200 import flavr
    g = _gen(seed)
    n_out = 4
    out_cl = torch.randn(row.x, device="cuda", generator=g)
    ue_cl = torch.randn((*row.x[:4], row.x[4] // 2), device="cuda", generator=g)
    head = torch.nn.Conv3d(row.w[1], 1, kernel_size=1).cuda()
    with torch.no_grad():
        head.weight.copy_(torch.randn(row.w, device="cuda", generator=g))
        head.bias.copy_(torch.randn((1,), device="cuda", generator=g))
    oe, ue = out_cl.clone().requires_grad_(True), ue_cl.clone().requires_grad_(True)
    n, _, h, wd, _ = row.x
    gr = torch.randn((n, 2, n_out, h, wd), device="cuda", generator=g).to(torch.bfloat16).float()
    gu = torch.randn((n, 1, n_out, h, wd), device="cuda", generator=g).to(torch.bfloat16).float()

    def engine():
        res, unc = flavr.uasr_mixture(oe, ue, head, n_out)
        return (res, unc) + torch.autograd.grad((res, unc), (oe, ue, head.weight, head.bias), (gr, gu))

    res, unc, d_out, d_ue, dw, db = engine()
    torch.cuda.synchronize()
    od, ud = out_cl.double().requires_grad_(True), ue_cl.double().requires_grad_(True)
    wd64, bd64 = head.weight.detach().double().requires_grad_(True), head.bias.detach().double().requires_grad_(True)
    rres, runc = _uasr_ref(od, ud, wd64, bd64, n_out)
    _check("res", res.detach(), rres.detach(), 1e-4)
    _check("unc", unc.detach(), runc.detach(), 1e-4)
    rd_out, rd_ue, rdw, rdb = torch.autograd.grad((rres, runc), (od, ud, wd64, bd64), (gr.double(), gu.double()))
    _check("d_out", d_out, rd_out, 1e-4)
    _check("d_ue", d_ue, rd_ue, 1e-4)
    _check("dW", dw, rdw, 1e-3)
    _check("db", db, rdb, 1e-3)
    return engine


RUNNERS = {"conv_act": _conv_act, "smallcin_conv_act": _smallcin, "conv_transpose": _conv_transpose, "se_gate": _se_gate,
           "uasr_mixture": _uasr}


def _row_id(row):
    parts = [row.fn, "x" + "x".join(map(str, row.x)), "w" + "x".join(map(str, row.w))]
    if row.k:
        parts += ["k" + "".join(map(str, row.k)), "s" + "".join(map(str, row.s))]
    parts += [row.act] if row.act != "none" else []
    parts += [f for f in ("want_pool", "out_f32", "residual", "pool") if getattr(row, f)] + ([] if row.bias else ["nobias"])
    return "-".join(parts)


@pytest.mark.parametrize("shape_key,row", [(k, r) for k in ("C2", "TRAIN") for r in TABLES[k]],
                         ids=[f"{k}-{_row_id(r)}" for k in ("C2", "TRAIN") for r in TABLES[k]])
def test_layer_vs_float64(monkeypatch, shape_key, row):
    """One table row alone, at its shape, against float64; then the same call again under kernel_timer, which must launch the
    conv kernel families and the number of engine launches the row had inside the network, after the same number of
    side-stream forks in the untimed run."""
    from rehrseg_b200 import functional as Fn
    net = network_routes(monkeypatch, shape_key, _heads_of(row)[-1])[row]
    cnt = _Counters(Fn, monkeypatch)
    engine = RUNNERS[row.fn](row, net["gpitch"], zlib.crc32(repr(row).encode()), Fn)
    assert cnt.forks == sum(net["forks"]), ("side-stream forks", cnt.forks, net["forks"])
    monkeypatch.undo()
    l0 = Fn.launches()
    with Fn.kernel_timer() as kt:
        engine()
        torch.cuda.synchronize()
    assert tuple(r[0] for r in kt.records if r[0] in FAMILIES) == net["families"][0] + net["families"][1], \
        ([r[0] for r in kt.records], net["families"])
    assert Fn.launches() - l0 == sum(net["launches"]), (Fn.launches() - l0, net["launches"])
    del engine
    torch.cuda.empty_cache()


# ----------------------------------------------------------------------------------------------------------------------
# the C2 training iteration at 256 x 256 against the oracle
# ----------------------------------------------------------------------------------------------------------------------
# Measured on an NVIDIA B200 (1000 W power limit): worst parameter tensor 3.10e-2 with the plain head
# (encoder.layer4.0.conv1.0.weight; global 3.4e-3) and 4.47e-2 with the UASR head (the same tensor; global 9.5e-5).  The bound is
# twice the worst, rounded up.  The deep encoder layers are the worst: their gradients pass through every decoder layer's bf16
# rounding, while the UASR head's global norm is dominated by its fp32 head layers.
PER_PARAM_BOUND = 9e-2


@pytest.mark.parametrize("unc", [False, True], ids=["plain", "uasr"])
def test_graphed_fused_sr_step_at_256_vs_oracle(unc):
    """GraphedSRStep with FusedSRLoss, the form the benchmark times, at C2's 256 x 256 planes (batch 2, so the fp32 CPU oracle
    stays near 10 s per head), against oracle.joint.ref_sr_step with the same weights.  Loss within 1e-2 and the global
    gradient within 8e-2 as at 64 x 64 (tests/test_sr_step_gpu.py), and every parameter tensor on its own within
    PER_PARAM_BOUND."""
    from oracle import flavr as of, joint as oj
    from rehrseg_b200 import flavr, loss_ops, train_step as ts
    ref = of.build(unc, seed=9).train()
    torch.manual_seed(9)
    mine = flavr.UNet_3D_3D(2, "unet_18", 4, 4, False, "concat", "transpose", use_uncertainty=unc)
    assert all(torch.equal(a, b) for a, b in zip(ref.state_dict().values(), mine.state_dict().values()))
    mine = mine.cuda().train()
    g = torch.Generator().manual_seed(13)
    lr = torch.rand((2, 2, 4, 256, 256), generator=g)
    lr[:, 1] = (lr[:, 1] > 0.8).float()
    hr = torch.rand((2, 2, 16, 256, 256), generator=g)
    hr[:, 1] = (hr[:, 1] > 0.8).float()
    want = float(oj.ref_sr_step(ref, lr.clone(), hr.clone(), torch.nn.L1Loss(), oj.RefBCEDiceLoss(1, 1), 4, 4, unc))
    step = ts.GraphedSRStep(mine, (lr.clone().cuda(), hr.clone().cuda()), slice_separation=4, num_slices=4, enable_uncertainty=unc,
                            fused_loss=loss_ops.FusedSRLoss(1.0, 1.0, enable_uncertainty=unc))
    try:
        got = float(step((lr.clone().cuda(), hr.clone().cuda()))["loss"])
        torch.cuda.synchronize()
        pr = dict(ref.named_parameters())
        num = den = 0.0
        per = {}
        for name, p in mine.named_parameters():
            assert (p.grad is None) == (pr[name].grad is None), name
            if p.grad is None:
                continue
            a, b = p.grad.double().cpu(), pr[name].grad.double()
            num += float((a - b).pow(2).sum())
            den += float(b.pow(2).sum())
            per[name] = float((a - b).norm() / (b.norm() + 1e-30))
    finally:
        step.close()
    glob = (num / den) ** 0.5
    print(f"\n256x256 graphed fused sr step {'uasr' if unc else 'plain'}: loss {got} vs {want}, global grad rel-L2 {glob:.3e}")
    for name, r in sorted(per.items(), key=lambda kv: -kv[1]):
        print(f"  {name:45s} {r:.3e}")
    assert abs(got - want) <= 1e-2 * abs(want), (got, want)
    assert glob <= 8e-2, glob
    worst = max(per, key=per.get)
    assert per[worst] <= PER_PARAM_BOUND, (worst, per[worst])
