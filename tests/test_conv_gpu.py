"""GPU parity of the conv engine (through the C-ABI) against torch fp32 convolutions on the same bf16-rounded
operands.  Tolerance: relative L2 <= 4e-3 -- about twice what the one 16-bit rounding of the result costs (2^-9 / sqrt(3) ~ 1.1e-3
relative per element), far below north_star's 1e-2 whole-network bound: a wrong halo row / tap of a 3x3x3 kernel moves > 1e-2 --
plus a max-abs bound of a few output ulps, which a single wrong voxel breaks."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

TOL = 4e-3


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return float((a.detach() - b.detach()).norm() / (b.detach().norm() + 1e-30))


def max_abs_ok(got, ref, ulps=3.0):
    """Every element within `ulps` bf16 ulps of the LARGEST reference magnitude (one ulp = 2^-8 relative): what one rounding of the
    result plus fp32 summation-order noise can cost; a voxel that misses a tap or reads a wrong halo row is off by far more."""
    err = float((got.double() - ref.double()).abs().max())
    return err <= ulps * 2.0 ** -8 * float(ref.abs().max())


def bf16r(t):
    return t.to(torch.bfloat16).float()


@pytest.fixture(autouse=True)
def _fp32_reference():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield


@pytest.fixture(params=["march", "generic"])
def engine(request):
    """Run the conv tests through both kernels: the halo-resident marching kernel (eligible k3/s1/p1 layers) and the
    generic tapped-GEMM kernel."""
    from rehrseg_b200 import functional as Fn
    old = Fn.USE_MARCH
    Fn.USE_MARCH = request.param == "march"
    yield request.param
    Fn.USE_MARCH = old


FWD_CASES = [
    # n, cin, cout, (d,h,w), k, s, p
    (1, 32, 32, (16, 16, 16), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (2, 64, 64, (8, 16, 16), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 16, 16, (8, 8, 16), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (2, 32, 64, (16, 16, 16), (3, 3, 3), (2, 2, 2), (1, 1, 1)),
    (2, 320, 320, (4, 4, 4), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (2, 256, 320, (8, 8, 8), (3, 3, 3), (2, 2, 2), (1, 1, 1)),
    (1, 32, 32, (4, 16, 16), (1, 3, 3), (1, 1, 1), (0, 1, 1)),
    (1, 64, 128, (4, 16, 16), (3, 3, 3), (1, 2, 2), (1, 1, 1)),
    (1, 32, 48, (7, 9, 11), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 16, 2, (8, 8, 8), (5, 5, 5), (1, 1, 1), (2, 2, 2)),
    (1, 64, 64, (1, 16, 16), (1, 1, 1), (1, 1, 1), (0, 0, 0)),
    (1, 128, 64, (4, 16, 16), (1, 1, 1), (1, 2, 2), (0, 0, 0)),
    (1, 256, 64, (1, 16, 16), (1, 3, 3), (1, 1, 1), (0, 1, 1)),
    # marching-kernel shapes: multi depth segments / TMEM slot wrap / Cout tiling / 2 channel chunks / ragged tiles
    (1, 32, 32, (40, 16, 8), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (2, 64, 64, (12, 32, 16), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 128, 64, (6, 16, 16), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 64, 128, (5, 20, 12), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 16, 16, (3, 5, 5), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 32, 16, (1, 8, 8), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    # stride-2 stage-entry convs big enough for the per-parity-class marching input gradient (even, odd and anisotropic)
    (1, 32, 64, (32, 32, 32), (3, 3, 3), (2, 2, 2), (1, 1, 1)),
    (1, 32, 64, (33, 31, 35), (3, 3, 3), (2, 2, 2), (1, 1, 1)),
    (1, 64, 128, (8, 64, 64), (3, 3, 3), (1, 2, 2), (1, 1, 1)),
    (2, 64, 32, (20, 32, 34), (3, 3, 3), (2, 2, 2), (1, 1, 1)),
    # 5x5x5 marching variant (sr_head.2, models/seg_model.py:199) and output-channel counts that do not fill a tile
    (1, 16, 16, (9, 20, 12), (5, 5, 5), (1, 1, 1), (2, 2, 2)),
    (2, 16, 2, (24, 16, 8), (5, 5, 5), (1, 1, 1), (2, 2, 2)),
    (1, 32, 2, (6, 16, 16), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 16, 40, (5, 9, 9), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    # planar k(1,3,3) layers of anisotropic plans through the marching kernels (centre depth tap only): channel chunks,
    # Cout tiling, ragged tiles, several depth segments, big enough for the marching weight gradient
    (2, 64, 32, (5, 20, 12), (1, 3, 3), (1, 1, 1), (0, 1, 1)),
    (1, 128, 64, (3, 16, 16), (1, 3, 3), (1, 1, 1), (0, 1, 1)),
    (1, 32, 48, (20, 9, 11), (1, 3, 3), (1, 1, 1), (0, 1, 1)),
    (2, 32, 32, (16, 64, 64), (1, 3, 3), (1, 1, 1), (0, 1, 1)),
    (1, 64, 64, (9, 40, 24), (1, 3, 3), (1, 1, 1), (0, 1, 1)),
]


def _mk(n, cin, cout, dhw, k, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn((n, cin, *dhw), generator=g)
    w = torch.randn((cout, cin, *k), generator=g) / (cin * k[0] * k[1] * k[2]) ** 0.5
    b = torch.randn((cout,), generator=g)
    return x.cuda(), w.cuda(), b.cuda()


@pytest.mark.parametrize("case", FWD_CASES)
def test_conv3d_fwd(case, engine):
    from rehrseg_b200 import functional as Fn
    n, cin, cout, dhw, k, s, p = case
    x, w, b = _mk(n, cin, cout, dhw, k)
    ref = F.conv3d(bf16r(x), bf16r(w), b, stride=s, padding=p)
    xcl = x.permute(0, 2, 3, 4, 1).contiguous().to(torch.bfloat16)
    y, _, _ = Fn.conv3d_raw(xcl, w, b, k, s, p)
    torch.cuda.synchronize()
    got = y.float().permute(0, 4, 1, 2, 3)
    assert got.shape == ref.shape
    assert rel_l2(got, ref) < TOL, (case, rel_l2(got, ref))
    assert max_abs_ok(got, ref), case


@pytest.mark.parametrize("case", FWD_CASES[:4] + FWD_CASES[6:9])
def test_conv3d_fwd_act_f32(case, engine):
    from rehrseg_b200 import functional as Fn
    from rehrseg_b200._lib import ACT_LRELU
    n, cin, cout, dhw, k, s, p = case
    x, w, b = _mk(n, cin, cout, dhw, k, seed=1)
    ref = F.leaky_relu(F.conv3d(bf16r(x), bf16r(w), b, stride=s, padding=p), 0.2)
    xcl = x.permute(0, 2, 3, 4, 1).contiguous().to(torch.bfloat16)
    y, _, _ = Fn.conv3d_raw(xcl, w, b, k, s, p, act=ACT_LRELU, slope=0.2, out_f32=True)
    torch.cuda.synchronize()
    assert y.dtype == torch.float32
    assert rel_l2(y.permute(0, 4, 1, 2, 3), ref) < 1e-4, case  # fp32 output: only accumulation-order noise


@pytest.mark.parametrize("case", [c for c in FWD_CASES if c[2] % 16 == 0])
def test_conv3d_dgrad(case, engine):
    from rehrseg_b200 import functional as Fn
    n, cin, cout, dhw, k, s, p = case
    x, w, _ = _mk(n, cin, cout, dhw, k, seed=2)
    x.requires_grad_(True)
    y = F.conv3d(x, bf16r(w), None, stride=s, padding=p)
    g = torch.randn(y.shape, generator=torch.Generator().manual_seed(3)).cuda()
    (ref,) = torch.autograd.grad(y, x, bf16r(g))
    gcl = g.permute(0, 2, 3, 4, 1).contiguous().to(torch.bfloat16)
    dx = Fn.conv3d_dgrad_raw(gcl, w, (n, *dhw, cin), k, s, p, cache=False)
    torch.cuda.synchronize()
    assert rel_l2(dx.float().permute(0, 4, 1, 2, 3), ref) < TOL, case
    assert max_abs_ok(dx.float().permute(0, 4, 1, 2, 3), ref), case


WGRAD_MARCH_CASES = [
    # marching weight-gradient shapes: role A / B, 32- and 64-channel halo pieces, channel splits, volume-edge planes,
    # ragged tiles, depth segments, a channel slice of a wider (concat) buffer is covered in test_wgrad_march_pitched
    (2, 32, 32, (20, 32, 16), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (2, 32, 32, (16, 32, 32), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 32, 32, (33, 40, 24), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 64, 32, (32, 64, 64), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 128, 64, (32, 32, 32), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 64, 32, (9, 16, 24), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 32, 64, (6, 32, 8), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (2, 64, 64, (5, 20, 12), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 128, 64, (8, 16, 16), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 128, 128, (4, 16, 16), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 64, 96, (4, 16, 8), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 32, 32, (1, 16, 16), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 256, 320, (4, 8, 8), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    # sr_head shapes: 32 -> 16 k3 (16-channel plain pieces) and 16 -> 16 k5 (16-channel halo pieces, N = 5 x 16)
    (1, 32, 16, (32, 32, 32), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 64, 16, (30, 40, 24), (3, 3, 3), (1, 1, 1), (1, 1, 1)),
    (1, 16, 16, (32, 32, 32), (5, 5, 5), (1, 1, 1), (2, 2, 2)),
    (2, 16, 16, (13, 24, 40), (5, 5, 5), (1, 1, 1), (2, 2, 2)),
]


@pytest.mark.parametrize("case", [c for c in FWD_CASES if c[2] % 16 == 0] + WGRAD_MARCH_CASES)
def test_conv3d_wgrad(case, engine):
    from rehrseg_b200 import functional as Fn
    n, cin, cout, dhw, k, s, p = case
    x, w, _ = _mk(n, cin, cout, dhw, k, seed=4)
    w.requires_grad_(True)
    y = F.conv3d(bf16r(x), w, None, stride=s, padding=p)
    g = torch.randn(y.shape, generator=torch.Generator().manual_seed(5)).cuda()
    (ref,) = torch.autograd.grad(y, w, bf16r(g))
    xcl = x.permute(0, 2, 3, 4, 1).contiguous().to(torch.bfloat16)
    gcl = g.permute(0, 2, 3, 4, 1).contiguous().to(torch.bfloat16)
    dw = Fn.conv3d_wgrad_raw(xcl, gcl, w.shape, k, s, p)
    torch.cuda.synchronize()
    assert dw.shape == ref.shape
    assert rel_l2(dw, ref) < 1e-3, (case, rel_l2(dw, ref))  # fp32 accumulate of exact bf16 products


def test_wgrad_march_routing():
    """The big k3/s1/p1 layers must take the marching weight-gradient kernel (and tiny volumes the split-K one), so the
    parity cases above really cover both kernels."""
    import ctypes as C
    from rehrseg_b200 import _lib as L
    desc = L.conv_desc((3, 3, 3), (1, 1, 1), (1, 1, 1))
    d5 = L.conv_desc((5, 5, 5), (1, 1, 1), (2, 2, 2))
    x5, y5 = L.RehrTensor(16, 1, 32, 32, 32, 16, 16), L.RehrTensor(16, 1, 32, 32, 32, 16, 16)
    assert L.lib().rehr_conv3d_wgrad_march_supported(C.byref(d5), C.byref(x5), C.byref(y5)) == 1
    for (n, ci, co, dhw), want in [((2, 32, 32, (16, 32, 32)), 1), ((1, 32, 16, (32, 32, 32)), 1), ((1, 64, 32, (32, 64, 64)), 1), ((1, 128, 64, (32, 32, 32)), 1),
                                   ((2, 32, 32, (128, 128, 128)), 1), ((2, 320, 320, (4, 4, 4)), 0), ((1, 16, 16, (32, 32, 32)), 0)]:
        x = L.RehrTensor(16, n, *dhw, ci, ci)
        dy = L.RehrTensor(16, n, *dhw, co, co)
        assert L.lib().rehr_conv3d_wgrad_march_supported(C.byref(desc), C.byref(x), C.byref(dy)) == want, (n, ci, co, dhw)


def test_planar_layers_take_the_marching_kernels():
    """k(1,3,3) / pad (0,1,1) layers must really be routed to conv_march_kernel / wgrad_march_kernel."""
    from rehrseg_b200 import functional as Fn
    x, w, b = _mk(2, 32, 32, (16, 64, 64), (1, 3, 3), seed=8)
    xcl = x.permute(0, 2, 3, 4, 1).contiguous().to(torch.bfloat16)
    with Fn.kernel_timer() as kt:
        y, _, _ = Fn.conv3d_raw(xcl, w, b, (1, 3, 3), (1, 1, 1), (0, 1, 1))
        Fn.conv3d_dgrad_raw(y, w, tuple(xcl.shape), (1, 3, 3), (1, 1, 1), (0, 1, 1), cache=False)
        Fn.conv3d_wgrad_raw(xcl, y, w.shape, (1, 3, 3), (1, 1, 1), (0, 1, 1))
    assert [r[0] for r in kt.rows()] == ["conv_march_kernel", "conv_march_kernel", "wgrad_march_kernel"]


TCONV_CASES = [
    (2, 64, 32, (8, 8, 8), (2, 2, 2), (2, 2, 2), (0, 0, 0)),
    (2, 320, 320, (4, 4, 4), (2, 2, 2), (2, 2, 2), (0, 0, 0)),
    (1, 64, 32, (4, 8, 8), (1, 2, 2), (1, 2, 2), (0, 0, 0)),
    (1, 128, 64, (4, 8, 8), (3, 4, 4), (1, 2, 2), (1, 1, 1)),   # FLAVR upConv3D (FLAVR_arch.py:49-51)
    # the three FLAVR up-convs of the C2 step ([8, 2, 4, 256, 256]): decoder.1, .2, .4; the last one's weight gradient is too
    # big for the side stream
    (8, 512, 128, (4, 32, 32), (3, 4, 4), (1, 2, 2), (1, 1, 1)),
    (8, 256, 64, (4, 64, 64), (3, 4, 4), (1, 2, 2), (1, 1, 1)),
    (8, 128, 64, (4, 128, 128), (3, 4, 4), (1, 2, 2), (1, 1, 1)),
]


@pytest.mark.parametrize("case", TCONV_CASES)
def test_conv_transpose_fwd_bwd(case):
    from rehrseg_b200 import functional as Fn
    n, cin, cout, dhw, k, s, p = case
    g = torch.Generator().manual_seed(6)
    x = torch.randn((n, cin, *dhw), generator=g).cuda()
    w = (torch.randn((cin, cout, *k), generator=g) / cin ** 0.5).cuda()
    b = torch.randn((cout,), generator=g).cuda()
    xr = bf16r(x).requires_grad_(True)
    wr = bf16r(w).requires_grad_(True)
    br = b.clone().requires_grad_(True)
    ref = F.conv_transpose3d(xr, wr, br, stride=s, padding=p)
    go = torch.randn(ref.shape, generator=g).cuda()
    rdx, rdw, rdb = torch.autograd.grad(ref, (xr, wr, br), bf16r(go))

    xcl = x.permute(0, 2, 3, 4, 1).contiguous().to(torch.bfloat16).requires_grad_(True)
    wp = w.clone().requires_grad_(True)
    bp = b.clone().requires_grad_(True)
    y = Fn.conv_transpose(xcl, wp, bp, k, s, p)
    assert rel_l2(y.float().permute(0, 4, 1, 2, 3), ref) < TOL, case
    gcl = go.permute(0, 2, 3, 4, 1).contiguous().to(torch.bfloat16)
    dx, dw, db = torch.autograd.grad(y, (xcl, wp, bp), gcl)
    torch.cuda.synchronize()
    assert rel_l2(dx.float().permute(0, 4, 1, 2, 3), rdx) < TOL, case
    assert rel_l2(dw, rdw) < 2e-3, case
    assert rel_l2(db, rdb) < 2e-3, case


@pytest.mark.parametrize("shape", [(2, 32, (16, 16, 16)), (1, 64, (8, 8, 8)), (2, 320, (4, 4, 4)), (1, 48, (7, 9, 11))])
@pytest.mark.parametrize("stride", [(1, 1, 1), (2, 2, 2)])
def test_conv_norm_act_block(shape, stride, engine):
    """Conv3d -> InstanceNorm3d(affine) -> LeakyReLU forward + full backward vs torch autograd (fp32)."""
    from rehrseg_b200 import functional as Fn
    n, c, dhw = shape
    cin = 32
    g = torch.Generator().manual_seed(7)
    x = torch.randn((n, cin, *dhw), generator=g).cuda()
    w = (torch.randn((c, cin, 3, 3, 3), generator=g) / (27 * cin) ** 0.5).cuda()
    b = torch.randn((c,), generator=g).cuda()
    ga = (1 + 0.1 * torch.randn((c,), generator=g)).cuda()
    be = (0.1 * torch.randn((c,), generator=g)).cuda()
    xr = bf16r(x).requires_grad_(True)
    wr = bf16r(w).requires_grad_(True)
    gar, ber = ga.clone().requires_grad_(True), be.clone().requires_grad_(True)
    ref = F.leaky_relu(F.instance_norm(F.conv3d(xr, wr, b, stride=stride, padding=1), weight=gar, bias=ber, eps=1e-5), 0.01)
    go = torch.randn(ref.shape, generator=g).cuda()
    rdx, rdw, rdg, rdb = torch.autograd.grad(ref, (xr, wr, gar, ber), bf16r(go))

    xcl = x.permute(0, 2, 3, 4, 1).contiguous().to(torch.bfloat16).requires_grad_(True)
    wp, bp = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    gap, bep = ga.clone().requires_grad_(True), be.clone().requires_grad_(True)
    a = Fn.conv_norm_act(xcl, wp, bp, gap, bep, (3, 3, 3), stride, (1, 1, 1), eps=1e-5, slope=0.01)
    assert rel_l2(Fn.to_float(a).permute(0, 4, 1, 2, 3), ref) < TOL
    gcl = go.permute(0, 2, 3, 4, 1).contiguous().to(torch.bfloat16)
    dx, dw, dbias, dg, dbeta = torch.autograd.grad(a, (xcl, wp, bp, gap, bep), gcl)
    torch.cuda.synchronize()
    # The engine stores the conv output in bf16, so ~0.1 % of the LeakyReLU masks (|z| below one bf16 ulp of y) differ
    # from the fp32 reference's; each flipped voxel carries a 100 % local gradient error => rel-L2 ~ sqrt(1e-3) ~ 3 %.
    # This is the gradient of the bf16 forward actually computed, not an error of the backward kernels (dgrad / wgrad
    # alone are checked at 1e-2 / 1e-3 above).
    GT = 6e-2
    assert rel_l2(dx.float().permute(0, 4, 1, 2, 3), rdx) < GT
    assert rel_l2(dw, rdw) < GT
    assert rel_l2(dg, rdg) < GT
    assert rel_l2(dbeta, rdb) < GT
    assert float(dbias.abs().max()) == 0.0


def test_smallcin_stem_block():
    """1-channel nnU-Net stem: NCDHW fp32 in, Conv3d(1->32,k3) -> IN -> LeakyReLU, weight gradient."""
    from rehrseg_b200 import functional as Fn
    g = torch.Generator().manual_seed(8)
    x = torch.randn((2, 1, 16, 24, 24), generator=g).cuda()
    w = (torch.randn((32, 1, 3, 3, 3), generator=g) / 27 ** 0.5).cuda()
    b = torch.randn((32,), generator=g).cuda()
    ga = (1 + 0.1 * torch.randn((32,), generator=g)).cuda()
    be = (0.1 * torch.randn((32,), generator=g)).cuda()
    wr, gar, ber = (t.clone().requires_grad_(True) for t in (w, ga, be))
    ref = F.leaky_relu(F.instance_norm(F.conv3d(x, wr, b, padding=1), weight=gar, bias=ber, eps=1e-5), 0.01)
    go = torch.randn(ref.shape, generator=g).cuda()
    rdw, rdg, rdb = torch.autograd.grad(ref, (wr, gar, ber), bf16r(go))
    wp, bp, gap, bep = (t.clone().requires_grad_(True) for t in (w, b, ga, be))
    a = Fn.conv_norm_act(x, wp, bp, gap, bep, (3, 3, 3), (1, 1, 1), (1, 1, 1), small_cin=True)
    assert rel_l2(Fn.to_float(a).permute(0, 4, 1, 2, 3), ref) < TOL
    gcl = go.permute(0, 2, 3, 4, 1).contiguous().to(torch.bfloat16)
    dw, dg, dbeta = torch.autograd.grad(a, (wp, gap, bep), gcl)
    torch.cuda.synchronize()
    assert rel_l2(dw, rdw) < 6e-2
    assert rel_l2(dg, rdg) < 6e-2
    assert rel_l2(dbeta, rdb) < 6e-2


@pytest.mark.parametrize("planar", [False, True])
@pytest.mark.parametrize("dhw", [(5, 11, 20), (3, 16, 128), (4, 9, 33)])
def test_stem_tensor_core_kernels_keep_fp32_accuracy(dhw, planar):
    """1 -> 32 k3 stem through the mma.sync kernels (csrc/stem_mma.cu): the fp32 image and weights are split into bf16 hi + lo
    parts, so forward and weight gradient must match fp32 torch far below bf16 resolution (output only rounded once to bf16)."""
    import ctypes as C
    from rehrseg_b200 import _lib as L
    g = torch.Generator().manual_seed(21)
    d, h, w_ = dhw
    x = torch.randn((2, 1, d, h, w_), generator=g).cuda()
    kern, pad = ((1, 3, 3), (0, 1, 1)) if planar else ((3, 3, 3), (1, 1, 1))   # planar: the stem of anisotropic plans
    w = (torch.randn((32, 1, *kern), generator=g) / 27 ** 0.5).cuda()
    b = torch.randn((32,), generator=g).cuda()
    wr = w.clone().requires_grad_(True)
    ref = F.conv3d(x, wr, b, padding=pad)
    desc = L.conv_desc(kern, (1, 1, 1), pad)
    y = torch.empty((2, d, h, w_, 32), dtype=torch.bfloat16, device="cuda")
    yt = L.rt(y)
    L.check(L.lib().rehr_conv3d_smallcin_fwd(C.byref(desc), L.ptr(x), 2, 1, d, h, w_, L.ptr(w), L.ptr(b), C.byref(yt),
                                             L.ACT_NONE, 0.0, None, L.stream_ptr()))
    got = y.float().permute(0, 4, 1, 2, 3)
    assert float((got - bf16r(ref)).abs().max()) <= 2.0 ** -7 * float(ref.abs().max())      # <= 1 bf16 ulp anywhere
    assert rel_l2(got, bf16r(ref)) < 5e-4                                                    # and almost always 0 ulp
    go = torch.randn(ref.shape, generator=g).cuda()
    (rdw,) = torch.autograd.grad(ref, wr, bf16r(go))
    gcl = go.permute(0, 2, 3, 4, 1).contiguous().to(torch.bfloat16)
    gt = L.rt(gcl)
    need = L.lib().rehr_conv3d_smallcin_wgrad_workspace(C.byref(desc), 1, C.byref(gt))
    ws = torch.empty((need,), dtype=torch.uint8, device="cuda")
    dw = torch.empty_like(w)
    L.check(L.lib().rehr_conv3d_smallcin_wgrad(C.byref(desc), L.ptr(x), 2, 1, d, h, w_, C.byref(gt), L.ptr(dw), 0, L.ptr(ws), need,
                                               L.stream_ptr()))
    torch.cuda.synchronize()
    assert rel_l2(dw, rdw) < 1e-4, rel_l2(dw, rdw)


def test_flavr_stem_smallcin_raw():
    """2-channel FLAVR stem k(3,7,7) s(1,2,2) p(1,3,3) + ReLU (resnet_3D.py:42-50) forward / wgrad / dgrad."""
    import ctypes as C
    from rehrseg_b200 import _lib as L
    g = torch.Generator().manual_seed(9)
    x = torch.randn((1, 2, 4, 32, 32), generator=g).cuda()
    w = (torch.randn((64, 2, 3, 7, 7), generator=g) / 294 ** 0.5).cuda()
    b = torch.randn((64,), generator=g).cuda()
    xr, wr = x.clone().requires_grad_(True), w.clone().requires_grad_(True)
    ref = F.relu(F.conv3d(xr, wr, b, stride=(1, 2, 2), padding=(1, 3, 3)))
    y = torch.empty((1, 4, 16, 16, 64), dtype=torch.bfloat16, device="cuda")
    desc = L.conv_desc((3, 7, 7), (1, 2, 2), (1, 3, 3))
    yt = L.rt(y)
    L.check(L.lib().rehr_conv3d_smallcin_fwd(C.byref(desc), L.ptr(x), 1, 2, 4, 32, 32, L.ptr(w), L.ptr(b), C.byref(yt),
                                             L.ACT_RELU, 0.0, None, L.stream_ptr()))
    assert rel_l2(y.float().permute(0, 4, 1, 2, 3), ref) < TOL
    go = torch.randn(ref.shape, generator=g).cuda()
    pre = F.conv3d(xr, wr, b, stride=(1, 2, 2), padding=(1, 3, 3))
    rdx, rdw = torch.autograd.grad(pre, (xr, wr), bf16r(go))
    gcl = go.permute(0, 2, 3, 4, 1).contiguous().to(torch.bfloat16)
    gt = L.rt(gcl)
    need = L.lib().rehr_conv3d_smallcin_wgrad_workspace(C.byref(desc), 2, C.byref(gt))
    ws = torch.empty((need,), dtype=torch.uint8, device="cuda")
    dw = torch.empty_like(w)
    L.check(L.lib().rehr_conv3d_smallcin_wgrad(C.byref(desc), L.ptr(x), 1, 2, 4, 32, 32, C.byref(gt), L.ptr(dw), 0, L.ptr(ws), need,
                                               L.stream_ptr()))
    dx = torch.empty_like(x)
    L.check(L.lib().rehr_conv3d_smallcin_dgrad(C.byref(desc), C.byref(gt), L.ptr(w), L.ptr(dx), 1, 2, 4, 32, 32, L.stream_ptr()))
    torch.cuda.synchronize()
    assert rel_l2(dw, rdw) < 1e-3
    assert rel_l2(dx, rdx) < 1e-3


@pytest.mark.parametrize("case", [(1, 32, 64, (16, 128, 128), (2, 2, 2)), (1, 64, 32, (15, 130, 126), (2, 2, 2)),
                                  (1, 32, 32, (8, 128, 128), (1, 2, 2)), (2, 32, 64, (33, 66, 70), (2, 2, 2)),
                                  (1, 32, 128, (32, 128, 128), (2, 2, 2))])
def test_wgrad_march_stride2(case):
    """Per-parity-class marching weight gradient of the stride-2 stage-entry convs (strided TMA views of x, offset masks),
    forced on for these mid-size shapes, against torch autograd."""
    from rehrseg_b200 import functional as Fn
    n, cin, cout, dhw, s = case
    x, w, _ = _mk(n, cin, cout, dhw, (3, 3, 3), seed=11)
    w.requires_grad_(True)
    y = F.conv3d(bf16r(x), w, None, stride=s, padding=1)
    g = torch.randn(y.shape, generator=torch.Generator().manual_seed(12)).cuda()
    (ref,) = torch.autograd.grad(y, w, bf16r(g))
    xcl = x.permute(0, 2, 3, 4, 1).contiguous().to(torch.bfloat16)
    gcl = g.permute(0, 2, 3, 4, 1).contiguous().to(torch.bfloat16)
    old = Fn.S2_WGRAD_MARCH_MIN_VOXELS
    Fn.S2_WGRAD_MARCH_MIN_VOXELS = 0
    try:
        with Fn.kernel_timer() as kt:
            dw = Fn.conv3d_wgrad_raw(xcl, gcl, w.shape, (3, 3, 3), s, (1, 1, 1))
        assert [r[0] for r in kt.rows()] == ["wgrad_march_kernel"]   # really took the marching path
    finally:
        Fn.S2_WGRAD_MARCH_MIN_VOXELS = old
    assert rel_l2(dw, ref) < 1e-3, (case, rel_l2(dw, ref))


FP16_CASES = [
    # n, cin, cout, (d,h,w), kernel, padding: marching-kernel shapes
    (2, 32, 32, (6, 16, 8), (3, 3, 3), (1, 1, 1)),
    (1, 64, 32, (5, 20, 12), (3, 3, 3), (1, 1, 1)),      # ragged tiles
    (2, 64, 64, (12, 32, 16), (3, 3, 3), (1, 1, 1)),     # Cout tiled 2 x 32
    (1, 128, 64, (6, 16, 16), (3, 3, 3), (1, 1, 1)),     # 2 channel chunks, tile 16
    (1, 32, 32, (4, 16, 16), (1, 3, 3), (0, 1, 1)),      # planar
    (1, 32, 16, (9, 7, 5), (3, 3, 3), (1, 1, 1)),        # everything ragged
]


@pytest.mark.parametrize("case", FP16_CASES)
def test_march_forward_fp16(case):
    """The forward activations of the InstanceNorm'ed SegModel path are fp16 (functional.FWD_FP16): the marching forward on fp16
    operands and fp16 output against F.conv3d on the same fp16-rounded operands, and the bf16 twin such an activation hands a
    weight gradient (converted on demand, cached on the tensor) against the bf16 rounding of its values."""
    from rehrseg_b200 import functional as Fn
    from rehrseg_b200._lib import conv_desc
    n, cin, cout, dhw, k, p = case
    assert Fn._march_route(conv_desc(k, (1, 1, 1), p), cin, cout)
    g = torch.Generator().manual_seed(31)
    x = torch.randn((n, *dhw, cin), generator=g).cuda().to(torch.float16)
    w = (torch.randn((cout, cin, *k), generator=g) / (cin * k[0] * k[1] * k[2]) ** 0.5).cuda()
    xh = Fn.mark_h(x.view(torch.bfloat16))
    y, stats, _ = Fn.conv3d_raw(xh, w, None, k, (1, 1, 1), p, want_stats=True, x_h=True, y_h=True)
    tw = Fn.bf_twin(xh)
    torch.cuda.synchronize()
    ref = F.conv3d(x.float().permute(0, 4, 1, 2, 3), w.to(torch.float16).float(), None, padding=p)
    got = y.view(torch.float16).float().permute(0, 4, 1, 2, 3)
    assert rel_l2(got, ref) < 2e-3, (case, rel_l2(got, ref))
    assert rel_l2(stats.sum(1)[..., 0], ref.sum((2, 3, 4))) < 2e-3     # InstanceNorm partial sums of the epilogue
    assert torch.equal(tw, x.float().to(torch.bfloat16)) and Fn.bf_twin(xh) is tw


@pytest.mark.parametrize("shape,out_d", [((2, 16, 24, 20, 32), 64), ((1, 5, 9, 7, 16), 18), ((1, 1, 8, 8, 8), 4), ((2, 7, 6, 6, 8), 7),
                                         ((1, 6, 5, 5, 8), 1), ((1, 3, 4, 4, 8), 2)])
def test_upsample_linear_d_matches_interpolate(shape, out_d):
    """models/seg_model.py:197-199: F.interpolate(scale_factor=(s, 1, 1), mode='trilinear', align_corners=True) = linear along depth
    only.  Forward against ATen on the same bf16-rounded input (one bf16 rounding of the result), backward against ATen's gradient of
    the same map; up-sampling shapes take the source-centric kernel, the down-sampling ones the output-centric one."""
    from rehrseg_b200 import functional as Fn
    g = torch.Generator().manual_seed(11)
    x = torch.randn(shape, generator=g).to(torch.bfloat16).cuda().requires_grad_(True)        # channels-last [N, D, H, W, C]
    n, d, h, w, c = shape
    y = Fn.upsample_linear_d(x, out_d)
    assert tuple(y.shape) == (n, out_d, h, w, c) and y.dtype == torch.bfloat16
    xr = x.detach().float().permute(0, 4, 1, 2, 3).contiguous().requires_grad_(True)           # NCDHW fp32
    want = F.interpolate(xr, size=(out_d, h, w), mode="trilinear", align_corners=True)
    got = y.detach().float().permute(0, 4, 1, 2, 3)
    assert torch.all((got - want.detach()).abs() <= 1.01 * 2.0 ** -8 * want.detach().abs() + 1e-6)   # half a bf16 ulp of the fp32 result
    if out_d < d:
        return                                           # the reference only up-samples (upscale >= 1): no gradient contract below that
    dy = torch.randn(y.shape, generator=g).to(torch.bfloat16).cuda()
    y.backward(dy)
    want.backward(dy.float().permute(0, 4, 1, 2, 3))
    dgot = x.grad.float().permute(0, 4, 1, 2, 3)
    assert torch.all((dgot - xr.grad).abs() <= 2.0 ** -7 * xr.grad.abs() + 1e-5)
