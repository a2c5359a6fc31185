"""CPU: host-side logic of the product (integer tile / pad / patch math, module trees, state_dict layout) against the
fixtures generated from the reference, and the C-ABI contract (library loads, every declared symbol exported, loud
failure without CUDA).  No GPU compute is called."""
import ctypes
import json
import os

import numpy as np
import pytest
import torch

from rehrseg_b200 import _lib, seg_model as sm, sliding_window as sw, volume_ops as vo

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_library_exports_every_declared_symbol():
    lib = _lib.lib()
    names = _lib.declared_symbols()
    assert len(names) >= 40
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing
    undeclared = [n for n in lib._rehr_signatures if n not in names]
    assert not undeclared, undeclared
    assert lib.rehr_version() == 6
    assert lib.rehr_strerror(-2).decode().startswith("configuration not supported")


def test_no_cpu_fallback():
    m = sm.SegModel(**{**__import__("oracle.seg_model", fromlist=["x"]).plan_kwargs("tiny")})
    with pytest.raises(_lib.RehrError):
        m(torch.zeros(1, 1, 8, 16, 16))
    with pytest.raises(_lib.RehrError):
        vo.rotate_vol_2d(torch.zeros(2, 2, 2), 90)
    with pytest.raises(NotImplementedError):
        vo.rotate_vol_2d(torch.zeros(2, 2, 2), 45)
    assert vo.rotate_vol_2d(torch.zeros(2, 2, 2), 0).shape == (2, 2, 2)  # identity never touches the device
    # the fused loss reductions are CUDA kernels only (the plain-PyTorch mirrors in train_step.py are separate, explicit classes)
    from rehrseg_b200 import loss_ops
    with pytest.raises(_lib.RehrError):
        loss_ops.build_fused_loss(False, 1)(torch.zeros(1, 2, 2, 4, 4), torch.zeros(1, 1, 2, 4, 4))
    with pytest.raises(_lib.RehrError):
        loss_ops.FusedDistiller(4, 4, 0.0, 1.0, 1.0)(torch.zeros(1, 4, 2, 4, 4), torch.zeros(1, 4, 2, 4, 4))


def test_index_math_matches_reference_fixtures():
    with open(os.path.join(G, "index_math.json")) as f:
        idx = json.load(f)
    for c in idx["steps"]:
        assert sw.compute_steps_for_sliding_window(c["image"], c["tile"], c["step"]) == c["out"], c
    for c in idx["n_slicers"]:
        sl = sw._internal_get_sliding_window_slicers(c["image"], patch_size=c["tile"])
        assert len(sl) == c["n"]
        assert [[[s.start, s.stop] for s in t[1:]] for t in sl[:3]] == c["first3"]
    for c in idx["find_integer_p"]:
        p = vo.find_integer_p(c["n"], c["s"])
        assert (p, vo.calc_slices_to_crop(p, c["s"]), vo.ideal_size(c["n"], c["s"]), vo.projected_size(c["n"], 0, c["s"])) == \
               (c["p"], c["crop"], c["ideal"], c["proj0"]), c
    for c in idx["get_pads"]:
        assert list(vo.get_pads(c["target"], c["d"])) == c["out"]
    for c in idx["get_patch"]:
        assert [[s.start, s.stop] for s in vo.get_patch(None, c["center"], c["size"], return_idx=True)] == c["idx"]


def test_sliding_window_edge_cases():
    assert sw.compute_steps_for_sliding_window((16, 16, 16), (16, 16, 16), 0.5) == [[0], [0], [0]]  # image == tile
    with pytest.raises(AssertionError):
        sw.compute_steps_for_sliding_window((8, 16, 16), (16, 16, 16), 0.5)                       # image < tile
    with pytest.raises(AssertionError):
        sw.compute_steps_for_sliding_window((32, 32, 32), (16, 16, 16), 0.0)
    # x-major, z-minor tile order (utils/seg_utils.py:232-234)
    sl = sw._internal_get_sliding_window_slicers((32, 16, 24), patch_size=[16, 16, 16])
    assert [(s[1].start, s[2].start, s[3].start) for s in sl] == [(0, 0, 0), (0, 0, 8), (8, 0, 0), (8, 0, 8), (16, 0, 0), (16, 0, 8)]
    assert len(sw.mirror_axes_combinations()) == 7


def test_pad_helpers_and_crop_roundtrip():
    z = np.load(os.path.join(G, "volume_ops.npz"))
    padded, pads = vo.target_pad(torch.from_numpy(z["pad_in"]), (10, 9, 7), mode="reflect")   # CPU tensor: numpy path
    assert np.array_equal(padded.numpy(), z["pad_out"]) and np.array_equal(np.array(pads), z["pad_pads"])
    assert np.array_equal(vo.crop(padded, pads).numpy(), z["pad_crop"])
    img = np.arange(24.).reshape(2, 3, 4)
    res, slicer = sw.pad_nd_image(img, (5, 4), 'constant', {'value': 0}, True)
    assert res.shape == (2, 5, 4) and np.array_equal(res[slicer], img) and slicer[1] == slice(1, 4)
    t, sl2 = sw.pad_nd_image(torch.from_numpy(img), (7, 9), 'constant', {'value': 0}, True)
    assert t.shape == (2, 7, 9) and torch.equal(t[sl2], torch.from_numpy(img))


def test_state_dict_layout_matches_reference_fixture():
    z = np.load(os.path.join(G, "segmodel_tiny.npz"))
    from oracle import seg_model as ref_seg
    torch.manual_seed(1234)
    m = sm.SegModel(**ref_seg.plan_kwargs("tiny"))
    assert sorted(m.state_dict().keys()) == list(z["keys"])
    # same construction order => same default-init weights as the reference module
    wsum = float(sum(p.detach().double().abs().sum() for p in m.parameters()))
    assert abs(wsum - float(z["weight_abs_sum"])) <= 1e-9 * wsum
    full = sm.plainconv_3d_fullres()
    assert len(full.state_dict()) == 296 and sum(p.numel() for p in full.parameters()) > 31_000_000
    assert 'sr_head' in "".join(n for n, _ in full.named_parameters())


def test_rehr_tensor_descriptor_of_channel_slice():
    buf = torch.zeros((1, 2, 3, 4, 64), dtype=torch.bfloat16)
    a = buf[..., 32:]
    assert _lib.cl_strides_ok(a) and _lib._pitch(a) == 64
    t = _lib.rt(a)
    assert (t.n, t.d, t.h, t.w, t.c, t.ld) == (1, 2, 3, 4, 32, 64) and t.ptr == buf.data_ptr() + 64
    assert not _lib.cl_strides_ok(buf.permute(0, 4, 1, 2, 3))


def test_weight_cache_drops_dead_entries():
    """Backward passes reach their weights through autograd's saved tensors (fresh objects every step): a training loop that never
    calls clear_weight_cache() must not accumulate their packed copies."""
    from rehrseg_b200 import functional as Fn
    Fn.clear_weight_cache()
    keep = []
    for i in range(600):
        w = torch.zeros(1)
        if i % 20 == 0:
            keep.append(w)
        Fn._cache_put((id(w), "dgrad", i), w, torch.zeros(1))
        del w
    live = sum(1 for v in Fn._wcache.values() if v[0]() is not None)
    assert live == len(keep) and len(Fn._wcache) <= 256 + len(keep)
    Fn.clear_weight_cache()


def test_get_random_centers_matches_reference_fixture():
    """utils/patch_ops.py:67-113: same numpy global-stream consumption (randint, per-axis choice, shuffle) and the same gradient
    magnitude marginals -> centre for centre equal to what the reference's own function drew under the same seed."""
    import json
    import numpy as np
    with open(os.path.join(G, "random_centers.json")) as f:
        cases = json.load(f)
    rng = np.random.RandomState(3)
    imgs = [rng.rand(20, 24, 9).astype(np.float32), rng.rand(20, 24, 9).astype(np.float32), rng.rand(18, 22, 9).astype(np.float32)]
    assert len(cases) == 4
    for c in cases:
        np.random.seed(c["seed"])
        got = vo.get_random_centers([im.copy() for im in imgs], tuple(c["patch_size"]), c["n"], c["weighted"])
        assert [[int(i), [int(v) for v in xyz]] for i, xyz in got] == c["centers"]
        ps = c["patch_size"]
        if c["weighted"]:   # no centre within p//2 + 1 of a border of an axis with p > 1
            for i, xyz in got:
                for ax, p in enumerate(ps):
                    if p > 1:
                        assert p // 2 + 1 <= xyz[ax] < imgs[i].shape[ax] - p // 2 - 1


def test_stitched_teacher_features_match_the_reference_loop(monkeypatch):
    """flavr._stitched_features_cl (engine teacher: only the kept depth slices leave the channels-last layout) against the generic loop
    of get_intermediate_features (train_all.py:85-112) on a stand-in encoder, CPU: same windows, same slices, same order."""
    import contextlib
    import torch
    from rehrseg_b200 import flavr

    def fake_encoder(enc, images, n_feats=5):            # NCDHW fp32 -> 5 channels-last "feature maps" that depend on every input slice
        x = images.permute(0, 2, 3, 4, 1)                # [n, 4, H, W, 2]
        f0 = torch.cat([x, x * 2.0 + 1.0], dim=4)
        f1 = (f0[:, :, ::2, ::2] * 3.0 - x.mean(dim=(1, 2, 3, 4), keepdim=True))
        f2 = f1[:, :, ::2, ::2].cumsum(dim=1)
        f3, f4 = f2 * f2, f2.flip(1) - 1.0
        return (f0, f1, f2, f3, f4)[:n_feats]

    class Fake(torch.nn.Module):
        encoder = None

        def forward(self, images, return_inetermediate_feature=False):
            mean_ = images[:, 0:1].mean(2, keepdim=True).mean(3, keepdim=True).mean(4, keepdim=True)
            images[:, 0:1] = images[:, 0:1] - mean_
            return tuple(f.permute(0, 4, 1, 2, 3).contiguous() for f in fake_encoder(None, images))

    monkeypatch.setattr(flavr, "encoder_forward", fake_encoder)
    monkeypatch.setattr(flavr, "device_of", lambda t: contextlib.nullcontext())
    monkeypatch.setattr(flavr.F_, "from_channels_last", lambda t: t.permute(0, 4, 1, 2, 3).contiguous().float())
    g = torch.Generator().manual_seed(7)
    for b, d, max_batch in ((2, 6, 2), (1, 2, 8), (3, 5, 1), (2, 9, 3)):
        img, lab = torch.randn((b, 1, d, 8, 12), generator=g), (torch.rand((b, 1, d, 8, 12), generator=g) > 0.8).float()
        want = flavr.get_intermediate_features(Fake(), img.clone(), lab, max_batch=max_batch)
        inp = torch.cat((img, lab), dim=1)
        win = flavr._windows(inp, 2)
        flat = win.reshape(win.shape[0] * b, *win.shape[2:])
        got = flavr._stitched_features_cl(Fake(), flat, win.shape[0], b, max_batch)
        assert got.keys() == want.keys()
        for k in want:
            assert got[k].shape == want[k].shape and got[k].shape[2] == d and torch.equal(got[k], want[k]), (b, d, max_batch, k)
        # opt-in `keys`: only the requested maps, the same values; the stand-in encoder is asked for no map behind the last one
        for keys in ((1,), (0, 3), (4,)):
            sub = flavr._stitched_features_cl(Fake(), flat, win.shape[0], b, max_batch, keys)
            assert sorted(sub) == sorted(keys) and all(torch.equal(sub[k], want[k]) for k in keys)
            gen = flavr.get_intermediate_features(Fake(), img.clone(), lab, max_batch=max_batch, keys=keys)   # generic (non-engine) path
            assert sorted(gen) == sorted(keys) and all(torch.equal(gen[k], want[k]) for k in keys)
    import pytest
    from rehrseg_b200._lib import RehrError
    with pytest.raises(RehrError):
        flavr._stitched_features_cl(Fake(), flat, win.shape[0], b, max_batch, (5,))


def test_product_package_never_touches_the_oracle_or_the_reference_tree():
    """The oracle is test infrastructure: nothing under rehrseg_b200/ may import it, and nothing there, in bench.py / bench_extras.py
    or in __graft_entry__.py may read /root/reference at run time (it does not exist on the GPU box).  bench.py and smoke() may use
    the oracle, but only as the CPU baseline / the checker."""
    import ast
    import glob
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

    def imported_roots(path):
        with open(path) as f:
            tree = ast.parse(f.read())
        roots = set()
        for node in ast.walk(tree):
            if isinstance(node, ast.Import):
                roots.update(a.name.split(".")[0] for a in node.names)
            elif isinstance(node, ast.ImportFrom) and node.level == 0 and node.module:
                roots.add(node.module.split(".")[0])
        return roots

    for path in glob.glob(os.path.join(root, "rehrseg_b200", "*.py")):
        assert "oracle" not in imported_roots(path), path
    for path in glob.glob(os.path.join(root, "rehrseg_b200", "*.py")) + [os.path.join(root, n) for n in
                                                                          ("bench.py", "bench_extras.py", "__graft_entry__.py")]:
        with open(path) as f:
            for line in f:      # citations in docstrings / messages are fine; path handling is not
                if "/root/reference" in line:
                    assert not any(tok in line for tok in ("open(", "sys.path", "os.path", "listdir", "exists(", "insert(", "import ")), (path, line)
