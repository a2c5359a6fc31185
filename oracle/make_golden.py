"""Generate tests/golden/* FROM THE REFERENCE ITSELF (imported unchanged from /root/reference through oracle/refimport.py).
Runs only in the build container (the GPU box has no /root/reference); the outputs are small and committed, the
script is committed so they can be regenerated:   python -m oracle.make_golden

The reference ships no tests, golden vectors or fixtures (SURVEY.md section 4), so these files -- outputs of the
reference's own functions / modules on seeded synthetic inputs -- are what pins the oracle and the CUDA path.
"""
from __future__ import annotations

import json
import os

import numpy as np
import torch
from torch import nn

from . import refimport
from . import seg_model as ref_seg

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

STEP_CASES = [((256, 256, 256), (128, 128, 128), 0.5), ((160, 512, 512), (128, 128, 128), 0.5), ((20, 455, 633), (14, 320, 384), 0.5),
              ((110, 64, 64), (64, 64, 64), 0.5), ((24, 20, 28), (16, 16, 16), 0.5), ((14, 320, 384), (14, 320, 384), 0.5),
              ((130, 130, 130), (128, 128, 128), 0.25), ((100, 99, 98), (32, 48, 64), 1.0), ((33, 65, 129), (32, 32, 32), 0.75)]
P_CASES = [(n, s) for n in (1, 2, 7, 20, 33, 40, 41, 57, 100, 160) for s in (1.0, 1.5, 2.0, 2.5, 3.2, 4.0, 4.8, 5.3)]
PAD_CASES = [(128, 100), (128, 101), (16, 16), (10, 20), (255, 0), (7, 6), (1000, 1), (33, 32)]
PATCH_CASES = [((10, 12, 5), (4, 6, 1)), ((3, 3, 3), (1, 1, 1)), ((20, 21, 22), (7, 8, 9)), ((5, 5, 0), (3, 3, 1))]


def conv_net(seed=7, half=False):
    torch.manual_seed(seed)
    conv = nn.Conv3d(1, 2, 3, padding=1)
    conv.requires_grad_(False)
    return (lambda x: conv(x).half()) if half else conv, conv


def joint_fixture() -> None:
    """The reference's own Distiller (models/seg_model.py:115-151) and _build_loss (utils/seg_utils.py:355-372) on seeded inputs."""
    sm = refimport.load("models.seg_model")
    seg_utils = refimport.load("utils.seg_utils")
    g = torch.Generator().manual_seed(21)
    fs = torch.randn((2, 64, 3, 12, 10), generator=g, requires_grad=True)
    ft = torch.randn((2, 64, 3, 12, 10), generator=g)
    arrs = {"feat_s": fs.detach().numpy(), "feat_t": ft.numpy()}
    for tag, lam in (("cos_struct", (0.0, 1.0, 1.0)), ("all", (0.5, 1.0, 2.0))):
        torch.manual_seed(77)
        d = sm.Distiller(64, 64, *lam)
        arrs[f"distill_keys"] = np.array(list(d.state_dict().keys()))
        arrs[f"distill_w"], arrs[f"distill_b"] = d.distill.weight.detach().numpy(), d.distill.bias.detach().numpy()
        fs.grad = None
        loss = d(fs, ft)
        loss.backward()
        arrs[f"distill_{tag}_loss"] = loss.detach().numpy()
        arrs[f"distill_{tag}_dfeat"] = fs.grad.numpy().copy()
        arrs[f"distill_{tag}_dw"] = d.distill.weight.grad.numpy().copy()
    logits = torch.randn((2, 2, 3, 8, 8), generator=g, requires_grad=True)
    target = (torch.rand((2, 1, 3, 8, 8), generator=g) > 0.7).float()
    unc = torch.rand((2, 1, 3, 8, 8), generator=g) * 0.99 + 0.01
    arrs.update(logits=logits.detach().numpy(), target=target.numpy(), unc=unc.numpy())
    for tag, wd, u in (("lr_unc", 0, unc), ("hr", 1, None), ("lr_nounc", 1, "omit")):
        obj = seg_utils._build_loss(enable_deep_supervision=False, weight_dice=wd)
        logits.grad = None
        loss = obj(logits, target) if isinstance(u, str) else obj(logits, target, u)
        loss.backward()
        arrs[f"loss_{tag}"] = loss.detach().numpy()
        arrs[f"loss_{tag}_dlogits"] = logits.grad.numpy().copy()
    np.savez_compressed(os.path.join(OUT, "joint_step.npz"), **arrs)


TINY_ANISO = dict(n_stages=3, features_per_stage=[32, 64, 128], kernel_sizes=[[1, 3, 3], [3, 3, 3], [3, 3, 3]],
                  strides=[[1, 1, 1], [1, 2, 2], [1, 2, 2]], n_conv_per_stage=[2] * 3, n_conv_per_stage_decoder=[2] * 2)


def joint_step_fixture() -> None:
    """One whole stage-2 iteration executed with the reference's OWN objects -- SegModel, UNet_3D_3D teacher, Distiller, _build_loss,
    train_all.get_intermediate_features -- following the loop body train_all.py:519-555 line by line (device = cpu, distillation and
    uncertainty on).  Stores the batch, the loss terms and a few gradients; tests/test_joint_cpu.py replays it through
    oracle.joint.ref_joint_step on oracle-built modules with the same default initialisation."""
    sm = refimport.load("models.seg_model")
    fa = refimport.load("models.FLAVR.FLAVR_arch")
    ta = refimport.load("train_all")
    seg_utils = refimport.load("utils.seg_utils")
    kw = ref_seg.plan_kwargs("tiny")
    kw.update(TINY_ANISO)
    torch.manual_seed(1234)
    model_seg = sm.SegModel(**kw)
    torch.manual_seed(1234)
    model_sr = fa.UNet_3D_3D(2, "unet_18", 4, 4, False, "concat", "transpose", use_uncertainty=True).eval()
    torch.manual_seed(5)
    distiller = sm.Distiller(64, 64, 0.0, 1.0, 1.0)
    g = torch.Generator().manual_seed(4)
    img = torch.randn((1, 1, 5, 32, 32), generator=g)
    label_lr = (torch.rand((1, 1, 5, 32, 32), generator=g) > 0.8).float()
    label = (torch.rand((1, 1, 20, 32, 32), generator=g) > 0.8).float()
    uncertainty_lr = torch.rand((1, 1, 5, 32, 32), generator=g) * 0.99 + 0.01
    arrs = {"img": img.numpy().copy(), "label_lr": label_lr.numpy(), "label": label.numpy(), "uncertainty_lr": uncertainty_lr.numpy()}
    device = torch.device("cpu")
    loss_obj_lr_seg = seg_utils._build_loss(enable_deep_supervision=False, weight_dice=0)      # enable_uncertainty = True
    loss_obj_hr_seg = seg_utils._build_loss(enable_deep_supervision=False, weight_dice=1)
    # ---- train_all.py:520-555 ----
    model_seg.train()
    pseudo_img_lr = img.to(device)
    pseudo_label_lr = label_lr.to(device)
    label_sr = label.to(device)
    with torch.no_grad():
        features_sr = ta.get_intermediate_features(model_sr, pseudo_img_lr, pseudo_label_lr, device)
    pseudo_seg_lr, seg_sr, features_seg = model_seg(pseudo_img_lr, return_inetermediate_feature=True)
    pseudo_uncertainty_lr = uncertainty_lr.to(device)
    loss_lr_seg = loss_obj_lr_seg(pseudo_seg_lr, pseudo_label_lr, pseudo_uncertainty_lr)
    loss_hr_seg = loss_obj_hr_seg(seg_sr, label_sr, None)
    loss = loss_lr_seg + loss_hr_seg
    distill_loss = 0
    distill_loss += distiller(features_seg[1], features_sr[1])
    loss += distill_loss
    loss.backward()
    # ------------------------------
    arrs.update(loss=loss.detach().numpy(), loss_lr_seg=loss_lr_seg.detach().numpy(), loss_hr_seg=loss_hr_seg.detach().numpy(),
                distill_loss=distill_loss.detach().numpy(), img_after=pseudo_img_lr.numpy(),
                grad_stem=model_seg.encoder.stages[0][0].convs[0].conv.weight.grad.numpy(),
                grad_sr_head0=model_seg.sr_head[0].weight.grad.numpy(), grad_distill=distiller.distill.weight.grad.numpy(),
                grad_abs_sum=np.array(float(sum(p.grad.double().abs().sum() for p in model_seg.parameters() if p.grad is not None))))
    np.savez_compressed(os.path.join(OUT, "joint_whole_step.npz"), **arrs)


def sr_sweep_fixture() -> None:
    """The reference's own `apply_to_vol_flavr` (utils/sr_utils.py:102-135) on its own UNet_3D_3D (plain head).  The function hard-codes
    `.cuda()` for its zero padding, so `torch.Tensor.cuda` is made the identity while it runs on the CPU; nothing else is touched."""
    fa = refimport.load("models.FLAVR.FLAVR_arch")
    sr_utils = refimport.load("utils.sr_utils")
    torch.manual_seed(1234)
    net = fa.UNet_3D_3D(2, "unet_18", 4, 4, False, "concat", "transpose", use_uncertainty=False).eval()
    g = torch.Generator().manual_seed(6)
    vol = torch.rand((5, 2, 20, 24), generator=g)          # [Z, C, X, Y]: ragged in-plane size -> zero-padded to 32 x 32
    vol[:, 1] = (vol[:, 1] > 0.8).float()
    orig = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        out = sr_utils.apply_to_vol_flavr(net, vol.clone())
    finally:
        torch.Tensor.cuda = orig
    np.savez_compressed(os.path.join(OUT, "sr_sweep.npz"), vol=vol.numpy(), out=out.numpy())


def sr_step_fixture() -> None:
    """ONE iteration of the reference's own `train_all.train_sr` (train_all.py:114-152) on its own UNet_3D_3D, L1Loss and
    BCEDiceLoss(1, 1), for the plain and the UASR head: a one-batch list stands in for the DataLoader, SGD(lr=0) keeps the weights
    so the gradients left in `.grad` belong to the stored loss, and `LossProgBar` is replaced by a recorder (it only displays)."""
    import tempfile
    fa = refimport.load("models.FLAVR.FLAVR_arch")
    ta = refimport.load("train_all")
    seg_utils = refimport.load("utils.seg_utils")
    seen = {}

    class Recorder:
        def __init__(self, *a, **k):
            pass

        def __enter__(self):
            return self

        def __exit__(self, *a):
            return False

        def update(self, d):
            seen["loss"] = float(d["loss"].detach())

    orig = ta.LossProgBar
    ta.LossProgBar = Recorder
    arrs = {}
    try:
        g = torch.Generator().manual_seed(8)
        lr = torch.rand((2, 2, 4, 32, 32), generator=g)
        lr[:, 1] = (lr[:, 1] > 0.8).float()
        hr = torch.rand((2, 2, 16, 32, 32), generator=g)
        hr[:, 1] = (hr[:, 1] > 0.8).float()
        arrs.update(patches_lr=lr.numpy().copy(), patches_hr=hr.numpy().copy())
        for tag, unc in (("plain", False), ("uasr", True)):
            torch.manual_seed(1234)
            net = fa.UNet_3D_3D(2, "unet_18", 4, 4, False, "concat", "transpose", use_uncertainty=unc)
            opt = torch.optim.SGD(net.parameters(), lr=0.0)
            sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda i: 1.0)
            with tempfile.TemporaryDirectory() as wd:
                ta.train_sr(1, 2, net, opt, sched, [(lr.clone(), hr.clone())], torch.device("cpu"), torch.nn.L1Loss(),
                            seg_utils.BCEDiceLoss(alpha=1, beta=1), 1, 4, 4, unc, wd, 1000)
            named = dict(net.named_parameters())
            arrs[f"{tag}_loss"] = np.array(seen["loss"])
            arrs[f"{tag}_grad_stem"] = named["encoder.stem.0.weight"].grad.numpy().copy()
            arrs[f"{tag}_grad_outconv"] = (named["outconv.1.weight"] if not unc else named["uncertainty_out.weight"]).grad.numpy().copy()
            arrs[f"{tag}_grad_abs_sum"] = np.array(float(sum(p.grad.double().abs().sum() for p in net.parameters() if p.grad is not None)))
    finally:
        ta.LossProgBar = orig
    np.savez_compressed(os.path.join(OUT, "sr_step.npz"), **arrs)


def wdsr_fixture() -> None:
    """The reference's own WDSR (models/wdsr.py) with the unavailable third-party `resize` replaced by the identity, which is what
    a resampling factor of 1 (integer scale) amounts to: forward on a seeded input + the gradient of the head for a seeded cotangent."""
    import warnings
    wd = refimport.load("models.wdsr")
    wd.resize = lambda x, factors, order=3: x
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        torch.manual_seed(1234)
        net = wd.WDSR(out_channel=2, n_resblocks=2, num_channels=32, scale=4.0)
    g = torch.Generator().manual_seed(9)
    x = torch.rand((2, 2, 16, 12), generator=g)
    out = net(x)
    cot = torch.randn(out.shape, generator=g)
    (out * cot).sum().backward()
    np.savez_compressed(os.path.join(OUT, "wdsr_small.npz"), x=x.numpy(), out=out.detach().numpy(), cot=cot.numpy(),
                        keys=np.array(list(net.state_dict().keys())), head_v=net.head.weight_v.detach().numpy(),
                        grad_head_g=net.head.weight_g.grad.numpy(), grad_tail_v=net.tail.conv0.weight_v.grad.numpy(),
                        patch=np.array(net.calc_out_patch_size([16, 12])))


def random_centers_fixture() -> None:
    """The reference's own `get_random_centers` (utils/patch_ops.py:67-113) under a fixed `np.random.seed`: images from the legacy
    RandomState(3) stream (stable across numpy versions), so the test can rebuild the inputs and compare centre by centre."""
    patch_ops = refimport.load("utils.patch_ops")
    rng = np.random.RandomState(3)
    imgs = [rng.rand(20, 24, 9).astype(np.float32), rng.rand(20, 24, 9).astype(np.float32), rng.rand(18, 22, 9).astype(np.float32)]
    cases = []
    for weighted in (True, False):
        for ps in ((8, 8, 1), (6, 10, 3)):
            np.random.seed(11)
            c = patch_ops.get_random_centers([im.copy() for im in imgs], ps, 25, weighted)
            cases.append({"weighted": weighted, "patch_size": list(ps), "n": 25, "seed": 11,
                          "centers": [[int(i), [int(v) for v in xyz]] for i, xyz in c]})
    with open(os.path.join(OUT, "random_centers.json"), "w") as f:
        json.dump(cases, f)


def sr_degrade_fixture() -> None:
    """The reference's OWN `TrainSetMultiple.__getitem__` (utils/train_set.py:337-434) and `load_img` pre-filter (:321-333) on a
    seeded synthetic volume, with the third-party `resize` replaced by the stand-in oracle/degrade.py defines (its source is not
    available; everything around it is the reference's code).  The dataset object is built without `__init__` (which reads NIfTI /
    HDF5 files through packages the image does not have): `__getitem__` only reads the attributes set below.  Python's `random`
    is seeded per case; the case list covers both transposition branches, both zero-slice branches, all flips and the final
    permutation, a patch larger than the volume (padding) and a non-integer slice separation."""
    import random
    from . import degrade as od
    refimport.install()
    import importlib
    importlib.import_module("resize.pytorch").resize = od.resize_standin
    train_set = refimport.load("utils.train_set")
    train_set.resize = od.resize_standin            # (the module did `from resize.pytorch import resize` at import time)
    rng = np.random.RandomState(21)
    X, Y, Z = 40, 36, 24
    img = rng.rand(X, Y, Z, 1).astype(np.float32)
    lab = (rng.rand(X, Y, Z, 1) > 0.7).astype(np.uint8)
    taps = np.exp(-0.5 * ((np.arange(9.0) - 4) / (3.873 / 2.355)) ** 2)
    kernel = torch.tensor(taps / taps.sum(), dtype=torch.float32).reshape(1, 1, 9, 1)
    image = np.concatenate([img, lab.astype(np.float32)], axis=-1)
    fx, fy = od.blur_prefilter(image, kernel)
    out = {"img": img, "lab": lab, "kernel": kernel.numpy(), "filtered_x": fx, "filtered_y": fy}
    cases = []
    configs = [((32, 32, 1), 4.0, True, True), ((16, 20, 3), 4.0, True, True), ((48, 32, 1), 4.0, True, False),
               ((32, 32, 1), 3.2, True, True), ((24, 24, 1), 4.0, False, True)]
    for ci, (ps, sep, blur, flip) in enumerate(configs):
        ds = object.__new__(train_set.TrainSetMultiple)
        ds.imgs_hr, ds.labels_hr = [img], [lab]
        ds.imgs_filtered_x, ds.imgs_filtered_y = [fx], [fy]
        ds.blur, ds.slice_separation, ds.patch_size = blur, sep, list(ps)
        ds.train_transform, ds.random_flip = None, flip
        for seed in range(8):
            random.seed(1000 * ci + seed)
            lr, hr = ds.__getitem__(0)
            key = f"c{ci}_s{seed}"
            out[key + "_lr"], out[key + "_hr"] = lr.numpy(), hr.numpy()
            cases.append({"key": key, "patch_size": list(ps), "slice_separation": sep, "blur": blur, "random_flip": flip,
                          "seed": 1000 * ci + seed})
    out["cases"] = np.frombuffer(json.dumps(cases).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, "sr_degrade.npz"), **out)


def spatial_aug_fixture() -> None:
    """The reference's OWN `augment_spatial` (utils/seg_utils.py:378-480) in the dummy-2D stage-2 configuration, with the
    batchgenerators helpers it imports replaced by the restatements of oracle/augment.py (the package is not installed) and
    scipy's real map_coordinates; `np.random` seeded per case.  Cases: the configured probabilities (0.2 / 0.2), forced rotation,
    forced scaling, both; a patch equal to and smaller than the image."""
    from . import augment as oa
    seg_utils = refimport.load("utils.seg_utils")
    for name in ("create_zero_centered_coordinate_mesh", "rotate_coords_2d", "rotate_coords_3d", "scale_coords", "interpolate_img",
                 "elastic_deform_coordinates"):
        setattr(seg_utils, name, getattr(oa, name))
    rng = np.random.RandomState(5)
    b, cz, X, Y = 2, 3, 28, 24
    data = rng.randn(b, cz, X, Y).astype(np.float32)
    blobs = rng.rand(b, 4 * cz, X, Y) > 0.6
    seg_sr = blobs.astype(np.float32)
    seg = seg_sr[:, ::4].copy()
    unc = (1 - rng.rand(b, cz, X, Y) * 0.99).astype(np.float32)
    out = {"data": data, "seg": seg, "seg_sr": seg_sr, "uncertainty": unc}
    cases = []
    configs = [((28, 24), 0.2, 0.2), ((28, 24), 1.0, 0.0), ((28, 24), 0.0, 1.0), ((20, 16), 1.0, 1.0), ((25, 24), 0.2, 0.2)]
    for ci, (ps, p_rot, p_scale) in enumerate(configs):
        for seed in range(3):
            np.random.seed(100 * ci + seed)
            d, segs = seg_utils.augment_spatial(data.copy(), [seg.copy(), seg_sr.copy(), unc.copy()], patch_size=ps,
                                                patch_center_dist_from_border=None, do_elastic_deform=False, alpha=(0, 0), sigma=(0, 0),
                                                do_rotation=True, angle_x=(-np.pi, np.pi), angle_y=(0, 0), angle_z=(0, 0),
                                                do_scale=True, scale=(0.7, 1.4), border_mode_data="constant", border_cval_data=0,
                                                order_data=3, border_mode_seg="constant", border_cval_seg=-1, order_seg=1,
                                                random_crop=False, p_el_per_sample=0, p_scale_per_sample=p_scale,
                                                p_rot_per_sample=p_rot, independent_scale_for_each_axis=False, p_rot_per_axis=1,
                                                enable_uncertainty=True)
            key = f"c{ci}_s{seed}"
            out[key + "_data"] = d
            for name, v in zip(("seg", "seg_sr", "uncertainty"), segs):
                out[key + "_" + name] = v
            cases.append({"key": key, "patch_size": list(ps), "p_rot": p_rot, "p_scale": p_scale, "seed": 100 * ci + seed})
    out["cases"] = np.frombuffer(json.dumps(cases).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, "spatial_aug.npz"), **out)


def stage2_sample_fixture() -> None:
    """The reference's OWN `TrainSetMultipleSegSREfficient.__getitem__` (utils/train_set.py:102-159) on a seeded synthetic subject.
    The dataset object is built without `__init__` (it reads HDF5 files); `train_transform` is the spatial part of what
    `get_training_transforms` composes (:652-676): the dummy-2D reshapes (nnunetv2, restated), the reference's OWN
    `MySpatialTransform` instance with the arguments of :660-673, and the float-tensor conversion -- the intensity transforms
    that follow are batchgenerators classes the image does not have."""
    import random
    from . import augment as oa
    seg_utils = refimport.load("utils.seg_utils")
    for name in ("create_zero_centered_coordinate_mesh", "rotate_coords_2d", "rotate_coords_3d", "scale_coords", "interpolate_img",
                 "elastic_deform_coordinates"):
        setattr(seg_utils, name, getattr(oa, name))
    train_set = refimport.load("utils.train_set")
    rng = np.random.RandomState(8)
    X, Y, Z, sep = 36, 30, 20, 4
    img = (rng.rand(X, Y, Z) * 300).astype(np.float32)
    lab = (rng.rand(X, Y, Z) > 0.6).astype(np.uint8)
    unc = (rng.rand(X, Y, Z) * 255).astype(np.uint8)
    out = {"img": img, "lab": lab, "unc": unc}
    cases = []
    for ci, (ps, p_rot, p_scale) in enumerate([((32, 24, 3), 0.2, 0.2), ((32, 24, 3), 1.0, 1.0), ((40, 24, 2), 1.0, 0.0)]):
        patch_zyx = (ps[2], ps[1], ps[0])        # target_patch_size[::-1] of utils/train_set.py:77
        mst = seg_utils.MySpatialTransform(
            patch_zyx[1:], patch_center_dist_from_border=None, do_elastic_deform=False, alpha=(0, 0), sigma=(0, 0), do_rotation=True,
            angle_x=(-np.pi, np.pi), angle_y=(0, 0), angle_z=(0, 0), p_rot_per_axis=1, do_scale=True, scale=(0.7, 1.4),
            border_mode_data="constant", border_cval_data=0, order_data=3, border_mode_seg="constant", border_cval_seg=-1, order_seg=1,
            random_crop=False, label_key=["seg", "seg_sr", "uncertainty"], p_el_per_sample=0, p_scale_per_sample=p_scale,
            p_rot_per_sample=p_rot, independent_scale_for_each_axis=False, enable_uncertainty=True)

        def transform(**dd):
            shapes = {}
            for k in list(dd):
                dd[k], shapes[k] = oa.convert_3d_to_2d(dd[k])
            dd = mst(**dd)
            return {k: torch.from_numpy(np.ascontiguousarray(oa.convert_2d_to_3d(v, shapes[k]))).float() for k, v in dd.items()}

        class H5Like:          # an h5py dataset: `d[:]` reads a FRESH array (the reference normalises what it reads in place)
            def __init__(self, a):
                self.a = a

            def __getitem__(self, k):
                return self.a[k].copy()

        ds = object.__new__(train_set.TrainSetMultipleSegSREfficient)
        ds.imgs, ds.labels, ds.uncertainties = [H5Like(img)], [H5Like(lab)], [H5Like(unc)]
        ds.norm, ds.patch_size, ds.separation, ds.uncertainty, ds.random_flip = True, list(ps), sep, True, True
        ds.train_transform = transform
        for seed in range(4):
            random.seed(50 * ci + seed)
            np.random.seed(50 * ci + seed)
            res = ds.__getitem__(0)
            key = f"c{ci}_s{seed}"
            for name, v in zip(("img", "label_lr", "label", "uncertainty_lr"), res):
                out[key + "_" + name] = v.numpy()
            cases.append({"key": key, "patch_size": list(ps), "separation": sep, "p_rot": p_rot, "p_scale": p_scale, "seed": 50 * ci + seed})
    out["cases"] = np.frombuffer(json.dumps(cases).encode(), dtype=np.uint8)
    np.savez_compressed(os.path.join(OUT, "stage2_sample.npz"), **out)


FBA_PS = ("infinity", "inf", 0.5, 2, "3")


def reference_helpers_fixture() -> None:
    """The reference's find_integer_p / projected_size / get_pads / compute_steps_for_sliding_window over the ranges
    tests/test_oracle_vs_reference.py sweeps, and rotate_vol_2d / fba on its seeded arrays -> tests/golden/reference_helpers.json
    + .npz, which that test compares against wherever no reference checkout is present.  The committed files were recorded
    through the oracle restatements (oracle/volume.py), which the live comparison had found bit-identical to the reference
    on every one of these inputs; with a checkout, this function records them from the reference itself."""
    po, pad, su = refimport.load("utils.patch_ops"), refimport.load("utils.pad"), refimport.load("utils.seg_utils")
    rot, fb = refimport.load("utils.rotate"), refimport.load("utils.fba")
    cases = {"find_integer_p": [], "get_pads": [], "steps": []}
    for n in range(1, 70):
        for s in (1.0, 1.25, 1.5, 2.0, 2.4, 3.0, 3.2, 4.0, 4.5, 6.0):
            cases["find_integer_p"].append([n, s, po.find_integer_p(n, s), po.projected_size(n, 3, s)])
    for t in range(0, 40):
        for d in range(0, 40):
            cases["get_pads"].append([t, d, *pad.get_pads(t, d)])
    rng = np.random.default_rng(0)
    for _ in range(200):
        tile = [int(v) for v in rng.integers(4, 40, 3)]
        img = [t + int(v) for t, v in zip(tile, rng.integers(0, 90, 3))]
        step = float(rng.choice([0.25, 0.5, 0.75, 1.0]))
        cases["steps"].append([img, tile, step, su.compute_steps_for_sliding_window(img, tile, step)])
    with open(os.path.join(OUT, "reference_helpers.json"), "w") as f:
        json.dump(cases, f)
    g = torch.Generator().manual_seed(3)
    v = torch.randn((4, 6, 5), generator=g)
    arrs = {"rot_in": v.numpy()}
    for a in (0, 90, -90, 180, -180, 270, -270, 360):
        arrs[f"rot_{a}"] = rot.rotate_vol_2d(v, a).contiguous().numpy()
    vols = [torch.randn((8, 6, 10), generator=g).numpy() for _ in range(4)]
    arrs["fba_in"] = np.stack(vols)
    for p in FBA_PS:
        arrs[f"fba_{p}"] = fb.fba(vols, p)
    np.savez_compressed(os.path.join(OUT, "reference_helpers.npz"), **arrs)


def main() -> None:
    os.makedirs(OUT, exist_ok=True)
    import sys
    if "--only-helpers" in sys.argv:
        reference_helpers_fixture()
        return
    if "--only-stage2" in sys.argv:
        stage2_sample_fixture()
        return
    if "--only-spatial" in sys.argv:
        spatial_aug_fixture()
        return
    if "--only-degrade" in sys.argv:
        sr_degrade_fixture()
        return
    if "--only-centers" in sys.argv:
        random_centers_fixture()
        return
    if "--only-wdsr" in sys.argv:
        wdsr_fixture()
        return
    if "--only-joint" in sys.argv:
        joint_fixture()
        joint_step_fixture()
        return
    if "--only-sweep" in sys.argv:
        sr_sweep_fixture()
        return
    if "--only-sr-step" in sys.argv:
        sr_step_fixture()
        return
    seg_utils = refimport.load("utils.seg_utils")
    patch_ops = refimport.load("utils.patch_ops")
    pad = refimport.load("utils.pad")
    rot = refimport.load("utils.rotate")
    fba = refimport.load("utils.fba")

    # ---- integer index math -------------------------------------------------------------------------------
    idx = {
        "steps": [{"image": list(i), "tile": list(t), "step": s, "out": seg_utils.compute_steps_for_sliding_window(i, t, s)}
                  for i, t, s in STEP_CASES],
        "n_slicers": [{"image": list(i), "tile": list(t),
                       "n": len(seg_utils._internal_get_sliding_window_slicers(i, patch_size=list(t))),
                       "first3": [[[sl.start, sl.stop] for sl in s[1:]] for s in
                                  seg_utils._internal_get_sliding_window_slicers(i, patch_size=list(t))[:3]]}
                      for i, t, _ in STEP_CASES],
        "find_integer_p": [{"n": n, "s": s, "p": patch_ops.find_integer_p(n, s),
                            "crop": patch_ops.calc_slices_to_crop(patch_ops.find_integer_p(n, s), s),
                            "ideal": patch_ops.ideal_size(n, s), "proj0": patch_ops.projected_size(n, 0, s)} for n, s in P_CASES],
        "get_pads": [{"target": t, "d": d, "out": list(pad.get_pads(t, d))} for t, d in PAD_CASES],
        "get_patch": [{"center": list(c), "size": list(p),
                       "idx": [[sl.start, sl.stop] for sl in patch_ops.get_patch(None, c, p, return_idx=True)]} for c, p in PATCH_CASES],
    }
    with open(os.path.join(OUT, "index_math.json"), "w") as f:
        json.dump(idx, f, indent=1)

    # ---- rotate / pad / fba ---------------------------------------------------------------------------------
    g = torch.Generator().manual_seed(11)
    vol = torch.randn((5, 7, 3, 2), generator=g)
    arrs = {"rot_in": vol.numpy()}
    for a in (0, 90, -90, 180, -180, 270, -270, 360):
        arrs[f"rot_{a}"] = rot.rotate_vol_2d(vol, a).contiguous().numpy()
    img = torch.randn((6, 9, 4), generator=g)
    padded, pads = pad.target_pad(img, (10, 9, 7), mode="reflect")
    arrs.update(pad_in=img.numpy(), pad_out=padded.numpy(), pad_pads=np.array(pads), pad_crop=pad.crop(padded, pads).numpy())
    vols = [torch.randn((12, 10, 8), generator=g).numpy() for _ in range(3)]
    vols_odd = [torch.randn((6, 5, 9), generator=g).numpy() for _ in range(2)]
    arrs.update(fba_in=np.stack(vols), fba_inf=fba.fba(vols, "infinity"), fba_p2=fba.fba(vols, 2), fba_p0=fba.fba(vols, 0),
                fba_odd_in=np.stack(vols_odd), fba_odd_inf=fba.fba(vols_odd, "inf"), fba_odd_p1=fba.fba(vols_odd, "1"))
    np.savez_compressed(os.path.join(OUT, "volume_ops.npz"), **arrs)

    # ---- sliding-window blend (reference function, CPU results device) --------------------------------------
    data = torch.randn((1, 24, 20, 28), generator=g)
    sw = {"data": data.numpy()}
    for half in (False, True):
        net, conv = conv_net(7, half)
        sw["conv_w"], sw["conv_b"] = conv.weight.numpy(), conv.bias.numpy()
        for gauss in (False, True):
            patch = [16, 16, 16]
            slicers = seg_utils._internal_get_sliding_window_slicers(data.shape[1:], patch_size=patch)
            out = seg_utils._internal_predict_sliding_window_return_logits(data.clone(), slicers, net, do_on_device=False, out_idx=None,
                                                                           slice_seperation=1, patch_size=patch, use_gaussian=gauss,
                                                                           deep_supervision=False)
            sw[f"logits_half{int(half)}_gauss{int(gauss)}"] = out.numpy()
    sw["gaussian_16"] = seg_utils.compute_gaussian((16, 16, 16), sigma_scale=1. / 8, value_scaling_factor=10, device=torch.device("cpu")).numpy()
    sw["gaussian_128_zero_count_before_fix"] = np.array(0)
    np.savez_compressed(os.path.join(OUT, "sliding_window.npz"), **sw)

    # ---- the reference's own SegModel (with the third-party shims) -----------------------------------------
    sm = refimport.load("models.seg_model")
    kw = ref_seg.plan_kwargs("tiny")
    torch.manual_seed(1234)
    model = sm.SegModel(**kw)
    model.eval()
    x = torch.randn((1, 1, 8, 16, 16), generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        out, up, skips = model(x, return_inetermediate_feature=True)
    wsum = float(sum(p.double().abs().sum() for p in model.parameters()))
    np.savez_compressed(os.path.join(OUT, "segmodel_tiny.npz"), x=x.numpy(), out=out.numpy(), up=up.numpy(), skip1=skips[1].numpy(),
                        weight_abs_sum=np.array(wsum), n_keys=np.array(len(model.state_dict())),
                        keys=np.array(sorted(model.state_dict().keys())))
    # ---- the reference's own FLAVR UNet_3D_3D (both heads) and train_all.get_intermediate_features ----------
    fa = refimport.load("models.FLAVR.FLAVR_arch")
    fl = {}
    xf = torch.rand((1, 2, 4, 32, 32), generator=torch.Generator().manual_seed(2))
    xf[:, 1] = (xf[:, 1] > 0.8).float()
    fl["x"] = xf.numpy()
    for unc in (False, True):
        torch.manual_seed(1234)
        net = fa.UNet_3D_3D(2, "unet_18", 4, 4, False, "concat", "transpose", use_uncertainty=unc)
        net.eval()
        tag = "uasr" if unc else "plain"
        fl[f"{tag}_weight_abs_sum"] = np.array(float(sum(p.detach().double().abs().sum() for p in net.parameters())))
        fl[f"{tag}_keys"] = np.array(list(net.state_dict().keys()))
        with torch.no_grad():
            xin = xf.clone()
            out = net(xin)
            feats = net(xf.clone(), return_inetermediate_feature=True)
        fl[f"{tag}_x_after"] = xin.numpy()            # the forward mutates its input in place
        if unc:
            fl["uasr_out"], fl["uasr_unc"] = out[0].numpy(), out[1].numpy()
        else:
            fl["plain_out"] = out.numpy()
            fl["plain_x1"], fl["plain_x4"] = feats[1].numpy(), feats[4].numpy()
    ta = refimport.load("train_all")
    torch.manual_seed(1234)
    teacher = fa.UNet_3D_3D(2, "unet_18", 4, 4, False, "concat", "transpose", use_uncertainty=True).eval()
    g2 = torch.Generator().manual_seed(4)
    img = torch.randn((1, 1, 5, 32, 32), generator=g2)
    lab = (torch.rand((1, 1, 5, 32, 32), generator=g2) > 0.8).float()
    fl["gif_img"], fl["gif_lab"] = img.numpy(), lab.numpy()
    with torch.no_grad():
        img_in = img.clone()
        feats = ta.get_intermediate_features(teacher, img_in, lab, torch.device("cpu"))
    fl["gif_img_after"] = img_in.numpy()               # zscore_normalization mutates the caller's tensor
    fl["gif_f1"], fl["gif_f3"] = feats[1].numpy(), feats[3].numpy()
    np.savez_compressed(os.path.join(OUT, "flavr_small.npz"), **fl)

    joint_fixture()
    joint_step_fixture()
    sr_sweep_fixture()
    sr_step_fixture()
    random_centers_fixture()
    wdsr_fixture()
    sr_degrade_fixture()
    spatial_aug_fixture()
    stage2_sample_fixture()
    reference_helpers_fixture()
    print("golden fixtures written to", OUT, {k: os.path.getsize(os.path.join(OUT, k)) for k in sorted(os.listdir(OUT))})


if __name__ == "__main__":
    main()
