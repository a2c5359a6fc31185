"""B200-native `SegModel` (nnU-Net PlainConvUNet + HR "SR head"), drop-in for the reference's
models/seg_model.py:153-210.

Two ways in:

* ``SegModel(...)`` -- same constructor signature, same module tree and therefore the same ``state_dict`` keys /
  shapes as the reference (``encoder.stages.S.0.convs.I.{conv,norm,all_modules.*}``, ``decoder.encoder.*`` aliases,
  ``decoder.{stages,transpconvs,seg_layers}``, ``sr_head.{0,2}``), without needing the third-party
  ``dynamic_network_architectures`` package (the reference imports it at models/seg_model.py:9-10).
* ``convert(model)`` -- takes an already-built reference ``SegModel`` (or any PlainConvUNet-shaped module tree) and
  re-routes its ``forward`` through the sm_100a engine, keeping every ``nn.Parameter`` object, so optimisers,
  ``load_state_dict`` (train_all.py:496-499) and ``torch.save(model.state_dict())`` (train_all.py:566-573) run
  unchanged.

The forward runs entirely in channels-last bf16 through rehrseg_b200.functional (tcgen05 implicit-GEMM convs with
fused InstanceNorm statistics, HBM kernels for normalise+LeakyReLU); there is no PyTorch fallback.
"""
from __future__ import annotations

from typing import List, Sequence, Union

import torch
import torch.nn as nn

from . import functional as F_
from ._lib import ACT_LRELU, ACT_NONE, ACT_RELU, RehrError, device_of

# ----------------------------------------------------------------------------------------------------------------
# generic "run this module tree on the engine" helpers (work on the reference's modules and on ours)
# ----------------------------------------------------------------------------------------------------------------


def _triple(v) -> tuple:
    if isinstance(v, int):
        return (v, v, v)
    v = tuple(int(i) for i in v)
    if len(v) == 2:  # Conv2d seen as D=1
        return (1,) + v
    return v


def _check_conv(conv: nn.Module) -> None:
    if getattr(conv, "groups", 1) != 1 or any(d != 1 for d in _triple(getattr(conv, "dilation", 1))):
        raise RehrError("grouped / dilated convolutions are not on the REHRSeg hot path and are not implemented")
    if getattr(conv, "padding_mode", "zeros") != "zeros":
        raise RehrError("only zero padding is implemented in the conv engine")


def _act_of(nonlin) -> tuple:
    """(act, slope) of an nn activation module; slope=1 <=> identity for the fused InstanceNorm apply."""
    if nonlin is None:
        return ACT_NONE, 1.0
    if isinstance(nonlin, nn.LeakyReLU):
        return ACT_LRELU, float(nonlin.negative_slope)
    if isinstance(nonlin, nn.ReLU):
        return ACT_RELU, 0.0
    raise RehrError(f"activation {type(nonlin).__name__} is not implemented")


def run_conv_block(block: nn.Module, x: torch.Tensor, first: bool = False, cat_room: bool = False) -> torch.Tensor:
    """One ConvDropoutNormReLU (conv -> [norm] -> [nonlin]).  `first`: x is the caller's NCDHW fp32 input.
    `cat_room`: produce the activation inside a 2C-channel buffer so the decoder can concatenate without a copy."""
    conv, norm, nonlin = block.conv, getattr(block, "norm", None), getattr(block, "nonlin", None)
    if getattr(block, "dropout", None) is not None:
        raise RehrError("dropout_op is None in the reference configuration (train_all.py:487-488); not implemented")
    _check_conv(conv)
    k, s, p = _triple(conv.kernel_size), _triple(conv.stride), _triple(conv.padding)
    act, slope = _act_of(nonlin)
    small = first and conv.in_channels <= 4
    if first and not small:
        x = F_.to_channels_last(x)
    if norm is not None:
        if not isinstance(norm, (nn.InstanceNorm3d, nn.InstanceNorm2d)) or norm.track_running_stats:
            raise RehrError("only InstanceNorm (no running stats) is implemented (train_all.py:485-486)")
        if act == ACT_RELU:
            slope = 0.0
        with F_.range_owner(block):
            return F_.conv_norm_act(x, conv.weight, conv.bias, norm.weight, norm.bias, k, s, p, eps=norm.eps, slope=slope,
                                    small_cin=small, cat_room=cat_room)
    if small:
        raise RehrError("small-Cin stem without InstanceNorm: use rehrseg_b200.flavr for the FLAVR stem")
    return F_.conv_act(x, conv.weight, conv.bias, k, s, p, act=act, slope=slope)


def run_stacked(blocks: nn.Module, x: torch.Tensor, first: bool = False, cat_room: bool = False) -> torch.Tensor:
    """StackedConvBlocks (has .convs) or an nn.Sequential wrapping one."""
    if hasattr(blocks, "convs"):
        last = len(blocks.convs) - 1
        for i, b in enumerate(blocks.convs):
            x = run_conv_block(b, x, first=first and i == 0, cat_room=cat_room and i == last)
        return x
    if isinstance(blocks, nn.Sequential):
        last = len(blocks) - 1
        for i, m in enumerate(blocks):
            x = run_stacked(m, x, first=first and i == 0, cat_room=cat_room and i == last)
        return x
    raise RehrError(f"unexpected module {type(blocks).__name__} in a PlainConvUNet stage (pooling variants are not "
                    "used by the reference, which builds pool='conv')")


def encoder_forward(encoder: nn.Module, x: torch.Tensor) -> List[torch.Tensor]:
    skips = []
    n = len(encoder.stages)
    for s, stage in enumerate(encoder.stages):
        # every stage output but the bottleneck is later concatenated with an up-sampled tensor of the same width
        x = run_stacked(stage, x, first=(s == 0), cat_room=(s < n - 1))
        skips.append(x)
    return skips


def run_transpconv(tc: nn.ConvTranspose3d, x: torch.Tensor, skip: torch.Tensor = None) -> torch.Tensor:
    """ConvTranspose3d; with `skip` returns torch.cat((up, skip), channel) (models/seg_model.py:36-37)."""
    _check_conv(tc)
    if any(o != 0 for o in _triple(tc.output_padding)):
        raise RehrError("output_padding is not implemented")
    k, s, p = _triple(tc.kernel_size), _triple(tc.stride), _triple(tc.padding)
    if skip is None:
        with F_.range_owner(tc):
            return F_.conv_transpose(x, tc.weight, tc.bias, k, s, p)
    room = F_.concat_room_of(skip)
    if room is not None and room == (2 * tc.out_channels, tc.out_channels):
        with F_.range_owner(tc):
            return F_.conv_transpose(x, tc.weight, tc.bias, k, s, p, skip=skip)
    # no concat room (a caller-built skip): plain copy; fp16 payloads concatenate bit-wise, their bf16 twins likewise
    with F_.range_owner(tc):
        up = F_.conv_transpose(x, tc.weight, tc.bias, k, s, p)
    if F_.is_h(up) != F_.is_h(skip):
        raise RehrError("run_transpconv: up-sampled tensor and skip use different 16-bit storage formats")
    cat = torch.cat((up, skip), dim=4)
    if F_.is_h(up):
        tu, ts = getattr(up, "_rehr_bf", None), getattr(skip, "_rehr_bf", None)
        F_.mark_h(cat, torch.cat((tu, ts), dim=4) if tu is not None and ts is not None else None)
    return cat


def decoder_forward(decoder: nn.Module, skips: Sequence[torch.Tensor]):
    """MyUnetDecoder.forward (models/seg_model.py:26-58) on channels-last skips."""
    lres = skips[-1]
    seg_outputs = []
    features = []
    n = len(decoder.stages)
    for s in range(n):
        x = run_transpconv(decoder.transpconvs[s], lres, skip=skips[-(s + 2)])  # [up | skip], seg_model.py:36-37
        x = run_stacked(decoder.stages[s], x)
        if getattr(decoder, "deep_features", False) and s == n - 1:
            features = x
        if decoder.deep_supervision:
            seg_outputs.append(_seg_layer(decoder.seg_layers[s], x))
        elif s == n - 1:
            seg_outputs.append(_seg_layer(decoder.seg_layers[-1], x))
        lres = x
    seg_outputs = seg_outputs[::-1]
    r = seg_outputs if decoder.deep_supervision else seg_outputs[0]
    if getattr(decoder, "deep_features", False):
        return r, features
    return r


def _seg_layer(layer: nn.Module, x: torch.Tensor) -> torch.Tensor:
    _check_conv(layer)
    if _triple(layer.kernel_size) != (1, 1, 1) or _triple(layer.stride) != (1, 1, 1):
        raise RehrError("seg layers are 1x1x1 convolutions in the reference decoder")
    return F_.seg_head(x, layer.weight, layer.bias)


def sr_head_forward(sr_head: nn.Sequential, features: torch.Tensor, upscale: int) -> torch.Tensor:
    """F.interpolate(features, (upscale,1,1), trilinear, align_corners=True) -> sr_head (models/seg_model.py:204-205)."""
    with F_.range_owner(sr_head):
        x = F_.upsample_linear_d(features, int(features.shape[1] * upscale))
    mods = list(sr_head)
    i = 0
    while i < len(mods):
        conv = mods[i]
        if not isinstance(conv, nn.Conv3d):
            raise RehrError("sr_head is Conv3d/ReLU/Conv3d in the reference (models/seg_model.py:197-199)")
        _check_conv(conv)
        act, slope = ACT_NONE, 0.0
        if i + 1 < len(mods) and not isinstance(mods[i + 1], nn.Conv3d):
            act, slope = _act_of(mods[i + 1])
            i += 1
        last = i == len(mods) - 1
        x = F_.conv_act(x, conv.weight, conv.bias, _triple(conv.kernel_size), _triple(conv.stride), _triple(conv.padding),
                        act=act, slope=slope, out_f32=last)
        i += 1
    return x.permute(0, 4, 1, 2, 3)  # NCDHW view of the fp32 NDHWC logits


class LazyNCDHW(Sequence):
    """`skips` as the reference returns them (NCDHW fp32, models/seg_model.py:207-208), converted on first access so that
    a caller that only reads skips[1] (train_all.py:550) pays for one tensor."""

    def __init__(self, cl: Sequence[torch.Tensor]):
        self._cl = list(cl)
        self._cache = {}

    def __len__(self):
        return len(self._cl)

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(len(self)))]
        i = range(len(self._cl))[i]
        if i not in self._cache:
            self._cache[i] = F_.from_channels_last(self._cl[i])
        return self._cache[i]

    def channels_last(self, i) -> torch.Tensor:
        return self._cl[i]


def segmodel_forward(model: nn.Module, x: torch.Tensor, return_inetermediate_feature: bool = False, want_hr: bool = True):
    """SegModel.forward (models/seg_model.py:201-210); the kwarg spelling is the reference's.  `want_hr=False` (not in the
    reference, whose forward has no switch) skips the x`upscale` SR head and returns None in its place: the LR logits do
    not depend on it, and the sliding-window evaluation only reads output 0 (utils/seg_utils.py:753)."""
    if not x.is_cuda:
        raise RehrError("rehrseg_b200 runs on CUDA (sm_100a) only; there is no CPU path")
    with device_of(x):
        skips = encoder_forward(model.encoder, x)
        out, features = decoder_forward(model.decoder, skips)
        out_up = sr_head_forward(model.sr_head, features, model.upscale) if want_hr else None
    if return_inetermediate_feature:
        return out, out_up, LazyNCDHW(skips)
    return out, out_up


class LRHeadOnly(nn.Module):
    """View of a SegModel whose forward skips the SR head: returns (out, None).  Used by the sliding-window driver when only
    output 0 is consumed."""

    def __init__(self, model: nn.Module):
        super().__init__()
        self.model = model

    @property
    def decoder(self):
        return self.model.decoder

    def forward(self, x):
        return segmodel_forward(self.model, x, want_hr=False)


class _EngineForward:
    """Mixin placed in front of a reference SegModel's class by convert()."""

    def forward(self, x, return_inetermediate_feature=False):  # noqa: D401
        return segmodel_forward(self, x, return_inetermediate_feature)


def convert(model: nn.Module) -> nn.Module:
    """Route `model.forward` through the sm_100a engine in place; parameters, buffers and state_dict are untouched."""
    for attr in ("encoder", "decoder", "sr_head", "upscale"):
        if not hasattr(model, attr):
            raise RehrError(f"convert(): {type(model).__name__} has no .{attr}; expected the reference SegModel")
    if isinstance(model, _EngineForward):
        return model
    cls = model.__class__
    model.__class__ = type("B200" + cls.__name__, (_EngineForward, cls), {})
    return model


# ----------------------------------------------------------------------------------------------------------------
# stand-alone module tree with the reference's state_dict layout
# ----------------------------------------------------------------------------------------------------------------
def _maybe_list(v, n):
    return [v] * n if isinstance(v, int) else list(v)


class ConvDropoutNormReLU(nn.Module):
    def __init__(self, conv_op, cin, cout, kernel_size, stride, conv_bias, norm_op, norm_op_kwargs, dropout_op,
                 dropout_op_kwargs, nonlin, nonlin_kwargs):
        super().__init__()
        if dropout_op is not None:
            raise RehrError("dropout_op must be None (train_all.py:487)")
        dim = 3 if conv_op is nn.Conv3d else 2
        kernel_size = _maybe_list(kernel_size, dim)
        stride = _maybe_list(stride, dim)
        self.stride = stride
        ops = []
        self.conv = conv_op(cin, cout, kernel_size, stride, padding=[(k - 1) // 2 for k in kernel_size], dilation=1,
                            bias=conv_bias)
        ops.append(self.conv)
        if norm_op is not None:
            self.norm = norm_op(cout, **(norm_op_kwargs or {}))
            ops.append(self.norm)
        if nonlin is not None:
            self.nonlin = nonlin(**(nonlin_kwargs or {}))
            ops.append(self.nonlin)
        self.all_modules = nn.Sequential(*ops)

    def forward(self, x):
        return run_conv_block(self, x)


class StackedConvBlocks(nn.Module):
    def __init__(self, num_convs, conv_op, cin, cout, kernel_size, initial_stride, conv_bias, norm_op, norm_op_kwargs,
                 dropout_op, dropout_op_kwargs, nonlin, nonlin_kwargs):
        super().__init__()
        couts = [cout] * num_convs if isinstance(cout, int) else list(cout)
        mk = lambda ci, co, st: ConvDropoutNormReLU(conv_op, ci, co, kernel_size, st, conv_bias, norm_op, norm_op_kwargs,
                                                    dropout_op, dropout_op_kwargs, nonlin, nonlin_kwargs)
        self.convs = nn.Sequential(mk(cin, couts[0], initial_stride),
                                   *[mk(couts[i - 1], couts[i], 1) for i in range(1, num_convs)])
        self.output_channels = couts[-1]

    def forward(self, x):
        return run_stacked(self, x)


class PlainConvEncoder(nn.Module):
    def __init__(self, input_channels, n_stages, features_per_stage, conv_op, kernel_sizes, strides, n_conv_per_stage,
                 conv_bias, norm_op, norm_op_kwargs, dropout_op, dropout_op_kwargs, nonlin, nonlin_kwargs):
        super().__init__()
        features_per_stage = _maybe_list(features_per_stage, n_stages)
        n_conv_per_stage = _maybe_list(n_conv_per_stage, n_stages)
        kernel_sizes = [kernel_sizes] * n_stages if isinstance(kernel_sizes, int) else list(kernel_sizes)
        strides = [strides] * n_stages if isinstance(strides, int) else list(strides)
        stages = []
        cin = input_channels
        for s in range(n_stages):
            stages.append(nn.Sequential(StackedConvBlocks(n_conv_per_stage[s], conv_op, cin, features_per_stage[s],
                                                          kernel_sizes[s], strides[s], conv_bias, norm_op, norm_op_kwargs,
                                                          dropout_op, dropout_op_kwargs, nonlin, nonlin_kwargs)))
            cin = features_per_stage[s]
        self.stages = nn.Sequential(*stages)
        self.output_channels = features_per_stage
        self.strides = [_maybe_list(i, 3 if conv_op is nn.Conv3d else 2) for i in strides]
        self.return_skips = True
        self.conv_op, self.norm_op, self.norm_op_kwargs = conv_op, norm_op, norm_op_kwargs
        self.nonlin, self.nonlin_kwargs = nonlin, nonlin_kwargs
        self.dropout_op, self.dropout_op_kwargs = dropout_op, dropout_op_kwargs
        self.conv_bias, self.kernel_sizes = conv_bias, kernel_sizes

    def forward(self, x):
        return encoder_forward(self, x)


class UNetDecoder(nn.Module):
    def __init__(self, encoder, num_classes, n_conv_per_stage, deep_supervision, nonlin_first=False, deep_features=True):
        super().__init__()
        self.deep_supervision = deep_supervision
        self.deep_features = deep_features
        self.encoder = encoder
        self.num_classes = num_classes
        n_enc = len(encoder.output_channels)
        n_conv_per_stage = _maybe_list(n_conv_per_stage, n_enc - 1)
        transp = nn.ConvTranspose3d if encoder.conv_op is nn.Conv3d else nn.ConvTranspose2d
        stages, transpconvs, seg_layers = [], [], []
        for s in range(1, n_enc):
            below, skip = encoder.output_channels[-s], encoder.output_channels[-(s + 1)]
            st = encoder.strides[-s]
            transpconvs.append(transp(below, skip, st, st, bias=encoder.conv_bias))
            stages.append(StackedConvBlocks(n_conv_per_stage[s - 1], encoder.conv_op, 2 * skip, skip,
                                            encoder.kernel_sizes[-(s + 1)], 1, encoder.conv_bias, encoder.norm_op,
                                            encoder.norm_op_kwargs, encoder.dropout_op, encoder.dropout_op_kwargs,
                                            encoder.nonlin, encoder.nonlin_kwargs))
            seg_layers.append(encoder.conv_op(skip, num_classes, 1, 1, 0, bias=True))
        self.stages = nn.ModuleList(stages)
        self.transpconvs = nn.ModuleList(transpconvs)
        self.seg_layers = nn.ModuleList(seg_layers)

    def forward(self, skips):
        return decoder_forward(self, skips)


class PlainConvUNet(nn.Module):
    """dynamic_network_architectures.architectures.unet.PlainConvUNet (the class the reference subclasses at
    models/seg_model.py:153): encoder -> decoder, forward returns the segmentation logits only."""

    def __init__(self, input_channels, n_stages, features_per_stage, conv_op, kernel_sizes, strides, n_conv_per_stage,
                 num_classes, n_conv_per_stage_decoder, conv_bias=False, norm_op=None, norm_op_kwargs=None,
                 dropout_op=None, dropout_op_kwargs=None, nonlin=None, nonlin_kwargs=None, deep_supervision=False,
                 nonlin_first=False):
        super().__init__()
        if conv_op is not nn.Conv3d:
            raise RehrError("the REHRSeg segmentation network is 3-D (train_all.py:479)")
        if nonlin_first:
            raise RehrError("nonlin_first=True is not used by the reference and is not implemented")
        self.encoder = PlainConvEncoder(input_channels, n_stages, features_per_stage, conv_op, kernel_sizes, strides,
                                        n_conv_per_stage, conv_bias, norm_op, norm_op_kwargs, dropout_op, dropout_op_kwargs,
                                        nonlin, nonlin_kwargs)
        self.decoder = UNetDecoder(self.encoder, num_classes, n_conv_per_stage_decoder, deep_supervision,
                                   nonlin_first=nonlin_first, deep_features=False)

    def forward(self, x):
        if not x.is_cuda:
            raise RehrError("rehrseg_b200 runs on CUDA (sm_100a) only; there is no CPU path")
        with device_of(x):
            return decoder_forward(self.decoder, encoder_forward(self.encoder, x))


class SegModel(nn.Module):
    """Same signature as the reference SegModel (models/seg_model.py:154-173)."""

    def __init__(self, input_channels, n_stages, features_per_stage, conv_op, kernel_sizes, strides, n_conv_per_stage,
                 num_classes, upscale, n_conv_per_stage_decoder, conv_bias=False, norm_op=None, norm_op_kwargs=None,
                 dropout_op=None, dropout_op_kwargs=None, nonlin=None, nonlin_kwargs=None, deep_supervision=False,
                 nonlin_first=False):
        super().__init__()
        if conv_op is not nn.Conv3d:
            raise RehrError("the REHRSeg segmentation network is 3-D (train_all.py:479)")
        if nonlin_first:
            raise RehrError("nonlin_first=True is not used by the reference and is not implemented")
        self.encoder = PlainConvEncoder(input_channels, n_stages, features_per_stage, conv_op, kernel_sizes, strides,
                                        n_conv_per_stage, conv_bias, norm_op, norm_op_kwargs, dropout_op, dropout_op_kwargs,
                                        nonlin, nonlin_kwargs)
        # The reference first builds PlainConvUNet's own decoder and then replaces it with MyUnetDecoder
        # (models/seg_model.py:174-193), drawing the decoder's default-init random numbers twice; do the same so that an
        # identically seeded construction yields identical weights.
        UNetDecoder(self.encoder, num_classes, n_conv_per_stage_decoder, deep_supervision, nonlin_first=nonlin_first)
        self.decoder = UNetDecoder(self.encoder, num_classes, n_conv_per_stage_decoder, deep_supervision,
                                   nonlin_first=nonlin_first, deep_features=True)
        self.upscale = upscale
        self.sr_head = nn.Sequential(nn.Conv3d(32, 16, kernel_size=3, stride=1, padding=1), nn.ReLU(),
                                     nn.Conv3d(16, num_classes, kernel_size=5, stride=1, padding=2))

    def forward(self, x, return_inetermediate_feature=False):
        return segmodel_forward(self, x, return_inetermediate_feature)


def fullres_kwargs(num_classes: int = 2, input_channels: int = 1) -> dict:
    """nnU-Net 3d_fullres defaults used by BASELINE configs 1 and 3 (SURVEY.md section 8(d))."""
    return dict(input_channels=input_channels, n_stages=6, features_per_stage=[32, 64, 128, 256, 320, 320],
                conv_op=nn.Conv3d, kernel_sizes=[[3, 3, 3]] * 6, strides=[[1, 1, 1]] + [[2, 2, 2]] * 5,
                n_conv_per_stage=[2] * 6, num_classes=num_classes, n_conv_per_stage_decoder=[2] * 5, conv_bias=True,
                norm_op=nn.InstanceNorm3d, norm_op_kwargs={"eps": 1e-5, "affine": True}, dropout_op=None,
                dropout_op_kwargs=None, nonlin=nn.LeakyReLU, nonlin_kwargs={"inplace": True}, deep_supervision=False)


def plainconv_3d_fullres(num_classes: int = 2, upscale: int = 4, input_channels: int = 1) -> SegModel:
    """The full REHRSeg SegModel (U-Net + x`upscale` SR head) on the 3d_fullres plan."""
    return SegModel(upscale=upscale, **fullres_kwargs(num_classes, input_channels))


def plainconv_unet_3d_fullres(num_classes: int = 2, input_channels: int = 1) -> PlainConvUNet:
    """The pure PlainConvUNet of BASELINE config 1 (no SR head)."""
    return PlainConvUNet(**fullres_kwargs(num_classes, input_channels))
