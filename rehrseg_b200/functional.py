"""autograd.Function wrappers over the C-ABI (include/rehrseg_b200.h).

Activations travel between these functions as channels-last bf16 tensors of logical shape [N, D, H, W, C]
(`_lib.as_cl`); parameters stay the caller's fp32 `nn.Parameter`s in PyTorch layout, so `state_dict()`,
optimisers and checkpoints of the reference (train_all.py:496-499,513,566-573) are untouched.  bf16 GEMM-operand
copies of the weights are derived caches keyed on the parameter's version counter.

Reference call sites replaced are listed per function.  There is no PyTorch fallback: every op calls the
library and raises `RehrError` on a non-zero status.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref
from typing import Optional, Sequence, Tuple

import torch

from . import _lib as L
from ._lib import ACT_LRELU, ACT_NONE, ACT_RELU, as_cl, check, conv_desc, lib, ptr, rt, stream_ptr

Triple = Tuple[int, int, int]

# --------------------------------------------------------------------------------------------------
# launch accounting (bench.py reports `gpu_launches`)
# --------------------------------------------------------------------------------------------------
_launches = 0
path_hits = {"tconv_bias_from_epilogue_sums": 0, "tconv_twin_from_epilogue": 0}   # which fused shortcuts really ran (tests read this)


def launches() -> int:
    return _launches


def _count(n: int = 1) -> None:
    global _launches
    _launches += n


# --------------------------------------------------------------------------------------------------
# optional per-kernel device timing (bench.py's roofline leg): CUDA events on the launching stream around each
# conv-engine launch, tagged with the kernel family and its ALGORITHMIC flops (2*M*N*K of the layer).
# --------------------------------------------------------------------------------------------------
_ktimer: Optional[list] = None


class kernel_timer:
    """with kernel_timer() as rec: ...; rec.summary() -> {family: (launches, total_ms, total_flops)}"""

    def __enter__(self):
        global _ktimer
        self.records: list = []
        _ktimer = self.records
        return self

    def __exit__(self, *exc):
        global _ktimer
        _ktimer = None
        return False

    def summary(self) -> dict:
        torch.cuda.synchronize()
        out: dict = {}
        for name, flops, e0, e1, _tag in self.records:
            n, ms, fl = out.get(name, (0, 0.0, 0.0))
            out[name] = (n + 1, ms + e0.elapsed_time(e1), fl + flops)
        return out

    def rows(self) -> list:
        """[(family, tag, ms, flops)] per launch, in launch order."""
        torch.cuda.synchronize()
        return [(name, tag, e0.elapsed_time(e1), flops) for name, flops, e0, e1, tag in self.records]


class _timed:
    def __init__(self, name: str, flops: float, tag: str = ""):
        self.name, self.flops, self.tag = name, flops, tag

    def __enter__(self):
        if _ktimer is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if _ktimer is not None:
            e1 = torch.cuda.Event(enable_timing=True)
            e1.record()
            _ktimer.append((self.name, self.flops, self.e0, e1, self.tag))
        return False


# --------------------------------------------------------------------------------------------------
# opt-in fp16 saturation check (rangecheck.RangeCheck): the active check, or None.  `_sink(kind)` wraps one fp16-producing
# launch of the SegModel forward; with no check active it does nothing and the kernels get a null slot.
# --------------------------------------------------------------------------------------------------
_range = None


class _sink:
    __slots__ = ("kind",)

    def __init__(self, kind: str):
        self.kind = kind

    def __enter__(self):
        if _range is not None:
            _range.arm(self.kind)
        return self

    def __exit__(self, *exc):
        if _range is not None:
            _range.disarm()
        return False


class range_owner:
    """Labels the fp16 stores issued inside the block with `module` (seg_model's conv blocks, transposed convs, sr_head)."""
    __slots__ = ("module", "prev")

    def __init__(self, module):
        self.module = module

    def __enter__(self):
        if _range is not None:
            self.prev, _range.owner = _range.owner, self.module
        return self

    def __exit__(self, *exc):
        if _range is not None:
            _range.owner = self.prev
        return False


# --------------------------------------------------------------------------------------------------
# 16-bit storage formats
# --------------------------------------------------------------------------------------------------
# Gradients (and every FLAVR activation) are bf16.  The forward activations of the InstanceNorm'ed SegModel path are stored in
# fp16: InstanceNorm bounds them, fp16 keeps 3 more mantissa bits than bf16 at the same tensor-core rate and the same bytes, and
# the logits land at ~1e-3 of the fp32 reference instead of ~9e-3 (tools/bf16_emulate.py; DESIGN.md section 4).  fp16 stores
# saturate (+-65504).  REHR_FWD_DTYPE=bf16 keeps bf16 MMA operands in the forward pass as well.
#
# PyTorch only sees bf16 tensors: an fp16 activation travels as a tensor of NOMINAL dtype bfloat16 whose Python object carries
# `_rehr_h = True` (its 16-bit payload is fp16).  That keeps autograd's dtype bookkeeping on bf16, which is what the gradient of
# such an activation really is.  Only engine functions may consume these tensors; `from_channels_last` converts at the boundary.
# One tcgen05.mma takes ONE 16-bit format (mixed fp16 x bf16 operands are an illegal instruction, tools/umma_mixed_probe.cu), so
# a weight-gradient GEMM (activation x bf16 gradient) needs a bf16 copy of the activation: `_rehr_bf` holds that twin, written
# by the same pass that writes the fp16 activation.
FWD_FP16 = os.environ.get("REHR_FWD_DTYPE", "fp16").lower() != "bf16"


def is_h(t) -> bool:
    """True if `t`'s 16-bit payload is fp16 (see above)."""
    return bool(getattr(t, "_rehr_h", False))


def mark_h(t: torch.Tensor, twin: Optional[torch.Tensor] = None) -> torch.Tensor:
    t._rehr_h = True
    if twin is not None:
        t._rehr_bf = twin
    return t


def to_float(t: torch.Tensor) -> torch.Tensor:
    """fp32 values of an engine activation (channels-last, either storage format) -- for tests and debugging."""
    h = is_h(t)
    t = t.detach()
    return t.view(torch.float16).float() if h else t.float()


def convert16_raw(x: torch.Tensor, x_h: bool, out_h: bool, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Copy of a channels-last 16-bit tensor in the other storage format (pitched channel slices allowed)."""
    x = as_cl(x)
    if out is None:
        out = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    xt, ot = rt(x, x_h), rt(out, out_h)
    check(lib().rehr_convert16(C.byref(xt), C.byref(ot), stream_ptr()), "convert16")
    _count()
    return out


def bf_twin(t: torch.Tensor) -> torch.Tensor:
    """The bf16 operand of `t` for a weight-gradient GEMM: `t` itself unless its payload is fp16, then its twin (converted on
    the spot and cached on `t` if the producer did not write one, e.g. a frozen producer feeding a trainable consumer)."""
    if not is_h(t):
        return as_cl(t)
    tw = getattr(t, "_rehr_bf", None)
    if tw is None:
        tw = t._rehr_bf = convert16_raw(t, True, False)
    return tw


# --------------------------------------------------------------------------------------------------
# packed-weight cache
# --------------------------------------------------------------------------------------------------
_wcache: dict = {}
USE_MARCH = True  # route eligible k3/s1/p1 layers through the halo-resident marching kernel (csrc/conv_march.cu)
S2_WGRAD_MARCH_MIN_VOXELS = 262144  # dy voxels from which the per-parity-class marching wgrad of a stride-2 conv wins


def _pack_into(weight: torch.Tensor, kind: str, h: bool, out: Optional[torch.Tensor] = None, extra=None) -> torch.Tensor:
    """Launch the pack kernel of `kind` for `weight` into `out` (allocated when None) on the current stream."""
    dt = L.F16 if h else L.BF16
    A, B = weight.shape[0], weight.shape[1]
    T = weight[0, 0].numel()
    w = weight.detach()
    if not w.is_contiguous():
        w = w.contiguous()
    if w.dtype != torch.float32:
        w = w.float()
    if _pack_keepalive is not None and w.data_ptr() != weight.data_ptr():
        _pack_keepalive.append(w)     # a recorded (batched) pack reads this temporary only when the batch is launched

    def buf(n_or_shape):
        if out is not None:
            return out
        shape = (n_or_shape,) if isinstance(n_or_shape, int) else n_or_shape
        return torch.empty(shape, dtype=torch.bfloat16, device=w.device)

    if kind == "march_fwd":      # conv A<-B, marching-kernel layout
        ks = int(weight.shape[2])
        o = buf(lib().rehr_conv3d_march_weight_bytes(B, A, ks) // 2)
        check(lib().rehr_pack_weight_march(ptr(w), ptr(o), A, B, ks, B * T, T, 0, dt, stream_ptr()), "pack_weight_march")
    elif kind == "march_dgrad":  # its input-gradient B<-A (transposed, taps flipped)
        ks = int(weight.shape[2])
        o = buf(lib().rehr_conv3d_march_weight_bytes(A, B, ks) // 2)
        check(lib().rehr_pack_weight_march(ptr(w), ptr(o), B, A, ks, T, B * T, 1, dt, stream_ptr()), "pack_weight_march")
    elif kind == "s2dgrad":      # parity-class weights of a stride-2 input gradient; extra = (kernel, stride, padding)
        desc = conv_desc(*extra)
        o = buf(lib().rehr_conv3d_march_s2dgrad_weight_bytes(C.byref(desc), B, A) // 2)
        check(lib().rehr_pack_weight_march_s2dgrad(C.byref(desc), ptr(w), ptr(o), B, A, stream_ptr()), "pack_weight_march_s2dgrad")
    elif kind == "tconv_fused":  # ConvTranspose weight [Cin=A][Cout=B][T] -> [T][Cout][Cin]
        o = buf((T, B, A))
        check(lib().rehr_pack_weight(ptr(w), ptr(o), T, A, B, 1, B * T, T, dt, stream_ptr()), "pack_weight")
    elif kind == "fwd":
        o = buf((A, T, B))
        check(lib().rehr_pack_weight(ptr(w), ptr(o), A, B, T, B * T, T, 1, dt, stream_ptr()), "pack_weight")
    else:
        o = buf((B, T, A))
        check(lib().rehr_pack_weight(ptr(w), ptr(o), B, A, T, T, B * T, 1, dt, stream_ptr()), "pack_weight")
    _count()
    return o


PACK_BATCHED = os.environ.get("REHR_PACK_BATCHED", "1") != "0"
_pack_keepalive: Optional[list] = None   # while pack calls are being recorded: fp32 / contiguous temporaries of the weights
PACK_BATCH_SPLITS = tuple(int(v) for v in os.environ.get("REHR_PACK_SPLITS", "200000,2000000,8000000").split(",") if v)   # cumulative elements
_pending_prepack = None   # fork object of refresh_weight_cache(): joined at the end of the step (or by clear_weight_cache)
_pack_events: dict = {}   # cache key -> event recorded on the pack stream right after that copy was re-packed


def _join_prepack() -> None:
    global _pending_prepack
    _pack_events.clear()
    if _pending_prepack is not None:
        fk, _pending_prepack = _pending_prepack, None
        fk.join()


def _await_pack(key) -> None:
    """Make the current stream wait for the refresh of ONE cached copy (not for the whole pack stream: the ~55 small pack kernels
    of a step take ~0.6 ms back to back, and the first convs would otherwise sit idle until the last of them has run)."""
    ev = _pack_events.pop(key, None)
    if ev is not None:
        torch.cuda.current_stream().wait_event(ev)


def _packed(weight: torch.Tensor, kind: str, cache: bool = True, h: bool = False, extra=None) -> torch.Tensor:
    """16-bit K-major operand of `weight` ([A][B][T...] fp32) -- kind 'fwd': [A][T][B], 'dgrad': [B][T][A], the marching layouts,
    ...; `h`: packed as fp16 (must match the activation tensor the GEMM contracts it with), else bf16.
    Cached per parameter object and version counter (an optimiser step bumps the version -> repack, or refresh_weight_cache()
    re-packs every cached copy in place at the start of a step)."""
    key = (id(weight), kind, h, extra)
    if weight.is_inference():      # tensors made under torch.inference_mode() carry no version counter: pack, never cache
        ver, cache = -1, False
    else:
        ver = weight._version
    if cache:
        hit = _wcache.get(key)
        if hit is not None and hit[0]() is weight and hit[1] == ver and hit[2].device == weight.device:
            _await_pack(key)
            return hit[2]
    out = _pack_into(weight, kind, h, None, extra)
    if cache:
        _cache_put(key, weight, out)
    return out


def clear_weight_cache() -> None:
    _join_prepack()
    _wcache.clear()


def refresh_weight_cache() -> int:
    """Re-pack every cached 16-bit operand copy IN PLACE from the current parameter values, on a side stream forked from the
    current one (events only: CUDA-graph capturable), and mark them current.  Called at the start of a training step after the
    optimiser update: the ~50 small pack kernels then run next to the first layers instead of in front of each conv, and the
    addresses the kernels see stay fixed (what a captured graph needs).  A cache hit waits for the event of its own copy only; the
    caller joins the pack stream at the end of the step (_join_prepack).
    Returns the number of copies refreshed (0 on the very first step: nothing is cached yet and the packs happen lazily)."""
    global _pending_prepack
    _join_prepack()
    live = [(k, v) for k, v in _wcache.items() if v[0]() is not None]
    for k in [k for k, v in _wcache.items() if v[0]() is None]:
        del _wcache[k]
    if not live:
        return 0
    fk = _fork(live[0][1][2].device, "pack")
    with fk:
        if PACK_BATCHED:
            # a few batched launches (csrc/pack_batch.cu: the calls below are recorded, not launched), one event per batch.  The
            # cache is in order of first use, so the first batches hold the small full-resolution layers the step needs at once;
            # the bulk (the 256-320 channel layers, the input-gradient layouts) follows in the last one and has ~2 ms to finish.
            global _launches
            bounds, acc = [], 0
            limits = list(PACK_BATCH_SPLITS)
            for i, (key, (wref, _ver, out)) in enumerate(live):
                acc += out.numel()
                if limits and acc > limits[0]:
                    bounds.append(i + 1)
                    limits.pop(0)
            bounds = sorted(set(b for b in bounds if b < len(live))) + [len(live)]
            first = 0
            global _pack_keepalive
            for last in bounds:
                check(lib().rehr_pack_batch_begin(), "pack_batch_begin")
                _pack_keepalive = []
                try:
                    for key, (wref, _ver, out) in live[first:last]:
                        w = wref()
                        _pack_into(w, key[1], key[2], out, key[3])
                        _wcache[key] = (wref, w._version, out)
                    check(lib().rehr_pack_batch_launch(stream_ptr()), "pack_batch_launch")
                except Exception:
                    lib().rehr_pack_batch_abort()
                    raise
                finally:
                    _pack_keepalive = None    # (the launch is stream-ordered before any later reuse of the temporaries' memory)
                _launches -= (last - first) - (last - first + 127) // 128      # _pack_into counted one launch per copy
                ev = torch.cuda.Event()
                ev.record(fk.side)
                for key, _ in live[first:last]:
                    _pack_events[key] = ev
                first = last
        else:
            for key, (wref, _ver, out) in live:
                w = wref()
                _pack_into(w, key[1], key[2], out, key[3])
                _wcache[key] = (wref, w._version, out)
                ev = torch.cuda.Event()
                ev.record(fk.side)
                _pack_events[key] = ev
    _pending_prepack = fk
    return len(live)


def _cache_put(key, weight: torch.Tensor, out: torch.Tensor) -> None:
    """Insert an operand copy; dead entries (weights that were garbage collected) are dropped once the table grows."""
    if weight.is_inference():
        return
    if len(_wcache) >= 256:
        for k in [k for k, v in _wcache.items() if v[0]() is None]:
            del _wcache[k]
    _wcache[key] = (weakref.ref(weight), weight._version, out)


def _orig_weight(ctx, saved: torch.Tensor) -> torch.Tensor:
    """The Parameter object the forward saw (autograd's saved tensor is a fresh Python object every step, which would miss the
    packed-weight cache and defeat refresh_weight_cache): kept as a weak reference on the ctx."""
    ref = getattr(ctx, "wref", None)
    w = ref() if ref is not None else None
    return w if (w is not None and w.data_ptr() == saved.data_ptr()) else saved


def _out_size(i: int, k: int, s: int, p: int) -> int:
    return (i + 2 * p - k) // s + 1


def _f32(t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
    if t is None:
        return None
    t = t.detach()
    if t.dtype != torch.float32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


def _alias(storage_of: torch.Tensor, offset: int, size, stride) -> torch.Tensor:
    """A fresh tensor over `storage_of`'s storage with NO autograd view relationship (the concat buffers below are
    written through raw pointers by the kernels, which autograd's view+inplace tracking cannot follow)."""
    t = torch.empty((0,), dtype=storage_of.dtype, device=storage_of.device)
    return t.set_(storage_of.untyped_storage(), offset, tuple(size), tuple(stride))


# Second gradient source of an encoder skip activation.  A skip `a` feeds the next encoder stage AND the decoder concat; autograd
# would add the two gradients with an extra full-tensor pass.  The InstanceNorm backward kernels take two gradient operands
# (da1, da2), so ConvTranspose.backward parks the concat-buffer half here (keyed by the skip's storage) instead of returning it,
# and the ConvNormAct.backward that produced the skip picks it up.  Autograd runs a node only after every consumer's backward,
# so the entry is always there in time; it is popped on use.
_skip_grads: dict = {}


def concat_room_of(t: torch.Tensor):
    """(total_channels, channel_offset) if `t` was produced inside a wider concat buffer (see conv_norm_act), else None."""
    return getattr(t, "_rehr_cat", None)


# Small and mid-size layers (<= 64^3): the weight gradient and the input gradient of a conv are independent consumers of dy and each is a
# latency-bound launch chain (GEMM + partial reduction) on a handful of CTAs, so the weight-gradient chain is forked onto a side
# stream and joined after the input gradient has been issued (events only: the fork/join is captured as two parallel branches by
# graphs.GraphedTrainStep).  Large layers fill the machine on their own and stay on one stream.
WGRAD_SIDE_STREAM = True
WGRAD_SIDE_MAX_VOXELS = 2 * 64 ** 3   # measured on the C1 step: 12.58 ms at 2 * 32^3, 12.46 ms at 2 * 64^3 and above
_side_streams: dict = {}


# Stream priorities.  The side stream of the weight-gradient chains has the HIGH priority graphs.GraphedTrainStep also gives its
# capture stream (kernel nodes of a captured graph keep the priority of the stream they were captured from), the re-pack stream
# ("pack") the default = lowest one: the one batched pack kernel of a step is ~36K small blocks, and at equal priority they queue
# in front of the blocks of the first forward kernels and hold them up (measured: the stem's statistics pass started 165 us late).
SIDE_PRIORITY = int(os.environ.get("REHR_SIDE_PRIORITY", "-1"))


class _fork:
    def __init__(self, device, kind: str = "wgrad"):
        self.main = torch.cuda.current_stream(device)
        key = (device.index if device.index is not None else torch.cuda.current_device(), kind)
        side = _side_streams.get(key)
        if side is None:
            side = _side_streams[key] = torch.cuda.Stream(device=device, priority=SIDE_PRIORITY if kind == "wgrad" else 0)
        self.side = side
        self.ctx = None

    def __enter__(self):
        ev = torch.cuda.Event()
        ev.record(self.main)
        self.side.wait_event(ev)
        self.ctx = torch.cuda.stream(self.side)
        self.ctx.__enter__()
        return self

    def __exit__(self, *exc):
        self.ctx.__exit__(*exc)
        return False

    def join(self):
        ev = torch.cuda.Event()
        ev.record(self.side)
        self.main.wait_event(ev)


# Deferred join: the weight gradient of a layer is needed by nobody until the optimiser (or the data-parallel all-reduce of its
# bucket) runs, so its chain stays on the side stream and the main stream goes straight on to the input gradient and to the
# InstanceNorm reduce / apply passes of the NEXT layer's backward -- HBM-bound kernels that fit next to a tensor-bound weight
# gradient CTA on every SM.  The side stream is joined once, by a final callback of the autograd engine (and before any bucket
# all-reduce, graphs.GraphedTrainStep).  Operands are kept alive until then (their memory must not be recycled by the main stream
# while the side stream still reads it).
# Order matters: two machine-filling GEMMs cannot share an SM, so whichever starts first runs first.  The input gradient must go
# first (the next layer's InstanceNorm passes depend on it); inside a replayed CUDA graph two independent branches start in no
# particular order, so for layers of >= DGRAD_FIRST_MIN_VOXELS voxels the weight gradient is made to WAIT for the input gradient
# (_dgrad_and_wgrad) -- the InstanceNorm passes of the next layer then run NEXT to it (tools/overlap_probe.py: about half of
# their time disappears behind a weight gradient).  Measured on the C1 step (tools/ab_step.py): 12.76 ms joined per layer,
# 12.41 ms deferred with the weight gradient launched first, 12.28-12.31 ms with the dependency.
# The window this opens: autograd's AccumulateGrad touches the returned dW on the MAIN stream whenever it cannot simply adopt the
# tensor (an existing .grad to add to, a hook that reads it).  So the deferral is (a) only taken for parameters whose .grad is
# None, and (b) only ON inside `deferred_wgrad()` -- entered by graphs.GraphedTrainStep, which owns the whole step, joins before
# its bucket all-reduces and at the end of the step.  Plain eager use keeps the per-layer join.  REHR_WGRAD_DEFER=1 forces it on
# everywhere, =0 off everywhere.
_DEFER_ENV = os.environ.get("REHR_WGRAD_DEFER", "")
WGRAD_DEFER_JOIN = _DEFER_ENV == "1"
DGRAD_FIRST_MIN_VOXELS = int(os.environ.get("REHR_DFIRST_MIN_VOXELS", str(2 * 32 ** 3)))


class deferred_wgrad:
    """Context: weight-gradient chains started inside stay on the side stream until `join_pending_wgrad()` / the end of the
    backward pass (see above).  The caller guarantees nothing reads a .grad on the main stream before that."""

    def __enter__(self):
        global WGRAD_DEFER_JOIN
        self.prev = WGRAD_DEFER_JOIN
        if _DEFER_ENV != "0":
            WGRAD_DEFER_JOIN = True
        return self

    def __exit__(self, *exc):
        global WGRAD_DEFER_JOIN
        WGRAD_DEFER_JOIN = self.prev
        join_pending_wgrad()      # also after an exception inside the pass: nothing may stay pending (and keep operands alive)
        return False


_wgrad_pending: list = []


def pending_wgrad_event():
    """An event that completes when every weight-gradient chain issued so far on the side stream has run (None if there is none
    pending).  For a consumer on ANOTHER stream (the communication stream of a bucketed all-reduce): it waits for this event
    instead of making the main stream join the side stream.  The chains stay pending: their operands are released by the join."""
    if not _wgrad_pending:
        return None
    fk = _wgrad_pending[-1][0]
    ev = torch.cuda.Event()
    ev.record(fk.side)
    return ev


def join_pending_wgrad() -> None:
    """Make the current stream wait for every weight-gradient chain still running on the side stream; release their operands."""
    if not _wgrad_pending:
        return
    fk = _wgrad_pending[-1][0]          # one in-order side stream: its latest event covers all earlier chains
    ev = torch.cuda.Event()
    ev.record(fk.side)
    torch.cuda.current_stream(fk.side.device).wait_event(ev)
    _wgrad_pending.clear()


def _dgrad_and_wgrad(x, dy, weight, wshape, kernel, stride, padding, need_dx: bool, cache: bool = True, want_chsum: bool = False):
    """(dx or None, dw) of a conv.  The weight-gradient chain runs on a side stream (events only: graph-capturable): joined right
    after the input gradient for small layers (two latency-bound chains side by side), or -- WGRAD_DEFER_JOIN, inside an autograd
    backward pass -- at the end of the pass."""
    voxels = dy.shape[0] * dy.shape[1] * dy.shape[2] * dy.shape[3]
    side_ok = need_dx and WGRAD_SIDE_STREAM and _ktimer is None
    if side_ok and (WGRAD_DEFER_JOIN or voxels <= WGRAD_SIDE_MAX_VOXELS):
        dw = torch.empty(tuple(wshape), dtype=torch.float32, device=dy.device)   # owned by the main stream's pool
        fk = _fork(dy.device)
        if WGRAD_DEFER_JOIN and voxels >= DGRAD_FIRST_MIN_VOXELS:
            # machine-filling layer: the two GEMMs cannot share an SM.  The input gradient goes first -- the NEXT layer's
            # InstanceNorm passes depend on it -- and the weight gradient is made to WAIT for it (fork point after the launch):
            # inside a replayed CUDA graph two independent branches start in no particular order, a dependency is the only
            # way to fix it.  The InstanceNorm passes then run next to the weight gradient.
            dx = conv3d_dgrad_raw(dy, weight, x.shape, kernel, stride, padding, cache=cache, want_chsum=want_chsum)
            with fk:
                conv3d_wgrad_raw(x, dy, wshape, kernel, stride, padding, out=dw)
        else:
            with fk:
                conv3d_wgrad_raw(x, dy, wshape, kernel, stride, padding, out=dw)
            dx = conv3d_dgrad_raw(dy, weight, x.shape, kernel, stride, padding, cache=cache, want_chsum=want_chsum)
        deferred = False
        # a leaf parameter without a .grad: AccumulateGrad adopts dw without touching it (a view of a parameter, e.g. FLAVR's 2-D
        # fuse convs seen as 5-D, sends dw through a ViewBackward first: joined per layer)
        if WGRAD_DEFER_JOIN and weight.is_leaf and weight.grad is None:
            try:
                if not _wgrad_pending:
                    torch.autograd.Variable._execution_engine.queue_callback(join_pending_wgrad)
                _wgrad_pending.append((fk, (x, dy)))   # NOT dw: an extra reference would force AccumulateGrad to clone it
                deferred = True
            except RuntimeError:      # not inside a backward pass: nobody would join later
                deferred = False
        if not deferred:
            fk.join()
        return dx, dw
    dx = conv3d_dgrad_raw(dy, weight, x.shape, kernel, stride, padding, cache=cache, want_chsum=want_chsum) if need_dx else None
    return dx, conv3d_wgrad_raw(x, dy, wshape, kernel, stride, padding)


MARCH_MAX_WIDE = int(os.environ.get("REHR_MARCH_MAX_WIDE", "128"))


def _march_route(desc, c_operand: int, c_result: int) -> bool:
    """Marching kernel or tapped GEMM for a stride-1 k3 / k5 conv (forward: operand = x, result = y; input gradient: operand = dy,
    result = dx).  With 128 operand channels the marching kernel keeps only a 16-channel result tile resident (N = 48 per A-read:
    operand-feed bound at ~500 TFLOP/s), so once the result has >= 128 channels the tapped GEMM (N = 128) wins -- measured,
    tools/route_probe.py: 128->128 @32^3 fwd 119 -> 88 us, dgrad 103 -> 83 us; dgrad 256<-128 @32^3 168 -> 92 us; while 128->64
    @64^3 stays on the marching kernel (319 vs 526 us)."""
    if not (USE_MARCH and lib().rehr_conv3d_march_supported(C.byref(desc), int(c_operand), int(c_result))):
        return False
    return not (c_operand >= 128 and c_result >= MARCH_MAX_WIDE)


# The exactly-zero bias gradients of the Conv -> InstanceNorm blocks (one per layer) are slices of ONE zero-filled buffer per
# backward pass instead of one fill kernel each (22 launches on the C1 step).  A fresh buffer per pass: whatever the caller does to
# a .grad in place can never leak into the next step.
_zero_pool: dict = {}


def _zero_pool_reset() -> None:
    _zero_pool.clear()


def _zero_grad_slice(n: int, device) -> torch.Tensor:
    st = _zero_pool.get(device)
    if st is None or st[1] + n > st[0].numel():
        try:
            if not _zero_pool:
                torch.autograd.Variable._execution_engine.queue_callback(_zero_pool_reset)
        except RuntimeError:      # not inside a backward pass: no pooling
            return torch.zeros((n,), dtype=torch.float32, device=device)
        st = _zero_pool[device] = [torch.zeros((max(8192, n),), dtype=torch.float32, device=device), 0]
    out = st[0][st[1]:st[1] + n]
    st[1] += (n + 3) // 4 * 4        # 16-byte aligned slices
    return out


def _ws(nbytes: int, device) -> torch.Tensor:
    return torch.empty((max(int(nbytes), 16),), dtype=torch.uint8, device=device)


# --------------------------------------------------------------------------------------------------
# raw (non-autograd) helpers
# --------------------------------------------------------------------------------------------------
def conv3d_raw(x: torch.Tensor, weight: torch.Tensor, bias: Optional[torch.Tensor], kernel: Triple, stride: Triple,
               padding: Triple, act: int = ACT_NONE, slope: float = 0.0, want_stats: bool = False,
               out_f32: bool = False, out: Optional[torch.Tensor] = None, x_h: bool = False, y_h: bool = False):
    """y = act(conv3d(x) + bias) on NDHWC 16-bit `x`; optionally per-tile InstanceNorm partial sums.  `x_h` / `y_h`: the payload
    of x / y is fp16 (the weights are packed in x's format).  Returns (y, stats_partial or None, tiles)."""
    x = as_cl(x)
    n, d, h, w, cin = x.shape
    cout = weight.shape[0]
    od, oh, ow = (_out_size(i, k, s, p) for i, k, s, p in zip((d, h, w), kernel, stride, padding))
    if out is None:
        out = torch.empty((n, od, oh, ow, cout), dtype=torch.float32 if out_f32 else torch.bfloat16, device=x.device)
    yt = rt(out, y_h)
    desc = conv_desc(kernel, stride, padding)
    stats = None
    tiles = 0
    flops = 2.0 * n * od * oh * ow * cout * cin * kernel[0] * kernel[1] * kernel[2]
    tag = f"fwd {cin}->{cout} in{d}x{h}x{w} k{kernel} s{stride}" if _ktimer is not None else ""
    if _march_route(desc, cin, cout):
        xt = rt(x, x_h)
        if want_stats:
            tiles = lib().rehr_conv3d_march_stats_tiles(C.byref(xt), C.byref(yt), int(kernel[0]))
            stats = torch.empty((n, tiles, cout, 2), dtype=torch.float32, device=x.device)
        wp = _packed(weight, "march_fwd", h=x_h)
        with _timed("conv_march_kernel", flops, tag):
            check(lib().rehr_conv3d_march_fwd(C.byref(xt), ptr(wp), ptr(_f32(bias)), C.byref(yt), int(kernel[0]), int(out_f32), act,
                                              float(slope), ptr(stats), stream_ptr()), "conv3d_march_fwd")
        _count()
        return out, stats, tiles
    if want_stats:
        tiles = lib().rehr_conv3d_stats_tiles(C.byref(yt))
        if tiles > 0:
            stats = torch.empty((n, tiles, cout, 2), dtype=torch.float32, device=x.device)
    wp = _packed(weight, "fwd", h=x_h)
    xt = rt(x, x_h)
    need = lib().rehr_conv3d_splitk_workspace(C.byref(desc), C.byref(xt), ptr(wp), C.byref(yt), 0)
    ws = _ws(need, x.device) if need else None
    with _timed("conv_tapped_gemm_kernel", flops, tag):
        check(lib().rehr_conv3d_fwd_ws(C.byref(desc), C.byref(xt), ptr(wp), ptr(_f32(bias)), C.byref(yt), int(out_f32), act,
                                       float(slope), ptr(stats), ptr(ws), need, stream_ptr()), "conv3d_fwd")
    _count(2 if need else 1)
    if want_stats and stats is None:
        stats, tiles = instnorm_stats_raw(out, y_h)
    return out, stats, tiles


def instnorm_stats_raw(y: torch.Tensor, y_h: bool = False):
    yt = rt(y, y_h)
    tiles = lib().rehr_instnorm_stats_tiles(C.byref(yt))
    stats = torch.empty((y.shape[0], tiles, y.shape[4], 2), dtype=torch.float32, device=y.device)
    check(lib().rehr_instnorm_stats(C.byref(yt), ptr(stats), stream_ptr()), "instnorm_stats")
    _count()
    return stats, tiles


def conv3d_dgrad_raw(dy: torch.Tensor, weight: torch.Tensor, in_shape: Sequence[int], kernel: Triple, stride: Triple,
                     padding: Triple, cache: bool = True, want_chsum: bool = False) -> torch.Tensor:
    """dx = conv^T(dy).  `want_chsum`: where the marching kernel runs, its epilogue also leaves the per-(sample, tile, channel) sums
    of the fp32 accumulators on the result (`dx._rehr_chsum`, f32 [n][tiles][cin][2]): the bias gradient of a transposed conv
    that produced (part of) the conv's input then needs no pass over dx."""
    dy = as_cl(dy)
    n, d, h, w, cin = in_shape
    dx = torch.empty((n, d, h, w, cin), dtype=torch.bfloat16, device=dy.device)
    desc = conv_desc(kernel, stride, padding)
    flops = 2.0 * dy.shape[0] * dy.shape[1] * dy.shape[2] * dy.shape[3] * dy.shape[4] * cin * kernel[0] * kernel[1] * kernel[2]
    tag = f"dgrad {cin}<-{dy.shape[4]} in{d}x{h}x{w} k{kernel} s{stride}" if _ktimer is not None else ""
    if _march_route(desc, dy.shape[4], cin):
        wp = _packed(weight, "march_dgrad", cache)
        dyt, dxt = rt(dy), rt(dx)
        stats = None
        if want_chsum:
            tiles = lib().rehr_conv3d_march_stats_tiles(C.byref(dyt), C.byref(dxt), int(kernel[0]))
            stats = torch.empty((n, tiles, cin, 2), dtype=torch.float32, device=dy.device)
        with _timed("conv_march_kernel", flops, tag):
            check(lib().rehr_conv3d_march_fwd(C.byref(dyt), ptr(wp), None, C.byref(dxt), int(kernel[0]), 0, ACT_NONE, 0.0, ptr(stats),
                                              stream_ptr()), "conv3d_march_dgrad")
        _count()
        if stats is not None:
            dx._rehr_chsum = stats
        return dx
    if USE_MARCH and lib().rehr_conv3d_march_s2dgrad_supported(C.byref(desc), cin, dy.shape[4]) \
            and dy.shape[1] * dy.shape[2] * dy.shape[3] >= 4096 and dy.shape[4] <= 64:
        # stride-2 stage-entry conv: one marching launch per output parity class (small volumes stay on the split-K path;
        # with more than 64 dy channels the resident-weight tile shrinks to 16 columns and the tapped kernel is faster)
        wp = _packed(weight, "s2dgrad", cache, extra=(tuple(kernel), tuple(stride), tuple(padding)))
        dyt, dxt = rt(dy), rt(dx)
        with _timed("conv_march_kernel", flops, tag):
            check(lib().rehr_conv3d_march_s2dgrad(C.byref(desc), C.byref(dyt), ptr(wp), C.byref(dxt), stream_ptr()),
                  "conv3d_march_s2dgrad")
        _count(stride[0] * stride[1] * stride[2])
        return dx
    wp = _packed(weight, "dgrad", cache)
    dyt, dxt = rt(dy), rt(dx)
    need = lib().rehr_conv3d_splitk_workspace(C.byref(desc), C.byref(dyt), ptr(wp), C.byref(dxt), 1)
    ws = _ws(need, dy.device) if need else None
    with _timed("conv_tapped_gemm_kernel", flops, tag):
        check(lib().rehr_conv3d_dgrad_ws(C.byref(desc), C.byref(dyt), ptr(wp), None, C.byref(dxt), 0, ACT_NONE, 0.0, ptr(ws), need,
                                         stream_ptr()), "conv3d_dgrad")
    _count(stride[0] * stride[1] * stride[2] * (2 if need else 1))
    return dx


def _wgrad_route(desc, xt, dyt) -> str:
    if USE_MARCH and lib().rehr_conv3d_wgrad_march_supported(C.byref(desc), C.byref(xt), C.byref(dyt)):
        return "march"
    # one marching pass per parity class of x; its fixed cost (TMEM drain + partial reduction per class) only pays off on
    # the full-resolution stage-entry conv (measured: 32->64 @128^3 0.86 -> 0.57 ms, 64->128 @64^3 0.14 -> 0.48 ms)
    if USE_MARCH and dyt.n * dyt.d * dyt.h * dyt.w >= S2_WGRAD_MARCH_MIN_VOXELS \
            and lib().rehr_conv3d_wgrad_march_s2_supported(C.byref(desc), C.byref(xt), C.byref(dyt)):
        return "march_s2"
    return "generic"


def wgrad_route(x_shape, dy_shape, kernel: Triple, stride: Triple, padding: Triple) -> str:
    """Which kernel conv3d_wgrad_raw picks for these (channels-last, unpitched) shapes: 'march', 'march_s2' or 'generic'."""
    xt = L.RehrTensor(0, *[int(v) for v in x_shape], int(x_shape[4]), 0)
    dyt = L.RehrTensor(0, *[int(v) for v in dy_shape], int(dy_shape[4]), 0)
    return _wgrad_route(conv_desc(kernel, stride, padding), xt, dyt)


def conv3d_wgrad_raw(x: torch.Tensor, dy: torch.Tensor, wshape: Sequence[int], kernel: Triple, stride: Triple,
                     padding: Triple, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    x, dy = as_cl(x), as_cl(dy)
    dw = out if out is not None else torch.empty(tuple(wshape), dtype=torch.float32, device=x.device)
    desc = conv_desc(kernel, stride, padding)
    xt, dyt = rt(x), rt(dy)
    flops = 2.0 * dy.shape[0] * dy.shape[1] * dy.shape[2] * dy.shape[3] * dy.shape[4] * x.shape[4] * kernel[0] * kernel[1] * kernel[2]
    tag = f"wgrad {x.shape[4]}->{dy.shape[4]} in{x.shape[1]}x{x.shape[2]}x{x.shape[3]} k{kernel} s{stride}" if _ktimer is not None else ""
    route = _wgrad_route(desc, xt, dyt)
    if route == "march":
        need = lib().rehr_conv3d_wgrad_march_workspace(C.byref(xt), C.byref(dyt), int(kernel[0]))
        ws = _ws(need, x.device)
        with _timed("wgrad_march_kernel", flops, tag):
            check(lib().rehr_conv3d_wgrad_march(C.byref(xt), C.byref(dyt), int(kernel[0]), int(wshape[0]), ptr(dw), 0, ptr(ws),
                                                need, stream_ptr()), "conv3d_wgrad_march")
        _count(2)
        return dw
    if route == "march_s2":
        need = lib().rehr_conv3d_wgrad_march_s2_workspace(C.byref(desc), C.byref(xt), C.byref(dyt))
        ws = _ws(need, x.device)
        with _timed("wgrad_march_kernel", flops, tag):
            check(lib().rehr_conv3d_wgrad_march_s2(C.byref(desc), C.byref(xt), C.byref(dyt), ptr(dw), 0, ptr(ws), need,
                                                   stream_ptr()), "conv3d_wgrad_march_s2")
        _count(2 * stride[0] * stride[1] * stride[2])
        return dw
    need = lib().rehr_conv3d_wgrad_workspace(C.byref(desc), C.byref(xt), C.byref(dyt))
    if need == 0:
        raise L.RehrError(f"conv3d_wgrad: unsupported configuration x={tuple(x.shape)} dy={tuple(dy.shape)}")
    ws = _ws(need, x.device)
    with _timed("conv_wgrad_kernel", flops, tag):
        check(lib().rehr_conv3d_wgrad(C.byref(desc), C.byref(xt), C.byref(dyt), ptr(dw), 0, ptr(ws), need, stream_ptr()),
              "conv3d_wgrad")
    _count(2)
    return dw


def channel_sum_raw(x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    x = as_cl(x)
    xt = rt(x)
    if out is None:
        out = torch.empty((x.shape[4],), dtype=torch.float32, device=x.device)
    need = lib().rehr_channel_sum_workspace(C.byref(xt))
    ws = _ws(need, x.device)
    check(lib().rehr_channel_sum(C.byref(xt), ptr(out), 0, ptr(ws), need, stream_ptr()), "channel_sum")
    _count(2)
    return out


def act_bwd_raw(a: torch.Tensor, da: torch.Tensor, act: int, slope: float, a_h: bool = False) -> torch.Tensor:
    """dy = da * act'(.) evaluated from the activation OUTPUT `a` (valid for ReLU and LeakyReLU with slope > 0)."""
    a, da = as_cl(a), as_cl(da)
    if act == ACT_NONE:
        return da
    dy = torch.empty(a.shape, dtype=torch.bfloat16, device=a.device)
    at, dat, dyt = rt(a, a_h), rt(da), rt(dy)
    check(lib().rehr_act_bwd(C.byref(at), C.byref(dat), act, float(slope), C.byref(dyt), stream_ptr()), "act_bwd")
    _count()
    return dy


# --------------------------------------------------------------------------------------------------
# Conv3d -> InstanceNorm3d(affine) -> LeakyReLU   (dynamic_network_architectures ConvDropoutNormReLU,
# constructed at models/seg_model.py:174-191 with the ops chosen at train_all.py:474-493)
# --------------------------------------------------------------------------------------------------
class ConvNormAct(torch.autograd.Function):
    """Returns the activation `a` (format FWD_FP16) and, when a gradient will be needed, its bf16 twin `a2` (the weight-gradient
    operand of the consumer; written by the same normalise pass).  `a2` is a non-differentiable side tensor; the gradient of
    output 0 is d(loss)/d(activation)."""

    @staticmethod
    def forward(ctx, x, weight, bias, gamma, beta, kernel, stride, padding, eps, slope, small_cin, cat_room):
        dev = x.device
        cout = weight.shape[0]
        desc = conv_desc(kernel, stride, padding)
        a_h = FWD_FP16
        train = any(ctx.needs_input_grad)
        ctx.set_materialize_grads(False)   # the twin output is non-differentiable: no zero-filled gradient tensor for it

        def alloc(shape5):
            if cat_room:
                # the output doubles as the skip half of the decoder's concat buffer [up | skip] (models/seg_model.py:37):
                # allocate 2C channels and write into the upper half, so torch.cat never runs
                buf = torch.empty((*shape5[:4], 2 * cout), dtype=torch.bfloat16, device=dev)
                return _alias(buf, cout, shape5, buf.stride())
            return torch.empty(tuple(shape5), dtype=torch.bfloat16, device=dev)

        # the pre-normalisation conv output y is stored as fp16 whatever FWD_FP16 says: it is never an MMA operand, only the
        # InstanceNorm kernels read it
        if small_cin:
            # x is the caller's NCDHW fp32 tensor (train_all.py:524)
            xs = _f32(x)
            n, cin, d, h, w = xs.shape
            od, oh, ow = (_out_size(i, k, s, p) for i, k, s, p in zip((d, h, w), kernel, stride, padding))
            y = torch.empty((n, od, oh, ow, cout), dtype=torch.bfloat16, device=dev)
            yt = rt(y, True)
            tiles = lib().rehr_instnorm_stats_tiles(C.byref(yt))
            stats = torch.empty((n, tiles, cout, 2), dtype=torch.float32, device=dev)
            # NB the conv bias is NOT added: a per-channel constant is removed exactly by the InstanceNorm that follows
            # (mean shifts by the same constant, variance is unchanged), so lrelu(IN(conv+b)) == lrelu(IN(conv)).
            with _sink("y"):
                check(lib().rehr_conv3d_smallcin_fwd(C.byref(desc), ptr(xs), n, cin, d, h, w, ptr(_f32(weight)), None,
                                                     C.byref(yt), ACT_NONE, 0.0, ptr(stats), stream_ptr()), "smallcin_fwd")
            _count(2)
            x_saved = xs
        else:
            xc = as_cl(x)
            x_saved = bf_twin(x) if train else None   # bf16 operand of this layer's weight gradient
            with _sink("y"):
                y, stats, tiles = conv3d_raw(xc, weight, None, kernel, stride, padding, want_stats=True, x_h=is_h(x), y_h=True)
        n = y.shape[0]
        vox = y.shape[1] * y.shape[2] * y.shape[3]
        mean = torch.empty((n, cout), dtype=torch.float32, device=dev)
        rstd = torch.empty((n, cout), dtype=torch.float32, device=dev)
        g32, b32 = _f32(gamma), _f32(beta)
        ctx.cfg = (kernel, stride, padding, slope, small_cin, bias is not None)
        ctx.wref = weakref.ref(weight)
        ctx.x_upcat = bool(getattr(x, "_rehr_upcat", False))   # x = [up | skip]: the transposed conv wants channel sums of dx
        check(lib().rehr_instnorm_finalize(ptr(stats), n, tiles, cout, vox, float(eps), ptr(mean), ptr(rstd), stream_ptr()),
              "instnorm_finalize")
        want_twin = a_h and train
        a = alloc(y.shape)
        a2 = alloc(y.shape) if want_twin else None
        yt, at = rt(y, True), rt(a, a_h)
        a2t = rt(a2, False) if a2 is not None else None
        with _sink("a"):
            check(lib().rehr_instnorm_lrelu_apply(C.byref(yt), ptr(mean), ptr(rstd), ptr(g32), ptr(b32), float(slope), C.byref(at),
                                                  C.byref(a2t) if a2t is not None else None, stream_ptr()), "instnorm_lrelu_apply")
        _count(2)
        ctx.save_for_backward(x_saved, weight, gamma, beta, y, mean, rstd)
        ctx.skip_key = (a.untyped_storage().data_ptr(), a.storage_offset()) if cat_room else None
        if a2 is not None:
            ctx.mark_non_differentiable(a2)
        return a, a2

    @staticmethod
    def backward(ctx, da, _twin_unused=None):
        if da is None:
            return (None,) * 12
        x, weight, gamma, beta, y, mean, rstd = ctx.saved_tensors
        weight = _orig_weight(ctx, weight)
        kernel, stride, padding, slope, small_cin, has_bias = ctx.cfg
        dev = y.device
        da = as_cl(da)
        n, cout = y.shape[0], y.shape[4]
        yt, dat = rt(y, True), rt(da)
        da2 = _skip_grads.pop(ctx.skip_key, None) if ctx.skip_key is not None else None
        da2t = rt(da2) if da2 is not None else None
        da2p = C.byref(da2t) if da2t is not None else None
        g32 = _f32(gamma) if gamma is not None else None
        b32 = _f32(beta) if beta is not None else None
        sums = torch.empty((n, cout, 2), dtype=torch.float32, device=dev)
        dgamma = torch.empty((cout,), dtype=torch.float32, device=dev)
        dbeta = torch.empty((cout,), dtype=torch.float32, device=dev)
        tiles = lib().rehr_instnorm_stats_tiles(C.byref(yt))
        partial = torch.empty((n, tiles, cout, 2), dtype=torch.float32, device=dev)
        check(lib().rehr_instnorm_lrelu_bwd_reduce(C.byref(yt), C.byref(dat), da2p, ptr(mean), ptr(rstd), ptr(g32), ptr(b32),
                                                   float(slope), ptr(partial), stream_ptr()), "instnorm_bwd_reduce")
        check(lib().rehr_instnorm_lrelu_bwd_finalize(ptr(partial), n, tiles, cout, ptr(rstd), ptr(sums), ptr(dgamma), ptr(dbeta),
                                                     0, stream_ptr()), "instnorm_bwd_finalize")
        dy = torch.empty_like(y)
        dyt = rt(dy)
        check(lib().rehr_instnorm_lrelu_bwd_apply(C.byref(yt), C.byref(dat), da2p, ptr(mean), ptr(rstd), ptr(g32), ptr(b32),
                                                  float(slope), ptr(sums), C.byref(dyt), stream_ptr()), "instnorm_bwd_apply")
        _count(3)
        desc = conv_desc(kernel, stride, padding)
        dx = None
        if small_cin:
            nb, cin, d, h, w = x.shape
            need = lib().rehr_conv3d_smallcin_wgrad_workspace(C.byref(desc), cin, C.byref(dyt))
            ws = _ws(need, dev)
            dw = torch.empty(weight.shape, dtype=torch.float32, device=dev)
            check(lib().rehr_conv3d_smallcin_wgrad(C.byref(desc), ptr(x), nb, cin, d, h, w, C.byref(dyt), ptr(dw), 0, ptr(ws),
                                                   need, stream_ptr()), "smallcin_wgrad")
            _count(2)
            if ctx.needs_input_grad[0]:
                dx = torch.empty(x.shape, dtype=torch.float32, device=dev)
                check(lib().rehr_conv3d_smallcin_dgrad(C.byref(desc), C.byref(dyt), ptr(_f32(weight)), ptr(dx), nb, cin, d, h, w,
                                                       stream_ptr()), "smallcin_dgrad")
                _count()
        else:
            dx, dw = _dgrad_and_wgrad(x, dy, weight, weight.shape, kernel, stride, padding, ctx.needs_input_grad[0],
                                      want_chsum=ctx.x_upcat)
        # A per-channel constant added before InstanceNorm is removed by the mean subtraction: d(loss)/d(bias) == 0
        # exactly (PyTorch's value is rounding noise of the same sum).
        dbias = _zero_grad_slice(cout, dev) if has_bias else None
        return dx, dw.to(weight.dtype), dbias, dgamma if gamma is not None else None, dbeta if beta is not None else None, \
            None, None, None, None, None, None, None


def conv_norm_act(x, weight, bias, gamma, beta, kernel, stride, padding, eps=1e-5, slope=0.01, small_cin=False,
                  cat_room=False):
    a, a2 = ConvNormAct.apply(x, weight, bias, gamma, beta, tuple(kernel), tuple(stride), tuple(padding), float(eps),
                              float(slope), bool(small_cin), bool(cat_room))
    if FWD_FP16:
        mark_h(a, a2)
    if cat_room:
        a._rehr_cat = (2 * weight.shape[0], weight.shape[0])
        if a2 is not None:
            a2._rehr_cat = a._rehr_cat
    return a


# --------------------------------------------------------------------------------------------------
# Conv3d (+bias) (+ReLU / LeakyReLU), no norm: sr_head (models/seg_model.py:197-199), FLAVR Conv3DSimple /
# Conv_3d / Conv_2d (models/FLAVR/resnet_3D.py:19-33, models/FLAVR/FLAVR_arch.py:24-88)
# --------------------------------------------------------------------------------------------------
class ConvAct(torch.autograd.Function):
    """`want_pool`: also return the per-(n, c) mean of the (pre-activation) output, taken from the conv epilogue's fused
    partial sums -- the global average pool of the SE gate that follows (resnet_3D.py:112-114).  It is a non-differentiable
    hint: `se_gate` recomputes nothing and owns the gradient through the pool."""

    @staticmethod
    def forward(ctx, x, weight, bias, kernel, stride, padding, act, slope, out_f32, want_pool):
        x = bf_twin(x)   # layers without InstanceNorm (sr_head, FLAVR) run on bf16 operands
        y, stats, tiles = conv3d_raw(x, weight, bias, kernel, stride, padding, act=act, slope=slope, out_f32=out_f32,
                                     want_stats=want_pool)
        ctx.save_for_backward(x, weight, y if act != ACT_NONE else None)
        ctx.cfg = (kernel, stride, padding, act, slope, bias is not None)
        ctx.wref = weakref.ref(weight)
        if want_pool:
            if act != ACT_NONE:
                raise L.RehrError("want_pool needs the pre-activation output (act=ACT_NONE)")
            n, cout = y.shape[0], y.shape[4]
            pool = torch.empty((n, cout), dtype=torch.float32, device=y.device)
            rstd = torch.empty((n, cout), dtype=torch.float32, device=y.device)
            check(lib().rehr_instnorm_finalize(ptr(stats), n, tiles, cout, y.shape[1] * y.shape[2] * y.shape[3], 1e-5, ptr(pool),
                                               ptr(rstd), stream_ptr()), "instnorm_finalize")
            _count()
            ctx.mark_non_differentiable(pool)
            return y, pool
        return y

    @staticmethod
    def backward(ctx, da, *_unused):
        x, weight, y = ctx.saved_tensors
        weight = _orig_weight(ctx, weight)
        kernel, stride, padding, act, slope, has_bias = ctx.cfg
        dy = act_bwd_raw(y, da, act, slope) if act != ACT_NONE else as_cl(da)
        cout = weight.shape[0]
        if cout % 16 != 0:
            # thin heads (sr_head.2: 16 -> 2, models/seg_model.py:199): the GEMM operands need >= 16 channels, so the
            # gradient is zero-padded to 16 channels (exact: the padded filters are zero)
            cp = (cout + 15) // 16 * 16
            dyp = torch.zeros((*dy.shape[:4], cp), dtype=torch.bfloat16, device=dy.device)
            dyp[..., :cout] = dy
            wpad = torch.zeros((cp, *weight.shape[1:]), dtype=torch.float32, device=dy.device)
            wpad[:cout] = weight.detach()
            dx = conv3d_dgrad_raw(dyp, wpad, x.shape, kernel, stride, padding, cache=False) if ctx.needs_input_grad[0] else None
            dw = conv3d_wgrad_raw(x, dyp, wpad.shape, kernel, stride, padding)[:cout]
            dy = dyp
        else:
            dx, dw = _dgrad_and_wgrad(x, dy, weight, weight.shape, kernel, stride, padding, ctx.needs_input_grad[0])
        db = channel_sum_raw(dy)[:cout] if has_bias else None
        return dx, dw.to(weight.dtype), db, None, None, None, None, None, None, None


def conv_act(x, weight, bias, kernel, stride, padding, act=ACT_NONE, slope=0.0, out_f32=False, want_pool=False):
    return ConvAct.apply(x, weight, bias, tuple(kernel), tuple(stride), tuple(padding), int(act), float(slope), bool(out_f32),
                         bool(want_pool))


# --------------------------------------------------------------------------------------------------
# SE "feature gating" tail (models/FLAVR/resnet_3D.py:100-116 and its users :140-151, FLAVR_arch.py:49-51,75-77):
#   y = act( x * sigmoid(W mean_v(x) + b) (+ residual) )
# --------------------------------------------------------------------------------------------------
class SEGate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, pool, attn_w, attn_b, residual, act, slope):
        x = as_cl(x)
        n, d, h, w, c = x.shape
        vox = d * h * w
        if pool is None:
            stats, tiles = instnorm_stats_raw(x)
            pool = torch.empty((n, c), dtype=torch.float32, device=x.device)
            rstd = torch.empty_like(pool)
            check(lib().rehr_instnorm_finalize(ptr(stats), n, tiles, c, vox, 1e-5, ptr(pool), ptr(rstd), stream_ptr()),
                  "instnorm_finalize")
            _count()
        w2 = attn_w.detach().reshape(c, c).float()
        gate = torch.sigmoid(torch.addmm(attn_b.detach().float(), pool, w2.t())).contiguous()  # [n, c], tiny
        res = as_cl(residual) if residual is not None else None
        y = torch.empty_like(x)
        xt, yt = rt(x), rt(y)
        rst = rt(res) if res is not None else None
        check(lib().rehr_segate_scale_add_act(C.byref(xt), ptr(gate), C.byref(rst) if rst is not None else None, act, float(slope),
                                              C.byref(yt), stream_ptr()), "segate_scale_add_act")
        _count()
        ctx.save_for_backward(x, gate, pool, attn_w, y if act != ACT_NONE else None)
        ctx.cfg = (act, slope, residual is not None)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, gate, pool, attn_w, y = ctx.saved_tensors
        act, slope, has_res = ctx.cfg
        dy = as_cl(dy)
        n, d, h, w, c = x.shape
        vox = d * h * w
        xt, dyt = rt(x), rt(dy)
        yt = rt(y) if y is not None else None
        tiles = lib().rehr_instnorm_stats_tiles(C.byref(xt))
        partial = torch.empty((n, tiles, c, 2), dtype=torch.float32, device=x.device)
        check(lib().rehr_segate_bwd_reduce(C.byref(xt), C.byref(yt) if yt is not None else None, C.byref(dyt), act, float(slope),
                                           ptr(partial), stream_ptr()), "segate_bwd_reduce")
        sums = torch.empty((n, c, 2), dtype=torch.float32, device=x.device)
        check(lib().rehr_instnorm_lrelu_bwd_finalize(ptr(partial), n, tiles, c, None, ptr(sums), None, None, 0, stream_ptr()),
              "segate_bwd_finalize")
        dgate = sums[..., 0]
        dz = dgate * gate * (1.0 - gate)                       # [n, c]
        w2 = attn_w.detach().reshape(c, c).float()
        dw = (dz.t() @ pool).reshape(attn_w.shape).to(attn_w.dtype)
        db = dz.sum(0)
        shift = ((dz @ w2) / float(vox)).contiguous()           # gradient through the average pool, per voxel
        dx = torch.empty_like(x)
        dxt = rt(dx)
        dres = None
        drt = None
        if has_res:
            if act == ACT_NONE:
                dres = dy
            else:
                dres = torch.empty_like(x)
                drt = rt(dres)
        check(lib().rehr_segate_bwd_apply(C.byref(yt) if yt is not None else None, C.byref(dyt), act, float(slope), ptr(gate), ptr(shift),
                                          C.byref(dxt), C.byref(drt) if drt is not None else None, stream_ptr()), "segate_bwd_apply")
        _count(3)
        return dx, None, dw, db, dres, None, None


def se_gate(x, attn_w, attn_b, residual=None, act=ACT_NONE, slope=0.0, pool=None):
    """SEGating (+ residual add + activation).  `pool` = the [n, c] mean of x if the producer already has it."""
    return SEGate.apply(x, pool, attn_w, attn_b, residual, int(act), float(slope))


# --------------------------------------------------------------------------------------------------
# small-Cin stem without normalisation: FLAVR BasicStem Conv3d(2, 64, k(3,7,7), s(1,2,2), p(1,3,3)) + ReLU
# (models/FLAVR/resnet_3D.py:42-50); x is the caller's NCDHW fp32 tensor
# --------------------------------------------------------------------------------------------------
class SmallCinConvAct(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, kernel, stride, padding, act, slope):
        xs = _f32(x)
        n, cin, d, h, w = xs.shape
        cout = weight.shape[0]
        od, oh, ow = (_out_size(i, k, s, p) for i, k, s, p in zip((d, h, w), kernel, stride, padding))
        y = torch.empty((n, od, oh, ow, cout), dtype=torch.bfloat16, device=xs.device)
        desc = conv_desc(kernel, stride, padding)
        yt = rt(y)
        check(lib().rehr_conv3d_smallcin_fwd(C.byref(desc), ptr(xs), n, cin, d, h, w, ptr(_f32(weight)), ptr(_f32(bias)), C.byref(yt),
                                             act, float(slope), None, stream_ptr()), "smallcin_fwd")
        _count()
        ctx.save_for_backward(xs, weight, y if act != ACT_NONE else None)
        ctx.cfg = (kernel, stride, padding, act, slope, bias is not None)
        return y

    @staticmethod
    def backward(ctx, da):
        xs, weight, y = ctx.saved_tensors
        kernel, stride, padding, act, slope, has_bias = ctx.cfg
        dy = act_bwd_raw(y, da, act, slope) if act != ACT_NONE else as_cl(da)
        desc = conv_desc(kernel, stride, padding)
        n, cin, d, h, w = xs.shape
        dyt = rt(dy)
        need = lib().rehr_conv3d_smallcin_wgrad_workspace(C.byref(desc), cin, C.byref(dyt))
        ws = _ws(need, xs.device)
        dw = torch.empty(weight.shape, dtype=torch.float32, device=xs.device)
        check(lib().rehr_conv3d_smallcin_wgrad(C.byref(desc), ptr(xs), n, cin, d, h, w, C.byref(dyt), ptr(dw), 0, ptr(ws), need,
                                               stream_ptr()), "smallcin_wgrad")
        _count(2)
        dx = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty(xs.shape, dtype=torch.float32, device=xs.device)
            check(lib().rehr_conv3d_smallcin_dgrad(C.byref(desc), C.byref(dyt), ptr(_f32(weight)), ptr(dx), n, cin, d, h, w,
                                                   stream_ptr()), "smallcin_dgrad")
            _count()
        db = channel_sum_raw(dy) if has_bias else None
        return dx, dw.to(weight.dtype), db, None, None, None, None, None


def smallcin_conv_act(x, weight, bias, kernel, stride, padding, act=ACT_NONE, slope=0.0):
    return SmallCinConvAct.apply(x, weight, bias, tuple(kernel), tuple(stride), tuple(padding), int(act), float(slope))


# --------------------------------------------------------------------------------------------------
# ConvTranspose3d: nnU-Net decoder up-sampling, kernel == stride (models/seg_model.py:36 via UNetDecoder.transpconvs),
# and FLAVR upConv3D k(3,4,4) s(1,2,2) p(1,1,1) (models/FLAVR/FLAVR_arch.py:49-51)
# --------------------------------------------------------------------------------------------------
class ConvTranspose(torch.autograd.Function):
    """`skip` (optional): an encoder activation that lives in the upper half of a 2C concat buffer (conv_norm_act with
    cat_room); the up-sampled tensor is then written straight into the lower half and the whole buffer is returned --
    `torch.cat((up, skip), 1)` of models/seg_model.py:37 without the copy."""

    @staticmethod
    def forward(ctx, x, weight, bias, skip, kernel, stride, padding, act, slope):
        x_h = is_h(x)
        train = any(ctx.needs_input_grad)
        ctx.set_materialize_grads(False)          # no zero-filled gradient for the non-differentiable twin output
        x_bf = bf_twin(x) if train else None      # the bf16 operand of the weight gradient
        x = as_cl(x)
        n, d, h, w, cin = x.shape
        cout = weight.shape[1]
        od, oh, ow = ((i - 1) * s - 2 * p + k for i, k, s, p in zip((d, h, w), kernel, stride, padding))
        desc = conv_desc(kernel, stride, padding)
        ctx.cat = skip is not None
        ctx.skip_key = None
        full2 = None

        def whole(t):   # the [up | skip] buffer a cat_room activation lives in
            tot, off = t._rehr_cat
            return _alias(t, t.storage_offset() - off, (n, od, oh, ow, tot), (od * oh * ow * tot, oh * ow * tot, ow * tot, tot, 1))

        if skip is not None:
            tot, off = skip._rehr_cat
            ctx.skip_key = (skip.untyped_storage().data_ptr(), skip.storage_offset())
            if tot != 2 * cout or off != cout or tuple(skip.shape) != (n, od, oh, ow, cout):
                raise L.RehrError("conv_transpose: skip does not sit in a matching [up | skip] concat buffer")
            if is_h(skip) != x_h:
                raise L.RehrError("conv_transpose: input and skip use different 16-bit storage formats")
            full = whole(skip)
            y = full[..., :cout]
        else:
            full = None
            y = torch.empty((n, od, oh, ow, cout), dtype=torch.bfloat16, device=x.device)
        xt, yt = rt(x, x_h), rt(y, x_h)
        twin_done = False
        with _sink("up"):
            if lib().rehr_convtranspose3d_fused_supported(C.byref(desc), cin, cout):
                wp = _packed(weight, "tconv_fused", h=x_h)  # [T][Cout][Cin]
                tw = getattr(skip, "_rehr_bf", None) if (skip is not None and x_h and train) else None
                if tw is not None and getattr(tw, "_rehr_cat", None) == skip._rehr_cat:
                    # the bf16 twin of the up-sampled half goes straight into the twin's [up | skip] buffer from the same epilogue
                    full2 = whole(tw)
                    y2t = rt(full2[..., :cout], False)
                    check(lib().rehr_convtranspose3d_fused_fwd2(C.byref(desc), C.byref(xt), ptr(wp), ptr(_f32(bias)), C.byref(yt),
                                                                C.byref(y2t), act, float(slope), stream_ptr()), "convtranspose3d_fused_fwd2")
                    twin_done = True
                    path_hits["tconv_twin_from_epilogue"] += 1
                else:
                    check(lib().rehr_convtranspose3d_fused_fwd(C.byref(desc), C.byref(xt), ptr(wp), ptr(_f32(bias)), C.byref(yt), act,
                                                               float(slope), stream_ptr()), "convtranspose3d_fused_fwd")
                _count()
            else:
                wp = _packed(weight, "dgrad", h=x_h)  # [Cout][T][Cin]
                check(lib().rehr_convtranspose3d_fwd(C.byref(desc), C.byref(xt), ptr(wp), ptr(_f32(bias)), C.byref(yt), act,
                                                     float(slope), stream_ptr()), "convtranspose3d_fwd")
                _count(stride[0] * stride[1] * stride[2])
        if x_h and train and not twin_done:
            # bf16 twin of the result for the weight-gradient GEMM of the consumer: the skip half already has one (written by
            # the skip's normalise pass), the up-sampled half is converted here
            if skip is not None:
                tw = getattr(skip, "_rehr_bf", None)
                if tw is not None and getattr(tw, "_rehr_cat", None) == skip._rehr_cat:
                    full2 = whole(tw)
                    convert16_raw(y, True, False, out=full2[..., :cout])
                else:
                    full2 = convert16_raw(full, True, False)
            else:
                full2 = convert16_raw(y, True, False)
        ctx.save_for_backward(x_bf, weight, y if act != ACT_NONE else None)
        ctx.cfg = (kernel, stride, padding, act, slope, bias is not None, x_h)
        ctx.wref = weakref.ref(weight)
        out = full if skip is not None else y
        if full2 is not None:
            ctx.mark_non_differentiable(full2)
        return out, full2

    @staticmethod
    def backward(ctx, da, _twin_unused=None):
        if da is None:
            return (None,) * 9
        x, weight, y = ctx.saved_tensors
        weight = _orig_weight(ctx, weight)
        kernel, stride, padding, act, slope, has_bias, y_h = ctx.cfg
        dskip = None
        chsum = getattr(da, "_rehr_chsum", None) if ctx.cat else None   # left by the marching input gradient that produced da
        if ctx.cat:  # da is the gradient of the whole [up | skip] buffer
            cout = weight.shape[1]
            da = as_cl(da)
            dskip = da[..., cout:]
            da = da[..., :cout]
            if ctx.skip_key is not None and ctx.needs_input_grad[3]:
                _skip_grads[ctx.skip_key] = dskip   # picked up by the skip producer's backward as its second gradient operand
                dskip = None
        dy = act_bwd_raw(y, da, act, slope, a_h=y_h) if act != ACT_NONE else as_cl(da)
        desc = conv_desc(kernel, stride, padding)
        dyt, xt = rt(dy), rt(x)
        need = lib().rehr_convtranspose3d_wgrad_workspace(C.byref(desc), C.byref(xt), C.byref(dyt))
        if need == 0:
            raise L.RehrError("convtranspose3d_wgrad: unsupported configuration")
        dw = torch.empty(weight.shape, dtype=torch.float32, device=x.device)
        db = torch.empty((weight.shape[1],), dtype=torch.float32, device=x.device) if has_bias else None

        def weight_and_bias_grads():
            ws = _ws(need, x.device)
            check(lib().rehr_convtranspose3d_wgrad(C.byref(desc), C.byref(xt), C.byref(dyt), ptr(dw), 0, ptr(ws), need, stream_ptr()),
                  "convtranspose3d_wgrad")
            _count(2)
            if has_bias:
                if chsum is not None and act == ACT_NONE and chsum.shape[2] >= weight.shape[1]:
                    # bias gradient = sum over voxels of d(up): the fp32 accumulator sums of the producing kernel's epilogue
                    torch.sum(chsum[:, :, :weight.shape[1], 0], dim=(0, 1), out=db)
                    path_hits["tconv_bias_from_epilogue_sums"] += 1
                else:
                    channel_sum_raw(dy, out=db)

        voxels = dy.shape[0] * dy.shape[1] * dy.shape[2] * dy.shape[3]
        fk = None
        if ctx.needs_input_grad[0] and WGRAD_SIDE_STREAM and _ktimer is None and voxels <= WGRAD_SIDE_MAX_VOXELS:
            fk = _fork(x.device)          # small layer: weight / bias gradients side by side with the input gradient
            with fk:
                weight_and_bias_grads()
        dx = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
            dxt = rt(dx)
            wp = _packed(weight, "fwd")  # [Cin][T][Cout]
            check(lib().rehr_convtranspose3d_dgrad(C.byref(desc), C.byref(dyt), ptr(wp), C.byref(dxt), stream_ptr()),
                  "convtranspose3d_dgrad")
            _count()
        if fk is not None:
            fk.join()
        else:
            weight_and_bias_grads()
        return dx, dw.to(weight.dtype), db, dskip, None, None, None, None, None


def conv_transpose(x, weight, bias, kernel, stride, padding=(0, 0, 0), act=ACT_NONE, slope=0.0, skip=None):
    """ConvTranspose3d; with `skip` (an activation produced with cat_room) returns the [up | skip] concat buffer."""
    if skip is not None and concat_room_of(skip) is None:
        raise L.RehrError("conv_transpose(skip=...): the skip tensor was not produced with cat_room=True")
    out, twin = ConvTranspose.apply(x, weight, bias, skip, tuple(kernel), tuple(stride), tuple(padding), int(act), float(slope))
    if is_h(x):
        mark_h(out, twin)
    if skip is not None:
        out._rehr_upcat = True
    return out


# --------------------------------------------------------------------------------------------------
# 1x1x1 segmentation head (decoder.seg_layers[-1], models/seg_model.py:44): NDHWC bf16 -> NCDHW fp32 logits
# --------------------------------------------------------------------------------------------------
class SegHead(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias):
        x_h = is_h(x)
        x = as_cl(x)
        n, d, h, w, cin = x.shape
        cout = weight.shape[0]
        y = torch.empty((n, cout, d, h, w), dtype=torch.float32, device=x.device)
        w2 = _f32(weight).reshape(cout, cin)
        xt = rt(x, x_h)
        ctx.x_h = x_h
        check(lib().rehr_pointwise_fwd(C.byref(xt), ptr(w2), ptr(_f32(bias)), ptr(y), cout, stream_ptr()), "pointwise_fwd")
        _count()
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        x, weight = ctx.saved_tensors
        cout, cin = weight.shape[0], weight.shape[1]
        dy = _f32(dy)
        xt = rt(x, ctx.x_h)
        dx = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
        dxt = rt(dx)
        dw = torch.empty((cout, cin), dtype=torch.float32, device=x.device)
        db = torch.empty((cout,), dtype=torch.float32, device=x.device)
        need = lib().rehr_pointwise_bwd_workspace(C.byref(xt), cout)
        ws = _ws(need, x.device)
        check(lib().rehr_pointwise_bwd(C.byref(xt), ptr(dy), ptr(_f32(weight).reshape(cout, cin)), cout, C.byref(dxt), ptr(dw), ptr(db),
                                       0, ptr(ws), need, stream_ptr()), "pointwise_bwd")
        _count(2)
        return dx, dw.reshape(weight.shape).to(weight.dtype), db if ctx.has_bias else None


def seg_head(x, weight, bias):
    return SegHead.apply(x, weight, bias)


# --------------------------------------------------------------------------------------------------
# F.interpolate(scale_factor=(s,1,1), mode='trilinear', align_corners=True)  (models/seg_model.py:204)
# --------------------------------------------------------------------------------------------------
class UpsampleD(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, out_d):
        x_h = is_h(x)
        x = as_cl(x)
        n, d, h, w, c = x.shape
        y = torch.empty((n, out_d, h, w, c), dtype=torch.bfloat16, device=x.device)   # bf16: the sr_head has no InstanceNorm
        xt, yt = rt(x, x_h), rt(y)
        with _sink("sr_up"):
            check(lib().rehr_upsample_linear_d(C.byref(xt), C.byref(yt), stream_ptr()), "upsample_linear_d")
        _count()
        ctx.in_shape = tuple(x.shape)
        return y

    @staticmethod
    def backward(ctx, dy):
        dy = as_cl(dy)
        dx = torch.empty(ctx.in_shape, dtype=torch.bfloat16, device=dy.device)
        dyt, dxt = rt(dy), rt(dx)
        check(lib().rehr_upsample_linear_d_bwd(C.byref(dyt), C.byref(dxt), stream_ptr()), "upsample_linear_d_bwd")
        _count()
        return dx, None


def upsample_linear_d(x, out_d: int):
    return UpsampleD.apply(x, int(out_d))


# --------------------------------------------------------------------------------------------------
# layout adapters at the model boundary
# --------------------------------------------------------------------------------------------------
class ToChannelsLast(torch.autograd.Function):
    """NCDHW fp32 -> NDHWC bf16."""

    @staticmethod
    def forward(ctx, x):
        xs = _f32(x)
        n, c, d, h, w = xs.shape
        y = torch.empty((n, d, h, w, c), dtype=torch.bfloat16, device=xs.device)
        yt = rt(y)
        check(lib().rehr_ncdhw_f32_to_ndhwc_bf16(ptr(xs), C.byref(yt), stream_ptr()), "ncdhw_to_ndhwc")
        _count()
        return y

    @staticmethod
    def backward(ctx, dy):
        return FromChannelsLast.apply(dy)


class FromChannelsLast(torch.autograd.Function):
    """NDHWC bf16 -> NCDHW fp32."""

    @staticmethod
    def forward(ctx, x):
        x_h = is_h(x)
        x = as_cl(x)
        n, d, h, w, c = x.shape
        y = torch.empty((n, c, d, h, w), dtype=torch.float32, device=x.device)
        xt = rt(x, x_h)
        check(lib().rehr_ndhwc_bf16_to_ncdhw_f32(C.byref(xt), ptr(y), stream_ptr()), "ndhwc_to_ncdhw")
        _count()
        return y

    @staticmethod
    def backward(ctx, dy):
        return ToChannelsLast.apply(dy)


def to_channels_last(x):
    return ToChannelsLast.apply(x)


def from_channels_last(x):
    return FromChannelsLast.apply(x)
