"""Opt-in report of fp16 saturation in the SegModel forward pass.

The SegModel forward stores its activations in fp16 (functional.FWD_FP16; the pre-normalisation conv output `y` always), and
an fp16 store saturates: a value of magnitude >= 65520 is written as +-65504 (NaN stays NaN).  Nothing else tells the user:
the InstanceNorm statistics come from the fp32 accumulators, but the normalise pass reads the clipped `y`.  Inputs that were
not z-scored, a large InstanceNorm gamma or weights that grew during training can get there.

    with RangeCheck(model) as rc:
        out, out_hr = model(x)
    rc.raise_if_saturated()            # or: for name, kind, count, max_abs in rc.report(): ...

Inside the context every fp16-producing engine call of the forward counts into its own slot, labelled with the module's
qualified name from `model.named_modules()` and a kind:

    y      the conv output before InstanceNorm (conv blocks)
    a      the normalised, activated output (conv blocks)
    up     the transposed-conv output written into the decoder's [up | skip] buffer (decoder.transpconvs.*)
    sr_up  the depth up-sampling in front of sr_head (its output is bf16 in the default configuration, so it only reports when
           that changes)

The kernels check the fp32 value just before each fp16 store (csrc/ptx.cuh range_check) and only observe: every stored value
is bit-identical with the check on or off.  Outside a RangeCheck nothing is checked and the kernels take a null slot.  The
slot buffer has a fixed size, so a CUDA graph captured inside the context bakes in a stable address (graphs.GraphedForward /
GraphedTrainStep with `range_check=True`).
"""
from __future__ import annotations

import struct
from typing import Dict, List, NamedTuple, Optional, Tuple

import numpy as np
import torch

from . import functional as F_
from ._lib import RehrError, check, lib, ptr, stream_ptr

SLOT_BYTES = 16          # { uint64 count; uint32 max_abs_bits; uint32 pad } (include/rehrseg_b200.h, rehr_range_sink)
DEFAULT_SLOTS = 256      # the 3d_fullres SegModel uses 50: 12 encoder conv blocks x 2, 5 decoder stages x (2 x 2 + 1), sr_up
KINDS = ("y", "a", "up", "sr_up")


class Saturation(NamedTuple):
    name: str        # qualified module name (model.named_modules())
    kind: str        # one of KINDS
    count: int       # values that saturated
    max_abs: float   # largest |v| among them (inf or nan possible)


def decode(slots: np.ndarray, labels: List[Tuple[str, str]]) -> List[Saturation]:
    """The non-zero records of a host copy of the slot array ([n, 2] int64), in slot (= forward) order."""
    out = []
    for i, (name, kind) in enumerate(labels):
        count = int(slots[i, 0])
        if count == 0:
            continue
        bits = int(slots[i, 1]) & 0xFFFFFFFF
        out.append(Saturation(name, kind, count, struct.unpack("<f", struct.pack("<I", bits))[0]))
    return out


class RangeCheck:
    """Context manager that records fp16 saturation per (module, kind) slot; see the module docstring.  Slots are assigned in
    forward order on first use and reused when the same module runs again (the counts then add up until `reset()`)."""

    def __init__(self, model: torch.nn.Module, slots: int = DEFAULT_SLOTS, device=None):
        if slots <= 0:
            raise ValueError("RangeCheck needs at least one slot")
        if device is None:
            device = next(model.parameters()).device
        self._names: Dict[int, str] = {id(m): n for n, m in model.named_modules()}
        self.capacity = int(slots)
        self.slots = torch.zeros((self.capacity, 2), dtype=torch.int64, device=device)
        self.labels: List[Tuple[str, str]] = []
        self._index: Dict[Tuple[str, str], int] = {}
        self.owner: Optional[torch.nn.Module] = None   # set by seg_model around each labelled engine call

    # ---- context ---------------------------------------------------------------------------------------------------------
    def __enter__(self):
        if F_._range is not None:
            raise RehrError("RangeCheck contexts do not nest")
        F_._range = self
        return self

    def __exit__(self, *exc):
        F_._range = None
        self.owner = None
        lib().rehr_range_sink(None, 0)
        return False

    # ---- called by functional around one fp16-producing launch ------------------------------------------------------------
    def slot_of(self, kind: str) -> Optional[int]:
        """Slot of (current owner, kind), assigned on first use; None when the owner is not a module of the checked model."""
        name = self._names.get(id(self.owner)) if self.owner is not None else None
        if name is None:
            return None
        key = (name, kind)
        s = self._index.get(key)
        if s is None:
            if len(self.labels) >= self.capacity:
                raise RehrError(f"RangeCheck: more than {self.capacity} labelled fp16 stores; construct it with a larger `slots`")
            s = self._index[key] = len(self.labels)
            self.labels.append(key)
        return s

    def arm(self, kind: str) -> None:
        s = self.slot_of(kind)
        if s is not None:
            check(lib().rehr_range_sink(ptr(self.slots), s), "range_sink")

    def disarm(self) -> None:
        lib().rehr_range_sink(None, 0)

    # ---- results ----------------------------------------------------------------------------------------------------------
    def reset(self) -> None:
        """Zero every slot (one memset on the current stream; inside a graph capture it becomes the graph's memset node)."""
        check(lib().rehr_range_clear(ptr(self.slots), self.capacity, stream_ptr(self.slots.device)), "range_clear")

    def report(self) -> List[Saturation]:
        """Copy the slots to the host (one synchronise) and return the non-zero records in forward order."""
        return decode(self.slots.cpu().numpy(), self.labels)

    def raise_if_saturated(self) -> None:
        rec = self.report()
        if rec:
            r = rec[0]
            raise RehrError(f"fp16 saturation in {r.name} ({r.kind}): {r.count} value(s) with |v| >= 65520, largest {r.max_abs:g}"
                            + (f"; {len(rec) - 1} later slot(s) saturated too" if len(rec) > 1 else ""))
