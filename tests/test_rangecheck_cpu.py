"""Host bookkeeping of the opt-in fp16 saturation check (rehrseg_b200.rangecheck): slot labels from named_modules, decoding of
the slot array, the fixed-size refusal and the C-ABI declaration.  No GPU needed."""
import re
import struct

import numpy as np
import pytest
import torch.nn as nn

from rehrseg_b200 import _lib, functional as F_
from rehrseg_b200.rangecheck import RangeCheck, decode


def _model():
    from oracle import seg_model as ref_seg
    from rehrseg_b200 import seg_model as sm
    return sm.SegModel(**ref_seg.plan_kwargs("tiny"))


def test_slots_are_labelled_with_qualified_names_in_first_use_order():
    m = _model()
    rc = RangeCheck(m, slots=8)
    stem = m.encoder.stages[0][0].convs[0]
    tc = m.decoder.transpconvs[0]
    rc.owner = stem
    assert rc.slot_of("y") == 0 and rc.slot_of("a") == 1
    rc.owner = tc
    assert rc.slot_of("up") == 2
    rc.owner = stem
    assert rc.slot_of("y") == 0          # the same module again reuses its slot
    rc.owner = m.sr_head
    assert rc.slot_of("sr_up") == 3
    assert rc.labels == [("encoder.stages.0.0.convs.0", "y"), ("encoder.stages.0.0.convs.0", "a"),
                         ("decoder.transpconvs.0", "up"), ("sr_head", "sr_up")]
    rc.owner = nn.Conv3d(1, 1, 1)        # not a module of the checked model: no slot
    assert rc.slot_of("y") is None
    rc.owner = None
    assert rc.slot_of("y") is None


def test_decoder_alias_of_the_encoder_keeps_the_first_name():
    m = _model()
    rc = RangeCheck(m, slots=4)
    rc.owner = m.decoder.encoder.stages[1][0].convs[0]
    rc.slot_of("y")
    assert rc.labels == [("encoder.stages.1.0.convs.0", "y")]


def test_fixed_size_refuses_overflow():
    m = _model()
    rc = RangeCheck(m, slots=2)
    rc.owner = m.encoder.stages[0][0].convs[0]
    rc.slot_of("y")
    rc.slot_of("a")
    with pytest.raises(_lib.RehrError, match="more than 2"):
        rc.slot_of("up")
    with pytest.raises(ValueError):
        RangeCheck(m, slots=0)


def test_decode_returns_nonzero_records_in_slot_order():
    bits = lambda f: struct.unpack("<I", struct.pack("<f", f))[0]
    slots = np.zeros((5, 2), dtype=np.int64)
    slots[1] = (7, bits(1.5e5))
    slots[3] = (1, 0x7F800000)            # inf
    slots[4] = (2, 0x7FC00000)            # NaN sorts above inf
    labels = [("l0", "y"), ("l1", "a"), ("l2", "up"), ("l3", "y"), ("l4", "a")]
    rec = decode(slots, labels)
    assert [(r.name, r.kind, r.count) for r in rec] == [("l1", "a", 7), ("l3", "y", 1), ("l4", "a", 2)]
    assert rec[0].max_abs == pytest.approx(1.5e5) and rec[1].max_abs == float("inf") and np.isnan(rec[2].max_abs)
    assert decode(np.zeros((3, 2), dtype=np.int64), labels[:3]) == []


def test_contexts_do_not_nest_and_leave_nothing_active():
    m = _model()
    assert F_._range is None
    a, b = RangeCheck(m, slots=2), RangeCheck(m, slots=2)
    F_._range = a                        # entered (without the library call of __exit__)
    try:
        with pytest.raises(_lib.RehrError, match="do not nest"):
            b.__enter__()
    finally:
        F_._range = None


def test_range_sink_is_declared_and_bound():
    with open(_lib.HEADER_PATH) as f:
        text = f.read()
    assert re.search(r"int rehr_range_sink\(void\* slots, int slot\);", text)
    assert re.search(r"int rehr_range_clear\(void\* slots, int n, rehr_stream stream\);", text)
    assert {"rehr_range_sink", "rehr_range_clear"} <= set(_lib.declared_symbols())
    src = open(_lib.__file__).read()
    assert '"rehr_range_sink": (i, [vp, i])' in src and '"rehr_range_clear": (i, [vp, i, vp])' in src
