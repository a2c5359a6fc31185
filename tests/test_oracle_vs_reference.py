"""CPU: the oracle restatements against the reference's integer helpers, rotate_vol_2d and fba over whole ranges and seeded
arrays, stored in tests/golden/reference_helpers.* (oracle/make_golden.py); with a checkout of the reference project
(REHRSEG_REFERENCE, oracle/refimport.py) the live functions are checked against the same stored results.  Also the
sliding FLAVR window logic against a hand-built expectation."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import make_golden, refimport
from oracle import volume as ov

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_integer_helpers_exhaustive():
    with open(os.path.join(G, "reference_helpers.json")) as f:
        cases = json.load(f)
    assert (len(cases["find_integer_p"]), len(cases["get_pads"]), len(cases["steps"])) == (690, 1600, 200)
    live = refimport.available()
    if live:
        po, pad, su = refimport.load("utils.patch_ops"), refimport.load("utils.pad"), refimport.load("utils.seg_utils")
    for n, s, p, proj3 in cases["find_integer_p"]:
        assert (ov.find_integer_p(n, s), ov.projected_size(n, 3, s)) == (p, proj3), (n, s)
        if live:
            assert (po.find_integer_p(n, s), po.projected_size(n, 3, s)) == (p, proj3), (n, s)
    for t, d, lo, hi in cases["get_pads"]:
        assert ov.get_pads(t, d) == (lo, hi), (t, d)
        if live:
            assert pad.get_pads(t, d) == (lo, hi), (t, d)
    for img, tile, step, out in cases["steps"]:
        assert ov.steps_for_sliding_window(img, tile, step) == out, (img, tile, step)
        if live:
            assert su.compute_steps_for_sliding_window(img, tile, step) == out, (img, tile, step)


def test_rotate_and_fba_random():
    z = np.load(os.path.join(G, "reference_helpers.npz"))
    live = refimport.available()
    if live:
        rot, fb = refimport.load("utils.rotate"), refimport.load("utils.fba")
    v = torch.from_numpy(z["rot_in"])
    for a in (0, 90, -90, 180, -180, 270, -270, 360):
        want = torch.from_numpy(z[f"rot_{a}"])
        assert torch.equal(ov.rotate_vol_2d(v, a), want), a
        if live:
            assert torch.equal(rot.rotate_vol_2d(v, a), want), a
    with pytest.raises(NotImplementedError):
        ov.rotate_vol_2d(v, 45)
    vols = list(z["fba_in"])
    assert len(vols) == 4
    for p in make_golden.FBA_PS:
        assert np.array_equal(ov.fba(vols, p), z[f"fba_{p}"]), p
        if live:
            assert np.array_equal(fb.fba(vols, p), z[f"fba_{p}"]), p


def test_apply_to_vol_flavr_window_logic():
    """utils/sr_utils.py:102-135 hard-codes .cuda(); compare the restatement against a hand-built expectation on a
    model that tags every window (identity on the middle slices)."""
    calls = []

    def model(x):  # x [1, C, 4, Y, X]
        calls.append(x.clone())
        return x[:, :, 1:3].repeat_interleave(2, dim=2)  # [1, C, 4, Y, X]: four output slices per window

    img = torch.arange(5 * 1 * 20 * 18, dtype=torch.float32).reshape(5, 1, 20, 18)
    out = ov.apply_to_vol_flavr(model, img)
    assert out.shape == (16, 1, 18, 20) and len(calls) == 4  # in-plane axes come back transposed, as in the reference
    assert calls[0].shape == (1, 1, 4, 32, 32)
    assert float(calls[0][0, 0, 0].abs().sum()) == 0.0 and float(calls[-1][0, 0, 3].abs().sum()) == 0.0
    # window st uses slices st-1..st+2; output slice 4*st+k comes from input slice st (k<2) or st+1 (k>=2)
    for st in range(4):
        assert torch.equal(out[4 * st, 0], img[st, 0].T) and torch.equal(out[4 * st + 3, 0], img[st + 1, 0].T)
