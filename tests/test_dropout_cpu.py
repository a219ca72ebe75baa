"""Dropout keep masks without a GPU: the numpy port of csrc/dropout.cuh (oracle/dropout_port.py) against the Random123
known-answer vectors of Philox4x32-10, the statistics of the masks, the probability checks of StepConfig, and the
C ABI surface of the dropout entry points."""
import importlib
import os
import re

import numpy as np
import pytest

from oracle import dropout_port as dp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW_EXPORTS = ("ep_dropout_keep_mask_u8", "ep_linear_fwd_dropout_f32", "ep_linear_bwd_dropout_f32",
               "ep_tc_linear_fwd_dropout_bf16", "ep_tc_linear_dx_dropout_bf16", "ep_tc_chain_fwd_dropout_bf16")


@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, want):
    got = dp.philox4x32_10(*ctr, *key)
    assert tuple(int(w) for w in got) == want


def test_lane_order_and_keep_rule():
    """feature 8c + 2j <- low half of word j, 8c + 2j + 1 <- high half; keep iff lane >= thr."""
    seed, step, layer, p = 0x0123456789ABCDEF, 7, 2, 0.3
    m = dp.keep_mask(3, 24, p, seed, step, layer, row0=5)
    thr = dp.threshold(p)
    for r in range(3):
        for c in range(3):
            w = dp.philox4x32_10(5 + r, c, layer, step, seed & 0xFFFFFFFF, seed >> 32)
            for j in range(4):
                assert m[r, 8 * c + 2 * j] == ((int(w[j]) & 0xFFFF) >= thr)
                assert m[r, 8 * c + 2 * j + 1] == ((int(w[j]) >> 16) >= thr)


@pytest.mark.parametrize("p", [0.05, 0.1, 0.5, 0.9])
def test_keep_fraction(p):
    n, width = 16384, 256                                   # 4 M draws
    m = dp.keep_mask(n, width, p, seed=1234, step=3, layer=1)
    q = 1.0 - dp.threshold(p) / 65536.0
    sigma = np.sqrt(q * (1 - q) / m.size)
    assert abs(m.mean() - q) < 5 * sigma
    assert abs(dp.threshold(p) / 65536.0 - np.float32(p)) <= 2.0 ** -17


@pytest.mark.parametrize("what", ["step", "layer", "row", "chunk"])
def test_masks_of_adjacent_counters_are_independent(what):
    p, n, width = 0.3, 8192, 256
    a = dp.keep_mask(n + 1, width + 8, p, seed=99, step=10, layer=2)
    if what == "step":
        b = dp.keep_mask(n + 1, width + 8, p, seed=99, step=11, layer=2)
    elif what == "layer":
        b = dp.keep_mask(n + 1, width + 8, p, seed=99, step=10, layer=3)
    else:
        b = a
    if what == "row":
        x, y = a[:-1, :width], b[1:, :width]
    elif what == "chunk":
        x, y = a[:n, :width], b[:n, 8:width + 8]
    else:
        x, y = a[:n, :width], b[:n, :width]
    q = dp.threshold(p) / 65536.0
    want = q * q + (1 - q) * (1 - q)
    agree = (x == y).mean()
    assert abs(agree - want) < 5 * np.sqrt(want * (1 - want) / x.size)


def test_p_zero_keeps_everything_and_scale_is_one():
    assert dp.keep_mask(777, 96, 0.0, seed=5, step=1, layer=0).all()
    assert dp.scale(0.0) == np.float32(1.0)
    assert dp.scale(0.5) == np.float32(2.0)


def test_step_config_checks_the_probability():
    engine = importlib.import_module("eigen-pinns_b200.engine")
    assert engine.StepConfig().dropout == 0.0
    assert engine.StepConfig(dropout=0.1, dropout_seed=3).dropout_seed == 3
    for bad in (-0.1, 1.0, 1.5, 1.0 - 2.0 ** -18, float("nan")):
        with pytest.raises(ValueError):
            engine.StepConfig(dropout=bad)


def test_header_and_library_export_the_dropout_entry_points():
    text = open(os.path.join(ROOT, "include", "eigenpinns_b200.h")).read()
    declared = set(re.findall(r"EP_API\s+[\w\s\*]+?\b(ep_\w+)\s*\(", text))
    cabi = importlib.import_module("eigen-pinns_b200._cabi")
    lib = cabi.load()
    for name in NEW_EXPORTS:
        assert name in declared and name in cabi.SIGNATURES and name in cabi.KERNELS_PER_CALL
        assert hasattr(lib, name)


def test_entry_points_reject_bad_probabilities_before_launching():
    """An invalid p returns EP_ERR_INVALID before any launch, so no GPU is needed to see it."""
    import ctypes
    cabi = importlib.import_module("eigen-pinns_b200._cabi")
    fake = ctypes.c_void_p(256)
    for p in (-0.5, 1.0):
        with pytest.raises(cabi.EpError, match="dropout probability"):
            cabi.call("ep_dropout_keep_mask_u8", 10, 32, p, 1, 1, None, 0, 0, fake, None)
        with pytest.raises(cabi.EpError, match="dropout probability"):
            cabi.call("ep_linear_fwd_dropout_f32", 10, 8, 8, fake, 8, fake, fake, fake, 8, p, 1, 1, None, 0, 0, None)
