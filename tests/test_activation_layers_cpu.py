"""Argument checks of the activation-epilogue layer entries (ep_linear_act_fwd_* / ep_linear_act_bwd_*) and of
ops.mlp_act.  They reject a bad call before anything touches a device, so no GPU is needed: the pointers are never
dereferenced."""
import ctypes
import importlib

import pytest

FAKE = ctypes.c_void_p(256)


def _cabi():
    return importlib.import_module("eigen-pinns_b200._cabi")


@pytest.mark.parametrize("sfx", ["f32", "f64"])
@pytest.mark.parametrize("n", [0, 100])
@pytest.mark.parametrize("act", [-1, 5, 1000])
def test_forward_rejects_unknown_activation(sfx, n, act):
    cabi = _cabi()
    with pytest.raises(cabi.EpError, match=r"status -1\).*ep_linear_act_fwd_%s: unknown activation" % sfx):
        cabi.call("ep_linear_act_fwd_" + sfx, n, 8, 16, FAKE, 8, FAKE, None, FAKE, 16, None, 0, act, None)


@pytest.mark.parametrize("sfx", ["f32", "f64"])
def test_backward_rejects_unknown_activation_and_missing_pre_activation(sfx):
    cabi = _cabi()
    name = "ep_linear_act_bwd_" + sfx

    def args(zx, act_x, dx=FAKE):
        return (100, 8, 16, FAKE, 8, zx, 8, act_x, FAKE, FAKE, 16, dx, 8, FAKE, FAKE, FAKE, 1 << 30, None)
    for act_x in (-1, 5):
        with pytest.raises(cabi.EpError, match="unknown activation"):
            cabi.call(name, *args(FAKE, act_x))
    for act_x in (2, 3):                      # SiLU and sin read act' from the pre-activation
        with pytest.raises(cabi.EpError, match=r"status -1\).*Zx is NULL"):
            cabi.call(name, *args(None, act_x))
    with pytest.raises(cabi.EpError, match="leading dimension"):
        cabi.call(name, 100, 8, 16, FAKE, 8, FAKE, 4, 2, FAKE, FAKE, 16, FAKE, 8, FAKE, FAKE, FAKE, 1 << 30, None)
    with pytest.raises(cabi.EpError, match="null pointer"):
        cabi.call(name, 100, 8, 16, FAKE, 8, FAKE, 8, 2, FAKE, FAKE, 16, FAKE, 8, None, FAKE, FAKE, 1 << 30, None)


def test_mlp_act_rejects_unknown_activation_and_mismatched_lists():
    import torch
    ops = importlib.import_module("eigen-pinns_b200.ops")
    W, b = torch.zeros(4, 3), torch.zeros(4)
    with pytest.raises(ValueError, match="activation"):
        ops.mlp_act(torch.zeros(2, 3), [W], [b], "gelu")
    with pytest.raises(ValueError, match="one bias per weight"):
        ops.mlp_act(torch.zeros(2, 3), [W, W], [b], "silu")
