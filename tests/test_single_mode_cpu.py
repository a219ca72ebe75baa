"""Argument checks of the single-mode entries (ep_single_mode_*, ep_grad_sqnorm_f64, ep_adam_clip_step_f64) and of
single_mode.SingleModeTrainer.  Every call here is rejected before anything touches a device, so no GPU is needed: the
pointers are never dereferenced."""
import ctypes
import importlib

import numpy as np
import pytest
import scipy.sparse as sp
import torch

FAKE = ctypes.c_void_p(256)
NEW = ["ep_single_mode_max_prev", "ep_single_mode_workspace_bytes", "ep_grad_sqnorm_f64", "ep_adam_clip_step_f64"] + [
    "ep_single_mode_%s_%s" % (what, sfx) for what in ("fwd", "bwd", "fold_fwd", "fold_bwd") for sfx in ("f32", "f64")]


def _pkg(name):
    return importlib.import_module("eigen-pinns_b200." + name)


def test_entries_are_bound_and_counted():
    cabi = _pkg("_cabi")
    for name in NEW:
        assert name in cabi.SIGNATURES
    for name in NEW[2:]:
        assert name in cabi.KERNELS_PER_CALL
    assert cabi.query("ep_single_mode_max_prev") == 64
    assert cabi.query("ep_single_mode_workspace_bytes", 0) > 0
    assert cabi.query("ep_single_mode_workspace_bytes", 65) == 0
    assert cabi.query("ep_single_mode_workspace_bytes", -1) == 0


def _fwd(sfx, n, P, ldq=None, Q=FAKE, u=FAKE, ws_bytes=1 << 30, loss=FAKE):
    return ("ep_single_mode_fwd_" + sfx, n, P, u, FAKE, FAKE, Q, P if ldq is None else ldq, FAKE, 1.0, loss, FAKE,
            FAKE, ws_bytes, None)


@pytest.mark.parametrize("sfx", ["f32", "f64"])
def test_forward_and_backward_reject_bad_arguments(sfx):
    cabi = _pkg("_cabi")
    for bad, status, msg in ((dict(n=0, P=0), -1, "n must be >= 1"),
                             (dict(n=-5, P=0), -1, "n must be >= 1"),
                             (dict(n=10, P=-1), -1, "P >= 0"),
                             (dict(n=10, P=65), -3, "not supported"),
                             (dict(n=10, P=3, Q=None), -1, "Q is NULL"),
                             (dict(n=10, P=3, ldq=2), -1, "ldq < P"),
                             (dict(n=10, P=0, u=None), -1, "null pointer"),
                             (dict(n=10, P=0, loss=None), -1, "null pointer"),
                             (dict(n=10, P=4, ws_bytes=8), -4, "workspace too small")):
        name, *args = _fwd(sfx, **bad)
        with pytest.raises(cabi.EpError, match=r"status %d\).*%s" % (status, msg)):
            cabi.call(name, *args)
    name = "ep_single_mode_bwd_" + sfx
    with pytest.raises(cabi.EpError, match=r"status -3\)"):
        cabi.call(name, 10, 65, FAKE, FAKE, FAKE, 65, FAKE, FAKE, FAKE, FAKE, FAKE, None)
    with pytest.raises(cabi.EpError, match=r"status -1\).*n must be"):
        cabi.call(name, -1, 0, FAKE, FAKE, None, 1, FAKE, FAKE, FAKE, FAKE, FAKE, None)
    with pytest.raises(cabi.EpError, match="null pointer"):
        cabi.call(name, 10, 0, FAKE, FAKE, None, 1, FAKE, None, FAKE, FAKE, FAKE, None)


@pytest.mark.parametrize("sfx", ["f32", "f64"])
def test_folding_rejects_bad_layer_tables(sfx):
    cabi = _pkg("_cabi")
    dims = (ctypes.c_int * 5)(3, 8, 8, 8, 1)
    bad_dims = (ctypes.c_int * 5)(3, 8, -8, 8, 1)
    fwd, bwd = "ep_single_mode_fold_fwd_" + sfx, "ep_single_mode_fold_bwd_" + sfx
    for n_layers in (0, -1, 9):
        with pytest.raises(cabi.EpError, match="layers"):
            cabi.call(fwd, n_layers, dims, FAKE, FAKE, None)
    with pytest.raises(cabi.EpError, match="layers"):
        cabi.call(fwd, 4, None, FAKE, FAKE, None)
    with pytest.raises(cabi.EpError, match="positive"):
        cabi.call(fwd, 4, bad_dims, FAKE, FAKE, None)
    with pytest.raises(cabi.EpError, match="null pointer"):
        cabi.call(fwd, 4, dims, None, FAKE, None)
    with pytest.raises(cabi.EpError, match="null pointer"):
        cabi.call(bwd, 4, dims, FAKE, None, None, FAKE, None)
    with pytest.raises(cabi.EpError, match="positive"):
        cabi.call(bwd, 4, bad_dims, FAKE, FAKE, None, FAKE, None)


def test_fp64_optimiser_entries_reject_bad_arguments():
    cabi = _pkg("_cabi")
    with pytest.raises(cabi.EpError, match="null pointer"):
        cabi.call("ep_grad_sqnorm_f64", 10, None, FAKE, None)
    with pytest.raises(cabi.EpError, match="null pointer"):
        cabi.call("ep_adam_clip_step_f64", 10, FAKE, None, FAKE, FAKE, 1e-3, None, 0.9, 0.999, 1e-8, 0.0, 1, 0.0,
                  None, None)
    with pytest.raises(cabi.EpError, match="step counts from 1"):
        cabi.call("ep_adam_clip_step_f64", 10, FAKE, FAKE, FAKE, FAKE, 1e-3, None, 0.9, 0.999, 1e-8, 0.0, 0, 0.0,
                  None, None)


def _cpu_pair(dtype=torch.float32):
    n = 12
    A = sp.random(n, n, density=0.3, random_state=0, format="csr") + sp.identity(n)
    S = (A + A.T).tocsr()
    return _pkg("sparse").OperatorPair(S, S, "cpu", dtype=dtype), n


def test_trainer_rejects_dtype_mismatch_cpu_tensors_and_too_many_modes():
    sm, v, cabi, ops = _pkg("single_mode"), _pkg("variants"), _pkg("_cabi"), _pkg("ops")
    pair, n = _cpu_pair()
    pair64, _ = _cpu_pair(torch.float64)
    X = torch.zeros((n, 3))
    net = v.EigenfunctionNN(8, 3, initial_eigenvalue=1.0)
    w_before = net.fc1.weight
    with pytest.raises(TypeError, match="one dtype"):
        sm.SingleModeTrainer(net, X, pair64)
    with pytest.raises(TypeError, match="one dtype"):
        sm.SingleModeTrainer(net, X.double(), pair)
    with pytest.raises(TypeError, match="float32 or float64"):
        sm.SingleModeTrainer(v.EigenfunctionNN(8, 3).half(), X.half(), pair)
    with pytest.raises(cabi.EpError, match="GPU"):
        sm.SingleModeTrainer(net, X, pair)
    assert net.fc1.weight is w_before                  # nothing adopted by a refused trainer
    with pytest.raises(cabi.EpError, match="0 .. 64"):
        ops.single_mode_workspace(65, "cpu")
    with pytest.raises(ValueError, match="one initial eigenvalue per mode"):
        sm.train_modes(X, pair, 3, 10, initial_eigenvalues=[1.0, 2.0])


def test_ops_wrappers_reject_cpu_tensors():
    ops, cabi = _pkg("ops"), _pkg("_cabi")
    col = torch.zeros((5, 1))
    with pytest.raises(cabi.EpError, match="CUDA tensors"):
        ops.single_mode_fwd(col, col, col, None, torch.ones(1), 1.0, torch.zeros(9, dtype=torch.float64),
                            torch.zeros(3, dtype=torch.float64), torch.zeros(8, dtype=torch.uint8))
    with pytest.raises(cabi.EpError, match="CUDA tensors"):
        ops.single_mode_fold_fwd([3, 4, 1], torch.zeros(26), torch.zeros(21))
    with pytest.raises(cabi.EpError, match="CUDA tensors"):
        ops.adam_clip_step(*(torch.zeros(4, dtype=torch.float64) for _ in range(4)), 1e-3, 0.9, 0.999, 1e-8, 0.0, 1,
                           0.0, None)
