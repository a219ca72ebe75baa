"""Dense layers with activation epilogues (ep_linear_act_fwd_* / ep_linear_act_bwd_*, ops.mlp_act) and the notebook
networks built on them (variants.CoordinateMLP, variants.EigenfunctionNN).

Single layers are compared with torch fp64 on the GPU, on the kernel's own inputs.  With u the unit roundoff of the
kernel's dtype (2^-24, 2^-53), gamma_m = m u / (1 - m u) and |.| elementwise, every output obeys the a-priori bound

    |got - ref| <= (E + C u (|ref_lin| + E)) * mag                                                    (assert_bound)

  Y  = act(z), z = X W^T + b   E = r gamma_{in+1} (|X| |W|^T + |b|), ref_lin = z, mag = L = 1.1 (|act'| <= 1.1)
  Z  = z                       same E, mag = 1, C = 1
  dX = (dY W) * act'           E = r gamma_out (|dY| |W|), ref_lin = dY W, mag = the size of act' and of its rounding:
                               SiLU s (1 + |z| (1 - s)), sin |cos z| + u, tanh 1 + x^2, ReLU / none 1
  dW = dY^T X, db = sum dY     E = r gamma_{n+1024} (|dY|^T |X|), (sum |dY|), mag = 1   (split-K partials then a
                               fixed-order sum: fewer than 1024 extra terms)

C = 8 covers the few-ulp error of the libm calls (expf / exp, sinf / sin, cosf / cos, tanhf / tanh), the final products
and, for tanh, the kernel reading act' from its stored x rather than from z.  r = 1 for fp32 (the fp64 reference's own
rounding is 2^-29 of E) and r = 2 for fp64, where the reference rounds as much as the kernel does: the fp64 kernels then
agree to a few ulp relative to |X| |W|.  Output buffers are NaN-filled and wider than the result, so an unwritten entry or
a write past the last column shows.
"""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

from gpu_util import pkg, dev

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import variants_port as vp          # noqa: E402

pytestmark = pytest.mark.gpu

ACTS = ["silu", "sin", "tanh", "relu", "none"]
DTYPES = [torch.float32, torch.float64]
C = 8.0
SLAB = 65535 * 64                # rows per launch of the layer kernels; larger n is processed in row slabs


def unit(dtype):
    return 2.0 ** -24 if dtype == torch.float32 else 2.0 ** -53


def gamma(m, dtype):
    u = unit(dtype)
    return m * u / (1 - m * u)


def act64(name, z):
    return {"silu": torch.nn.functional.silu, "sin": torch.sin, "tanh": torch.tanh, "relu": torch.relu,
            "none": lambda t: t}[name](z)


def assert_bound(got, ref, E, ref_lin, mag, dtype, what, c=C):
    u = unit(dtype)
    got = got.double()
    bound = (E + c * u * (ref_lin.abs() + E)) * mag
    bad = ~((got - ref).abs() <= bound)
    if bad.any():
        i = tuple(int(v) for v in bad.nonzero()[0])
        raise AssertionError("%s: %d of %d entries out of bound, first at %s: got %r ref %r bound %r" % (
            what, int(bad.sum()), bad.numel(), i, got[i].item(), ref[i].item(), bound[i].item()))


def strided(n, k, dtype, pad, gen, scale=1.0, fill=None):
    """n x k view with row stride k + pad, one element into its allocation (unaligned base)."""
    buf = torch.empty(n * (k + pad) + 2, dtype=dtype, device=dev())
    view = buf[1:1 + n * (k + pad)].view(n, k + pad)
    if fill is None:
        view.copy_(torch.randn(n, k + pad, generator=gen, dtype=torch.float64).to(dev()) * scale)
    else:
        view.fill_(fill)
    return view[:, :k], view


def act_grad_mag(name, z64, x64, dtype):
    if name == "silu":
        s = torch.sigmoid(z64)
        return s * (1 + z64.abs() * (1 - s))
    if name == "sin":
        return torch.cos(z64).abs() + unit(dtype)
    if name == "tanh":
        return 1 + x64 * x64
    return torch.ones_like(z64)


def check_layer(n, d_in, d_out, act, dtype, seed=0):
    """Forward of one layer with `act`, then the backward of the layer above it (input X = act(Zx)), both through ops on
    strided NaN-filled buffers, against torch fp64."""
    ops = pkg("ops")
    g = torch.Generator().manual_seed(seed)
    W = (torch.randn(d_out, d_in, generator=g, dtype=torch.float64) / np.sqrt(d_in)).to(dev(), dtype)
    b = (0.5 * torch.randn(d_out, generator=g, dtype=torch.float64)).to(dev(), dtype)
    X, _ = strided(n, d_in, dtype, 3, g)
    Y, Yfull = strided(n, d_out, dtype, 5, g, fill=float("nan"))
    Z, Zfull = strided(n, d_out, dtype, 2, g, fill=float("nan"))
    ops.linear_act_fwd(X, W, b, act, Y=Y, Z=Z)
    X64, W64, b64 = X.double(), W.double(), b.double()
    z = X64 @ W64.t() + b64
    Ez = gamma(d_in + 1, dtype) * (X64.abs() @ W64.abs().t() + b64.abs()) * (1 if dtype == torch.float32 else 2)
    assert_bound(Z, z, Ez, z, 1.0, dtype, "Z", c=1.0)
    assert_bound(Y, act64(act, z), Ez, z, 1.1, dtype, "Y")
    assert torch.isnan(Yfull[:, d_out:]).all() and torch.isnan(Zfull[:, d_out:]).all()

    # backward of a layer whose input X2 = act(Zx) is this activation's output
    Zx, _ = strided(n, d_in, dtype, 2, g, scale=1.5)
    X2 = act64(act, Zx.double()).to(dtype)                 # what the forward kernel stores (rounded to dtype)
    dY, _ = strided(n, d_out, dtype, 4, g)
    dX, dXfull = strided(n, d_in, dtype, 7, g, fill=float("nan"))
    _, dW, db = ops.linear_act_bwd(X2, Zx if act in ("silu", "sin") else None, act, W, dY, True, dX=dX)
    dY64, Zx64 = dY.double(), Zx.double().requires_grad_(True)
    act64(act, Zx64).matmul(W64.t()).backward(dY64)       # torch autograd: dZx = (dY W) * act'(Zx)
    G = dY64 @ W64
    EG = gamma(d_out, dtype) * (dY64.abs() @ W64.abs()) * (1 if dtype == torch.float32 else 2)
    mag = act_grad_mag(act, Zx64.detach(), X2.double(), dtype)
    assert_bound(dX, Zx64.grad, EG, G, mag, dtype, "dX")
    assert torch.isnan(dXfull[:, d_in:]).all()
    X2_64 = X2.double()
    r = 1 if dtype == torch.float32 else 2
    EW = r * gamma(n + 1024, dtype) * (dY64.abs().t() @ X2_64.abs())
    assert_bound(dW, dY64.t() @ X2_64, EW, dY64.t() @ X2_64, 1.0, dtype, "dW")
    Eb = r * gamma(n + 1024, dtype) * dY64.abs().sum(0)
    assert_bound(db, dY64.sum(0), Eb, dY64.sum(0), 1.0, dtype, "db")
    return X, W, b, Y, X2, Zx, dY, dX, dW, db


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("act", ACTS)
@pytest.mark.parametrize("n", [1, 63, 65, 777, 4097])
def test_single_layer_within_rounding_bound(n, act, dtype):
    check_layer(n, 37, 83, act, dtype, seed=n)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("act", ["silu", "sin", "tanh"])
def test_single_layer_wide_ragged(act, dtype):
    check_layer(1000, 130, 257, act, dtype, seed=11)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_row_slab_fold(dtype):
    """n above 65535 * 64: the forward and dX kernels run in two row slabs."""
    check_layer(SLAB + 333, 5, 7, "silu", dtype, seed=5)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("act", ["none", "relu"])
def test_relu_and_none_match_the_plain_layer_entries_bit_for_bit(act, dtype):
    """act 0 / 1 of the new entries computes what ep_linear_fwd_* / ep_linear_bwd_* compute, bit for bit."""
    ops = pkg("ops")
    X, W, b, Y, X2, _, dY, dX, dW, db = check_layer(777, 37, 83, act, dtype, seed=3)
    assert torch.equal(ops.linear_fwd(X, W, b, act == "relu"), Y)
    dX0, dW0, db0 = ops.linear_bwd(X2, W, dY, True, relu_mask=act == "relu")
    assert torch.equal(dX0, dX) and torch.equal(dW0, dW) and torch.equal(db0, db)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_input_layer_without_dx(dtype):
    """act_x = none with dX = NULL (the network input): only dW and db, equal to ep_linear_bwd_*."""
    ops = pkg("ops")
    g = torch.Generator().manual_seed(2)
    X = torch.randn(513, 3, generator=g, dtype=torch.float64).to(dev(), dtype)
    W = torch.randn(50, 3, generator=g, dtype=torch.float64).to(dev(), dtype)
    dY = torch.randn(513, 50, generator=g, dtype=torch.float64).to(dev(), dtype)
    dX, dW, db = ops.linear_act_bwd(X, None, "none", W, dY, False)
    _, dW0, db0 = ops.linear_bwd(X, W, dY, False, relu_mask=False)
    assert dX is None and torch.equal(dW, dW0) and torch.equal(db, db0)


def test_argument_errors_do_not_launch():
    """An unknown act, or a NULL Zx where act_x needs the pre-activation, is an error and leaves every output as it was."""
    cabi = pkg("_cabi")
    n, d_in, d_out = 100, 8, 16
    for dtype, sfx in ((torch.float32, "f32"), (torch.float64, "f64")):
        X = torch.randn(n, d_in, device=dev(), dtype=dtype)
        W = torch.randn(d_out, d_in, device=dev(), dtype=dtype)
        Y = torch.full((n, d_out), float("nan"), device=dev(), dtype=dtype)
        Z = Y.clone()
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        p = lambda t: ctypes.c_void_p(t.data_ptr())                   # noqa: E731
        for act in (-1, 5, 99):
            with pytest.raises(cabi.EpError, match="unknown activation"):
                cabi.call("ep_linear_act_fwd_" + sfx, n, d_in, d_out, p(X), d_in, p(W), None, p(Y), d_out, p(Z), d_out,
                          act, st)
        dY = torch.randn(n, d_out, device=dev(), dtype=dtype)
        dX = torch.full((n, d_in), float("nan"), device=dev(), dtype=dtype)
        dW = torch.full((d_out, d_in), float("nan"), device=dev(), dtype=dtype)
        db = torch.full((d_out,), float("nan"), device=dev(), dtype=dtype)
        ws = torch.empty(cabi.query("ep_linear_bwd_workspace_bytes" + ("_f64" if sfx == "f64" else ""), n, d_in, d_out),
                         dtype=torch.uint8, device=dev())
        args = lambda zx, act_x: (n, d_in, d_out, p(X), d_in, zx, d_in, act_x, p(W), p(dY), d_out, p(dX), d_in,  # noqa
                                  p(dW), p(db), p(ws), ws.numel(), st)
        for act_x in (2, 3):
            with pytest.raises(cabi.EpError, match="Zx is NULL"):
                cabi.call("ep_linear_act_bwd_" + sfx, *args(None, act_x))
        for act_x in (-1, 5):
            with pytest.raises(cabi.EpError, match="unknown activation"):
                cabi.call("ep_linear_act_bwd_" + sfx, *args(p(X), act_x))
        torch.cuda.synchronize()
        for t in (Y, Z, dX, dW, db):
            assert torch.isnan(t).all()
    with pytest.raises(ValueError, match="activation"):
        pkg("ops").mlp_act(X, [W], [W[:, 0].contiguous()], "gelu")


# ------------------------------------------------------------------------------------------------------ networks
def _rel(a, b):
    a, b = a.detach().double().cpu(), b.detach().double().cpu()
    return (a - b).abs().max().item() / max(b.abs().max().item(), 1e-300)


TOL = {torch.float32: (2e-5, 2e-4), torch.float64: (1e-12, 1e-10)}       # (output, gradients), relative to the max


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("act", ["silu", "sin", "tanh", "relu"])
def test_coordinate_mlp_matches_the_oracle(act, dtype):
    v = pkg("variants")
    torch.manual_seed(7)
    ref = vp.CoordinateMLP(3, 12, (64, 48, 33), act).double()
    net = v.CoordinateMLP(3, 12, (64, 48, 33), act).to(dev(), dtype)
    net.load_state_dict({k: t.to(dtype) for k, t in ref.state_dict().items()})
    g = torch.Generator().manual_seed(8)
    x = torch.randn(1999, 3, generator=g, dtype=torch.float64).to(dtype)
    R = torch.randn(1999, 12, generator=g, dtype=torch.float64)
    xr = x.double().clone().requires_grad_(True)
    out_ref = ref(xr)
    (out_ref * R).sum().backward()
    xd = x.to(dev()).requires_grad_(True)
    out = net(xd)
    (out * R.to(dev(), dtype)).sum().backward()
    tol_out, tol_grad = TOL[dtype]
    assert out.dtype == dtype and _rel(out, out_ref) < tol_out
    assert _rel(xd.grad, xr.grad) < tol_grad
    for (name, p), (_, q) in zip(net.named_parameters(), ref.named_parameters()):
        assert _rel(p.grad, q.grad) < tol_grad, name


@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_eigenfunction_nn_matches_the_oracle(dtype):
    v = pkg("variants")
    torch.manual_seed(9)
    ref = vp.EigenfunctionNN(64, 3, initial_eigenvalue=-1.3).double()
    net = v.EigenfunctionNN(64, 3, initial_eigenvalue=-1.3).to(dev(), dtype)
    net.load_state_dict({k: t.to(dtype) for k, t in ref.state_dict().items()})
    g = torch.Generator().manual_seed(10)
    x = torch.randn(3001, 3, generator=g, dtype=torch.float64).to(dtype)
    R = torch.randn(3001, 1, generator=g, dtype=torch.float64)
    u_ref, lam_ref = ref(x.double())
    ((u_ref * R).sum() + 0.3 * lam_ref.sum()).backward()
    u, lam = net(x.to(dev()))
    ((u * R.to(dev(), dtype)).sum() + 0.3 * lam.sum()).backward()
    tol_out, tol_grad = TOL[dtype]
    assert u.dtype == dtype and _rel(u, u_ref) < tol_out and _rel(lam, lam_ref) < tol_out
    names = [name for name, _ in net.named_parameters()]
    assert names == [name for name, _ in ref.named_parameters()]
    for (name, p), (_, q) in zip(net.named_parameters(), ref.named_parameters()):
        assert _rel(p.grad, q.grad) < tol_grad, name                 # eigenvalue_layer.weight.grad is d lambda
