"""fp64 kernels of the notebook variants against an extended-precision reference, and the fp64 notebook functionals
against the fp64 restatement (oracle/variants_port.py) on the UNROUNDED operators.

Every kernel result y^ is checked against the a-priori bound |y^ - y| <= gamma_m (|A| |x|), gamma_m = m u / (1 - m u),
u = 2^-53, m = number of terms in each sum; y and |A| |x| are computed in numpy longdouble (64-bit mantissa), so the
reference's own rounding is 2^-11 of the bound.  Rounding to fp32 anywhere would exceed it by about 10^7."""
import ctypes
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from gpu_util import pkg, dev, bunny_levels, random_csr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import variants_port as vp          # noqa: E402

pytestmark = pytest.mark.gpu

U64 = 2.0 ** -53
LD = np.longdouble
SIZES = [0, 1, 127, 129, 777, 4097, "bunny"]
KS = [1, 3, 8, 50, 64, 65, 128]


def gamma(m):
    return m * U64 / (1 - m * U64)


def _assert_bound(got, ref, absref, m):
    got = np.asarray(got, dtype=LD)
    err = np.abs(got - ref)
    bound = gamma(m) * absref * (1 + 2.0 ** -10)
    assert np.all(err <= bound), "max err / bound = %g" % float(np.max(err / np.maximum(bound, 1e-300)))


def _csr_pair(n, seed, empty_every=0):
    """Two operators on one pattern: the bunny K / M, or random square CSR (values with full 53-bit mantissas)."""
    if n == "bunny":
        _, (K, M), _ = bunny_levels()
        return K.tocsr(), M.tocsr()
    if n == 0:
        Z = sp.csr_matrix((0, 0), dtype=np.float64)
        return Z, Z.copy()
    A = random_csr(n, n, min(8, n), seed, empty_every)
    B = A.copy()
    B.data = np.random.default_rng(seed + 1).standard_normal(B.nnz) / 3.0
    return A, B


def _dense(n, k, seed, ld=None, offset=0):
    """n x k fp64 CUDA tensor, row stride ld (>= k), base pointer `offset` elements into its allocation."""
    ld = k if ld is None else ld
    buf = torch.zeros(n * ld + offset + 1, dtype=torch.float64, device=dev())
    view = buf[offset:offset + n * ld].view(n, ld)[:, :k]
    view.copy_(torch.from_numpy(np.random.default_rng(seed).standard_normal((n, k))))
    return view


def _host(t):
    return t.detach().cpu().numpy().astype(LD)


def _nnz_max(A):
    return int(np.diff(A.indptr).max()) if A.shape[0] and A.nnz else 0


# ------------------------------------------------------------------------------------------------------------ SpMM
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("k", KS)
def test_spmm_family_within_rounding_bound(n, k):
    sparse, ops = pkg("sparse"), pkg("ops")
    A, B = _csr_pair(n, 7 + k)
    rows = A.shape[0]
    pair = sparse.OperatorPair(A, B, dev(), dtype=torch.float64)
    X = _dense(rows, k, k)
    m = _nnz_max(A) + 1
    Al, Bl, Xl = A.astype(LD), B.astype(LD), _host(X)
    aA, aB, aX = abs(Al), abs(Bl), np.abs(Xl)
    Y = ops.spmm(pair.K, X)
    assert Y.dtype == torch.float64
    _assert_bound(_host(Y), Al @ Xl, aA @ aX, m)
    KU, MU = ops.spmm2(pair, X)
    _assert_bound(_host(KU), Al @ Xl, aA @ aX, m)
    _assert_bound(_host(MU), Bl @ Xl, aB @ aX, m)
    XB = _dense(rows, k, k + 100)
    XBl = _host(XB)
    # spmm2_sum takes the transposed operators (pair.KT, pair.MT); the random matrices are not symmetric
    At, Bt = abs(Al.T.tocsr()), abs(Bl.T.tocsr())
    mt = _nnz_max(A.T.tocsr()) + 1
    for with_d, scale, dev_scale in ((False, 1.0, False), (True, -0.37, False), (True, 2.5, True)):
        D = _dense(rows, k, k + 200) if with_d else None
        sdev = torch.tensor([scale], dtype=torch.float64, device=dev()) if dev_scale else None
        Y = ops.spmm2_sum(pair.KT, pair.MT, X, XB, D, 123.0 if dev_scale else scale, scale_dev=sdev)
        ref = Al.T @ Xl + Bl.T @ XBl
        absref = At @ aX + Bt @ np.abs(XBl)
        if with_d:
            ref = ref + _host(D)
            absref = absref + np.abs(_host(D))
        _assert_bound(_host(Y), LD(scale) * ref, abs(scale) * absref, 2 * mt + 2)


@pytest.mark.parametrize("layout", ["ld", "offset", "empty_rows"])
def test_spmm_family_layouts(layout):
    sparse, ops = pkg("sparse"), pkg("ops")
    n, k = 777, 50
    A, B = _csr_pair(n, 3, empty_every=5 if layout == "empty_rows" else 0)
    pair = sparse.OperatorPair(A, B, dev(), dtype=torch.float64)
    ld, off = (k + 3, 0) if layout == "ld" else (k, 1) if layout == "offset" else (k, 0)
    X = _dense(n, k, 1, ld, off)
    outK, outM = _dense(n, k, 2, ld, off), _dense(n, k, 3, ld, off)
    outK.fill_(np.nan)
    outM.fill_(np.nan)
    if layout != "offset":
        assert X.data_ptr() % 16 == 0
    else:
        assert X.data_ptr() % 16 == 8
    m = _nnz_max(A) + 1
    Al, Bl, Xl = A.astype(LD), B.astype(LD), _host(X)
    ops.spmm2(pair, X, out_K=outK, out_M=outM)
    _assert_bound(_host(outK), Al @ Xl, abs(Al) @ np.abs(Xl), m)
    _assert_bound(_host(outM), Bl @ Xl, abs(Bl) @ np.abs(Xl), m)
    Y = _dense(n, k, 4, ld, off)
    ops.spmm(pair.K, X, out=Y)
    _assert_bound(_host(Y), Al @ Xl, abs(Al) @ np.abs(Xl), m)
    if layout == "empty_rows":
        assert np.all(_host(Y)[::5] == 0)
    D = _dense(n, k, 5, ld, off)
    Z = _dense(n, k, 6, ld, off)
    ops.spmm2_sum(pair.KT, pair.MT, X, X, D, 0.5, out=Z)          # transposed operators
    ref = Al.T @ Xl + Bl.T @ Xl + _host(D)
    mt = _nnz_max(A.T.tocsr()) + 1
    absref = (abs(Al.T) + abs(Bl.T)) @ np.abs(Xl) + np.abs(_host(D))
    _assert_bound(_host(Z), LD(0.5) * ref, LD(0.5) * absref, 2 * mt + 2)


# ------------------------------------------------------------------------------------------------------ partials
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("k", KS)
def test_eigen_partials_within_rounding_bound(n, k):
    ops = pkg("ops")
    rows = bunny_levels()[1][0].shape[0] if n == "bunny" else n
    U, KU, MU = _dense(rows, k, 1), _dense(rows, k, 2), _dense(rows, k, 3)
    P = ops.eigen_partials(U, KU, MU)
    assert P.dtype == torch.float64 and P.numel() == k * k + 5 * k
    P = P.cpu().numpy().astype(LD)
    u, ku, mu = _host(U), _host(KU), _host(MU)
    m = max(rows, 1)
    _assert_bound(P[:k * k].reshape(k, k), u.T @ mu, np.abs(u).T @ np.abs(mu), m)
    blocks = [(u, ku), (ku, ku), (ku, mu), (mu, mu)]
    for q, (a, b) in enumerate(blocks):
        _assert_bound(P[k * k + q * k:k * k + (q + 1) * k], (a * b).sum(0), np.abs(a * b).sum(0), m)
    _assert_bound(P[k * k + 4 * k:], mu.sum(0), np.abs(mu).sum(0), m)


def test_eigen_partials_layouts():
    ops = pkg("ops")
    n, k = 4097, 65
    for ld, off in ((k + 7, 0), (k + 1, 1)):
        U = _dense(n, k, 1, ld, off)
        buf = torch.zeros(n * (2 * k + 2) + 2, dtype=torch.float64, device=dev())
        KM = buf[off:off + n * (2 * k + 2)].view(n, 2 * k + 2)          # KU / MU share one row stride
        KM.copy_(torch.from_numpy(np.random.default_rng(9).standard_normal((n, 2 * k + 2))))
        KU, MU = KM[:, :k], KM[:, k + 1:2 * k + 1]
        P = ops.eigen_partials(U, KU, MU).cpu().numpy().astype(LD)
        u, mu = _host(U), _host(MU)
        _assert_bound(P[:k * k].reshape(k, k), u.T @ mu, np.abs(u).T @ np.abs(mu), n)


# ---------------------------------------------------------------------------------------------------- dense layers
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("k", KS)
def test_linear_layers_within_rounding_bound(n, k):
    ops = pkg("ops")
    rows = bunny_levels()[1][0].shape[0] if n == "bunny" else n
    d_in, d_out = k, 64 + k % 7
    X, W, b = _dense(rows, d_in, 1), _dense(d_out, d_in, 2).contiguous(), _dense(1, d_out, 3).reshape(-1).contiguous()
    x, w, bb = _host(X), _host(W), _host(b)
    for bias, relu in ((False, False), (True, False), (True, True)):
        Y = ops.linear_fwd(X, W, b if bias else None, relu)
        ref = x @ w.T + (bb if bias else 0)
        absref = np.abs(x) @ np.abs(w).T + (np.abs(bb) if bias else 0)
        got = _host(Y)
        if relu:
            assert np.all(got >= 0)
            keep = ref > gamma(d_in + 1) * absref            # clearly positive: the ReLU keeps the value
            got, ref, absref = got[keep], ref[keep], absref[keep]
        _assert_bound(got, ref, absref, d_in + 1)
    if rows == 0:
        return
    dY = _dense(rows, d_out, 4)
    dy = _host(dY)
    for mask in (False, True):
        dX, dW, db = ops.linear_bwd(X, W, dY, True, relu_mask=mask)
        refx = dy @ w
        absx = np.abs(dy) @ np.abs(w)
        if mask:
            refx, absx = refx * (x > 0), absx * (x > 0)
        _assert_bound(_host(dX), refx, absx, d_out)
        _assert_bound(_host(dW), dy.T @ x, np.abs(dy).T @ np.abs(x), rows)
        _assert_bound(_host(db), dy.sum(0), np.abs(dy).sum(0), rows)


def test_linear_layer_layouts():
    ops = pkg("ops")
    n, d_in, d_out = 4097, 65, 128
    X = _dense(n, d_in, 1, d_in + 3, 1)
    W, b = _dense(d_out, d_in, 2).contiguous(), _dense(1, d_out, 3).reshape(-1).contiguous()
    Y = _dense(n, d_out, 4, d_out + 1, 1)
    ops.linear_fwd(X, W, b, False, out=Y)
    x, w = _host(X), _host(W)
    _assert_bound(_host(Y), x @ w.T + _host(b), np.abs(x) @ np.abs(w).T + np.abs(_host(b)), d_in + 1)
    dY = _dense(n, d_out, 5, d_out + 5, 1)
    dX = _dense(n, d_in, 6, d_in + 2, 1)
    _, dW, db = ops.linear_bwd(X, W, dY, True, relu_mask=False, dX=dX)
    dy = _host(dY)
    _assert_bound(_host(dX), dy @ w, np.abs(dy) @ np.abs(w), d_out)
    _assert_bound(_host(dW), dy.T @ x, np.abs(dy).T @ np.abs(x), n)


# ------------------------------------------------------------------------------------------- determinism, errors
def test_every_fp64_entry_is_deterministic():
    sparse, ops = pkg("sparse"), pkg("ops")
    A, B = _csr_pair("bunny", 0)
    pair = sparse.OperatorPair(A, B, dev(), dtype=torch.float64)
    n, k = A.shape[0], 50
    X, XB, D = _dense(n, k, 1), _dense(n, k, 2), _dense(n, k, 3)
    W, b = _dense(96, k, 4).contiguous(), _dense(1, 96, 5).reshape(-1).contiguous()
    dY = _dense(n, 96, 6)

    def run():
        out = [ops.spmm(pair.K, X)]
        out += list(ops.spmm2(pair, X))
        out.append(ops.spmm2_sum(pair.KT, pair.MT, X, XB, D, 0.75))
        out.append(ops.eigen_partials(X, XB, D))
        out.append(ops.linear_fwd(X, W, b, True))
        out += list(ops.linear_bwd(X, W, dY, True, relu_mask=True))
        return [t.clone() for t in out]
    for a, c in zip(run(), run()):
        assert torch.equal(a, c)


def test_fp64_errors_on_the_device():
    sparse, ops, cabi = pkg("sparse"), pkg("ops"), pkg("_cabi")
    _, _, (Kc, Mc) = bunny_levels()
    p64 = sparse.OperatorPair(Kc, Mc, dev(), dtype=torch.float64)
    p32 = sparse.OperatorPair(Kc, Mc, dev())
    n = Kc.shape[0]
    U64, U32 = _dense(n, 4, 1), _dense(n, 4, 1).float()
    for pair, U in ((p32, U64), (p64, U32)):
        with pytest.raises(TypeError, match="float"):
            ops.spmm2(pair, U)
        with pytest.raises(TypeError):
            pkg("variants").operator_stats(U, pair)
    with pytest.raises(TypeError):
        ops.eigen_partials(U64, U32, U32)
    with pytest.raises(TypeError):
        ops.linear_fwd(U64, torch.zeros(3, 4, device=dev()), None, False)
    with pytest.raises(cabi.EpError, match="k > 128"):
        U = _dense(n, 129, 2)
        ops.eigen_partials(U, U, U)
    with pytest.raises(TypeError):                # stays fp32-only
        ops.m_normalize_columns(U64, p64.M)


# ------------------------------------------------------------------------------------- notebook functionals, fp64
def _setup(k, seed=0, coarse=False):
    fem, (K, M), (Kc, Mc) = bunny_levels()
    K, M, verts = (Kc, Mc, fem["coarse_verts"]) if coarse else (K, M, fem["verts"])
    rng = np.random.default_rng(seed)
    n = K.shape[0]
    return verts, K.tocsr(), M.tocsr(), rng.standard_normal((n, k)) / np.sqrt(n) * 30.0


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


ERRORS = {}        # largest measured error per quantity (printed with -s)


def _record(name, value):
    ERRORS[name] = max(ERRORS.get(name, 0.0), float(value))
    print("measured %-40s %.3e" % (name, value))


@pytest.mark.parametrize("k", [8, 16, 50])
def test_dense_rayleigh_loss_fp64(k):
    v = pkg("variants")
    _, K, M, U0 = _setup(k)
    pair = pkg("sparse").OperatorPair(K, M, dev(), dtype=torch.float64)
    U = torch.from_numpy(U0).to(dev()).requires_grad_(True)
    loss, l1, dl, ol, lam = v.dense_rayleigh_loss(U, pair)
    loss.backward()
    Ur = torch.from_numpy(U0).requires_grad_(True)
    rloss, rl1, rdl, rol, rlam = vp.dense_rayleigh_loss(Ur, vp.to_torch_sparse(K), vp.to_torch_sparse(M))
    rloss.backward()
    for name, a, b in (("loss", loss, rloss), ("loss_1", l1, rl1), ("diag", dl, rdl), ("off_diag", ol, rol)):
        err = abs(a.item() - b.item()) / abs(b.item())
        _record("dense_rayleigh %s" % name, err)
        assert err <= 2e-8
    _record("dense_rayleigh lambda", _rel(lam.detach().cpu(), rlam.detach()))
    assert _rel(lam.detach().cpu(), rlam.detach()) < 2e-8
    _record("dense_rayleigh dL/dU", _rel(U.grad.cpu(), Ur.grad))
    assert _rel(U.grad.cpu(), Ur.grad) < 5e-8


@pytest.mark.parametrize("k", [8, 32])
def test_whitened_subspace_loss_fp64(k):
    v = pkg("variants")
    _, K, M, U0 = _setup(k, seed=1)
    Kn, Mn, _, _ = v.frobenius_normalised(K, M)
    pair = pkg("sparse").OperatorPair(Kn, Mn, dev(), dtype=torch.float64)
    U = torch.from_numpy(U0).to(dev()).requires_grad_(True)
    loss, terms, eigs = v.whitened_subspace_loss(U, pair, lambda_orth=0.1)
    loss.backward()
    Ur = torch.from_numpy(U0).requires_grad_(True)
    rloss, rterms, reigs = vp.whitened_subspace_loss(Ur, vp.to_torch_sparse(Kn), vp.to_torch_sparse(Mn), lambda_orth=0.1)
    rloss.backward()
    _record("whitened loss", abs(loss.item() - rloss.item()) / abs(rloss.item()))
    assert abs(loss.item() - rloss.item()) <= 1e-8 * abs(rloss.item())
    hinge_atol = 1e-8 * reigs.abs().max().item()
    for name in ("zero", "trace", "diversity", "offdiag", "ordering", "stability"):
        atol = hinge_atol if name in ("diversity", "ordering") else 1e-15
        assert abs(terms[name].item() - rterms[name].item()) <= 1e-8 * abs(rterms[name].item()) + atol, name
    assert terms["orth"].item() < 1e-12 and rterms["orth"].item() < 1e-12
    _record("whitened eigs", _rel(eigs.detach().cpu(), reigs.detach()))
    assert _rel(eigs.detach().cpu(), reigs.detach()) < 1e-8
    _record("whitened dL/dU", _rel(U.grad.cpu(), Ur.grad))
    assert _rel(U.grad.cpu(), Ur.grad) < 1e-7


def test_single_mode_loss_and_network_gradients_fp64():
    v = pkg("variants")
    verts, K, M, _ = _setup(1, coarse=True)
    pair = pkg("sparse").OperatorPair(K, M, dev(), dtype=torch.float64)
    torch.manual_seed(3)
    ref = vp.EigenfunctionNN(32, 3, initial_eigenvalue=0.7).double()
    net = v.EigenfunctionNN(32, 3, initial_eigenvalue=0.7).double().to(dev())
    net.load_state_dict(ref.state_dict())
    X = torch.from_numpy(np.ascontiguousarray(verts, dtype=np.float64))
    prev = [torch.from_numpy(np.random.default_rng(5).standard_normal(K.shape[0])) for _ in range(2)]
    u, lam = net(X.to(dev()))
    total, eig, norm, ortho = v.single_mode_loss(u, lam, pair, [p.to(dev()) for p in prev], ortho_weight=2.0)
    total.backward()
    ru, rlam = ref(X)
    rtotal, reig, rnorm, rortho = vp.single_mode_loss(ru, rlam.reshape(()), vp.to_torch_sparse(K), vp.to_torch_sparse(M),
                                                      prev, ortho_weight=2.0)
    rtotal.backward()
    _record("single_mode u", _rel(u.detach().cpu(), ru.detach()))
    assert _rel(u.detach().cpu(), ru.detach()) < 1e-8
    for name, a, b in (("total", total, rtotal), ("eig", eig, reig), ("norm", norm, rnorm), ("ortho", ortho, rortho)):
        _record("single_mode %s" % name, abs(a.item() - b.item()) / max(abs(b.item()), 1e-300))
        assert abs(a.item() - b.item()) <= 1e-7 * abs(b.item()) + 1e-13, name
    for (name, p), (_, q) in zip(net.named_parameters(), ref.named_parameters()):
        _record("single_mode grad", _rel(p.grad.cpu(), q.grad))
        assert _rel(p.grad.cpu(), q.grad) < 2e-7, name


def test_smoothness_loss_fp64():
    v = pkg("variants")
    _, K, M, U0 = _setup(8, seed=4, coarse=True)
    pair = pkg("sparse").OperatorPair(K, M, dev(), dtype=torch.float64)
    c0 = np.random.default_rng(12).standard_normal(U0.shape) * 0.05
    corr = torch.from_numpy(c0).to(dev()).requires_grad_(True)
    a, b = v.smoothness_loss(corr, torch.from_numpy(U0).to(dev()) + corr, pair)
    (3.0 * (a + b)).backward()
    rcorr = torch.from_numpy(c0).requires_grad_(True)
    ra, rb = vp.smoothness_loss(rcorr, torch.from_numpy(U0) + rcorr, vp.to_torch_sparse(K))
    (3.0 * (ra + rb)).backward()
    for name, x, y in (("corr", a, ra), ("total", b, rb)):
        _record("smoothness %s" % name, abs(x.item() - y.item()) / abs(y.item()))
        assert abs(x.item() - y.item()) <= 1e-8 * abs(y.item())
    _record("smoothness grad", _rel(corr.grad.cpu(), rcorr.grad))
    assert _rel(corr.grad.cpu(), rcorr.grad) < 1e-7


def test_coordinate_mlp_trains_in_lock_step_with_the_fp64_oracle():
    """CoordinateMLP.double() + whitened_subspace_loss on the coarse bunny, 20 Adam steps from the oracle's weights:
    the loss agrees to 1e-8 relative at every step, and so do the final parameters."""
    v = pkg("variants")
    verts, K, M, _ = _setup(1, coarse=True)
    Kn, Mn, _, _ = v.frobenius_normalised(K, M)
    pair = pkg("sparse").OperatorPair(Kn, Mn, dev(), dtype=torch.float64)
    Kt, Mt = vp.to_torch_sparse(Kn), vp.to_torch_sparse(Mn)
    torch.manual_seed(0)
    ref = vp.CoordinateMLP(3, 6, (64, 64), "silu").double()
    net = v.CoordinateMLP(3, 6, (64, 64), "silu").double().to(dev())
    net.load_state_dict(ref.state_dict())
    Xr = torch.from_numpy(np.ascontiguousarray(verts, dtype=np.float64))
    X = Xr.to(dev())
    opt, ropt = torch.optim.Adam(net.parameters(), lr=3e-3), torch.optim.Adam(ref.parameters(), lr=3e-3)
    worst = 0.0
    for it in range(20):
        opt.zero_grad()
        ropt.zero_grad()
        loss, _, _ = v.whitened_subspace_loss(net(X), pair)
        loss.backward()
        rloss, _, _ = vp.whitened_subspace_loss(ref(Xr), Kt, Mt)
        rloss.backward()
        if it == 0:
            for (name, p), (_, q) in zip(net.named_parameters(), ref.named_parameters()):
                _record("coordinate_mlp grad (step 0)", _rel(p.grad.cpu(), q.grad))
                assert _rel(p.grad.cpu(), q.grad) < 2e-6, name
        rel = abs(loss.item() - rloss.item()) / abs(rloss.item())
        worst = max(worst, rel)
        assert rel <= 1e-8, (it, loss.item(), rloss.item())
        opt.step()
        ropt.step()
    _record("lock-step loss (20 steps)", worst)
    for (name, p), (_, q) in zip(net.named_parameters(), ref.named_parameters()):
        _record("lock-step final params", _rel(p.detach().cpu(), q.detach()))
        assert _rel(p.detach().cpu(), q.detach()) <= 1e-8, name
