"""The single-mode training step (csrc/single_mode.cu, single_mode.py) against the fp64 restatement of
delta_pinns_validation/iterative_eigenvalues_on_cloud.ipynb cell 1 (oracle/variants_port.py) and against the autograd
path it replaces (variants.EigenfunctionNN + variants.single_mode_loss + torch.optim.Adam).

Stated tolerances.  fp64: loss terms within 1e-12 relative of the oracle on the same bytes, dL/du within 1e-9, the
parameter gradients within 1e-8 (the only differences are summation orders and libm's sin), twenty Adam steps within
1e-10.  fp32: the kernels widen to fp64 for every sum, so what is left is the fp32 rounding of L u, M u
(ep_spmm2_csr_f32) and of the layers: loss terms within 1e-4 relative, dL/du within 1e-4, the rest to the tolerances
of tests/test_gpu_variants.py."""
import os
import sys

import numpy as np
import pytest
import scipy.linalg
import scipy.sparse as sp
import torch

from gpu_util import pkg, dev, bunny_levels

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import variants_port as vp          # noqa: E402

pytestmark = pytest.mark.gpu

GUARD = 64
DTYPES = {"f32": torch.float32, "f64": torch.float64}


def _rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)


def _sym_pair(n, seed):
    """Symmetric L (indefinite) and M (diagonally dominant) on one random pattern."""
    rng = np.random.default_rng(seed)
    rows, cols = np.repeat(np.arange(n), 3), rng.integers(0, n, 3 * n)
    C = (sp.coo_matrix((rng.standard_normal(3 * n), (rows, cols)), shape=(n, n)) + sp.identity(n)).tocsr()
    L = (C + C.T).tocsr()
    M = (abs(C) + abs(C).T + 4.0 * sp.identity(n)).tocsr()
    return L, M


def _rounded(A, dtype):
    return A.astype(np.float32).astype(np.float64) if dtype == torch.float32 else A


def _nan(shape, dtype, guard=GUARD):
    """NaN-filled buffer with a NaN guard region behind the first prod(shape) entries."""
    size = int(np.prod(shape))
    buf = torch.full((size + guard,), float("nan"), dtype=dtype, device=dev())
    return buf, buf[:size].view(shape)


def _guard_intact(buf, size):
    assert torch.isnan(buf[size:]).all(), "write past the end of an output"


def _case(n, P, dtype, seed=0):
    L, M = _sym_pair(n, seed)
    rng = np.random.default_rng(seed + 1)
    u = rng.standard_normal(n) / np.sqrt(n) * 3.0
    prev = [rng.standard_normal(n) / np.sqrt(n) for _ in range(P)]
    np_t = np.float32 if dtype == torch.float32 else np.float64
    u, prev = u.astype(np_t), [p.astype(np_t) for p in prev]
    return L, M, u, prev


def _kernel_loss(pair, u, prev, w, ortho_weight, dtype):
    ops = pkg("ops")
    n, P = u.shape[0], len(prev)
    ud = torch.from_numpy(u).to(dev()).reshape(n, 1)
    Lu, Mu = ops.spmm2(pair, ud)
    Q = ops.spmm(pair.M, torch.from_numpy(np.stack(prev, 1)).to(dev())) if P else None
    wd = torch.tensor([w], dtype=dtype, device=dev())
    lbuf, loss = _nan((4,), torch.float64)
    cbuf, coef = _nan((3 + P,), torch.float64)
    ops.single_mode_fwd(ud, Lu, Mu, Q, wd, ortho_weight, loss, coef, ops.single_mode_workspace(P, dev()))
    _guard_intact(lbuf, 4)
    _guard_intact(cbuf, 3 + P)
    return ud, Lu, Mu, Q, wd, loss, coef


@pytest.mark.parametrize("sfx", ["f32", "f64"])
@pytest.mark.parametrize("P", [0, 1, 5, 64])
@pytest.mark.parametrize("n", [1, 127, 2503, 40001, 300001])
def test_forward_kernel_against_fp64(n, P, sfx):
    """n = 300001 is more than 4 x 148 CTAs of 256 rows: every CTA of the capped grid loops."""
    dtype = DTYPES[sfx]
    L, M, u, prev = _case(n, P, dtype, seed=n + P)
    pair = pkg("sparse").OperatorPair(L, M, dev(), dtype=dtype)
    Lt, Mt = vp.to_torch_sparse(_rounded(L, dtype)), vp.to_torch_sparse(_rounded(M, dtype))
    tol = 1e-12 if dtype == torch.float64 else 1e-4
    for w in (0.8, -0.8, 0.0):
        w_t = float(np.float32(w)) if dtype == torch.float32 else w
        _, _, _, _, _, loss, coef = _kernel_loss(pair, u, prev, w_t, 1.5, dtype)
        if n > 1:
            ref = vp.single_mode_loss(torch.from_numpy(u.astype(np.float64)).reshape(n, 1),
                                      torch.tensor(abs(w_t), dtype=torch.float64), Lt, Mt,
                                      [torch.from_numpy(p.astype(np.float64)) for p in prev], ortho_weight=1.5)
            ref = [t.item() for t in ref]
        else:                       # the restatement's u.squeeze() makes one vertex a 0-d tensor: same formulas inline
            l_, m_ = _rounded(L, dtype)[0, 0], _rounded(M, dtype)[0, 0]
            u0 = float(u[0])
            eig, norm = (l_ * u0 - abs(w_t) * (m_ * u0)) ** 2, (u0 * (m_ * u0) - 1.0) ** 2
            ortho = sum((u0 * (m_ * float(p[0]))) ** 2 for p in prev)
            ref = [eig + norm + 1.5 * ortho, eig, norm, ortho]
        got = loss.cpu().numpy()
        for name, a, b in zip(("total", "eig", "norm", "ortho"), got, ref):
            assert np.isfinite(a) and abs(a - b) <= tol * abs(b) + 1e-300, (name, w, a, b)
        assert coef[0].item() == 2.0 / n


@pytest.mark.parametrize("sfx", ["f32", "f64"])
@pytest.mark.parametrize("P", [0, 3])
@pytest.mark.parametrize("w", [0.9, -0.9, 0.0])
def test_du_and_dlambda_against_fp64_autograd(w, P, sfx):
    dtype = DTYPES[sfx]
    ops = pkg("ops")
    n = 2503
    L, M, u, prev = _case(n, P, dtype, seed=7)
    pair = pkg("sparse").OperatorPair(L, M, dev(), dtype=dtype)
    w_t = float(np.float32(w)) if dtype == torch.float32 else w
    ud, Lu, Mu, Q, wd, loss, coef = _kernel_loss(pair, u, prev, w_t, 2.0, dtype)
    bufs = [_nan((n, 1), dtype) for _ in range(3)]
    gL, gM, D = (b[1] for b in bufs)
    ops.single_mode_bwd(Lu, Mu, Q, wd, coef, gL, gM, D)
    for b, _ in bufs:
        _guard_intact(b, n)
    du = ops.spmm2_sum(pair.KT, pair.MT, gL, gM, D=D)
    ur = torch.from_numpy(u.astype(np.float64)).reshape(n, 1).requires_grad_(True)
    lam = torch.tensor(abs(w_t), dtype=torch.float64, requires_grad=True)
    Lt, Mt = vp.to_torch_sparse(_rounded(L, dtype)), vp.to_torch_sparse(_rounded(M, dtype))
    total, _, _, _ = vp.single_mode_loss(ur, lam, Lt, Mt, [torch.from_numpy(p.astype(np.float64)) for p in prev],
                                         ortho_weight=2.0)
    total.backward()
    tol = 1e-9 if dtype == torch.float64 else 1e-4
    assert _rel(du.cpu(), ur.grad) < tol
    assert abs(coef[2].item() - lam.grad.item()) <= tol * abs(lam.grad.item())


def _net_pair(dtype, hidden=32, w0=0.7, seed=3, coarse=True):
    fem, (K, M), (Kc, Mc) = bunny_levels()
    K, M, verts = (Kc, Mc, fem["coarse_verts"]) if coarse else (K, M, fem["verts"])
    torch.manual_seed(seed)
    ref = vp.EigenfunctionNN(hidden, 3, initial_eigenvalue=w0).double()
    return ref, K.tocsr(), M.tocsr(), np.ascontiguousarray(verts, dtype=np.float64)


def _kernel_net(ref, dtype):
    net = pkg("variants").EigenfunctionNN(ref.fc1.out_features, 3).to(device=dev(), dtype=dtype)
    net.load_state_dict({k: t.to(dtype) for k, t in ref.state_dict().items()})
    return net


def _split_grad(tr):
    """The trainer's flat gradient per named parameter of the module."""
    out, off = {}, 0
    for i in range(1, 5):
        fc = getattr(tr.net, "fc%d" % i)
        for name, p in (("weight", fc.weight), ("bias", fc.bias)):
            out["fc%d.%s" % (i, name)] = tr.grad[off:off + p.numel()].view(p.shape)
            off += p.numel()
    out["eigenvalue_layer.weight"] = tr.grad[off:].view(1, 1)
    return out


@pytest.mark.parametrize("sfx", ["f32", "f64"])
@pytest.mark.parametrize("w0", [0.7, -0.7, 0.0])
def test_parameter_gradients_against_fp64_autograd(w0, sfx):
    dtype = DTYPES[sfx]
    sm = pkg("single_mode")
    ref, K, M, verts = _net_pair(dtype, w0=w0)
    net = _kernel_net(ref, dtype)
    pair = pkg("sparse").OperatorPair(K, M, dev(), dtype=dtype)
    rng = np.random.default_rng(5)
    prev = [rng.standard_normal(K.shape[0]) for _ in range(2)]
    X = torch.from_numpy(verts).to(device=dev(), dtype=dtype)
    tr = sm.SingleModeTrainer(net, X, pair, previous=[torch.from_numpy(p).to(device=dev(), dtype=dtype) for p in prev],
                              ortho_weight=2.0)
    tr.forward()
    loss = tr.loss_forward().cpu().numpy()[:4]
    tr.backward()
    Xr = torch.from_numpy(verts.astype(np.float32).astype(np.float64) if dtype == torch.float32 else verts)
    ru, rlam = ref(Xr)
    prev_r = [torch.from_numpy(p.astype(np.float32).astype(np.float64) if dtype == torch.float32 else p) for p in prev]
    rtot = vp.single_mode_loss(ru, rlam.reshape(()), vp.to_torch_sparse(_rounded(K, dtype)),
                               vp.to_torch_sparse(_rounded(M, dtype)), prev_r, ortho_weight=2.0)
    rtot[0].backward()
    tol_u, tol_l, tol_g = (1e-10, 1e-10, 1e-8) if dtype == torch.float64 else (1e-5, 1e-4, 2e-4)
    assert _rel(tr.u.cpu(), ru.detach()) < tol_u
    for a, b in zip(loss, rtot):
        assert abs(a - b.item()) <= tol_l * abs(b.item()) + 1e-300
    grads = _split_grad(tr)
    for name, q in ref.named_parameters():
        g = grads[name].cpu()
        if w0 == 0.0 and name == "eigenvalue_layer.weight":
            assert g.item() == 0.0 and q.grad.item() == 0.0          # d|w|/dw = 0 at w = 0, as torch
            continue
        assert _rel(g, q.grad) < tol_g, name


def _autograd_run(ref, K, M, verts, prev, steps, dtype, lr):
    """The path the trainer replaces: variants.EigenfunctionNN + variants.single_mode_loss + torch.optim.Adam."""
    v = pkg("variants")
    net = _kernel_net(ref, dtype)
    pair = pkg("sparse").OperatorPair(K, M, dev(), dtype=dtype)
    X = torch.from_numpy(verts).to(device=dev(), dtype=dtype)
    opt = torch.optim.Adam(net.parameters(), lr=lr, betas=(0.999, 0.9999), eps=1e-8)
    losses = []
    for _ in range(steps):
        opt.zero_grad()
        u, lam = net(X)
        terms = v.single_mode_loss(u, lam, pair, [p.to(device=dev(), dtype=dtype) for p in prev], ortho_weight=1.0)
        terms[0].backward()
        opt.step()
        losses.append([t.item() for t in terms])
    return np.array(losses), {k: t.detach().double().cpu() for k, t in net.state_dict().items()}


def _trainer_run(ref, K, M, verts, prev, steps, dtype, lr, graph=False):
    sm = pkg("single_mode")
    net = _kernel_net(ref, dtype)
    pair = pkg("sparse").OperatorPair(K, M, dev(), dtype=dtype)
    X = torch.from_numpy(verts).to(device=dev(), dtype=dtype)
    tr = sm.SingleModeTrainer(net, X, pair, previous=[p.to(device=dev(), dtype=dtype) for p in prev], lr=lr)
    losses = []
    for i in range(steps):
        if graph and i == 1:
            tr.enable_graph()
        losses.append(tr.step().clone())
    torch.cuda.synchronize()
    return tr, losses


@pytest.mark.parametrize("w0", [0.7, 0.0])
def test_twenty_steps_match_the_autograd_path(w0):
    ref, K, M, verts = _net_pair(torch.float64, w0=w0, coarse=False)
    rng = np.random.default_rng(9)
    prev = [torch.from_numpy(rng.standard_normal(K.shape[0]) / 40.0) for _ in range(2)]
    lr = 1e-3
    want_l, want_p = _autograd_run(ref, K, M, verts, prev, 20, torch.float64, lr)
    tr, got = _trainer_run(ref, K, M, verts, prev, 20, torch.float64, lr)
    got_l = torch.stack(got).cpu().numpy()[:, :4]
    assert _rel(got_l, want_l) < 1e-10
    got_p = tr.net.state_dict()
    for k, t in want_p.items():
        assert _rel(got_p[k].cpu(), t) < 1e-10, k
    # fp32 trainer against the fp64 autograd run: the tolerances of tests/test_gpu_variants.py
    tr32, got32 = _trainer_run(ref, K, M, verts, prev, 20, torch.float32, lr)
    l32 = torch.stack(got32).cpu().numpy()[:, :4]
    for j in range(3):                                      # total, eig, norm (ortho is checked with an absolute part)
        assert _rel(l32[:, j], want_l[:, j]) < 1e-4, j
    assert np.abs(l32[:, 3] - want_l[:, 3]).max() <= 1e-4 * np.abs(want_l[:, 3]).max() + 1e-8
    p32 = tr32.net.state_dict()
    for k, t in want_p.items():
        assert _rel(p32[k].double().cpu(), t) < 2e-4, k


@pytest.mark.parametrize("sfx", ["f32", "f64"])
def test_graph_replay_is_bit_identical_to_eager_and_runs_repeat(sfx):
    dtype = DTYPES[sfx]
    ref, K, M, verts = _net_pair(dtype, w0=0.5, coarse=False, hidden=64)
    rng = np.random.default_rng(4)
    prev = [torch.from_numpy(rng.standard_normal(K.shape[0]) / 40.0) for _ in range(3)]
    runs = [_trainer_run(ref, K, M, verts, prev, 12, dtype, 1e-3, graph=g) for g in (False, True, False)]
    (a, la), (b, lb), (c, lc) = runs
    for other, lo in ((b, lb), (c, lc)):
        for x, y in zip(la, lo):
            assert torch.equal(x, y)
        for name in ("flat", "m", "v"):
            assert torch.equal(getattr(a, name), getattr(other, name)), name
    assert a.step_count == b.step_count == 12


def test_train_modes_on_the_bunny_deflates():
    sm, fem = pkg("single_mode"), pkg("fem")
    g, (K, M), _ = bunny_levels()
    K, M = K.tocsr(), M.tocsr()
    pair = pkg("sparse").OperatorPair(K, M, dev())
    exact = scipy.linalg.eigh(K.toarray(), M.toarray(), eigvals_only=True, subset_by_index=[0, 3])
    torch.manual_seed(0)
    losses = []
    X = torch.from_numpy(np.ascontiguousarray(g["verts"], dtype=np.float32))
    eigs, U = sm.train_modes(X, pair, 3, 300, initial_eigenvalues=[0.0, 1.2 * exact[1], 1.2 * exact[2]],
                             hidden_dim=64, losses=losses)
    assert eigs.shape == (3,) and U.shape == (K.shape[0], 3)
    assert len(losses) == 3 and all(l.shape == (300, 4) for l in losses)
    assert (losses[0][:, 3] == 0).all()
    assert (losses[1][:, 3] > 0).any() and (losses[2][:, 3] > 0).any()     # the deflation term acts on modes 1, 2
    for l in losses:
        assert np.isfinite(l).all() and l[-1, 0] < l[0, 0]
    Ud = U.double().cpu().numpy()
    B = Ud.T @ (M @ Ud)
    A = Ud.T @ (K @ Ud)
    d = np.sqrt(np.diag(B))
    C = B / np.outer(d, d)
    off = np.abs(C - np.diag(np.diag(C))).max()
    print("train_modes: eigenvalues %s, exact %s, max |normalised U^T M U off-diagonal| %.3e" % (
        eigs.cpu().numpy(), exact[:3], off))
    assert off < 0.3
    ritz = scipy.linalg.eigh(A, B, eigvals_only=True)              # Rayleigh-Ritz on the span of the three modes
    assert np.all(ritz >= exact[:3] - 1e-6 * max(1.0, abs(exact[2])))


def test_errors_launch_nothing():
    sm, sparse, ops, cabi, v = (pkg(m) for m in ("single_mode", "sparse", "ops", "_cabi", "variants"))
    _, _, (Kc, Mc) = bunny_levels()
    n = Kc.shape[0]
    X = torch.zeros((n, 3), device=dev())
    net = v.EigenfunctionNN(16, 3, initial_eigenvalue=1.0).to(dev())
    before = cabi.launch_counter
    Kn = Kc.tolil()
    Kn[0, 1] = Kn[0, 1] + 1.0
    with pytest.raises(ValueError, match="symmetric"):
        sm.SingleModeTrainer(net, X, sparse.OperatorPair(Kn.tocsr(), Mc, dev()))
    with pytest.raises(TypeError):
        sm.SingleModeTrainer(net, X, sparse.OperatorPair(Kc, Mc, dev(), dtype=torch.float64))
    with pytest.raises(TypeError):
        sm.SingleModeTrainer(net, X.double(), sparse.OperatorPair(Kc, Mc, dev()))
    pair = sparse.OperatorPair(Kc, Mc, dev())
    with pytest.raises(cabi.EpError, match="at most 64"):
        sm.SingleModeTrainer(net, X, pair, previous=[torch.zeros(n, device=dev())] * 65)
    with pytest.raises(cabi.EpError, match="GPU"):
        sm.SingleModeTrainer(v.EigenfunctionNN(16, 3), X.cpu(), pair)
    assert cabi.launch_counter == before
    # the C ABI itself: P > P_max is EP_ERR_UNSUPPORTED, nothing is written
    ws = ops.single_mode_workspace(64, dev())
    lbuf, loss = _nan((4,), torch.float64)
    cbuf, coef = _nan((67,), torch.float64)
    col = torch.zeros((n, 1), device=dev())
    Q = torch.zeros((n, 65), device=dev())
    with pytest.raises(cabi.EpError, match=r"status -3"):
        ops.single_mode_fwd(col, col, col, Q, torch.ones(1, device=dev()), 1.0, loss, coef, ws)
    torch.cuda.synchronize()
    assert torch.isnan(lbuf).all() and torch.isnan(cbuf).all()


def test_fp64_optimiser_entries():
    """ep_adam_clip_step_f64 against torch.optim.Adam (fp64, betas of the notebook) over five steps, with clipping off;
    ep_grad_sqnorm_f64 against the fp64 sum; clipping on scales the gradient by max_norm / (norm + 1e-6)."""
    ops = pkg("ops")
    torch.manual_seed(1)
    n = 100003
    p0 = torch.randn(n, dtype=torch.float64, device=dev())
    grads = [torch.randn(n, dtype=torch.float64, device=dev()) for _ in range(5)]
    ref = p0.clone().requires_grad_(True)
    opt = torch.optim.Adam([ref], lr=1e-3, betas=(0.999, 0.9999), eps=1e-8)
    p, m, v = p0.clone(), torch.zeros_like(p0), torch.zeros_like(p0)
    sq = torch.full((1,), float("nan"), dtype=torch.float64, device=dev())
    for t, g in enumerate(grads, 1):
        ref.grad = g.clone()
        opt.step()
        ops.adam_clip_step(p, g, m, v, 1e-3, 0.999, 0.9999, 1e-8, 0.0, t, 0.0, None)
        ops.grad_sqnorm(g, sq)
        assert abs(sq.item() - (g * g).sum().item()) <= 1e-13 * sq.item()
    assert _rel(p.cpu(), ref.detach().cpu()) < 1e-13
    # clipping: one step with max_norm = norm / 4 equals an unclipped step on g * max_norm / (norm + 1e-6)
    g = grads[0]
    ops.grad_sqnorm(g, sq)
    norm = sq.item() ** 0.5
    pa, ma, va = p0.clone(), torch.zeros_like(p0), torch.zeros_like(p0)
    pb, mb, vb = p0.clone(), torch.zeros_like(p0), torch.zeros_like(p0)
    ops.adam_clip_step(pa, g, ma, va, 1e-3, 0.9, 0.999, 1e-8, 0.0, 1, norm / 4, sq)
    ops.adam_clip_step(pb, g * ((norm / 4) / (norm + 1e-6)), mb, vb, 1e-3, 0.9, 0.999, 1e-8, 0.0, 1, 0.0, None)
    assert _rel(va.cpu(), vb.cpu()) < 1e-14 and _rel(pa.cpu(), pb.cpu()) < 1e-14
