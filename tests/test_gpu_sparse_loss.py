"""GPU parity: CSR SpMM family and the eigen-loss (forward, analytic backward) against the CPU
oracle and the golden fixtures written by the reference.  Everything goes through the C ABI."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from gpu_util import pkg, dev, bunny_levels, random_csr
from oracle import step_port

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("k", [1, 3, 10, 16, 32, 64, 128, 130])
def test_spmm_matches_scipy(k):
    ops, sparse = pkg("ops"), pkg("sparse")
    A = random_csr(777, 500, 11, seed=k, empty_every=13)
    X = np.random.default_rng(k).standard_normal((500, k)).astype(np.float32)
    Ad = sparse.CsrMatrix.from_scipy(A, dev())
    Y = ops.spmm(Ad, torch.from_numpy(X).to(dev())).cpu().numpy()
    ref = (A.astype(np.float32) @ X.astype(np.float64))
    np.testing.assert_allclose(Y, ref, rtol=2e-5, atol=2e-5)


def test_spmm_strided_views_and_empty():
    ops, sparse = pkg("ops"), pkg("sparse")
    A = random_csr(300, 300, 7, seed=5)
    Ad = sparse.CsrMatrix.from_scipy(A, dev())
    big = torch.randn(300, 50, device=dev())
    X = big[:, 3:35]                       # k = 32 but unaligned base and ld = 50
    out = torch.zeros(300, 40, device=dev())
    ops.spmm(Ad, X, out=out[:, 1:33])
    ref = A.astype(np.float32) @ X.cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(out[:, 1:33].cpu().numpy(), ref, rtol=2e-5, atol=2e-5)
    assert out[:, 0].abs().max() == 0 and out[:, 33:].abs().max() == 0
    E = sparse.CsrMatrix.from_scipy(random_csr(0, 10, 1, 0), dev())
    assert ops.spmm(E, torch.randn(10, 8, device=dev())).shape == (0, 8)


@pytest.mark.parametrize("k", [10, 32, 64])
def test_dual_and_sum_kernels(k):
    ops, sparse = pkg("ops"), pkg("sparse")
    fem, (K, M), _ = bunny_levels()
    pair = sparse.OperatorPair(K, M, dev())
    assert pair.shared and pair.symmetric
    U = torch.randn(K.shape[0], k, device=dev())
    KU, MU = ops.spmm2(pair, U)
    Un = U.cpu().numpy().astype(np.float64)
    K32, M32 = K.astype(np.float32).astype(np.float64), M.astype(np.float32).astype(np.float64)
    np.testing.assert_allclose(KU.cpu().numpy(), K32 @ Un, rtol=1e-5, atol=1e-4)
    np.testing.assert_allclose(MU.cpu().numpy(), M32 @ Un, rtol=1e-5, atol=1e-6)
    D = torch.randn_like(U)
    Y = ops.spmm2_sum(pair.KT, pair.MT, KU, MU, D, 0.37)
    ref = 0.37 * (K32 @ KU.cpu().numpy().astype(np.float64) + M32 @ MU.cpu().numpy().astype(np.float64)
                  + D.cpu().numpy())
    np.testing.assert_allclose(Y.cpu().numpy(), ref, rtol=2e-5, atol=2e-3)


def test_operator_pair_unifies_different_patterns_and_transposes():
    ops, sparse = pkg("ops"), pkg("sparse")
    A, B = random_csr(200, 200, 6, 1), random_csr(200, 200, 4, 2)
    pair = sparse.OperatorPair(A, B, dev())
    assert pair.shared and not pair.symmetric
    X = torch.randn(200, 16, device=dev())
    YA, YB = ops.spmm2(pair, X)
    Xn = X.cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(YA.cpu().numpy(), A.astype(np.float32) @ Xn, rtol=2e-5, atol=2e-5)
    np.testing.assert_allclose(YB.cpu().numpy(), B.astype(np.float32) @ Xn, rtol=2e-5, atol=2e-5)
    Z = ops.spmm2_sum(pair.KT, pair.MT, YA, YB, None, 1.0)
    ref = A.T.astype(np.float32) @ YA.cpu().numpy().astype(np.float64) + B.T.astype(np.float32) @ YB.cpu().numpy().astype(np.float64)
    np.testing.assert_allclose(Z.cpu().numpy(), ref, rtol=2e-5, atol=2e-4)


@pytest.mark.parametrize("k", [5, 16, 32, 48, 64, 128])
def test_eigen_partials_against_fp64(k):
    ops = pkg("ops")
    n = 3001
    g = torch.Generator().manual_seed(k)
    U, KU, MU = [torch.randn(n, k, generator=g) for _ in range(3)]
    P = ops.eigen_partials(U.to(dev()), KU.to(dev()), MU.to(dev())).cpu().numpy()
    U64, KU64, MU64 = U.double().numpy(), KU.double().numpy(), MU.double().numpy()
    ref = np.concatenate([(U64.T @ MU64).ravel(), (U64 * KU64).sum(0), (KU64 * KU64).sum(0),
                          (KU64 * MU64).sum(0), (MU64 * MU64).sum(0), MU64.sum(0)])
    np.testing.assert_allclose(P, ref, rtol=0, atol=2e-6 * np.sqrt(n) * 4)
    # run twice: deterministic reduction order
    P2 = ops.eigen_partials(U.to(dev()), KU.to(dev()), MU.to(dev())).cpu().numpy()
    assert np.array_equal(P, P2)


@pytest.mark.parametrize("tag,k", [("k16_1lvl", 16), ("k64_1lvl", 64), ("k16_2lvl", 16)])
def test_eigen_loss_matches_reference_fixture(tag, k):
    """loss_res, loss_orth, lambda within 1e-5 relative of the reference's CPU fp32 values; gradient vs autograd."""
    ops, sparse = pkg("ops"), pkg("sparse")
    g = load_golden("eigen_loss.npz")
    fem, (K, M), (Kc, Mc) = bunny_levels()
    levels = [(Kc, Mc), (K, M)] if tag.endswith("2lvl") else [(K, M)]
    pairs = [sparse.OperatorPair(a, b, dev()) for a, b in levels]
    U = torch.from_numpy(g[f"{tag}_U"]).to(dev()).requires_grad_(True)
    l_res, l_orth, lams = ops.eigen_loss(U, pairs, [int(o) for o in g[f"{tag}_offsets"]], 1000.0, 10.0)
    lam_t = torch.from_numpy(g[f"{tag}_lam_target"]).to(dev())
    lam0 = lams[0]
    extra = (0.5 * lam0.mean() + 2.0 * torch.relu(lam0[:-1] - lam0[1:]).sum() + 3.0 * ((lam0 - lam_t) ** 2).mean())
    total = l_res + l_orth + extra
    total.backward()
    assert l_res.item() == pytest.approx(float(g[f"{tag}_loss_res"]), rel=1e-5)
    assert l_orth.item() == pytest.approx(float(g[f"{tag}_loss_orth"]), rel=1e-5)
    assert total.item() == pytest.approx(float(g[f"{tag}_total"]), rel=1e-5)
    for i, l in enumerate(lams):
        ref = g[f"{tag}_lam{i}"]
        np.testing.assert_allclose(l.detach().cpu().numpy(), ref, rtol=1e-5, atol=1e-5 * np.abs(ref).max())
    gref = g[f"{tag}_grad"]
    err = np.abs(U.grad.cpu().numpy() - gref).max()
    assert err <= 2e-5 * np.abs(gref).max(), err


def test_engine_fused_loss_equals_autograd_path():
    """The explicit engine (level-0 eigenvalue terms inside the finalize kernel) and the autograd
    Function (terms in torch) must give the same loss and the same dL/dU."""
    ops, sparse, engine = pkg("ops"), pkg("sparse"), pkg("engine")
    g = load_golden("eigen_loss.npz")
    fem, (K, M), (Kc, Mc) = bunny_levels()
    pairs = [sparse.OperatorPair(Kc, Mc, dev()), sparse.OperatorPair(K, M, dev())]
    k = 16
    U = torch.from_numpy(g["k16_2lvl_U"]).to(dev())
    offs = [int(o) for o in g["k16_2lvl_offsets"]]
    lam_t = torch.from_numpy(g["k16_2lvl_lam_target"]).to(dev())
    W = [torch.zeros(k, 4, device=dev())]
    b = [torch.zeros(k, device=dev())]
    cfg = engine.StepConfig(w_trace=0.5, w_order=2.0, w_eigen=3.0)
    eng = engine.TrainStepEngine(torch.zeros(U.shape[0], 4, device=dev()), U, pairs, offs,
                                 engine.FlatParams(W, b, dev()), cfg, lam_target=lam_t)
    eng.U_pred.copy_(U)
    eng.loss_forward()
    eng.loss_backward(1.0)
    acc = eng.loss_acc.cpu().numpy()
    assert acc[5] == pytest.approx(float(g["k16_2lvl_total"]), rel=1e-5)
    np.testing.assert_allclose(acc[2:5] / np.array([0.5, 2.0, 3.0]),
                               g["k16_2lvl_extra"][1:] / np.array([0.5, 2.0, 3.0]), rtol=1e-5, atol=1e-7)
    gref = g["k16_2lvl_grad"]
    assert np.abs(eng.dCorr.cpu().numpy() - gref).max() <= 2e-5 * np.abs(gref).max()


def test_m_normalize_and_rayleigh_ritz():
    ops, sparse = pkg("ops"), pkg("sparse")
    g = load_golden("corrector_train.npz")
    fem, (K, M), _ = bunny_levels()
    U0 = torch.from_numpy(g["U0_1"]).to(dev())
    out = ops.m_normalize_columns(U0, sparse.CsrMatrix.from_scipy(M, dev()))
    np.testing.assert_allclose(out.cpu().numpy(), g["U_norm_1"], rtol=1e-5, atol=1e-7)
    A, B = ops.gram_pair(U0, sparse.OperatorPair(K, M, dev()))
    from scipy.linalg import eigh
    vals, _ = eigh(A.cpu().numpy(), B.cpu().numpy())
    np.testing.assert_allclose(vals, g["rr_vals"], rtol=1e-4, atol=2e-5)


def test_large_mesh_properties():
    """1 M-vertex icosphere (BASELINE config 4 size): linearity, symmetry <x, K y> = <K x, y>, constant
    vector in the null space of K, and M 1 = lumped areas (sum = 2 * 4 pi)."""
    ops, sparse, fem_mod, syn = pkg("ops"), pkg("sparse"), pkg("fem"), pkg("synthetic")
    v, t = syn.icosphere(316)
    K, M = fem_mod.assemble_stiffness_mass(v, t)
    pair = sparse.OperatorPair(K, M, dev())
    n, k = v.shape[0], 32
    g = torch.Generator(device="cuda").manual_seed(0)
    X = torch.randn(n, k, device=dev(), generator=g)
    Y = torch.randn(n, k, device=dev(), generator=g)
    KX, MX = ops.spmm2(pair, X)
    KY, MY = ops.spmm2(pair, Y)
    KXY, _ = ops.spmm2(pair, X + 2.0 * Y)
    assert (KXY - (KX + 2.0 * KY)).abs().max().item() <= 1e-3 * KX.abs().max().item()
    a = (X.double() * KY.double()).sum().item()
    b = (KX.double() * Y.double()).sum().item()
    assert abs(a - b) <= 1e-6 * max(abs(a), abs(b), (X.double().norm() * KY.double().norm()).item())
    ones = torch.ones(n, k, device=dev())
    K1, M1 = ops.spmm2(pair, ones)
    assert K1.abs().max().item() < 2e-2 * float(abs(K).max())
    assert M1[:, 0].double().sum().item() == pytest.approx(8.0 * np.pi, rel=1e-4)


@pytest.mark.parametrize("k", [16, 32, 64, 128])
def test_fused_symmetric_backward_equals_general_path(k):
    """One-pass backward (symmetric K, M) against prepare + transposed dual SpMM (the same matrices declared
    non-symmetric), and partials for every tiling."""
    ops, sparse, engine = pkg("ops"), pkg("sparse"), pkg("engine")
    fem, (K, M), _ = bunny_levels()
    pairs = [sparse.OperatorPair(K, M, dev()), sparse.OperatorPair(K, M, dev(), assume_symmetric=False)]
    assert pairs[0].symmetric and not pairs[1].symmetric
    n = K.shape[0]
    g = torch.Generator().manual_seed(k)
    U = (0.3 * torch.randn(n, k, generator=g)).to(dev())
    cfg = engine.StepConfig(w_trace=0.5, w_order=2.0, w_eigen=3.0)
    outs = []
    for pair in pairs:                                 # one-pass form, then the general path
        eng = engine.TrainStepEngine(torch.zeros(n, 4, device=dev()), U, [pair], [0],
                                     engine.FlatParams([torch.zeros(k, 4)], [torch.zeros(k)], dev()), cfg,
                                     lam_target=torch.linspace(0, 2, k).to(dev()))
        eng.U_pred.copy_(U)
        eng.loss_forward()
        eng.loss_backward(0.7)
        outs.append((eng.dCorr.clone(), eng.loss_acc.clone()))
    assert torch.equal(outs[0][1], outs[1][1])
    ref = outs[1][0]
    assert (outs[0][0] - ref).abs().max().item() <= 2e-5 * ref.abs().max().item()
    # and against torch autograd on the CPU oracle
    Uc = U.cpu().requires_grad_(True)
    l_res, l_orth, lams = step_port.residual_ortho_loss(Uc, [K], [M], [0], cfg.w_res, cfg.w_orth, k)
    extra = step_port.eigenvalue_losses(lams[0], torch.linspace(0, 2, k), 0.0, 0.5, 2.0, 3.0)
    (l_res + l_orth + sum(extra)).backward()
    gref = 0.7 * Uc.grad
    assert (outs[0][0].cpu() - gref).abs().max().item() <= 5e-5 * gref.abs().max().item()


@pytest.mark.parametrize("symmetric", [True, False])
def test_notebook_variant_terms_against_autograd(symmetric):
    """Zero-mean, smoothness and projection terms (SURVEY 8a-bis; notebooks multigrid_gnn_farthest_point_sampling cell 0,
    multigrid_gnn_refine_fixed cells 0 and 4) as flags of the engine's eigen-loss: loss terms and dL/dU against a
    torch-autograd (fp64) restatement of the notebook formulas on the coarse + bunny pair.  symmetric=False declares the
    operators non-symmetric, so the backward takes the general path instead of the one-pass form."""
    import scipy.sparse as sp
    ops, sparse, engine = pkg("ops"), pkg("sparse"), pkg("engine")
    from sklearn.neighbors import NearestNeighbors
    fem, (K, M), (Kc, Mc) = bunny_levels()
    n, nc, k = K.shape[0], Kc.shape[0], 16
    g = torch.Generator().manual_seed(4)
    U = 0.05 * torch.randn(nc + n, k, generator=g)
    U[:, 0] += 0.02                                                   # a mean component for the zero-mean term
    dist_, idx = NearestNeighbors(n_neighbors=6).fit(fem["coarse_verts"]).kneighbors(fem["verts"])
    w = 1.0 / (dist_ + 1e-12)
    w /= w.sum(1, keepdims=True)
    P = sp.coo_matrix((w.ravel(), (np.repeat(np.arange(n), 6), idx.ravel())), shape=(n, nc)).tocsr()
    U_c = 0.05 * torch.randn(nc, k, generator=g)
    w_res, w_orth, w_mean, w_smooth, w_proj = 1000.0, 10.0, 7.0, 3.0, 11.0
    # ---- reference: the notebook formulas in fp64 with autograd
    Ud = U.double().requires_grad_(True)
    total = torch.zeros((), dtype=torch.float64)
    terms = {"mean": 0.0, "smooth": 0.0}
    for (Kl, Ml, off) in ((Kc, Mc, 0), (K, M, nc)):
        nl = Kl.shape[0]
        Kt = torch.from_numpy(Kl.astype(np.float32).toarray().astype(np.float64))
        Mt = torch.from_numpy(Ml.astype(np.float32).toarray().astype(np.float64))
        Ul = Ud[off:off + nl]
        Lu, Mu = Kt @ Ul, Mt @ Ul
        lam = (Ul * Lu).sum(0) / ((Ul * Mu).sum(0) + 1e-12)
        l_res = ((Lu - Mu * lam) ** 2).mean()
        l_orth = ((Ul.t() @ Mu - torch.eye(k, dtype=torch.float64)) ** 2).sum() / k
        l_mean = ((torch.ones(1, nl, dtype=torch.float64) @ Mu[:, 1:]) ** 2).mean()
        l_smooth = (Ul * Lu).sum() / (nl * k)
        total = total + w_res * l_res + w_orth * l_orth + w_mean * l_mean + w_smooth * l_smooth
        terms["mean"] += w_mean * float(l_mean)
        terms["smooth"] += w_smooth * float(l_smooth)
    Pt = torch.from_numpy(P.toarray())
    l_proj = ((Pt.t() @ Ud[nc:] - U_c.double()) ** 2).sum() / (nc * k)
    total = total + w_proj * l_proj
    total.backward()
    # ---- engine
    h = torch.zeros(nc + n, 4, device=dev())
    params = engine.FlatParams([torch.zeros(8, 4), torch.zeros(k, 8)], [torch.zeros(8), torch.zeros(k)], dev())
    cfg = engine.StepConfig(w_res=w_res, w_orth=w_orth, w_mean=w_mean, w_smooth=w_smooth)
    assume = None if symmetric else False
    pairs = [sparse.OperatorPair(a, b, dev(), assume_symmetric=assume) for a, b in ((Kc, Mc), (K, M))]
    assert all(p.symmetric == symmetric for p in pairs)
    eng = engine.TrainStepEngine(h, U.to(dev()), pairs, [0, nc], params, cfg)
    eng.add_projection_term(1, P, U_c, w_proj)
    eng.U_pred.copy_(U.to(dev()))
    eng.loss_forward()
    eng.loss_backward(1.0)
    acc = eng.loss_acc.cpu().numpy()
    assert acc[5] == pytest.approx(float(total), rel=2e-5)
    assert acc[6] == pytest.approx(w_proj * float(l_proj), rel=2e-5)
    assert acc[7] == pytest.approx(terms["mean"], rel=2e-5) and acc[8] == pytest.approx(terms["smooth"], rel=2e-5)
    gref = Ud.grad.numpy()
    err = np.abs(eng.dCorr.cpu().numpy() - gref).max()
    assert err <= 3e-5 * np.abs(gref).max(), err


@pytest.mark.parametrize("k", [64])
@pytest.mark.parametrize("n", [1, 127, 2503, 40001])
def test_tensor_core_gram_term_matches_fp64(n, k):
    """ep_eigen_bwd_gram_term_tf32x3: dU = s * MU (Gp + Gp^T) on tcgen05 (TF32 x 3) against fp64, strided inputs.  It is
    built for k = 64 only; tests/test_cabi_cpu.py checks that every other k is rejected."""
    import ctypes
    cabi, ops = pkg("_cabi"), pkg("ops")
    g = torch.Generator().manual_seed(100 * k + n % 97)
    KUMU = torch.randn(n, 2 * k, generator=g).to(dev())                # MU is the right half of an interleaved row
    MU = KUMU[:, k:]
    clen = cabi.query("ep_eigen_coef_len", k)
    coef = torch.randn(clen, generator=g).to(dev())
    out = torch.full((n + 3, k), float("nan"), device=dev())           # rows [2, 2 + n) of a larger array are written
    P = lambda t: ctypes.c_void_p(t.data_ptr())
    cabi.call("ep_eigen_bwd_gram_term_tf32x3", 0, n, k, P(MU), MU.stride(0), P(coef), 0.37, None, P(out[2:]), out.stride(0),
              ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    c = coef.double().cpu()
    G = c[1 + 3 * k:1 + 3 * k + k * k].view(k, k)
    S = G + G.t() + 2.0 * torch.diag(c[1 + 2 * k:1 + 3 * k])
    ref = 0.37 * (MU.double().cpu() @ S)
    got = out[2:2 + n].double().cpu()
    assert torch.isnan(out[:2]).all() and torch.isnan(out[2 + n:]).all()
    assert (got - ref).abs().max().item() <= 4e-6 * ref.abs().max().item() * np.sqrt(k / 16.0)


def test_one_pass_backward_row_ranges_and_general_path_at_k64():
    """k = 64, where the k x k term runs on the tensor cores before the gather pass: the row ranges (0, 1000) + (1000, n)
    give the whole-range result bit for bit, and that equals the general path (prepare + transposed dual SpMM, which
    takes no row range)."""
    ops, sparse = pkg("ops"), pkg("sparse")
    fem, (K, M), _ = bunny_levels()
    pair = sparse.OperatorPair(K, M, dev())
    general = sparse.OperatorPair(K, M, dev(), assume_symmetric=False)
    n, k = K.shape[0], 64
    U = (0.3 * torch.randn(n, k, generator=torch.Generator().manual_seed(k))).to(dev())
    KUMU = torch.empty(n, 2 * k, device=dev())
    KU, MU = KUMU[:, :k], KUMU[:, k:]
    ops.spmm2(pair, U, out_K=KU, out_M=MU)
    Pp = ops.eigen_partials(U, KU, MU)
    acc = torch.zeros(ops.N_LOSS_TERMS, dtype=torch.float64, device=dev())
    _, coef = ops.eigen_finalize(k, n, Pp, 1000.0, 10.0, acc, w_mean=2.0, w_smooth=1.5)
    whole = ops.eigen_loss_bwd(pair, U, KU, MU, coef, 0.7, torch.zeros(n, k, device=dev()))
    split = torch.zeros(n, k, device=dev())
    ops.eigen_loss_bwd(pair, U, KU, MU, coef, 0.7, split, rows=(0, 1000))
    ops.eigen_loss_bwd(pair, U, KU, MU, coef, 0.7, split, rows=(1000, n))
    ref = ops.eigen_loss_bwd(general, U, KU, MU, coef, 0.7, torch.zeros(n, k, device=dev()))
    assert torch.equal(split, whole)
    assert (whole - ref).abs().max().item() <= 1e-5 * ref.abs().max().item()
    with pytest.raises(NotImplementedError):
        ops.eigen_loss_bwd(general, U, KU, MU, coef, 0.7, split, rows=(0, 1000))
