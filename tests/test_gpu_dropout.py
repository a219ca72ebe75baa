"""Dropout in the fused training step (csrc/dropout.cuh): device masks against the numpy port, the fp32 and bf16 layer
kernels against fp64 with the same masks, the chain against the layer-by-layer kernels bit for bit, one whole step
against an fp64 restatement, graph replay against eager, p = 0 unchanged, the drop-in entry point, and the sharded
engine's refusal."""
import numpy as np
import pytest
import torch

from gpu_util import pkg, dev, dropin, bunny_levels
from oracle import dropout_port as port

pytestmark = pytest.mark.gpu


def _drop(p, seed):
    return pkg("ops").Dropout(p, seed)


@pytest.mark.parametrize("n", [1, 127, 129, 777, 4097])
@pytest.mark.parametrize("width", [32, 82, 256])
def test_keep_mask_equals_port(n, width):
    ops = pkg("ops")
    for seed, step, layer, p, row0 in ((1, 1, 0, 0.1, 0), (2 ** 63 + 12345, 77, 3, 0.5, 1000), (42, 2 ** 20, 5, 0.9, 7)):
        got = ops.dropout_keep_mask(n, width, _drop(p, seed), step, layer, row0=row0, device=dev()).cpu().numpy()
        assert np.array_equal(got.astype(bool), port.keep_mask(n, width, p, seed, step, layer, row0=row0))


@pytest.mark.parametrize("n,d_in,d_out", [(1, 7, 5), (300, 82, 256), (4097, 146, 64), (129, 256, 256)])
def test_fp32_layers_match_fp64_with_the_same_masks(n, d_in, d_out):
    ops = pkg("ops")
    g = torch.Generator().manual_seed(n + d_out)
    X = torch.randn(n, d_in, generator=g).abs() - 0.3
    W = torch.randn(d_out, d_in, generator=g) / np.sqrt(d_in)
    b = torch.randn(d_out, generator=g)
    dY = torch.randn(n, d_out, generator=g)
    d, step, layer = _drop(0.25, 9), 5, 1
    keep = torch.from_numpy(port.keep_mask(n, d_out, d.p, d.seed, step, layer)).double()
    s = float(port.scale(d.p))
    Y = ops.linear_fwd_dropout(X.to(dev()), W.to(dev()), b.to(dev()), d, step, layer)
    ref = torch.relu(torch.nn.functional.linear(X.double(), W.double(), b.double())) * keep * s
    np.testing.assert_allclose(Y.cpu().numpy(), ref.numpy(), rtol=1e-5, atol=1e-5)
    # backward of the NEXT layer, whose input is this dropped activation: dX = (dZ W2) * [Y > 0] * s
    W2 = torch.randn(d_in, d_out, generator=g) / np.sqrt(d_out)
    dZ = torch.randn(n, d_in, generator=g)
    dX, dW, db = ops.linear_bwd_dropout(Y, W2.to(dev()), dZ.to(dev()), d)
    Yd = Y.cpu().double()
    np.testing.assert_allclose(dX.cpu().numpy(), ((dZ.double() @ W2.double()) * (Yd > 0) * s).numpy(), rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(dW.cpu().numpy(), (dZ.double().t() @ Yd).numpy(), rtol=1e-5, atol=1e-5 * np.sqrt(n))
    np.testing.assert_allclose(db.cpu().numpy(), dZ.double().sum(0).numpy(), rtol=1e-5, atol=1e-5 * np.sqrt(n))


def _tc_pair(n, dims, seed, drop):
    eng, tcm = pkg("engine"), pkg("mlp_tc")
    g = torch.Generator().manual_seed(seed)
    Ws = [torch.randn(dims[i + 1], dims[i], generator=g) / np.sqrt(dims[i]) for i in range(len(dims) - 1)]
    bs = [0.1 * torch.randn(dims[i + 1], generator=g) for i in range(len(dims) - 1)]
    h = torch.randn(n, dims[0], generator=g).to(dev())
    U = torch.randn(n, dims[-1], generator=g).to(dev())
    out = []
    for chain in (True, False):
        fp = eng.FlatParams(Ws, bs, dev())
        out.append((fp, tcm.TcMlp(n, fp, dev(), h, chain_fwd=chain, dropout=drop)))
    return h, U, out


@pytest.mark.parametrize("n,dims", [(1, [82, 256, 32]), (300, [82, 256, 256, 256, 32]), (4097, [146, 128, 256, 64]),
                                    (998, [82, 256, 256, 256, 256, 256, 256, 32])])
def test_bf16_chain_equals_layers_with_dropout(n, dims):
    d = _drop(0.1, 2024)
    h, U, ((_, chain), (_, layers)) = _tc_pair(n, dims, n, d)
    res = []
    for m in (chain, layers):
        Up = torch.empty_like(U)
        m.forward(h, U_base=U, scale=0.7, U_pred=Up, step=3)
        torch.cuda.synchronize()
        res.append((m, m.corr.clone(), Up))
    (a, ca, ua), (b, cb, ub) = res
    assert torch.equal(ca, cb) and torch.equal(ua, ub)
    tcm = pkg("mlp_tc")
    for l in range(len(dims) - 2):
        assert torch.equal(a.acts[l], b.acts[l]) and torch.equal(a.masks[l], b.masks[l])
        act = tcm.unpack_rows(a.acts[l], n, a.pd[l + 1])[:, :dims[l + 1]].cpu()
        keep = torch.from_numpy(port.keep_mask(n, dims[l + 1], d.p, d.seed, 3, l))
        assert not bool((act[~keep] != 0).any())                 # dropped units are stored as zero
        frac = (act != 0).double().mean().item()
        assert frac <= keep.double().mean().item() + 1e-9


def test_bf16_chain_with_dropout_differs_from_plain_and_p0_equals_plain():
    n, dims = 515, [82, 256, 256, 32]
    outs = []
    for d in (None, _drop(0.0, 5), _drop(0.2, 5)):
        h, U, ((_, chain), _) = _tc_pair(n, dims, 1, d)
        Up = torch.empty_like(U)
        chain.forward(h, U_base=U, scale=0.5, U_pred=Up, step=1)
        outs.append(Up.clone())
    assert torch.equal(outs[0], outs[1])
    assert not torch.equal(outs[0], outs[2])


def test_bf16_dx_with_dropout_within_a_priori_bound():
    """dZprev = bf16((dZ WT) * s) & mask, checked against fp64 from the same bf16 operands: one fp32 accumulation
    (K <= 256 terms) and one bf16 rounding of the scaled value."""
    tcm, cabi = pkg("mlp_tc"), pkg("_cabi")
    n, n_out, n_in = 777, 256, 256
    d = _drop(0.3, 11)
    h, U, ((fp, m), _) = _tc_pair(n, [82, n_in, n_out, 32], 3, d)
    m.forward(h, step=4)
    g = torch.Generator().manual_seed(5)
    dz = torch.randn(n, n_out, generator=g).to(dev())
    dz_p = tcm.pack_rows(dz, n_out)
    out = torch.zeros_like(m.dz[0])
    cabi.call("ep_tc_linear_dx_dropout_bf16", n, n_out, n_in, tcm._p(dz_p), tcm._p(m.WTp[1]), tcm._p(m.masks[0]),
              tcm._p(out), d.p, 0, tcm._stream())
    got = tcm.unpack_rows(out, n, n_in).double().cpu()
    dzb = tcm.unpack_rows(dz_p, n, n_out).double().cpu()
    Wb = fp.W[1].detach().to(torch.bfloat16).double().cpu()             # (n_out, n_in)
    act = tcm.unpack_rows(m.acts[0], n, n_in).cpu()
    s = float(port.scale(d.p))
    exact = (dzb @ Wb) * s * (act > 0)
    mag = (dzb.abs() @ Wb.abs()) * s
    bound = 2.0 ** -8 * exact.abs() + 256 * 2.0 ** -23 * mag + 1e-30
    assert bool(((got - exact).abs() <= bound).all()), ((got - exact).abs() / bound).max().item()


def _engine(mlp_mode, p, model="simple", seed=0):
    eng, sparse = pkg("engine"), pkg("sparse")
    fem, (K, M), (Kc, Mc) = bunny_levels()
    g = torch.Generator().manual_seed(seed)
    k = 16
    n = K.shape[0]
    h = torch.randn(n, 2 * 41, generator=g).to(dev())
    U = (0.1 * torch.randn(n, k, generator=g)).to(dev())
    dims = [82, 128, 128, 128, k]
    Ws = [torch.randn(dims[i + 1], dims[i], generator=g) / np.sqrt(dims[i]) for i in range(len(dims) - 1)]
    bs = [0.05 * torch.randn(dims[i + 1], generator=g) for i in range(len(dims) - 1)]
    scales = torch.ones(k) + 0.1 * torch.randn(k, generator=g) if model == "adaptive" else None
    fp = eng.FlatParams(Ws, bs, dev(), mode_scales=scales)
    cfg = eng.StepConfig(corr_scale=1.0, ramp_epochs=1.0, w_res=1000.0, w_orth=10.0, dropout=p, dropout_seed=77)
    pair = sparse.OperatorPair(K, M, dev())
    e = eng.TrainStepEngine(h, U, [pair], [0], fp, cfg, mlp_mode=mlp_mode)
    return e, (K, M), h, U, Ws, bs, scales


def _fp64_step(e, KM, h, U, Ws, bs, scales, p, step):
    """Loss terms and gradient of one step in fp64 torch autograd, with the kernels' keep masks."""
    K, M = KM
    n, k = U.shape
    Ws = [w.double().requires_grad_() for w in Ws]
    bs = [b.double().requires_grad_() for b in bs]
    x = h.double().cpu()
    s = float(port.scale(p))
    for l, (W, b) in enumerate(zip(Ws, bs)):
        x = torch.nn.functional.linear(x, W, b)
        if l + 1 < len(Ws):
            keep = torch.from_numpy(port.keep_mask(n, W.shape[0], p, 77, step, l)).double()
            x = torch.relu(x) * keep * s
    leaves = Ws + bs
    if scales is not None:
        sc = scales.double().requires_grad_()
        x = x * sc[None, :]
        leaves = leaves + [sc]
    Up = U.double().cpu() + x
    Kd = torch.sparse_csr_tensor(torch.from_numpy(K.indptr).long(), torch.from_numpy(K.indices).long(),
                                 torch.from_numpy(K.data).double(), size=K.shape)
    Md = torch.sparse_csr_tensor(torch.from_numpy(M.indptr).long(), torch.from_numpy(M.indices).long(),
                                 torch.from_numpy(M.data).double(), size=M.shape)
    KU, MU = Kd @ Up, Md @ Up
    lam = (Up * KU).sum(0) / ((Up * MU).sum(0) + 1e-12)
    res = 1000.0 * ((KU - MU * lam[None, :]) ** 2).mean()
    orth = 10.0 * ((Up.t() @ MU - torch.eye(k, dtype=torch.float64)) ** 2).sum() / k
    total = res + orth
    grads = torch.autograd.grad(total, leaves)
    flat = []
    for W, b, gw, gb in zip(Ws, bs, grads[:len(Ws)], grads[len(Ws):2 * len(Ws)]):
        flat += [gw.reshape(-1), gb.reshape(-1)]
    if scales is not None:
        flat.append(grads[-1])
    return np.array([res.item(), orth.item(), total.item()]), torch.cat(flat).numpy()


@pytest.mark.parametrize("model", ["simple", "adaptive"])
def test_whole_step_matches_fp64_restatement_and_bf16_tracks_fp32(model):
    p = 0.1
    res = {}
    for mode in ("fp32", "bf16"):
        e, KM, h, U, Ws, bs, scales = _engine(mode, p, model)
        acc = e.step(1.0).cpu().numpy()
        torch.cuda.synchronize()
        res[mode] = (np.array([acc[0], acc[1], acc[5]]), e.params.grad.cpu().numpy().copy())
        if mode == "fp32":
            ref_loss, ref_grad = _fp64_step(e, KM, h.cpu(), U.cpu(), Ws, bs, scales, p, 1)
    np.testing.assert_allclose(res["fp32"][0], ref_loss, rtol=1e-5)
    np.testing.assert_allclose(res["fp32"][1], ref_grad, rtol=1e-4, atol=1e-4 * np.abs(ref_grad).max())
    rel = np.abs(res["bf16"][0] - res["fp32"][0]) / np.abs(res["fp32"][0])
    assert rel[:2].max() < 2.5e-2 and rel[2] < 5e-3, rel


@pytest.mark.parametrize("mlp_mode", ["fp32", "bf16"])
def test_graph_replay_equals_eager_with_dropout(mlp_mode):
    p = 0.1
    runs = []
    for graphed in (False, True):
        e = _engine(mlp_mode, p)[0]
        hist = [e.step(1.0).cpu().numpy().copy()]
        if graphed:
            e.enable_graph()
        for ep_ in range(11):
            hist.append(e.step(1.0, lr=1e-3 if ep_ < 5 else 5e-4).cpu().numpy().copy())
        runs.append((np.array(hist), e.params.flat.clone(), e.params.m.clone(), e.params.v.clone()))
    assert np.array_equal(runs[0][0], runs[1][0]), np.abs(runs[0][0] - runs[1][0]).max()
    for a, b in zip(runs[0][1:], runs[1][1:]):
        assert torch.equal(a, b), (a - b).abs().max().item()
    # masks of consecutive steps differ in about 2 p_q (1 - p_q) of the entries
    ops = pkg("ops")
    d = _drop(p, 77)
    a = ops.dropout_keep_mask(4096, 256, d, 5, 0, device=dev())
    b = ops.dropout_keep_mask(4096, 256, d, 6, 0, device=dev())
    q = port.threshold(p) / 65536.0
    want = 2 * q * (1 - q)
    assert abs((a != b).double().mean().item() - want) < 5 * np.sqrt(want * (1 - want) / a.numel())


@pytest.mark.parametrize("mlp_mode", ["fp32", "bf16"])
def test_p0_launches_the_plain_kernels(mlp_mode):
    tables = []
    for kw in ({}, {"dropout": 0.0}):
        eng = pkg("engine")
        e, _, h, U, Ws, bs, _ = _engine(mlp_mode, 0.0)
        if not kw:
            cfg = eng.StepConfig(corr_scale=1.0, ramp_epochs=1.0, w_res=1000.0, w_orth=10.0)
            e = eng.TrainStepEngine(e.h, e.U_base, e.pairs, [0], eng.FlatParams(Ws, bs, dev()), cfg, mlp_mode=mlp_mode)
        assert e.dropout is None
        e.step(1.0)
        e.enable_graph()
        e.step(1.0)
        tables.append(dict(e.launches_by_entry))
    assert tables[0] == tables[1]
    assert not any("dropout" in k for k in tables[0])


@pytest.mark.parametrize("mlp_mode", ["fp32", "bf16"])
def test_dropin_main_trains_with_dropout(mlp_mode, tmp_path):
    import sys
    from conftest import load_golden
    from test_gpu_dropin_e2e import _write_obj, _write_config
    for m in ("main", "samplers", "multigrid_model", "diagnostics"):
        sys.modules.pop(m, None)
    main_mod = dropin("main")
    fem = load_golden("bunny_fem.npz")
    mesh_file, coarse_file = str(tmp_path / "bunny.obj"), str(tmp_path / "coarse.obj")
    _write_obj(mesh_file, fem["verts"], fem["tris"])
    _write_obj(coarse_file, fem["coarse_verts"], fem["coarse_tris"])
    k = 12
    cfg_file = _write_config(tmp_path, mesh_file=mesh_file, coarse_mesh_files=[coarse_file],
                             vtu_file=str(tmp_path / "out" / "model.vtu"), diagnostics_viz=None, n_modes=k,
                             hierarchy=[300, 900], k_neighbors=8, prolongation_neighbors=8, hidden_layers=[128, 128],
                             epochs=300, log_every=100, sampler_type="farthest_point", mlp_mode=mlp_mode,
                             cgc_mode="regularized", seed=0, fps_start=5, operator_type="auto", dropout=0.1)
    U = main_mod.main(cfg_file)
    assert U.shape == (fem["verts"].shape[0], k) and np.isfinite(U).all()
    rep = main_mod.main.last_report
    assert np.isfinite(rep["rel_errors"]).all()


def test_eval_mode_inference_is_deterministic_with_dropout_in_the_module():
    cm = dropin("corrector_model")
    torch.manual_seed(0)
    model = cm.SimpleCorrector(20, 8, [64, 64], 0.1).to(dev())
    model.eval()
    x = torch.randn(300, 40, device=dev())
    with torch.no_grad():
        a, b = cm._run_net(model.net, x, model.training), cm._run_net(model.net, x, model.training)
    assert torch.equal(a, b)


def test_sharded_engine_refuses_dropout():
    dist, eng = pkg("dist_engine"), pkg("engine")
    with pytest.raises(NotImplementedError, match="dropout"):
        dist._refuse_dropout(eng.StepConfig(dropout=0.1).dropout)
    dist._refuse_dropout(0.0)
