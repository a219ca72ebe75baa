"""Learnable per-mode scales (AdaptiveCorrector) and the smoothness of the correction in the fused training step:
ep_mode_scale_fwd_f32 / ep_mode_scale_bwd_f32 against fp64 torch, the loss level against fp64 autograd, six training
epochs against the fp64 restatement of the notebook step (oracle/adaptive_port.py), graph replay, and that the plain
step is unchanged when neither option is on."""
import ctypes
import os
import types

import numpy as np
import pytest
import torch

from conftest import load_golden
from gpu_util import pkg, dev, dropin, bunny_levels, SRC

pytestmark = pytest.mark.gpu

W_SMOOTH, W_SMOOTH_CORR = 10.0, 2000.0


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _block(n, k, layout, fill=None, g=None):
    """An n x k view inside a NaN-filled buffer with one guard row above and below.
    dense: ld = k; pad: ld = k + 4, 16-byte aligned rows; offset: ld = k + 6, rows start 8 bytes into the line."""
    ld, c0 = {"dense": (k, 0), "pad": (k + 4, 4), "offset": (k + 6, 2)}[layout]
    buf = torch.full((n + 2, ld), float("nan"), device=dev())
    view = buf[1:1 + n, c0:c0 + k]
    if fill is not None:
        view.copy_(fill)
    elif g is not None:
        view.copy_(torch.randn(n, k, generator=g).to(dev()))
    return buf, view


def _guards_intact(buf, n, k, layout):
    _, c0 = {"dense": (k, 0), "pad": (k + 4, 4), "offset": (k + 6, 2)}[layout]
    inner = torch.zeros_like(buf, dtype=torch.bool)
    inner[1:1 + n, c0:c0 + k] = True
    return bool(torch.isnan(buf[~inner]).all())


def _run_bwd(n, k, n_global, c, Kc, s, w, dcorr, grad_s, acc, loss):
    cabi = pkg("_cabi")
    ws = pkg("ops").mode_scale_workspace(k, dev())
    cabi.call("ep_mode_scale_bwd_f32", n, k, float(n_global), _p(c), c.stride(0), _p(Kc), Kc.stride(0) if Kc is not None else k,
              _p(s), float(w), _p(dcorr), dcorr.stride(0), _p(grad_s), acc, _p(loss), _p(ws), ws.numel(), _stream())


@pytest.mark.parametrize("k", [1, 3, 16, 32, 50, 64, 128])
@pytest.mark.parametrize("n", [0, 1, 127, 129, 4097, 40001])
def test_kernels_match_fp64(n, k):
    cabi, ops = pkg("_cabi"), pkg("ops")
    g = torch.Generator().manual_seed(1000 * k + n % 997)
    sigma, w, n_global = 3.75, 0.75, n + 7              # exact in fp32: the kernels take float arguments
    s_dev = (0.5 + torch.rand(k, generator=g)).to(dev())
    for layout in ("dense", "pad", "offset"):
        _, c = _block(n, k, layout, g=g)
        _, U_base = _block(n, k, layout, g=g)
        _, Kc_t = _block(n, k, layout, g=g)
        for s in (s_dev, None):
            sd = s.double() if s is not None else torch.ones(k, dtype=torch.float64, device=dev())
            # ---- forward
            outs = []
            for _ in range(2):
                obuf, out = _block(n, k, layout)
                cabi.call("ep_mode_scale_fwd_f32", n, k, _p(c), c.stride(0), _p(U_base), U_base.stride(0), _p(s),
                          sigma, None, _p(out), out.stride(0), _stream())
                assert _guards_intact(obuf, n, k, layout)
                outs.append(out.clone())
            assert torch.equal(outs[0], outs[1])
            cs = c.double() * sd
            ref = U_base.double() + sigma * cs
            bound = 3e-7 * (U_base.double().abs() + sigma * cs.abs()) + 1e-30
            assert bool(((outs[0].double() - ref).abs() <= bound).all())
            if s is None and layout == "dense":                     # unit scales: bit-identical to ep_axpy_out_f32
                assert torch.equal(outs[0], ops.axpy_out(U_base.contiguous(), c.contiguous(), sigma))
            sig_dev = torch.tensor([sigma], device=dev())
            _, out_d = _block(n, k, layout)
            cabi.call("ep_mode_scale_fwd_f32", n, k, _p(c), c.stride(0), _p(U_base), U_base.stride(0), _p(s),
                      -99.0, _p(sig_dev), _p(out_d), out_d.stride(0), _stream())
            assert torch.equal(out_d, outs[0])                        # the device scalar overrides the argument
            # ---- backward
            for Kc in (Kc_t, None):
                for acc in (0, 1):
                    gbuf0, g0 = _block(n, k, layout, g=g)
                    gs0 = torch.randn(k, generator=g).to(dev())
                    loss0 = torch.randn(9, generator=g, dtype=torch.float64).to(dev())
                    runs = []
                    for _ in range(2):
                        gbuf = gbuf0.clone()
                        dcorr = gbuf.as_strided(g0.shape, g0.stride(), g0.storage_offset())
                        grad_s = gs0.clone() if s is not None else None
                        loss = loss0.clone()
                        _run_bwd(n, k, n_global, c, Kc, s, w, dcorr, grad_s, acc, loss)
                        assert _guards_intact(gbuf, n, k, layout)
                        runs.append((dcorr.clone(), grad_s, loss))
                    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][2], runs[1][2])
                    if s is not None:
                        assert torch.equal(runs[0][1], runs[1][1])
                    dcorr, grad_s, loss = runs[0]
                    gd, cd = g0.double(), c.double()
                    w2 = 2.0 * w / (n_global * k)
                    kd = Kc.double() if Kc is not None else torch.zeros_like(cd)
                    wk = w2 if Kc is not None else 0.0
                    dc_ref = sd * gd + wk * sd * sd * kd
                    bound = 4e-7 * ((sd * gd).abs() + wk * sd * sd * kd.abs()) + 1e-30
                    assert bool(((dcorr.double() - dc_ref).abs() <= bound).all())
                    P = (cd * kd).sum(0)
                    if s is not None:
                        ds_ref = (cd * gd).sum(0) + wk * sd * P
                        base = gs0.double() if acc else torch.zeros_like(ds_ref)
                        scale = (cd * gd).abs().sum(0) + wk * sd * (cd * kd).abs().sum(0) + base.abs()
                        assert bool(((grad_s.double() - (base + ds_ref)).abs() <= 2e-7 * scale + 1e-30).all())
                    L = (w / (n_global * k)) * float((sd * sd * P).sum()) if Kc is not None else 0.0
                    Lb = (w / (n_global * k)) * float((sd * sd * (cd * kd).abs().sum(0)).sum()) * 1e-9 + 1e-300
                    l0 = loss0.cpu().numpy()
                    got = loss.cpu().numpy()
                    assert abs((got[8] - l0[8]) - L) <= Lb + 1e-12 * abs(l0[8])
                    assert abs((got[5] - l0[5]) - L) <= Lb + 1e-12 * abs(l0[5])
                    others = [0, 1, 2, 3, 4, 6, 7]
                    assert np.array_equal(got[others], l0[others])


def test_kernel_argument_errors():
    cabi, ops = pkg("_cabi"), pkg("ops")
    c = torch.zeros(8, 4, device=dev())
    ws = ops.mode_scale_workspace(4, dev())
    with pytest.raises(cabi.EpError):              # grad_s without scales
        cabi.call("ep_mode_scale_bwd_f32", 8, 4, 8.0, _p(c), 4, None, 4, None, 0.0, _p(c), 4, _p(c), 0, None, _p(ws),
                  ws.numel(), _stream())
    with pytest.raises(cabi.EpError):              # workspace too small
        cabi.call("ep_mode_scale_bwd_f32", 8, 4, 8.0, _p(c), 4, None, 4, None, 0.0, _p(c), 4, None, 0, None, _p(ws), 8,
                  _stream())
    with pytest.raises(cabi.EpError):              # k beyond the supported range
        cabi.call("ep_mode_scale_fwd_f32", 1, 300, _p(c), 300, _p(c), 300, None, 1.0, None, _p(c), 300, _stream())


@pytest.mark.parametrize("fused", [True, False])
def test_loss_level_against_autograd(fused):
    """Mode scales, both smoothness parts, the projection term, fused and unfused eigen-loss backward, on the coarse +
    bunny pair: loss slots 5 and 8, dL/dc and dL/ds against fp64 autograd.  For the unfused (general) backward the same
    matrices, declared non-symmetric, replace the pairs after construction: the constructor refuses w_smooth_corr on a
    non-symmetric pair, and since these matrices are symmetric the gradient it protects still holds."""
    import scipy.sparse as sp
    from sklearn.neighbors import NearestNeighbors
    sparse, engine = pkg("sparse"), pkg("engine")
    fem, (K, M), (Kc, Mc) = bunny_levels()
    n, nc, k = K.shape[0], Kc.shape[0], 16
    g = torch.Generator().manual_seed(5)
    U_base = 0.05 * torch.randn(nc + n, k, generator=g)
    c = 0.03 * torch.randn(nc + n, k, generator=g)
    s = 0.5 + torch.rand(k, generator=g)
    sigma = 0.7
    dist_, idx = NearestNeighbors(n_neighbors=6).fit(fem["coarse_verts"]).kneighbors(fem["verts"])
    wts = 1.0 / (dist_ + 1e-12)
    wts /= wts.sum(1, keepdims=True)
    P = sp.coo_matrix((wts.ravel(), (np.repeat(np.arange(n), 6), idx.ravel())), shape=(n, nc)).tocsr()
    U_c = 0.05 * torch.randn(nc, k, generator=g)
    w_res, w_orth, w_smooth, w_sc, w_proj = 1000.0, 10.0, 3.0, 500.0, 11.0
    # ---- reference: fp64 autograd
    cd = c.double().requires_grad_(True)
    sd = s.double().requires_grad_(True)
    corr = cd * sd
    Ud = U_base.double() + sigma * corr
    total = torch.zeros((), dtype=torch.float64)
    smooth = 0.0
    for (Kl, Ml, off) in ((Kc, Mc, 0), (K, M, nc)):
        nl = Kl.shape[0]
        Kt = torch.from_numpy(Kl.astype(np.float32).toarray().astype(np.float64))
        Mt = torch.from_numpy(Ml.astype(np.float32).toarray().astype(np.float64))
        Ul, cl = Ud[off:off + nl], corr[off:off + nl]
        Lu, Mu = Kt @ Ul, Mt @ Ul
        lam = (Ul * Lu).sum(0) / ((Ul * Mu).sum(0) + 1e-12)
        l_res = ((Lu - Mu * lam) ** 2).mean()
        l_orth = ((Ul.t() @ Mu - torch.eye(k, dtype=torch.float64)) ** 2).sum() / k
        l_smooth = (Ul * Lu).sum() / (nl * k)
        l_sc = (cl * (Kt @ cl)).sum() / (nl * k)
        total = total + w_res * l_res + w_orth * l_orth + w_smooth * l_smooth + w_sc * l_sc
        smooth += w_smooth * float(l_smooth) + w_sc * float(l_sc)
    Pt = torch.from_numpy(P.toarray())
    total = total + w_proj * ((Pt.t() @ Ud[nc:] - U_c.double()) ** 2).sum() / (nc * k)
    total.backward()
    # ---- engine
    h = torch.zeros(nc + n, 4, device=dev())
    params = engine.FlatParams([torch.zeros(8, 4), torch.zeros(k, 8)], [torch.zeros(8), torch.zeros(k)], dev(),
                               mode_scales=s)
    cfg = engine.StepConfig(w_res=w_res, w_orth=w_orth, w_smooth=w_smooth, w_smooth_corr=w_sc)
    eng = engine.TrainStepEngine(h, U_base.to(dev()), [sparse.OperatorPair(Kc, Mc, dev()), sparse.OperatorPair(K, M, dev())],
                                 [0, nc], params, cfg)
    assert eng.adaptive and eng.Kc is not None
    if not fused:
        eng.pairs = [sparse.OperatorPair(a, b, dev(), assume_symmetric=False) for a, b in ((Kc, Mc), (K, M))]
    eng.add_projection_term(1, P, U_c, w_proj)
    eng.corr_raw.copy_(c.to(dev()))
    eng.mode_scale_forward(sigma)
    eng.loss_forward()
    eng.loss_backward(sigma)
    acc = eng.loss_acc.cpu().numpy()
    assert acc[5] == pytest.approx(float(total), rel=2e-5)
    assert acc[8] == pytest.approx(smooth, rel=2e-5)
    dc_ref, ds_ref = cd.grad.numpy(), sd.grad.numpy()
    err = np.abs(eng.dCorr.cpu().numpy() - dc_ref).max()
    assert err <= 3e-5 * np.abs(dc_ref).max(), err
    err_s = np.abs(params.d_mode_scales.cpu().numpy() - ds_ref).max()
    assert err_s <= 3e-5 * np.abs(ds_ref).max(), err_s


def _adaptive_gnn(mlp_mode, w_smooth=W_SMOOTH, w_smooth_corr=W_SMOOTH_CORR, scales=None):
    """MultigridGNN with model_type 'adaptive' on the golden bunny trainer: the simple-model initial weights, per-mode
    scales spread over [0.5, 1.5] so that every mode sees a different one."""
    mg, cfgm = dropin("multigrid_model"), dropin("config")
    g = load_golden("corrector_train.npz")
    fem, (K, M), (Kc, Mc) = bunny_levels()
    cfg = cfgm.PINNConfig.from_yaml(os.path.join(SRC, "parameters.yml"))
    cfg.n_modes, cfg.hidden_layers, cfg.model_type, cfg.mlp_mode = 16, [int(h) for h in g["hidden"]], "adaptive", mlp_mode
    cfg.weight_smooth, cfg.weight_smooth_corr = w_smooth, w_smooth_corr
    gnn = mg.MultigridGNN(cfg)
    x = torch.from_numpy(g["simple_x_feats"]).to(dev())
    ei = torch.from_numpy(g["edge_index_all"])
    gnn._initialize_model(x.shape[1], 16, gnn.hidden_layers, 0.0)
    state = {k_[12:]: torch.from_numpy(g[k_]) for k_ in g.files if k_.startswith("simple_init_")}
    state["mode_scales"] = torch.linspace(0.5, 1.5, 16) if scales is None else scales
    gnn.model.load_state_dict(state)
    opt, _ = gnn._create_optimizer(gnn.lr, gnn.weight_decay)
    U_all = torch.cat([torch.from_numpy(g["U_norm_0"]), torch.from_numpy(g["U_norm_1"])])
    offs = [0, g["U_norm_0"].shape[0]]
    eng = gnn._make_engine(x, ei, None, U_all, [Kc, K], [Mc, M], torch.from_numpy(g["lam_0"]), offs, opt)
    return types.SimpleNamespace(gnn=gnn, eng=eng, opt=opt, g=g, x=x, ei=ei, U_all=U_all, K=K, M=M, Kc=Kc, Mc=Mc,
                                 state=state)


def _oracle(t, w_smooth=W_SMOOTH, w_smooth_corr=W_SMOOTH_CORR):
    from oracle import adaptive_port
    names = sorted({k_.rsplit(".", 1)[0] for k_ in t.state if k_.startswith("net.")}, key=lambda s: int(s.split(".")[1]))
    gnn = t.gnn
    return adaptive_port.AdaptiveTrainer(
        t.g["simple_x_feats"], t.g["edge_index_all"], t.U_all, [t.Kc, t.K], [t.Mc, t.M], t.g["lam_0"],
        [t.state[n_ + ".weight"] for n_ in names], [t.state[n_ + ".bias"] for n_ in names], t.state["mode_scales"],
        lr=gnn.lr, weight_decay=gnn.weight_decay, corr_scale=gnn.corr_scale, w_res=gnn.w_res, w_orth=gnn.w_orth,
        w_trace=gnn.w_trace, w_order=gnn.w_order, w_eigen=gnn.w_eigen, w_smooth=w_smooth, w_smooth_corr=w_smooth_corr,
        grad_clip=gnn.grad_clip)


def test_six_adaptive_epochs_follow_the_fp64_notebook_step():
    t = _adaptive_gnn("fp32")
    ref = _oracle(t)
    hist, want = [], []
    for epoch in range(2500, 2506):
        acc = t.eng.step(epoch, lr=t.opt.param_groups[0]["lr"]).cpu().numpy()
        hist.append([acc[5], acc[0], acc[1], acc[8]])
        want.append(ref.step(epoch))
    np.testing.assert_allclose(np.array(hist), np.array(want), rtol=2e-4)
    sd = t.gnn.model.state_dict()                    # module parameters are views of the flat buffer
    ref_lin = [m for m in ref.model.net if isinstance(m, torch.nn.Linear)]
    names = sorted({k_.rsplit(".", 1)[0] for k_ in sd if k_.startswith("net.")}, key=lambda s: int(s.split(".")[1]))
    for name, lin in zip(names, ref_lin):
        np.testing.assert_allclose(sd[name + ".weight"].cpu().numpy(), lin.weight.detach().numpy(), rtol=0, atol=3e-5)
    np.testing.assert_allclose(sd["mode_scales"].cpu().numpy(), ref.model.mode_scales.detach().numpy(), rtol=1e-4)
    assert not np.allclose(sd["mode_scales"].cpu().numpy(), t.state["mode_scales"].numpy(), rtol=1e-6, atol=0)
    # the drop-in's final predictions (AdaptiveCorrector.forward, corr_scale) and the engine's U_pred at that scale
    U_norm = [torch.from_numpy(t.g["U_norm_0"]), torch.from_numpy(t.g["U_norm_1"])]
    U_final = t.gnn._generate_final_predictions(t.x, t.ei, None, t.U_all, U_norm, [t.Mc, t.M])
    t.eng.forward(t.gnn.corr_scale)
    ops, utils = pkg("ops"), dropin("utils")
    nc = U_norm[0].shape[0]
    U_eng = torch.cat([ops.m_normalize_columns(t.eng.U_pred[:nc], utils.device_operator(t.Mc, dev())),
                       ops.m_normalize_columns(t.eng.U_pred[nc:], utils.device_operator(t.M, dev()))]).cpu().numpy()
    np.testing.assert_allclose(U_final, U_eng, rtol=0, atol=1e-6)


def test_bf16_step_within_stated_tolerance():
    t = _adaptive_gnn("bf16")
    ref = _oracle(t)
    acc = t.eng.step(2500, lr=t.opt.param_groups[0]["lr"]).cpu().numpy()
    want = ref.step(2500)
    assert acc[5] == pytest.approx(want[0], rel=5e-3)
    for got, w in zip((acc[0], acc[1], acc[8]), want[1:]):
        assert got == pytest.approx(w, rel=2.5e-2)


@pytest.mark.parametrize("mlp_mode", ["fp32", "bf16"])
def test_cuda_graph_replay_equals_eager(mlp_mode):
    runs = []
    for graphed in (False, True):
        t = _adaptive_gnn(mlp_mode)
        eng = t.eng
        hist = [eng.step(2500).cpu().numpy().copy()]
        if graphed:
            eng.enable_graph()
        for e in range(2501, 2512):
            lr = 1e-3 if e < 2506 else 5e-4
            hist.append(eng.step(e, lr=lr).cpu().numpy().copy())
        if graphed:
            launches = eng.launches_by_entry
            assert launches["ep_mode_scale_fwd_f32"] == 1 and launches["ep_mode_scale_bwd_f32"] == 2 * 2
        runs.append((np.array(hist), eng.params.flat.clone(), eng.params.m.clone(), eng.params.v.clone()))
    assert np.array_equal(runs[0][0], runs[1][0]), np.abs(runs[0][0] - runs[1][0]).max()
    for a, b in zip(runs[0][1:], runs[1][1:]):
        assert torch.equal(a, b), (a - b).abs().max().item()


def test_off_means_off():
    """Neither option: the captured step launches exactly what a plain engine launches, and no new entry point."""
    engine, sparse = pkg("engine"), pkg("sparse")
    mg, cfgm = dropin("multigrid_model"), dropin("config")
    g = load_golden("corrector_train.npz")
    fem, (K, M), (Kc, Mc) = bunny_levels()
    cfg = cfgm.PINNConfig.from_yaml(os.path.join(SRC, "parameters.yml"))
    cfg.n_modes, cfg.hidden_layers, cfg.model_type = 16, [int(h) for h in g["hidden"]], "simple"
    cfg.weight_smooth_corr = 0.0
    gnn = mg.MultigridGNN(cfg)
    x = torch.from_numpy(g["simple_x_feats"]).to(dev())
    ei = torch.from_numpy(g["edge_index_all"])
    gnn._initialize_model(x.shape[1], 16, gnn.hidden_layers, 0.0)
    opt, _ = gnn._create_optimizer(gnn.lr, gnn.weight_decay)
    U_all = torch.cat([torch.from_numpy(g["U_norm_0"]), torch.from_numpy(g["U_norm_1"])])
    offs = [0, g["U_norm_0"].shape[0]]
    a = gnn._make_engine(x, ei, None, U_all, [Kc, K], [Mc, M], torch.from_numpy(g["lam_0"]), offs, opt)
    lin = [m for m in gnn.model.net if isinstance(m, torch.nn.Linear)]
    params = engine.FlatParams([l.weight.detach().clone() for l in lin], [l.bias.detach().clone() for l in lin], dev())
    b = engine.TrainStepEngine(a.h, a.U_base, [sparse.OperatorPair(Kc, Mc, dev()), sparse.OperatorPair(K, M, dev())],
                               offs, params, engine.StepConfig(), lam_target=torch.from_numpy(g["lam_0"]).to(dev()))
    for eng in (a, b):
        assert not eng.adaptive and eng.Kc is None
        eng.step(2500)
        eng.enable_graph()
        eng.step(2501)
    assert a.launches_by_entry == b.launches_by_entry
    assert a.launches_per_step == b.launches_per_step
    assert not any(name.startswith("ep_mode_scale") for name in a.launches_by_entry)
    # the option on: the same step gains exactly the new launches (and K c per level)
    t = _adaptive_gnn("fp32")
    t.eng.step(2500)
    t.eng.enable_graph()
    t.eng.step(2501)
    extra = dict(t.eng.launches_by_entry)
    assert extra.pop("ep_mode_scale_fwd_f32") == 1 and extra.pop("ep_mode_scale_bwd_f32") == 4
    assert extra.pop("ep_spmm_csr_f32") - a.launches_by_entry.get("ep_spmm_csr_f32", 0) == 2
    base = dict(a.launches_by_entry)
    base.pop("ep_spmm_csr_f32", None)
    assert base.pop("ep_axpy_out_f32") == 1                      # U_pred: ep_mode_scale_fwd_f32 instead
    assert extra == base


def _sampler(k, fem, K, M, Kc, Mc):
    """What reference Sampler.preprocess_mesh leaves behind, built from the FEM operators (as in test_gpu_dropin_e2e)."""
    utils = dropin("utils")
    from scipy.sparse.linalg import eigsh
    s = types.SimpleNamespace()
    s.X_list = [fem["coarse_verts"], fem["verts"]]
    s.K_list, s.M_list = [Kc.tocoo(), K.tocoo()], [Mc.tocoo(), M.tocoo()]
    s.edge_index_list = [utils.build_knn_graph(X, k=8) for X in s.X_list]
    _, U0 = eigsh(Kc.tocsc(), k=k, M=Mc.tocsc(), sigma=-1e-6, which="LM")
    P = utils.build_prolongation(s.X_list[0], s.X_list[1], k=8)
    U1 = utils.jacobi_smooth(M, K, P @ U0, alpha=0.1, n_iters=10)
    s.P_list, s.U_list = [P], [U0, U1]
    s.actual_hierarchy = [X.shape[0] for X in s.X_list]
    return s


def test_train_multiresolution_adaptive_end_to_end():
    cfgm, mg = dropin("config"), dropin("multigrid_model")
    fem, (K, M), (Kc, Mc) = bunny_levels()
    k = 16
    cfg = cfgm.PINNConfig.from_yaml(os.path.join(SRC, "parameters.yml"))
    cfg.n_modes, cfg.hidden_layers, cfg.epochs, cfg.log_every = k, [128, 128], 200, 100
    cfg.mlp_mode, cfg.cgc_mode, cfg.seed, cfg.model_type = "fp32", "skip", 0, "adaptive"
    cfg.weight_smooth, cfg.weight_smooth_corr = 1.0, 1.0
    gnn = mg.MultigridGNN(cfg)
    U = gnn.train_multiresolution(_sampler(k, fem, K, M, Kc, Mc))
    assert U.shape == (fem["verts"].shape[0], k) and np.isfinite(U).all()
    hist = np.array(gnn.loss_history)
    assert hist.size == 200 and np.isfinite(hist).all()
    scales = gnn.model.mode_scales.detach().cpu().numpy()
    assert np.isfinite(scales).all() and np.abs(scales - 0.01).max() > 1e-4
    assert gnn.model.mode_scales.data_ptr() == gnn.engine.params.mode_scales.data_ptr()
