"""CPU-side checks of the per-mode scale support: the flat parameter layout with the AdaptiveCorrector's scales,
the StepConfig default, the workspace query, the config keys, and the vertex-sharded engine's refusal."""
import importlib
import os
import sys
import types

import pytest
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def pkg(name):
    return importlib.import_module("eigen-pinns_b200." + name)


class _Adaptive(nn.Module):
    """Same parameter layout as corrector_model.AdaptiveCorrector (net.<i>.weight|bias, mode_scales)."""

    def __init__(self, dims, k, init_scale=0.01):
        super().__init__()
        layers = []
        for a, b in zip(dims[:-1], dims[1:]):
            layers += [nn.Linear(a, b), nn.ReLU()]
        layers.append(nn.Linear(dims[-1], k))
        self.net = nn.Sequential(*layers)
        self.mode_scales = nn.Parameter(torch.linspace(0.5, 1.5, k) * init_scale)


def _linears(model):
    return [m for m in model.net if isinstance(m, nn.Linear)]


def test_flat_params_adopt_appends_the_scales():
    engine = pkg("engine")
    torch.manual_seed(0)
    model = _Adaptive([6, 16, 8], 5)
    before = {k: v.detach().clone() for k, v in model.state_dict().items()}
    plain = engine.FlatParams([l.weight for l in _linears(model)], [l.bias for l in _linears(model)], "cpu")
    fp = engine.FlatParams.adopt(_linears(model), mode_scales=model.mode_scales)
    n_net = sum(p.numel() for name, p in model.named_parameters() if name.startswith("net."))
    assert plain.mode_scales is None and plain.d_mode_scales is None and plain.flat.numel() == n_net
    assert fp.flat.numel() == n_net + 5 and fp.grad.numel() == fp.m.numel() == fp.v.numel() == n_net + 5
    # layout: [W0 | b0 | W1 | b1 | W2 | b2 | mode_scales]; the layer blocks and dims are those of the plain buffer
    assert fp.layer_range == plain.layer_range and fp.dims == plain.dims == [6, 16, 8, 5]
    assert fp.layer_range[-1][1] == n_net
    assert torch.equal(fp.flat[n_net:], before["mode_scales"])
    assert torch.equal(fp.flat[:n_net], plain.flat)
    # the module's parameters are views of the flat buffers, state_dict keys and values unchanged
    sd = model.state_dict()
    assert sorted(sd) == sorted(before) and "mode_scales" in sd
    for k in sd:
        assert torch.equal(sd[k], before[k]), k
    base = fp.flat.data_ptr()
    assert model.mode_scales.data_ptr() == base + 4 * n_net
    assert fp.mode_scales.data_ptr() == base + 4 * n_net
    assert fp.d_mode_scales.data_ptr() == fp.grad.data_ptr() + 4 * n_net
    for lin, W, b in zip(_linears(model), fp.W, fp.b):
        assert lin.weight.data_ptr() == W.data_ptr() and lin.bias.data_ptr() == b.data_ptr()
    fp.flat[n_net:] = 2.0                              # an optimiser update of the flat buffer reaches the module
    assert torch.equal(model.mode_scales.detach(), torch.full((5,), 2.0))
    fp.d_mode_scales.fill_(3.0)
    assert torch.equal(fp.grad[n_net:], torch.full((5,), 3.0))


def test_flat_params_adopt_without_scales_is_unchanged():
    engine = pkg("engine")
    torch.manual_seed(1)
    model = _Adaptive([4, 8], 3)
    a = engine.FlatParams.adopt(_linears(model))
    assert a.mode_scales is None and a.d_mode_scales is None
    assert a.flat.numel() == sum(p.numel() for n, p in model.named_parameters() if n.startswith("net."))


def test_step_config_default_leaves_the_correction_smoothness_off():
    engine = pkg("engine")
    cfg = engine.StepConfig()
    assert cfg.w_smooth_corr == 0.0 and cfg.w_smooth == 0.0
    assert engine.StepConfig(w_smooth_corr=2.5).w_smooth_corr == 2.5


def test_workspace_size_depends_on_k_only():
    cabi = pkg("_cabi")
    assert cabi.query("ep_mode_scale_bwd_workspace_bytes", 32) == 8 * 2 * 32 * 1024
    assert cabi.query("ep_mode_scale_bwd_workspace_bytes", 256) == 8 * 2 * 256 * 1024
    assert cabi.query("ep_mode_scale_bwd_workspace_bytes", 0) == 0
    assert cabi.query("ep_mode_scale_bwd_workspace_bytes", 257) == 0
    assert cabi.KERNELS_PER_CALL["ep_mode_scale_fwd_f32"] == 1 and cabi.KERNELS_PER_CALL["ep_mode_scale_bwd_f32"] == 2


def test_config_accepts_the_adaptive_keys():
    src = os.path.join(ROOT, "eigen-pinns_b200", "src")
    sys.path.insert(0, src)
    try:
        sys.modules.pop("config", None)
        import config
        cfg = config.PINNConfig.from_yaml(os.path.join(src, "parameters.yml"))
        assert (cfg.mode_scale_init, cfg.weight_smooth, cfg.weight_smooth_corr) == (0.01, 0.0, 0.0)
        fields = dict(vars(cfg), model_type="adaptive", mode_scale_init=0.1, weight_smooth=1.0, weight_smooth_corr=2.0)
        cfg2 = config.PINNConfig(**fields)
        assert (cfg2.model_type, cfg2.mode_scale_init, cfg2.weight_smooth, cfg2.weight_smooth_corr) == \
            ("adaptive", 0.1, 1.0, 2.0)
    finally:
        sys.path.remove(src)


def test_sharded_engine_refuses_mode_scales_and_correction_smoothness():
    engine, dist_engine = pkg("engine"), pkg("dist_engine")
    model = _Adaptive([4, 8], 3)
    lin = _linears(model)
    with_scales = engine.FlatParams([l.weight for l in lin], [l.bias for l in lin], "cpu", mode_scales=model.mode_scales)
    plain = engine.FlatParams([l.weight for l in lin], [l.bias for l in lin], "cpu")
    h, U = torch.zeros(10, 4), torch.zeros(10, 3)
    with pytest.raises(NotImplementedError):
        dist_engine.ShardedTrainStepEngine(h, U, [], with_scales, engine.StepConfig())
    with pytest.raises(NotImplementedError):
        dist_engine.ShardedTrainStepEngine(h, U, [], plain, engine.StepConfig(w_smooth_corr=1.0))
    gnn = types.SimpleNamespace(model=model, w_smooth_corr=0.0)
    with pytest.raises(NotImplementedError):
        dist_engine.make_sharded_engine(gnn, None, None, None, None, None, None, None, 0, 2)
    gnn = types.SimpleNamespace(model=types.SimpleNamespace(net=model.net), w_smooth_corr=1.0)
    with pytest.raises(NotImplementedError):
        dist_engine.make_sharded_engine(gnn, None, None, None, None, None, None, None, 0, 2)


def test_sharded_engine_refuses_projection_terms():
    """The sharded forward and backward have no projection term, so adding one raises instead of being ignored."""
    import scipy.sparse as sp
    dist_engine = pkg("dist_engine")
    eng = object.__new__(dist_engine.ShardedTrainStepEngine)          # the refusal needs no engine state
    with pytest.raises(NotImplementedError):
        eng.add_projection_term(0, sp.eye(4, 2, format="csr"), torch.zeros(2, 3), 1.0)
