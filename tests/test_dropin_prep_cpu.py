"""CPU: the reference-shaped pre-processing helpers (src/utils.py here) against fixtures written by the reference's
own utils.py (oracle/make_golden_prep.py): prolongation, kNN graph, Jacobi smoothing, Gram-Schmidt, config surface."""
import os
import sys

import numpy as np
import pytest
import scipy.sparse as sp

from conftest import load_golden, csr_from_golden, ROOT

SRC = os.path.join(ROOT, "eigen-pinns_b200", "src")


@pytest.fixture(scope="module")
def mods():
    sys.path.insert(0, SRC)
    for m in ("utils", "config", "mesh_helpers", "Mesh", "samplers"):
        sys.modules.pop(m, None)
    import config
    import utils
    import Mesh
    import mesh_helpers
    yield dict(utils=utils, config=config, Mesh=Mesh, mesh_helpers=mesh_helpers)
    sys.path.remove(SRC)


def test_prolongation_knn_smoothing_match_reference(mods, monkeypatch):
    # the scikit-learn kNN path, also on a host with a GPU (the GPU kernel breaks distance ties by index and is checked
    # against the same fixtures in test_gpu_knn.py)
    import torch
    monkeypatch.setattr(torch.cuda, "is_available", lambda: False)
    utils = mods["utils"]
    g, fem = load_golden("prep_cgc.npz"), load_golden("bunny_fem.npz")
    n = fem["verts"].shape[0]
    K, M = csr_from_golden(fem, "K", n), csr_from_golden(fem, "M", n)
    P = utils.build_prolongation(fem["coarse_verts"], fem["verts"], k=8).tocsr()
    Pref = sp.coo_matrix((g["P_data"], (g["P_row"], g["P_col"])), shape=P.shape).tocsr()
    assert abs(P - Pref).max() < 1e-12
    np.testing.assert_allclose(np.asarray(P.sum(1)).ravel(), 1.0, rtol=1e-12)
    U1 = utils.jacobi_smooth(M, K, P @ g["U0"], alpha=0.1, n_iters=10)
    np.testing.assert_allclose(U1, g["U1"], rtol=1e-9, atol=1e-12)
    knn = utils.build_knn_graph(fem["coarse_verts"], k=5).numpy()
    assert knn.shape == g["knn_coarse"].shape and np.array_equal(knn[0], g["knn_coarse"][0])
    # neighbour SETS per node are pinned (order inside equal-distance ties is sklearn's)
    same = [set(knn[1, i * 5:(i + 1) * 5]) == set(g["knn_coarse"][1, i * 5:(i + 1) * 5]) for i in range(knn.shape[1] // 5)]
    assert np.mean(same) > 0.999


def test_orthonormalize_and_column_norms(mods):
    utils = mods["utils"]
    g = load_golden("prep_cgc.npz")
    Ms = sp.diags(g["ortho_M"])
    np.testing.assert_allclose(utils.orthonormalize(g["ortho_in"], Ms), g["ortho_out"], rtol=1e-10, atol=1e-12)
    ncol, nrm = utils.normalize_columns_np(g["ortho_in"])
    np.testing.assert_allclose(ncol, g["ncol"], rtol=1e-14)
    np.testing.assert_allclose(nrm, g["nrm"], rtol=1e-14)


def test_config_surface(mods, tmp_path):
    config = mods["config"]
    cfg = config.PINNConfig.from_yaml(os.path.join(SRC, "parameters.yml"))
    assert (cfg.n_modes, cfg.hierarchy, cfg.k_neighbors) == (64, [256, 512, 1024], 21)
    assert cfg.hidden_layers == [256] * 6 and cfg.model_type == "simple" and cfg.epochs == 10000
    assert cfg.normalization_eps == "1E-9"                       # PyYAML quirk Q8 kept
    bad = tmp_path / "bad.yml"
    bad.write_text(open(os.path.join(SRC, "parameters.yml")).read() + "\nextra:\n  unknown_key: 1\n")
    with pytest.raises(TypeError):
        config.PINNConfig.from_yaml(str(bad))
    missing = tmp_path / "missing.yml"
    missing.write_text("runner:\n  n_modes: 4\n")
    with pytest.raises(TypeError):
        config.PINNConfig.from_yaml(str(missing))


def test_mesh_surface(mods, tmp_path):
    Mesh, mh = mods["Mesh"], mods["mesh_helpers"]
    fem = load_golden("bunny_fem.npz")
    obj = tmp_path / "m.obj"
    with open(obj, "w") as f:
        for v in fem["coarse_verts"]:
            f.write("v %.17g %.17g %.17g\n" % tuple(v))
        for t in fem["coarse_tris"]:
            f.write("f %d/1/1 %d/2/2 %d/3/3\n" % tuple(t + 1))
    m = mh.load_mesh(str(obj), normalize=False)
    assert np.array_equal(m.connectivity, fem["coarse_tris"]) and np.allclose(m.verts, fem["coarse_verts"], rtol=0, atol=0)
    Kd, Md = m.computeLaplacian()
    np.testing.assert_allclose(np.abs(Kd).sum(1), fem["Kc_rowsum_abs"], rtol=1e-11)
    np.testing.assert_allclose(Md.sum(1), fem["Mc_rowsum"], rtol=1e-12)
    mn = mh.normalize_mesh(m)
    assert abs(mn.verts.mean(0)).max() < 1e-12 and mn.verts.std(0).max() == pytest.approx(1.0, abs=1e-9)
    ei = mh.mesh_to_edge_index(m).numpy()
    assert ei.shape[0] == 2 and np.array_equal(np.unique(ei[0] * 10000 + ei[1]), np.sort(ei[0] * 10000 + ei[1]))


def test_every_optional_config_key_is_consumed(mods):
    """Each B200-only key of config.OPTIONAL_FIELDS must be read somewhere in the drop-in modules (an advertised
    switch that nothing reads is a bug), and the shipped YAML must carry every one of them."""
    import re
    config = mods["config"]
    sources = ""
    for name in os.listdir(SRC):
        if name.endswith(".py") and name != "config.py":
            sources += open(os.path.join(SRC, name)).read()
    cfg = config.PINNConfig.from_yaml(os.path.join(SRC, "parameters.yml"))
    for key in config.OPTIONAL_FIELDS:
        assert re.search(r"\b%s\b" % key, sources), "config key %r is never read" % key
        assert hasattr(cfg, key)
    assert cfg.operator_type == "auto"


def test_galerkin_level_operators_are_consistent(mods):
    """operator_type 'fem' fallback of the point samplers: P^T K P keeps constants in its null space, P^T M P
    keeps the total mass; the finest level is the mesh's own FEM pair."""
    import types
    sys.modules.pop("samplers", None)
    import importlib
    try:
        samplers = importlib.import_module("samplers")
    except Exception as exc:                      # the sampling back end needs the CUDA library at import
        pytest.skip("samplers module needs the built library: %r" % (exc,))
    fem = load_golden("bunny_fem.npz")
    mesh = mods["Mesh"].Mesh(verts=fem["verts"], connectivity=fem["tris"])
    cfg = mods["config"].PINNConfig.from_yaml(os.path.join(SRC, "parameters.yml"))
    cfg.operator_type = "fem"
    s = samplers.Sampler(cfg)
    assert s._use_point_cloud_operators() is False
    idx = np.arange(0, fem["verts"].shape[0], 7)
    Kl, Ml = s._galerkin_operators(mesh, fem["verts"][idx])
    Kl, Ml = Kl.tocsr(), Ml.tocsr()
    n = fem["verts"].shape[0]
    M = csr_from_golden(fem, "M", n)
    assert abs(Kl @ np.ones(idx.size)).max() < 1e-9
    assert Ml.sum() == pytest.approx(M.sum(), rel=1e-12)
    assert abs(Kl - Kl.T).max() < 1e-12 and abs(Ml - Ml.T).max() < 1e-12
    Kf, Mf = s._galerkin_operators(mesh, fem["verts"])
    assert abs(Kf.tocsr() - csr_from_golden(fem, "K", n)).max() < 1e-12


def test_diagnostics_alignment_matches_reference(mods):
    """align_eigenvectors / Procrustes / Rayleigh quotients against fixtures written by the reference's own
    src/diagnostics.py (oracle/make_golden_diag.py), with sparse operators instead of the reference's dense ones."""
    sys.modules.pop("diagnostics", None)
    import diagnostics
    g, fem = load_golden("diagnostics.npz"), load_golden("bunny_fem.npz")
    n = fem["verts"].shape[0]
    K, M = csr_from_golden(fem, "K", n), csr_from_golden(fem, "M", n)
    U_al, perm, signs = diagnostics.align_eigenvectors(g["U_pred"], fem["evec10"], M)
    assert np.array_equal(perm, g["permutation"]) and np.array_equal(signs, g["signs"])
    np.testing.assert_allclose(U_al, g["U_aligned"], rtol=0, atol=1e-14)
    U_e, perm_e, signs_e = diagnostics.align_eigenvectors(g["U_pred"], fem["evec10"], None)
    assert np.array_equal(perm_e, g["permutation_euclid"]) and np.array_equal(signs_e, g["signs_euclid"])
    U_pa, err = diagnostics.get_subspace_error_and_alignment(g["U_pred"], fem["evec10"], M)
    assert err == pytest.approx(float(g["subspace_error"]), rel=1e-9)
    np.testing.assert_allclose(U_pa, g["U_procrustes"], rtol=0, atol=1e-10)
    np.testing.assert_allclose(diagnostics.compute_rayleigh_quotients(g["U_pred"], K, M), g["lam_pred"], rtol=1e-9)
    np.testing.assert_allclose(diagnostics.compute_rayleigh_quotients(fem["evec10"], K, M), g["lam_exact"], rtol=1e-8,
                               atol=1e-12)
