"""fp64 operators of the notebook variants, host side: CsrMatrix / OperatorPair keep scipy's fp64 values bit for bit
(duplicates merged in fp64, union-pattern padding in fp64), report their dtype, leave fp32 construction unchanged, and
the fp64 wrappers refuse mixed dtypes, CPU tensors and k > 128 before any kernel runs."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from gpu_util import pkg, bunny_levels


def _canonical_f64(A):
    B = sp.csr_matrix(A, dtype=np.float64)
    B.sum_duplicates()
    B.sort_indices()
    return B


def _with_duplicates(seed=0, n=40):
    """COO with repeated (row, col) entries whose fp32 and fp64 sums differ."""
    rng = np.random.default_rng(seed)
    rows = rng.integers(0, n, 400)
    cols = rng.integers(0, n, 400)
    vals = rng.standard_normal(400) * (1 + 1e-9 * rng.standard_normal(400))
    return sp.coo_matrix((vals, (rows, cols)), shape=(n, n))


def _host_equal(t, ref):
    return np.array_equal(t.cpu().numpy(), ref) and t.cpu().numpy().dtype == ref.dtype


def test_fp64_csr_keeps_scipy_values_bit_for_bit():
    sparse = pkg("sparse")
    A = _with_duplicates()
    C = sparse.CsrMatrix.from_scipy(A, "cpu", dtype=torch.float64)
    ref = _canonical_f64(A)
    assert C.dtype == torch.float64 and C.val.dtype == torch.float64
    assert _host_equal(C.rowptr, ref.indptr.astype(np.int32)) and _host_equal(C.col, ref.indices.astype(np.int32))
    assert np.array_equal(C.val.numpy().view(np.int64), ref.data.view(np.int64))
    # the fp32 rounding-then-merging of the reference would give other values here
    assert not np.array_equal(C.val.numpy(), sparse._to_csr_f32(A).data.astype(np.float64))
    T = sparse.CsrMatrix.from_scipy(sp.random(30, 20, 0.2, random_state=1), "cpu", dtype=torch.float64).transpose()
    assert T.dtype == torch.float64 and T.val.dtype == torch.float64 and T.shape == (20, 30)


def test_fp32_construction_unchanged():
    sparse = pkg("sparse")
    A = _with_duplicates(1)
    C = sparse.CsrMatrix.from_scipy(A, "cpu")
    ref = sparse._to_csr_f32(A)
    assert C.dtype == torch.float32 and C.val.dtype == torch.float32
    assert np.array_equal(C.val.numpy(), ref.data) and np.array_equal(C.col.numpy(), ref.indices)
    P = sparse.OperatorPair(A, A * 2.0, "cpu")
    assert P.dtype == torch.float32 and P.K.val.dtype == torch.float32
    with pytest.raises(TypeError):
        sparse.CsrMatrix.from_scipy(A, "cpu", dtype=torch.float16)


def test_fp64_pair_unify_pads_in_fp64():
    sparse = pkg("sparse")
    rng = np.random.default_rng(2)
    n = 50
    K = sp.random(n, n, 0.1, random_state=3, data_rvs=lambda m: rng.standard_normal(m) * np.pi).tocsr()
    M = sp.random(n, n, 0.1, random_state=4, data_rvs=lambda m: rng.standard_normal(m) / 3.0).tocsr()
    P = sparse.OperatorPair(K, M, "cpu", dtype=torch.float64)
    assert P.dtype == torch.float64 and P.K.dtype == P.M.dtype == torch.float64
    assert torch.equal(P.K.rowptr, P.M.rowptr) and torch.equal(P.K.col, P.M.col)
    rowptr, col = P.K.rowptr.numpy(), P.K.col.numpy()
    for A, got in ((K, P.K.val.numpy()), (M, P.M.val.numpy())):
        back = sp.csr_matrix((got, col, rowptr), shape=(n, n))
        ref = _canonical_f64(A)
        assert np.array_equal(back.toarray().view(np.int64), ref.toarray().view(np.int64))
    assert P.KT.dtype == P.MT.dtype == torch.float64 and P.KT.val.dtype == torch.float64


def test_bunny_operators_are_symmetric_in_fp64():
    sparse, v = pkg("sparse"), pkg("variants")
    _, (K, M), (Kc, Mc) = bunny_levels()
    for A, B in ((K, M), (Kc, Mc), v.frobenius_normalised(K, M)[:2], v.frobenius_normalised(Kc, Mc)[:2]):
        P = sparse.OperatorPair(A, B, "cpu", dtype=torch.float64)
        assert P.symmetric and P.KT is P.K and P.MT is P.M


def test_mixed_dtypes_cpu_tensors_and_large_k_are_refused():
    sparse, ops, cabi = pkg("sparse"), pkg("ops"), pkg("_cabi")
    _, _, (Kc, Mc) = bunny_levels()
    n = Kc.shape[0]
    p64 = sparse.OperatorPair(Kc, Mc, "cpu", dtype=torch.float64)
    p32 = sparse.OperatorPair(Kc, Mc, "cpu")
    U64, U32 = torch.zeros(n, 4, dtype=torch.float64), torch.zeros(n, 4)
    for pair, U in ((p32, U64), (p64, U32)):
        with pytest.raises(TypeError, match="float"):
            ops.spmm2(pair, U)
        with pytest.raises(TypeError):
            ops.spmm(pair.K, U)
        with pytest.raises(TypeError):
            ops.spmm2_sum(pair.KT, pair.MT, U, U)
    with pytest.raises(cabi.EpError):           # same dtype, but on the CPU: no fallback
        ops.spmm2(p64, U64)
    with pytest.raises(cabi.EpError):
        ops.linear_fwd(U64, torch.zeros(3, 4, dtype=torch.float64), None, False)
    fake = ctypes.c_void_p(256)
    with pytest.raises(cabi.EpError, match="k > 128"):
        cabi.call("ep_eigen_partials_f64", 10, 129, fake, 129, fake, fake, 129, fake, fake, 1 << 20, None)


def test_library_version_and_fp64_entries():
    cabi = pkg("_cabi")
    assert cabi.query("ep_version") == 400
    for name in ("ep_spmm_csr_f64", "ep_spmm2_csr_f64", "ep_spmm2_sum_csr_f64", "ep_eigen_partials_f64",
                 "ep_linear_fwd_f64", "ep_linear_bwd_f64"):
        assert name in cabi.SIGNATURES and name in cabi.KERNELS_PER_CALL
    b32 = cabi.query("ep_linear_bwd_workspace_bytes", 1000, 64, 32)
    b64 = cabi.query("ep_linear_bwd_workspace_bytes_f64", 1000, 64, 32)
    assert b32 > 0 and b64 == 2 * b32
