"""Device-resident CSR operators (fp32 values, or fp64 for the notebook variants; int32 indices).

The reference converts every scipy matrix to a torch COO tensor on EVERY epoch
(reference src/utils.py:14-20, called from src/multigrid_model.py:306-307); here the
conversion happens once and the CSR arrays stay in HBM.
"""
import numpy as np
import scipy.sparse as sp
import torch


def _to_csr_f32(A):
    """scipy -> canonical CSR with fp32 values (cast first, then merge duplicates, like
    `torch.FloatTensor(A.data)` followed by `.coalesce()` in the reference)."""
    A = A.tocoo()
    B = sp.coo_matrix((A.data.astype(np.float32), (A.row, A.col)), shape=A.shape).tocsr()
    B.sum_duplicates()
    B.sort_indices()
    return B


def _to_csr_f64(A):
    """scipy -> canonical CSR with fp64 values: duplicates are merged in fp64, values stay scipy's bit for bit."""
    A = A.tocoo()
    B = sp.coo_matrix((A.data.astype(np.float64), (A.row, A.col)), shape=A.shape).tocsr()
    B.sum_duplicates()
    B.sort_indices()
    return B


_NP_DTYPE = {torch.float32: np.float32, torch.float64: np.float64}


def _np_dtype(dtype):
    if dtype not in _NP_DTYPE:
        raise TypeError("CSR values are torch.float32 or torch.float64, not %s" % dtype)
    return _NP_DTYPE[dtype]


class CsrMatrix:
    """CSR matrix on one CUDA device; `dtype` is the type of its values (torch.float32 or torch.float64)."""

    def __init__(self, host_csr, device, dtype=torch.float32):
        if host_csr.nnz >= 2 ** 31 or max(host_csr.shape) >= 2 ** 31:
            raise ValueError("CsrMatrix uses int32 indices")
        self.shape = tuple(host_csr.shape)
        self.nnz = int(host_csr.nnz)
        self.device = torch.device(device)
        self.dtype = dtype
        self._host = host_csr
        self.rowptr = torch.from_numpy(host_csr.indptr.astype(np.int32)).to(self.device)
        self.col = torch.from_numpy(host_csr.indices.astype(np.int32)).to(self.device)
        self.val = torch.from_numpy(host_csr.data.astype(_np_dtype(dtype))).to(self.device)
        self._T = None
        self._symmetric = None

    @classmethod
    def from_scipy(cls, A, device, dtype=torch.float32):
        """fp32 rounds the values first and then merges duplicates, as the reference's torch.FloatTensor + coalesce
        does; fp64 keeps scipy's values."""
        if dtype == torch.float64:
            return cls(_to_csr_f64(A), device, dtype)
        _np_dtype(dtype)
        return cls(_to_csr_f32(A), device)

    @classmethod
    def from_device_arrays(cls, rowptr, col, val, shape, symmetric=None):
        """Wrap CSR arrays that already live on the GPU (e.g. from fem_device.assemble)."""
        obj = cls.__new__(cls)
        obj.shape, obj.nnz, obj.device = tuple(shape), int(col.numel()), rowptr.device
        obj.dtype = val.dtype if val is not None else torch.float32
        obj._host, obj.rowptr, obj.col, obj.val = None, rowptr, col, val
        obj._T, obj._symmetric = None, symmetric
        return obj

    @classmethod
    def from_torch_sparse(cls, A, device):
        A = A.coalesce().cpu()
        idx = A.indices().numpy()
        return cls.from_scipy(sp.coo_matrix((A.values().numpy(), (idx[0], idx[1])), shape=tuple(A.shape)), device)

    @classmethod
    def from_edge_index(cls, edge_index, n, device):
        """Adjacency pattern for the neighbour-mean aggregation: row = destination, columns in
        the ORIGINAL edge order (stable sort), duplicates kept - reference
        src/corrector_model.py:24-27 sums with index_add_ in edge order."""
        ei = edge_index.detach().cpu().numpy() if torch.is_tensor(edge_index) else np.asarray(edge_index)
        row, col = ei[0].astype(np.int64), ei[1].astype(np.int64)
        order = np.argsort(row, kind="stable")
        counts = np.bincount(row, minlength=n)
        obj = cls.__new__(cls)
        obj.shape = (n, n)
        obj.nnz = int(row.size)
        obj.device = torch.device(device)
        obj.dtype = torch.float32
        obj._host = None
        rowptr = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(counts, out=rowptr[1:])
        obj.rowptr = torch.from_numpy(rowptr.astype(np.int32)).to(obj.device)
        obj.col = torch.from_numpy(col[order].astype(np.int32)).to(obj.device)
        obj.val = None
        obj._T, obj._symmetric = None, None
        return obj

    def _need_host(self, what):
        if self._host is None:
            raise ValueError("CsrMatrix.%s needs the host copy, which device-built matrices (from_device_arrays / "
                             "from_edge_index) do not keep: pass symmetric=True/False to from_device_arrays" % what)
        return self._host

    @property
    def symmetric(self):
        if self._symmetric is None:
            A = self._need_host("symmetric")
            if A.shape[0] != A.shape[1]:
                self._symmetric = False
            else:
                T = A.T.tocsr()
                T.sort_indices()
                self._symmetric = (np.array_equal(T.indptr, A.indptr) and np.array_equal(T.indices, A.indices)
                                   and np.array_equal(T.data, A.data))
        return self._symmetric

    def transpose(self):
        if self.symmetric:
            return self
        if self._T is None:
            T = self._need_host("transpose()").T.tocsr()
            T.sort_indices()
            self._T = CsrMatrix(T, self.device, self.dtype)
        return self._T


class OperatorPair:
    """Stiffness K and mass M of one resolution level.  When both share one sparsity pattern
    (always true for the FEM operators of src/Mesh.py) the dual kernel reads each gathered
    row of U once for both products."""

    def __init__(self, K, M, device, assume_symmetric=None, dtype=torch.float32):
        """assume_symmetric=True: the GLOBAL operators are symmetric although these (possibly rectangular,
        rank-local [owned | halo] column space) blocks cannot be checked - skips the transposes.
        dtype: value type of operators given as scipy matrices (torch.float64 for the notebook variants); operators
        given as CsrMatrix keep their own, which must agree."""
        self.K = K if isinstance(K, CsrMatrix) else CsrMatrix.from_scipy(K, device, dtype)
        self.M = M if isinstance(M, CsrMatrix) else CsrMatrix.from_scipy(M, device, dtype)
        assert self.K.shape == self.M.shape
        if self.K.dtype != self.M.dtype:
            raise TypeError("K is %s but M is %s" % (self.K.dtype, self.M.dtype))
        self.dtype = self.K.dtype
        self.n = self.K.shape[0]
        self.shared = (self.K.rowptr is self.M.rowptr and self.K.col is self.M.col) or (
            self.K.nnz == self.M.nnz and torch.equal(self.K.rowptr, self.M.rowptr) and torch.equal(self.K.col, self.M.col))
        if not self.shared:
            self._unify()
        self.symmetric = bool(assume_symmetric) if assume_symmetric is not None else (self.K.symmetric and self.M.symmetric)
        if self.symmetric:
            self.KT, self.MT = self.K, self.M
        else:
            KT, MT = self.K._need_host("transpose()").T.tocsr(), self.M._need_host("transpose()").T.tocsr()
            self.KT, self.MT = CsrMatrix(_sorted(KT), device, self.dtype), CsrMatrix(_sorted(MT), device, self.dtype)

    def _unify(self):
        """Pad both operators to the union pattern (explicit zeros) so one rowptr/col serves both."""
        K, M = self.K._host.tocoo(), self.M._host.tocoo()
        rows = np.concatenate([K.row, M.row])
        cols = np.concatenate([K.col, M.col])
        zK, zM = np.zeros(K.nnz, K.data.dtype), np.zeros(M.nnz, M.data.dtype)
        Ku = sp.coo_matrix((np.concatenate([K.data, zM]), (rows, cols)), shape=K.shape).tocsr()
        Mu = sp.coo_matrix((np.concatenate([zK, M.data]), (rows, cols)), shape=K.shape).tocsr()
        dev = self.K.device
        self.K, self.M = CsrMatrix(_sorted(Ku), dev, self.dtype), CsrMatrix(_sorted(Mu), dev, self.dtype)
        assert np.array_equal(Ku.indices, Mu.indices) and np.array_equal(Ku.indptr, Mu.indptr)
        self.shared = True


def _sorted(A):
    A.sort_indices()
    return A
