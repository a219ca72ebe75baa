"""Tensor-level wrappers of the C ABI plus the autograd Functions the drop-in modules use.

Every function here enqueues hand-written sm_100a kernels on torch's current CUDA stream;
torch is only the allocator / stream / autograd plumbing.  CPU tensors are rejected: there is
no fallback path.

The SpMM, partials and dense-layer wrappers also take float64 tensors (the notebook variants train in double):
the dtype of the inputs selects the _f64 entry point, and operators must have the same dtype as the dense
operands (OperatorPair(..., dtype=torch.float64)).  Nothing is cast implicitly.
"""
import ctypes

import numpy as np
import torch

from . import _cabi
from ._cabi import call, query
from .sparse import CsrMatrix, OperatorPair


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _check(t, dtype=torch.float32):
    if not t.is_cuda:
        raise _cabi.EpError("eigenpinns_b200 ops need CUDA tensors (no CPU fallback exists)")
    if t.dtype != dtype:
        raise TypeError("expected %s, got %s" % (dtype, t.dtype))
    if t.dim() == 2 and t.stride(1) != 1:
        raise ValueError("matrices must be row-major (unit stride in the last dimension)")
    return t


def _rowmajor(t):
    t = t if (t.dim() != 2 or t.stride(1) == 1) else t.contiguous()
    return t


_SUFFIX = {torch.float32: "f32", torch.float64: "f64"}


def _scalar(t):
    """Entry-point suffix for a tensor of the fp32 / fp64 families."""
    if t.dtype not in _SUFFIX:
        raise TypeError("expected torch.float32 or torch.float64, got %s" % t.dtype)
    return _SUFFIX[t.dtype]


def _check_op(t, op):
    """Dense operand t of a product with CSR operator(s) op (CsrMatrix or OperatorPair): same dtype, no cast."""
    if t.dtype != op.dtype:
        raise TypeError("operator values are %s but the dense operand is %s" % (op.dtype, t.dtype))
    return _check(t, op.dtype)


# ------------------------------------------------------------------------------- SpMM
def spmm(A: CsrMatrix, X, out=None):
    """Y = A X (fp32, or fp64 for an fp64 A).  reference: torch.sparse.mm, src/multigrid_model.py:309-310."""
    X = _check_op(_rowmajor(X), A)
    k = X.shape[1]
    Y = out if out is not None else torch.empty((A.shape[0], k), device=X.device, dtype=A.dtype)
    call("ep_spmm_csr_" + _scalar(X), A.shape[0], k, _ptr(A.rowptr), _ptr(A.col), _ptr(A.val), _ptr(X), X.stride(0),
         _ptr(Y), Y.stride(0), _stream())
    return Y


def _off(t, elements):
    """Device pointer `elements` items into tensor t."""
    return ctypes.c_void_p(t.data_ptr() + elements * t.element_size())


def spmm2(pair: OperatorPair, X, out_K=None, out_M=None, rows=None):
    """(K X, M X) with one pass over the shared sparsity pattern.  rows=(a, b) restricts the product to that row
    range (outputs are still indexed by the full row number): the sharded engine computes interior rows while
    the halo exchange is in flight, then the boundary rows."""
    X = _check_op(_rowmajor(X), pair)
    k = X.shape[1]
    n = pair.n
    KU = out_K if out_K is not None else torch.empty((n, k), device=X.device, dtype=pair.dtype)
    MU = out_M if out_M is not None else torch.empty((n, k), device=X.device, dtype=pair.dtype)
    assert KU.stride(0) == MU.stride(0)
    a, b = (0, n) if rows is None else rows
    if b <= a:
        return KU, MU
    ld = KU.stride(0)
    call("ep_spmm2_csr_" + _scalar(X), b - a, k, _off(pair.K.rowptr, a), _ptr(pair.K.col), _ptr(pair.K.val), _ptr(pair.M.val),
         _ptr(X), X.stride(0), _off(KU, a * ld), _off(MU, a * ld), ld, _stream())
    return KU, MU


def spmm2_sum(KT: CsrMatrix, MT: CsrMatrix, XA, XB, D=None, scale=1.0, out=None, scale_dev=None):
    """out = scale * (KT XA + MT XB + D); KT and MT share a pattern."""
    XA, XB = _check_op(XA, KT), _check_op(XB, MT)
    if D is not None and D.dtype != KT.dtype:
        raise TypeError("operator values are %s but D is %s" % (KT.dtype, D.dtype))
    k = XA.shape[1]
    assert XA.stride(0) == XB.stride(0)
    Y = out if out is not None else torch.empty((KT.shape[0], k), device=XA.device, dtype=KT.dtype)
    call("ep_spmm2_sum_csr_" + _scalar(XA), KT.shape[0], k, _ptr(KT.rowptr), _ptr(KT.col), _ptr(KT.val), _ptr(MT.val),
         _ptr(XA), _ptr(XB), XA.stride(0), _ptr(D), D.stride(0) if D is not None else 0,
         float(scale), _ptr(scale_dev), _ptr(Y), Y.stride(0), _stream())
    return Y


class _SpmmFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, X, A):
        ctx.A = A
        return spmm(A, X)

    @staticmethod
    def backward(ctx, gY):
        return spmm(ctx.A.transpose(), gY.contiguous()), None


def spmm_autograd(A, X):
    return _SpmmFn.apply(X, A)


# ------------------------------------------------------------------------------- aggregation
def neighbor_mean_concat(x, adj: CsrMatrix, out=None):
    """h = cat([x, mean_{j in N(i)} x_j]); reference src/corrector_model.py:23-30."""
    x = _check(_rowmajor(x))
    n, d = adj.shape[0], x.shape[1]             # adj may be a rank-local block: rows = owned vertices, columns index x
    H = out if out is not None else torch.empty((n, 2 * d), device=x.device, dtype=torch.float32)
    call("ep_neighbor_mean_concat_f32", n, d, _ptr(adj.rowptr), _ptr(adj.col), _ptr(x), x.stride(0), _ptr(H),
         H.stride(0), _stream())
    return H


def spmm_concat(x, A: CsrMatrix, out=None):
    """h = cat([x, A x]); reference src/corrector_model.py:76-79."""
    x = _check(_rowmajor(x))
    n, d = x.shape
    H = out if out is not None else torch.empty((n, 2 * d), device=x.device, dtype=torch.float32)
    call("ep_spmm_concat_f32", n, d, _ptr(A.rowptr), _ptr(A.col), _ptr(A.val), _ptr(x), x.stride(0), _ptr(H),
         H.stride(0), _stream())
    return H


# ------------------------------------------------------------------------------- eigen-loss pieces
class EigenWorkspace:
    """Per-device scratch shared by all eigen-loss calls with the same k."""
    _cache = {}

    @classmethod
    def get(cls, k, device):
        key = (k, str(device))
        ws = cls._cache.get(key)
        if ws is None:
            ws = cls(k, device)
            cls._cache[key] = ws
        return ws

    def __init__(self, k, device):
        self.k = k
        self.plen = query("ep_eigen_partials_len", k)
        self.clen = query("ep_eigen_coef_len", k)
        self.bytes = query("ep_eigen_partials_workspace_bytes", k)
        self.buf = torch.empty(self.bytes, dtype=torch.uint8, device=device)


def eigen_partials(U, KU, MU, out=None):
    """fp64 [G (k*k) | num | sKK | sKM | sMM] for one level (see include/eigenpinns_b200.h).  U, KU, MU are all fp32
    or all fp64."""
    dtype = torch.float64 if U.dtype == torch.float64 else torch.float32
    U, KU, MU = _check(U, dtype), _check(KU, dtype), _check(MU, dtype)
    n, k = U.shape
    ws = EigenWorkspace.get(k, U.device)
    P = out if out is not None else torch.empty(ws.plen, dtype=torch.float64, device=U.device)
    assert KU.stride(0) == MU.stride(0)
    call("ep_eigen_partials_" + _scalar(U), n, k, _ptr(U), U.stride(0), _ptr(KU), _ptr(MU), KU.stride(0), _ptr(P),
         _ptr(ws.buf), ws.bytes, _stream())
    return P


N_LOSS_TERMS = 9      # [res, orth, trace, order, eigen, TOTAL, projection, zero-mean, smoothness]


def eigen_finalize(k, n_global, P, w_res, w_orth, loss_acc, coef=None, lam_out=None, level0=False,
                   lam_target=None, w_trace=0.0, w_order=0.0, w_eigen=0.0, lam_bar_extra=None, overwrite=False,
                   w_mean=0.0, w_smooth=0.0):
    """level0: add the eigenvalue terms (:326-348); overwrite: loss_acc is set, not accumulated (first level)."""
    ws = EigenWorkspace.get(k, P.device)
    coef = coef if coef is not None else torch.empty(ws.clen, dtype=torch.float32, device=P.device)
    lam_out = lam_out if lam_out is not None else torch.empty(k, dtype=torch.float32, device=P.device)
    flags = (1 if level0 else 0) | (2 if overwrite else 0)
    call("ep_eigen_finalize_f32", k, float(n_global), _ptr(P), float(w_res), float(w_orth), flags,
         _ptr(lam_target), float(w_trace), float(w_order), float(w_eigen), float(w_mean), float(w_smooth),
         _ptr(lam_bar_extra), _ptr(lam_out), _ptr(coef), _ptr(loss_acc), _stream())
    return lam_out, coef


def eigen_bwd_prepare(U, KU, MU, coef, KU_bar=None, MU_bar=None, D=None):
    n, k = U.shape

    def like_KU():                                # same row stride as KU (which may be one half of an interleaved row)
        return torch.empty((n, KU.stride(0)), dtype=torch.float32, device=KU.device)[:, :k]
    KU_bar = KU_bar if KU_bar is not None else like_KU()
    MU_bar = MU_bar if MU_bar is not None else like_KU()
    D = D if D is not None else like_KU()
    assert KU.stride(0) == MU.stride(0) == KU_bar.stride(0) == MU_bar.stride(0) == D.stride(0)
    call("ep_eigen_bwd_prepare_f32", n, k, _ptr(U), U.stride(0), _ptr(KU), _ptr(MU), KU.stride(0), _ptr(coef),
         _ptr(KU_bar), _ptr(MU_bar), _ptr(D), _stream())
    return KU_bar, MU_bar, D


def eigen_loss_bwd(pair, U, KU, MU, coef, scale, out, scale_dev=None, rows=None, scratch=None):
    """out = scale * dL/dU of one level (scale_dev: device scalar that overrides scale) from K U, M U and the coefficients
    of eigen_finalize.  Symmetric (K, M), k % 4 == 0, k <= 128 and 16-byte aligned rows of KU, MU and out: one gather
    pass over the pattern, reading every row of KU / MU the pattern references (owned and halo).  Otherwise
    eigen_bwd_prepare + the transposed dual SpMM; scratch, if given, is called on that path only and returns the
    (KU_bar, MU_bar, D) buffers to use (default: new ones per call).  rows=(a, b) restricts the OUTPUT rows to that range
    (one-pass form only): the sharded engine computes the interior rows while the halo rows of KU / MU are in flight."""
    k = KU.shape[1]
    assert KU.stride(0) == MU.stride(0)
    if not (pair.symmetric and k % 4 == 0 and k <= 128
            and all(t.stride(0) % 4 == 0 and t.data_ptr() % 16 == 0 for t in (KU, MU, out))):
        if rows is not None:
            raise NotImplementedError("a row range needs the one-pass backward: symmetric K, M and k a multiple of 4 "
                                      "(<= 128)")
        KU_bar, MU_bar, D = eigen_bwd_prepare(U, KU, MU, coef, *(scratch() if scratch is not None else ()))
        return spmm2_sum(pair.KT, pair.MT, KU_bar, MU_bar, D, scale, out=out, scale_dev=scale_dev)
    a, b = (0, out.shape[0]) if rows is None else rows
    if b <= a:
        return out
    # the kernels read row i of KU / MU for output row i and gather neighbours through absolute column indices, so all
    # pointers keep their row-0 bases and the range is passed as (row0, n_rows)
    gather = (a, b - a, k, _ptr(pair.K.rowptr), _ptr(pair.K.col), _ptr(pair.K.val), _ptr(pair.M.val), _ptr(KU),
              _ptr(MU), KU.stride(0), _ptr(coef), float(scale), _ptr(scale_dev), _ptr(out), out.stride(0))
    if k == 64:
        # k x k product on the tensor cores (TF32 x 3, fp32 accuracy), then the gather pass adds the sparse terms.
        # Measured on B200: at k = 64 this wins (15.8 vs 16.4 ms at 16.7 M vertices); at k = 32 the SIMT product of the
        # one-kernel form hides behind the gather (0.45 vs 0.54 ms at 1 M vertices)
        call("ep_eigen_bwd_gram_term_tf32x3", a, b - a, k, _ptr(MU), MU.stride(0), _ptr(coef), float(scale),
             _ptr(scale_dev), _ptr(out), out.stride(0), _stream())
        call("ep_eigen_bwd_gather_sym_rows_f32", *gather, 1, _stream())
    else:
        call("ep_eigen_bwd_fused_sym_rows_f32", *gather, _stream())
    return out


class ProjectionTerm:
    """w_proj * sum (P^T U - U_coarse)^2 / (n_coarse k) for one fine level (notebook variant, SURVEY 8a-bis:
    multigrid_gnn_refine_fixed.ipynb cell 0 `train_gnn`).  Forward and analytic backward are assembled from the
    existing kernels: SpMM with R = P^T, axpy, the partials kernel (its `num` block = column-wise sum of squares),
    and for the gradient  dL/dU += P (2 w / (n_c k)) (R U - U_c)  one more SpMM."""

    def __init__(self, P_csr: CsrMatrix, R_csr: CsrMatrix, U_coarse, w_proj):
        self.P, self.R, self.U_c, self.w = P_csr, R_csr, _check(U_coarse.contiguous()), float(w_proj)
        n_c, k = U_coarse.shape
        self.denom = float(max(1, n_c * k))
        dev = U_coarse.device
        self.proj = torch.empty((n_c, k), dtype=torch.float32, device=dev)
        self.diff = torch.empty_like(self.proj)
        self.part = torch.empty(EigenWorkspace.get(k, dev).plen, dtype=torch.float64, device=dev)
        self.back = torch.empty((P_csr.shape[0], k), dtype=torch.float32, device=dev)

    def forward(self, U, loss_acc):
        k = U.shape[1]
        spmm(self.R, U, out=self.proj)
        axpy_out(self.proj, self.U_c, -1.0, out=self.diff)
        eigen_partials(self.diff, self.diff, self.diff, out=self.part)            # part[k*k : k*k + k] = sum_i diff^2
        call("ep_loss_add_sum_f64", k, _off(self.part, k * k), self.w / self.denom, 6, _ptr(loss_acc), _stream())

    def backward(self, dU, scale, scale_dev=None):
        """dU += scale * P (2 w / denom) diff."""
        spmm(self.P, self.diff, out=self.back)
        c = 2.0 * self.w / self.denom
        if scale_dev is not None:
            dU.add_(self.back * (scale_dev * c))          # plumbing-level update (device scalar: graph-capturable)
        else:
            call("ep_axpy_out_f32", dU.numel(), float(scale) * c, None, _ptr(dU), _ptr(self.back), _ptr(dU), _stream())
        return dU


def m_normalize_columns(U, M: CsrMatrix, eps=1e-12):
    """u_j / sqrt(u_j^T M u_j + eps); reference src/multigrid_model.py:120-130."""
    U = _check(_rowmajor(U))
    n, k = U.shape
    MU = spmm(M, U)
    P = eigen_partials(U, MU, MU)                 # G = U^T M U (only the diagonal is used)
    out = torch.empty_like(U)
    call("ep_scale_columns_rsqrt_f32", n, k, _ptr(U), U.stride(0), _ptr(P), k, float(eps), _ptr(out),
         out.stride(0), _stream())
    return out


def gram_pair(U, pair: OperatorPair):
    """(U^T K U, U^T M U) as fp64 k x k tensors; reference src/multigrid_model.py:403-404."""
    U = _check(_rowmajor(U))
    k = U.shape[1]
    KU, MU = spmm2(pair, U)
    A = eigen_partials(U, KU, KU)[: k * k].view(k, k).clone()
    B = eigen_partials(U, MU, MU)[: k * k].view(k, k).clone()
    return A, B


def axpy_out(a, b, alpha, out=None, alpha_dev=None):
    a, b = _check(a), _check(b)
    assert a.is_contiguous() and b.is_contiguous() and a.shape == b.shape
    out = out if out is not None else torch.empty_like(a)
    call("ep_axpy_out_f32", a.numel(), float(alpha), _ptr(alpha_dev), _ptr(a), _ptr(b), _ptr(out), _stream())
    return out


def mode_scale_fwd(c, U_base, s, sigma, out=None, sigma_dev=None):
    """out = U_base + sigma * (c o s): the AdaptiveCorrector's per-mode scales (s None = unit scales)."""
    c, U_base = _check(c), _check(U_base)
    n, k = c.shape
    assert U_base.shape == (n, k) and (s is None or (s.numel() == k and s.is_contiguous()))
    out = out if out is not None else torch.empty((n, k), device=c.device, dtype=torch.float32)
    call("ep_mode_scale_fwd_f32", n, k, _ptr(c), c.stride(0), _ptr(U_base), U_base.stride(0),
         _ptr(_check(s) if s is not None else None), float(sigma), _ptr(sigma_dev), _ptr(_check(out)), out.stride(0),
         _stream())
    return out


_mode_scale_ws = {}


def mode_scale_workspace(k, device):
    """Device scratch of ep_mode_scale_bwd_f32 for this k (one per device and k; calls on one stream share it)."""
    key = (k, str(device))
    ws = _mode_scale_ws.get(key)
    if ws is None:
        ws = torch.empty(query("ep_mode_scale_bwd_workspace_bytes", k), dtype=torch.uint8, device=device)
        _mode_scale_ws[key] = ws
    return ws


def mode_scale_bwd(c, Kc, s, w_smooth_corr, dcorr, n_global=None, grad_s=None, accumulate=False, loss_acc=None):
    """In place: dcorr (= dL/dcorr) -> dL/dc; grad_s (k) = or += dL/ds; loss_acc[8], [5] += the smoothness of the
    correction, w / (n k) sum corr o (K corr).  Kc = K c (None when w_smooth_corr = 0), s None = unit scales."""
    c, dcorr = _check(c), _check(dcorr)
    n, k = c.shape
    assert dcorr.shape == (n, k) and (Kc is None or Kc.shape == (n, k))
    ws = mode_scale_workspace(k, c.device)
    call("ep_mode_scale_bwd_f32", n, k, float(n if n_global is None else n_global), _ptr(c), c.stride(0),
         _ptr(_check(Kc) if Kc is not None else None), Kc.stride(0) if Kc is not None else k,
         _ptr(_check(s) if s is not None else None), float(w_smooth_corr), _ptr(dcorr), dcorr.stride(0),
         _ptr(_check(grad_s) if grad_s is not None else None), 1 if accumulate else 0, _ptr(loss_acc), _ptr(ws),
         ws.numel(), _stream())
    return dcorr


class _EigenLossFn(torch.autograd.Function):
    """(w_res * sum_levels L_res, w_orth * sum_levels L_orth, lam_0, lam_1, ...) with the analytic
    backward of SURVEY Appendix A.  Reference: src/multigrid_model.py:291-324."""

    @staticmethod
    def forward(ctx, U_pred, pairs, offsets, w_res, w_orth):
        U_pred = _check(_rowmajor(U_pred))
        k = U_pred.shape[1]
        dev = U_pred.device
        loss_acc = torch.zeros(N_LOSS_TERMS, dtype=torch.float64, device=dev)
        saved = []
        lams = []
        for pair, off in zip(pairs, offsets):
            U = U_pred[int(off):int(off) + pair.n]
            KU, MU = spmm2(pair, U)
            P = eigen_partials(U, KU, MU)
            lam, _ = eigen_finalize(k, pair.n, P, w_res, w_orth, loss_acc)
            saved.append((KU, MU, P))
            lams.append(lam)
        ctx.pairs, ctx.offsets, ctx.saved = pairs, [int(o) for o in offsets], saved
        ctx.w = (float(w_res), float(w_orth))
        ctx.save_for_backward(U_pred)
        out = loss_acc.to(torch.float32)
        return (out[0], out[1]) + tuple(lams)

    @staticmethod
    def backward(ctx, g_res, g_orth, *g_lams):
        (U_pred,) = ctx.saved_tensors
        k = U_pred.shape[1]
        w_res, w_orth = ctx.w
        # upstream scalars (1.0 when the caller just sums the terms, as the reference does)
        gr = float(g_res) if g_res is not None else 0.0
        go = float(g_orth) if g_orth is not None else 0.0
        dU = torch.zeros_like(U_pred)
        scratch_acc = torch.zeros(N_LOSS_TERMS, dtype=torch.float64, device=U_pred.device)
        for li, (pair, off) in enumerate(zip(ctx.pairs, ctx.offsets)):
            KU, MU, P = ctx.saved[li]
            U = U_pred[off:off + pair.n]
            extra = g_lams[li].contiguous() if (li < len(g_lams) and g_lams[li] is not None) else None
            _, coef = eigen_finalize(k, pair.n, P, w_res * gr, w_orth * go, scratch_acc, lam_bar_extra=extra)
            eigen_loss_bwd(pair, U, KU, MU, coef, 1.0, dU[off:off + pair.n])
        return dU, None, None, None, None


def eigen_loss(U_pred, pairs, offsets, w_res, w_orth):
    out = _EigenLossFn.apply(U_pred, pairs, offsets, w_res, w_orth)
    return out[0], out[1], list(out[2:])


# ------------------------------------------------------------------------------- MLP, fp32 path
def _layer_dtype(X):
    """fp64 activations run the fp64 layer kernels; everything else is checked against fp32 as before."""
    return torch.float64 if X.dtype == torch.float64 else torch.float32


def linear_fwd(X, W, b, relu, out=None):
    dtype = _layer_dtype(X)
    X, W = _check(_rowmajor(X), dtype), _check(W, dtype)
    if b is not None and b.dtype != dtype:
        raise TypeError("X is %s but the bias is %s" % (dtype, b.dtype))
    n, d_in = X.shape
    d_out = W.shape[0]
    assert W.is_contiguous() and W.shape[1] == d_in
    Y = out if out is not None else torch.empty((n, d_out), device=X.device, dtype=dtype)
    call("ep_linear_fwd_" + _scalar(X), n, d_in, d_out, _ptr(X), X.stride(0), _ptr(W), _ptr(b), _ptr(Y), Y.stride(0),
         1 if relu else 0, _stream())
    return Y


_bwd_ws = {}


def _linear_bwd_workspace(n, d_in, d_out, device, dtype=torch.float32):
    need = query("ep_linear_bwd_workspace_bytes" + ("_f64" if dtype == torch.float64 else ""), n, d_in, d_out)
    key = str(device)
    buf = _bwd_ws.get(key)
    if buf is None or buf.numel() < need:
        buf = torch.empty(need, dtype=torch.uint8, device=device)
        _bwd_ws[key] = buf
    return buf, need


def linear_bwd(X, W, dY, need_dX, relu_mask, dW=None, db=None, dX=None):
    """dX = (dY W) * [X > 0] (if need_dX), dW = dY^T X, db = colsum(dY)."""
    dtype = _layer_dtype(X)
    X, W, dY = _check(_rowmajor(X), dtype), _check(W, dtype), _check(_rowmajor(dY), dtype)
    n, d_in = X.shape
    d_out = W.shape[0]
    dW = dW if dW is not None else torch.empty_like(W)
    db = db if db is not None else torch.empty(d_out, device=X.device, dtype=dtype)
    if need_dX and dX is None:
        dX = torch.empty((n, d_in), device=X.device, dtype=dtype)
    buf, need = _linear_bwd_workspace(n, d_in, d_out, X.device, dtype)
    call("ep_linear_bwd_" + _scalar(X), n, d_in, d_out, _ptr(X), X.stride(0), _ptr(W), _ptr(dY), dY.stride(0),
         _ptr(dX) if need_dX else None, dX.stride(0) if need_dX else 0, 1 if relu_mask else 0, _ptr(dW), _ptr(db),
         _ptr(buf), need, _stream())
    return dX, dW, db


ACTIVATIONS = {"none": 0, "relu": 1, "silu": 2, "sin": 3, "tanh": 4}     # the `act` codes of ep_linear_act_*
_NEEDS_Z = ("silu", "sin")                      # act' is read from the pre-activation; relu and tanh read the output


def linear_act_fwd(X, W, b, act, Y=None, Z=None):
    """Y = act(X W^T + b) with act one of ACTIVATIONS; Z (optional) receives X W^T + b.  fp32 or fp64 by X's dtype."""
    dtype = _layer_dtype(X)
    X, W = _check(_rowmajor(X), dtype), _check(W, dtype)
    if b is not None:
        _check(b, dtype)
    n, d_in = X.shape
    d_out = W.shape[0]
    assert W.is_contiguous() and W.shape[1] == d_in and (b is None or (b.is_contiguous() and b.numel() == d_out))
    Y = Y if Y is not None else torch.empty((n, d_out), device=X.device, dtype=dtype)
    call("ep_linear_act_fwd_" + _scalar(X), n, d_in, d_out, _ptr(X), X.stride(0), _ptr(W), _ptr(b), _ptr(_check(Y, dtype)),
         Y.stride(0), _ptr(Z if Z is None else _check(Z, dtype)), Z.stride(0) if Z is not None else 0, ACTIVATIONS[act],
         _stream())
    return Y


def linear_act_bwd(X, Zx, act_x, W, dY, need_dX, dW=None, db=None, dX=None, workspace=None):
    """Backward of one layer whose input is X = act_x(Zx) ("none" for the network input): dX = (dY W) * act_x' (if
    need_dX; the gradient w.r.t. the layer below's pre-activation), dW = dY^T X, db = colsum(dY).  Zx: the
    pre-activation saved by linear_act_fwd, needed for silu and sin.  workspace: the caller's scratch of at least
    ep_linear_bwd_workspace_bytes (default: the shared per-device buffer)."""
    dtype = _layer_dtype(X)
    X, W, dY = _check(_rowmajor(X), dtype), _check(W, dtype), _check(_rowmajor(dY), dtype)
    n, d_in = X.shape
    d_out = W.shape[0]
    assert W.is_contiguous() and W.shape[1] == d_in and dY.shape == (n, d_out)
    dW = dW if dW is not None else torch.empty_like(W)
    db = db if db is not None else torch.empty(d_out, device=X.device, dtype=dtype)
    if need_dX and dX is None:
        dX = torch.empty((n, d_in), device=X.device, dtype=dtype)
    if Zx is not None:
        _check(Zx, dtype)
    if workspace is None:
        buf, need = _linear_bwd_workspace(n, d_in, d_out, X.device, dtype)
    else:
        buf, need = workspace, workspace.numel()
    call("ep_linear_act_bwd_" + _scalar(X), n, d_in, d_out, _ptr(X), X.stride(0), _ptr(Zx),
         Zx.stride(0) if Zx is not None else 0, ACTIVATIONS[act_x], _ptr(W), _ptr(dY), dY.stride(0),
         _ptr(dX) if need_dX else None, dX.stride(0) if need_dX else 0, _ptr(dW), _ptr(db), _ptr(buf), need, _stream())
    return (dX if need_dX else None), dW, db


class _MlpActFn(torch.autograd.Function):
    """x -> L_{m-1}(act(... act(L_0(x)))) with L_i(h) = h W_i^T + b_i: one ep_linear_act_fwd per layer; the backward is
    one ep_linear_act_bwd per layer with act' of the layer below folded into its dX, so no element-wise pass and no
    n x h temporary beyond the saved outputs (and pre-activations for silu / sin)."""

    @staticmethod
    def forward(ctx, act, x, *params):
        m = len(params) // 2
        Ws = [W.contiguous() for W in params[:m]]
        bs = [b.contiguous() for b in params[m:]]
        keep_z = act in _NEEDS_Z
        h, hs, zs = x, [], []
        for i in range(m):
            hidden = i < m - 1
            z = torch.empty((h.shape[0], Ws[i].shape[0]), device=x.device, dtype=x.dtype) if hidden and keep_z else None
            h = linear_act_fwd(h, Ws[i], bs[i], act if hidden else "none", Z=z)
            if hidden:
                hs.append(h)
                zs.append(z)
        ctx.act, ctx.m, ctx.keep_z = act, m, keep_z
        ctx.save_for_backward(x, *Ws, *hs, *(zs if keep_z else ()))
        return h

    @staticmethod
    def backward(ctx, g):
        m, act = ctx.m, ctx.act
        saved = ctx.saved_tensors
        x, Ws, hs = saved[0], saved[1:1 + m], saved[1 + m:2 * m]
        zs = saved[2 * m:] if ctx.keep_z else (None,) * (m - 1)
        dWs, dbs = [None] * m, [None] * m
        g = g.contiguous()
        for i in reversed(range(m)):
            if i > 0:
                g, dWs[i], dbs[i] = linear_act_bwd(hs[i - 1], zs[i - 1], act, Ws[i], g, True)
            else:
                g, dWs[i], dbs[i] = linear_act_bwd(x, None, "none", Ws[i], g, ctx.needs_input_grad[1])
        return (None, g, *dWs, *dbs)


def mlp_act(x, weights, biases, act):
    """The network x -> L_{m-1}(act(... act(L_0(x)))), L_i(h) = h W_i^T + b_i (last layer linear), differentiable in x,
    the weights and the biases; act in {"none", "relu", "silu", "sin", "tanh"}.  x's dtype selects the fp32 / fp64
    kernels."""
    if act not in ACTIVATIONS:
        raise ValueError("activation must be one of %s (got %r)" % (sorted(ACTIVATIONS), act))
    if len(weights) != len(biases) or not weights:
        raise ValueError("need one bias per weight and at least one layer")
    return _MlpActFn.apply(act, _rowmajor(x), *weights, *biases)


class Dropout:
    """Dropout after every hidden ReLU of the fused step (nn.Dropout(p) of corrector_model.py::_build_net in training
    mode).  Keep masks are a pure function of (seed, step, layer, row, col) (csrc/dropout.cuh), regenerated by every
    kernel; they are NOT torch's RNG stream, so a dropout run matches the reference in distribution only."""

    def __init__(self, p, seed):
        self.p = check_dropout_p(p)
        self.seed = int(seed) % (1 << 64)

    @property
    def thr(self):
        return round(float(self.p) * 65536.0)

    @property
    def scale(self):
        """s = 1 / (1 - thr / 65536) in fp32, as the kernels use it."""
        return float(np.float32(1.0) / (np.float32(1.0) - np.float32(self.thr) / np.float32(65536.0)))


def check_dropout_p(p):
    """p as the kernels see it (fp32); raises ValueError unless 0 <= p < 1 with round(p * 65536) < 65536."""
    p32 = float(np.float32(p))
    if not (0.0 <= p32 < 1.0) or round(p32 * 65536.0) >= 65536:
        raise ValueError("dropout must lie in [0, 1) (got %r)" % (p,))
    return p32


def dropout_keep_mask(n, width, drop, step, layer, row0=0, device="cuda"):
    """(n, width) uint8 keep mask of hidden layer `layer` at Adam step `step` (1 = kept)."""
    out = torch.empty((n, width), dtype=torch.uint8, device=device)
    call("ep_dropout_keep_mask_u8", n, width, drop.p, drop.seed, int(step), None, int(layer), int(row0), _ptr(out),
         _stream())
    return out


def linear_fwd_dropout(X, W, b, drop, step, layer, step_dev=None, out=None):
    """Y = keep ? relu(X W^T + b) * s : 0 (fp32); step_dev (device int32) overrides step."""
    X, W = _check(_rowmajor(X)), _check(W)
    n, d_in = X.shape
    d_out = W.shape[0]
    assert W.is_contiguous() and W.shape[1] == d_in
    Y = out if out is not None else torch.empty((n, d_out), device=X.device, dtype=torch.float32)
    call("ep_linear_fwd_dropout_f32", n, d_in, d_out, _ptr(X), X.stride(0), _ptr(W), _ptr(b), _ptr(Y), Y.stride(0),
         drop.p, drop.seed, int(step), _ptr(step_dev), int(layer), 0, _stream())
    return Y


def linear_bwd_dropout(X, W, dY, drop, dW=None, db=None, dX=None):
    """linear_bwd for a layer whose input X came out of a hidden layer with dropout: dX = (dY W) * [X > 0] * s."""
    X, W, dY = _check(_rowmajor(X)), _check(W), _check(_rowmajor(dY))
    n, d_in = X.shape
    d_out = W.shape[0]
    dW = dW if dW is not None else torch.empty_like(W)
    db = db if db is not None else torch.empty(d_out, device=X.device, dtype=torch.float32)
    dX = dX if dX is not None else torch.empty((n, d_in), device=X.device, dtype=torch.float32)
    buf, need = _linear_bwd_workspace(n, d_in, d_out, X.device)
    call("ep_linear_bwd_dropout_f32", n, d_in, d_out, _ptr(X), X.stride(0), _ptr(W), _ptr(dY), dY.stride(0), _ptr(dX),
         dX.stride(0), drop.p, _ptr(dW), _ptr(db), _ptr(buf), need, _stream())
    return dX, dW, db


class _LinearFn(torch.autograd.Function):
    """y = relu?(x W^T + b) as one kernel; used layer by layer by the drop-in correctors."""

    @staticmethod
    def forward(ctx, x, W, b, relu):
        y = linear_fwd(x, W.contiguous(), b, relu)
        ctx.relu = relu
        ctx.save_for_backward(x, W, y)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, W, y = ctx.saved_tensors
        gy = gy.contiguous()
        if ctx.relu:
            gy = gy * (y > 0).to(gy.dtype)       # plumbing-level mask; the fused engine folds it into the GEMM
        need_dx = ctx.needs_input_grad[0]
        dX, dW, db = linear_bwd(x, W.contiguous(), gy, need_dx, relu_mask=False)
        return dX, dW, db, None


def linear(x, W, b, relu=False):
    return _LinearFn.apply(x, W, b, relu)


# ------------------------------------------------------------------------------- optimiser
def grad_sqnorm(g, out):
    """out (fp64, device) = sum g^2; g fp32 or fp64."""
    call("ep_grad_sqnorm_" + ("f64" if g.dtype == torch.float64 else "f32"), g.numel(), _ptr(g), _ptr(out), _stream())
    return out


def adam_clip_step(p, g, m, v, lr, beta1, beta2, eps, weight_decay, step, max_norm, sq_norm, hyper_dev=None):
    """hyper_dev: device buffer overriding lr / step (graph replay): {float lr, int32 step} for fp32 p, {double lr,
    double step} for fp64 p.  max_norm <= 0 or sq_norm None: no clipping."""
    if p.dtype == torch.float64:
        for t in (p, g, m, v):
            _check(t, torch.float64)
        call("ep_adam_clip_step_f64", p.numel(), _ptr(p), _ptr(g), _ptr(m), _ptr(v), float(lr), _ptr(hyper_dev),
             float(beta1), float(beta2), float(eps), float(weight_decay), int(step), float(max_norm), _ptr(sq_norm),
             _stream())
        return
    call("ep_adam_clip_step_f32", p.numel(), _ptr(p), _ptr(g), _ptr(m), _ptr(v), float(lr), _ptr(hyper_dev),
         float(beta1), float(beta2), float(eps), float(weight_decay), int(step), float(max_norm), _ptr(sq_norm),
         _stream())


# ------------------------------------------------------------------------------- single mode with learnable eigenvalue
def single_mode_max_prev():
    """Largest number of earlier modes P the single-mode kernels take."""
    return query("ep_single_mode_max_prev")


def single_mode_workspace(P, device):
    """Device scratch of ep_single_mode_fwd_* for P earlier modes."""
    if not 0 <= P <= single_mode_max_prev():
        raise _cabi.EpError("P = %d earlier modes: the single-mode kernels take 0 .. %d" % (P, single_mode_max_prev()))
    return torch.empty(query("ep_single_mode_workspace_bytes", P), dtype=torch.uint8, device=device)


def _column(t, dtype, n):
    _check(t, dtype)
    if t.numel() != n or (t.dim() == 2 and t.shape[1] != 1) or not t.is_contiguous():
        raise ValueError("expected a contiguous n x 1 column of %d values" % n)
    return t


def _prev_block(Q, dtype, n):
    """(P, ldq) of the n x P block of the earlier modes' M u_p (None: P = 0)."""
    if Q is None:
        return 0, 1
    _check(Q, dtype)
    if Q.dim() != 2 or Q.shape[0] != n:
        raise ValueError("Q must be n x P")
    return Q.shape[1], Q.stride(0)


def single_mode_fwd(u, Lu, Mu, Q, w, ortho_weight, loss, coef, workspace):
    """loss[0:4] = [total, eig, norm, ortho] and coef[0:3+P] (fp64, device) of the single-mode functional
    (include/eigenpinns_b200.h).  u, Lu, Mu: n x 1; Q: n x P (None for P = 0); w: the eigenvalue weight (1 value)."""
    dtype = _layer_dtype(u)
    n = u.shape[0]
    u, Lu, Mu = (_column(t, dtype, n) for t in (u, Lu, Mu))
    _check(w, dtype)
    P, ldq = _prev_block(Q, dtype, n)
    _check(loss, torch.float64)
    _check(coef, torch.float64)
    call("ep_single_mode_fwd_" + _scalar(u), n, P, _ptr(u), _ptr(Lu), _ptr(Mu), _ptr(Q), ldq, _ptr(w),
         float(ortho_weight), _ptr(loss), _ptr(coef), _ptr(workspace), workspace.numel(), _stream())
    return loss, coef


def single_mode_bwd(Lu, Mu, Q, w, coef, gL, gM, D):
    """gL = (2/n) r, gM = -(2/n) lambda r, D = 4 (u^T M u - 1) Mu + Q c from the coefficients of single_mode_fwd;
    dL/du = spmm2_sum(L, M, gL, gM, D) for symmetric L, M."""
    dtype = _layer_dtype(Lu)
    n = Lu.shape[0]
    Lu, Mu, gL, gM, D = (_column(t, dtype, n) for t in (Lu, Mu, gL, gM, D))
    _check(w, dtype)
    _check(coef, torch.float64)
    P, ldq = _prev_block(Q, dtype, n)
    call("ep_single_mode_bwd_" + _scalar(Lu), n, P, _ptr(Lu), _ptr(Mu), _ptr(Q), ldq, _ptr(w), _ptr(coef), _ptr(gL),
         _ptr(gM), _ptr(D), _stream())
    return gL, gM, D


def _dims_array(dims):
    return (ctypes.c_int * len(dims))(*[int(d) for d in dims])


def single_mode_fold_fwd(dims, params, eff):
    """eff = [W_l[:, :d] | b_l + lambda W_l[:, d]] per layer from the flat params [W_l | b_l ... | w]
    (include/eigenpinns_b200.h); dims: the len(layers) + 1 widths, input first."""
    dtype = _layer_dtype(params)
    _check(params, dtype)
    _check(eff, dtype)
    call("ep_single_mode_fold_fwd_" + _scalar(params), len(dims) - 1, _dims_array(dims), _ptr(params), _ptr(eff),
         _stream())
    return eff


def single_mode_fold_bwd(dims, params, grad_eff, dloss_dlam, grad):
    """grad (layout of params) from grad_eff (layout of eff) and dL/dlambda of the loss (fp64 device scalar or None)."""
    dtype = _layer_dtype(params)
    for t in (params, grad_eff, grad):
        _check(t, dtype)
    if dloss_dlam is not None:
        _check(dloss_dlam, torch.float64)
    call("ep_single_mode_fold_bwd_" + _scalar(params), len(dims) - 1, _dims_array(dims), _ptr(params),
         _ptr(grad_eff), _ptr(dloss_dlam), _ptr(grad), _stream())
    return grad


# ------------------------------------------------------------------------------- halo rows
def gather_rows(src, idx, out=None):
    src = _check(_rowmajor(src))
    k = src.shape[1]
    out = out if out is not None else torch.empty((idx.numel(), k), device=src.device, dtype=torch.float32)
    call("ep_gather_rows_f32", idx.numel(), k, _ptr(idx), _ptr(src), src.stride(0), _ptr(out), out.stride(0),
         _stream())
    return out


def scatter_add_rows(dst, idx, src):
    call("ep_scatter_add_rows_f32", idx.numel(), src.shape[1], _ptr(idx), _ptr(src), src.stride(0), _ptr(dst),
         dst.stride(0), _stream())
    return dst
