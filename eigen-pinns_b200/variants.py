"""Loss / model variants of the reference's notebooks (SURVEY.md section 8 a-bis) on the B200 kernels.

The notebooks train other networks against other functionals of the same two operators K and M.  What is expensive
in all of them is what the main path already has kernels for - K U and M U (dual CSR SpMM), the k x k Gram matrices
U^T K U and U^T M U (fp64-accumulated partials kernel), the dense layers (fp32 GEMM kernels) - while the rest is
algebra on k x k matrices or element-wise work.  This module exposes the expensive parts as autograd Functions over
the C ABI and writes each notebook's functional on top of them with torch for the k x k / element-wise glue:

  dense_rayleigh_loss      scripts/simplified_loss.ipynb cell 0 (training loop body): element-wise k x k Rayleigh
                           matrix, residual of all modes, mean + MAX orthogonality term
  whitened_subspace_loss   scripts/loss_with_rigid_body.ipynb cell 0: B = U^T M U, B^-1/2 by a k x k SVD, loss on the
                           whitened Rayleigh matrix (zero mode, trace, gap hinge, off-diagonal, ordering, conditioning)
  single_mode_loss         delta_pinns_validation/iterative_eigenvalues_on_cloud.ipynb cell 1: one eigenfunction at a
                           time with a learnable eigenvalue, normalisation and deflation against earlier modes
  smoothness_loss          delta_pinns_validation/multigrid_gnn_refine_fixed.ipynb cell 4 `train_gnn`: Laplacian energy of
                           the correction and of the prediction (the per-mode scales of its AdaptiveCorrector live in
                           src/corrector_model.py)
  CoordinateMLP            the coordinate networks of the first two (x in R^3 -> U in R^k, SiLU)
  EigenfunctionNN          the network of the third (sin activations, lambda = |w| appended to every layer's input)

Every piece runs in fp32 (fp64 accumulation in the Gram partials) or, as the notebooks train, in fp64: the dtype of
the tensors selects the kernels.  For fp64 build the operators with OperatorPair(K, M, device, dtype=torch.float64)
and call .double() on the networks.  The networks run on ops.mlp_act in either precision: SiLU, sin, tanh and ReLU are
epilogues of the layer GEMMs, forward and backward (ep_linear_act_fwd_* / ep_linear_act_bwd_*).  Parity with the
restated formulas (oracle/variants_port.py, fp64) is checked to fp32 tolerances in tests/test_gpu_variants.py and
on the unrounded operators to fp64 tolerances in tests/test_gpu_variants_f64.py.
Operators must be symmetric (FEM K and M are): the backward uses K^T = K.
"""
import torch
import torch.nn as nn

from . import ops
from .sparse import OperatorPair


# ------------------------------------------------------------------------------------- differentiable operator products
class _OperatorStatsFn(torch.autograd.Function):
    """U -> (K U, M U, U^T K U, U^T M U); the last two as fp64 k x k.  One dual SpMM, two Gram passes.
    Backward: dU = K gKU + M gMU + KU (gA + gA^T) + MU (gB + gB^T)  (K, M symmetric)."""

    @staticmethod
    def forward(ctx, U, pair, want_gram):
        if not pair.symmetric:
            raise ValueError("variants need symmetric operators (K^T = K, M^T = M)")
        U = ops._check_op(ops._rowmajor(U), pair)
        k = U.shape[1]
        KU, MU = ops.spmm2(pair, U)
        ctx.pair = pair
        ctx.set_materialize_grads(False)            # unused outputs arrive as None, not as n x k zeros
        ctx.save_for_backward(KU, MU)
        if want_gram:
            A = ops.eigen_partials(U, KU, KU)[: k * k].view(k, k).clone()
            B = ops.eigen_partials(U, MU, MU)[: k * k].view(k, k).clone()
        else:
            A = B = torch.zeros((0, 0), dtype=torch.float64, device=U.device)
        if not want_gram:
            ctx.mark_non_differentiable(A, B)
        return KU, MU, A, B

    @staticmethod
    def backward(ctx, gKU, gMU, gA, gB):
        KU, MU = ctx.saved_tensors
        direct = None
        if gA is not None:
            direct = ops.linear_fwd(KU, (gA + gA.t()).to(KU.dtype).contiguous(), None, False)   # KU S, S symmetric
        if gB is not None:
            d = ops.linear_fwd(MU, (gB + gB.t()).to(KU.dtype).contiguous(), None, False)
            direct = d if direct is None else direct + d
        if gKU is None and gMU is None:
            return direct, None, None
        gKU = gKU.contiguous() if gKU is not None else torch.zeros_like(KU)
        gMU = gMU.contiguous() if gMU is not None else torch.zeros_like(MU)
        return ops.spmm2_sum(ctx.pair.KT, ctx.pair.MT, gKU, gMU, D=direct), None, None


def operator_products(U, pair: OperatorPair):
    """(K U, M U), differentiable with respect to U."""
    KU, MU, _, _ = _OperatorStatsFn.apply(U, pair, False)
    return KU, MU


def operator_stats(U, pair: OperatorPair):
    """(K U, M U, U^T K U, U^T M U), differentiable; the Gram matrices are fp64."""
    return _OperatorStatsFn.apply(U, pair, True)


# ------------------------------------------------------------------------------------- notebook functionals
def dense_rayleigh_loss(U, pair: OperatorPair, eps=1e-6):
    """scripts/simplified_loss.ipynb cell 0, loop body:
        rayleigh = UKU / (UMU + 1e-6)                     (element-wise, k x k)
        loss_1   = mean(norm((KU - diag(rayleigh) * MU)**2))          = sqrt(sum residual^4)
        orth     = mean((UMU - I)^2) + max((UMU - I)^2)
    Returns (loss, loss_1, diag_loss, off_diag_loss, lambdas)."""
    KU, MU, UKU, UMU = operator_stats(U, pair)
    k = U.shape[1]
    rayleigh = UKU / (UMU + eps)
    lam = torch.diagonal(rayleigh)
    res2 = (KU - lam.to(KU.dtype) * MU) ** 2
    loss_1 = torch.linalg.norm(res2.double())
    d2 = (UMU - torch.eye(k, dtype=UMU.dtype, device=UMU.device)) ** 2
    off_diag_loss = d2.max()
    diag_loss = d2.mean()
    return loss_1 + diag_loss + off_diag_loss, loss_1, diag_loss, off_diag_loss, lam


def whitened_subspace_loss(U, pair: OperatorPair, lambda_orth=1.0, lambda_zero=100.0, lambda_order=0.05,
                           lambda_stability=0.1, min_gap=1e-4):
    """scripts/loss_with_rigid_body.ipynb cell 0, loop body.  With A = U^T K U, B = U^T M U and W = B^-1/2 (k x k SVD,
    singular values clamped at 1e-7) the notebook's U_orth = U W gives rayleigh_matrix = W A W and B_orth = W B W, so
    the whole functional lives on two k x k matrices; no n x k product with W is formed.  The caller passes the
    operators the notebook trains on ((K + 1e-4 I) / ||.||_F and M / ||M||_F: `frobenius_normalised`).
    Returns (loss, dict of the named terms, sorted eigenvalue estimates)."""
    _, _, A, B = operator_stats(U, pair)
    k = U.shape[1]
    eye = torch.eye(k, dtype=B.dtype, device=B.device)
    V, S, _ = torch.linalg.svd(B)
    W = V @ torch.diag_embed(1.0 / torch.sqrt(torch.clamp(S, min=1e-7))) @ V.t()
    R = W @ A @ W
    sorted_eigs, _ = torch.sort(torch.diagonal(R))
    zero_eig = sorted_eigs[0] ** 2
    trace = sorted_eigs[1:].sum() / (k - 1)
    gaps = sorted_eigs[1:] - sorted_eigs[:-1]
    diversity = torch.relu(min_gap - gaps).sum() / (k - 1)
    offdiag = ((R * (1 - eye)) ** 2).sum() / (k * (k - 1))
    eig_loss = lambda_zero * zero_eig + 5.0 * trace + 2.0 * diversity + offdiag
    orth = torch.linalg.norm(W @ B @ W - eye) ** 2
    ordering = torch.relu(sorted_eigs[:-1] - sorted_eigs[1:]).sum() / k
    stability = torch.relu(S.max() / (S.min() + 1e-10) - 1e3) / 1e3
    loss = eig_loss + lambda_orth * orth + lambda_order * ordering + lambda_stability * stability
    terms = {"zero": zero_eig, "trace": trace, "diversity": diversity, "offdiag": offdiag, "orth": orth,
             "ordering": ordering, "stability": stability}
    return loss, terms, sorted_eigs


def frobenius_normalised(K, M, epsilon=1e-4):
    """(K + epsilon I) / ||K + epsilon I||_F and M / ||M||_F as scipy CSR plus the two scales - the operator
    preparation of scripts/loss_with_rigid_body.ipynb cell 0 (done there on dense matrices)."""
    import numpy as np
    import scipy.sparse as sp
    K_reg = (sp.csr_matrix(K) + epsilon * sp.identity(K.shape[0], format="csr")).tocsr()
    K_scale = float(np.sqrt((K_reg.data.astype(np.float64) ** 2).sum()))
    Mc = sp.csr_matrix(M)
    M_scale = float(np.sqrt((Mc.data.astype(np.float64) ** 2).sum()))
    return K_reg / K_scale, Mc / M_scale, K_scale, M_scale


def single_mode_loss(u, eigenvalue, pair: OperatorPair, previous=(), ortho_weight=1.0):
    """delta_pinns_validation/iterative_eigenvalues_on_cloud.ipynb cell 1 (compute_eigenvalue_loss,
    compute_normalization_loss, compute_orthogonality_loss):
        mean((L u - lambda M u)^2) + (u^T M u - 1)^2 + w * sum_prev (u^T M u_prev)^2
    u: n x 1; previous: earlier eigenfunctions (n x 1 each, constants).  Returns (total, eig, norm, ortho)."""
    Lu, Mu = operator_products(u, pair)
    uf, Luf, Muf = u.squeeze(1), Lu.squeeze(1), Mu.squeeze(1)
    eig = ((Luf - eigenvalue.reshape(()) * Muf) ** 2).mean()
    norm = (torch.dot(uf, Muf) - 1.0) ** 2
    ortho = torch.zeros((), dtype=u.dtype, device=u.device)
    for u_prev in previous:
        Mp = ops.spmm(pair.M, u_prev.detach().reshape(-1, 1).contiguous()).squeeze(1)
        ortho = ortho + torch.dot(uf, Mp) ** 2
    return eig + norm + ortho_weight * ortho, eig, norm, ortho


def smoothness_loss(corr, U_pred, pair: OperatorPair, denom=None):
    """delta_pinns_validation/multigrid_gnn_refine_fixed.ipynb cell 4 (`train_gnn` loop body):
        L_smooth_corr = sum(corr * (L corr)) / denom_res,  L_smooth_total = sum(U_pred * (L U_pred)) / denom_res
    with denom_res = n * n_modes.  Returns (L_smooth_corr, L_smooth_total); the notebook adds w_smooth * (both)."""
    n, k = U_pred.shape
    denom = float(n * k) if denom is None else float(denom)
    L_corr = ops.spmm_autograd(pair.K, corr)
    Lu = ops.spmm_autograd(pair.K, U_pred)
    return (corr * L_corr).sum() / denom, (U_pred * Lu).sum() / denom


# ------------------------------------------------------------------------------------- networks
class KernelLinear(nn.Module):
    """nn.Linear whose products run on the GEMM kernels of the C ABI (ep_linear_fwd_f32 / ep_linear_bwd_f32, or the
    _f64 entries after .double())."""

    def __init__(self, in_features, out_features):
        super().__init__()
        ref = nn.Linear(in_features, out_features)
        self.weight, self.bias = ref.weight, ref.bias
        self.in_features, self.out_features = in_features, out_features

    def forward(self, x):
        return ops.linear(x, self.weight, self.bias, False)


class Sin(nn.Module):
    def forward(self, x):
        return torch.sin(x)


_ACTIVATIONS = {"silu": nn.SiLU, "sin": Sin, "relu": nn.ReLU, "tanh": nn.Tanh}


class CoordinateMLP(nn.Module):
    """x (n x in_dim) -> U (n x out_dim): Linear + activation per hidden width, then Linear.  `net` is a Sequential
    with the reference's indexing (state_dict keys net.<2i>.weight / .bias), scripts/simplified_loss.ipynb cell 0
    `MLP`, scripts/loss_with_rigid_body.ipynb cell 0 `MLP`.  forward runs the whole network as ops.mlp_act: the
    activation is the epilogue of each hidden layer's GEMM, and act' that of the dX GEMM above it."""

    def __init__(self, in_dim=3, out_dim=50, hidden=(256, 256, 128), activation="silu"):
        super().__init__()
        layers, last = [], in_dim
        for h in hidden:
            layers += [KernelLinear(last, h), _ACTIVATIONS[activation]()]
            last = h
        layers.append(KernelLinear(last, out_dim))
        self.net = nn.Sequential(*layers)
        self.activation = activation

    def forward(self, x):
        linear = self.net[::2]
        return ops.mlp_act(x, [m.weight for m in linear], [m.bias for m in linear], self.activation)


class EigenfunctionNN(nn.Module):
    """delta_pinns_validation/iterative_eigenvalues_on_cloud.ipynb cell 1: u(x) with sin activations and a learnable
    eigenvalue lambda = |w| that is appended to the input of every layer.  forward -> (u (n x 1), lambda (1 x 1)).
    The appended column is folded into the bias, layer(h (+) lambda) = h W[:, :d]^T + (b + lambda W[:, d]), so the
    four layers run as one ops.mlp_act with sin and no n x (d + 1) concatenation is formed; autograd on the k-sized
    bias pieces gives d lambda and dW[:, d]."""

    def __init__(self, hidden_dim=64, input_dim=3, initial_eigenvalue=0.0):
        super().__init__()
        self.activation = Sin()
        self.eigenvalue_layer = nn.Linear(1, 1, bias=False)
        with torch.no_grad():
            self.eigenvalue_layer.weight.fill_(initial_eigenvalue)
        self.fc1 = KernelLinear(input_dim + 1, hidden_dim)
        self.fc2 = KernelLinear(hidden_dim + 1, hidden_dim)
        self.fc3 = KernelLinear(hidden_dim + 1, hidden_dim)
        self.fc4 = KernelLinear(hidden_dim + 1, 1)

    def forward(self, x):
        eigenvalue = torch.abs(self.eigenvalue_layer.weight).reshape(1, 1)
        lam = eigenvalue.reshape(())
        fcs = (self.fc1, self.fc2, self.fc3, self.fc4)
        u = ops.mlp_act(x, [fc.weight[:, :-1] for fc in fcs], [fc.bias + lam * fc.weight[:, -1] for fc in fcs], "sin")
        return u, eigenvalue
