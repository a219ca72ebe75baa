"""TEST INFRASTRUCTURE ONLY (imported by tests/, never by the product): fp64 torch-CPU restatement of one epoch of the
`train_gnn` loop of delta_pinns_validation/multigrid_gnn_refine_fixed.ipynb cell 4 with its AdaptiveCorrector,
on the loss the fused step computes:

    corr   = net([x | mean_nbr x]) * mode_scales                     variants_port.AdaptiveCorrector
    U_pred = U_base + scale * corr,  scale = corr_scale * min(1, epoch / ramp_epochs)
    per level l:  w_res L_res + w_orth L_orth                       step_port.residual_ortho_loss (in fp64 here)
                  + w_smooth sum U_pred o (K U_pred) / (n_l k)
                  + w_smooth_corr sum corr o (K corr) / (n_l k)       variants_port.smoothness_loss
    level 0:      the eigenvalue terms                               step_port.eigenvalue_losses
    clip_grad_norm_ over every parameter (mode_scales included), then torch.optim.Adam(weight_decay)

The operators are the scipy matrices rounded to fp32 and widened back, i.e. the values the CUDA path holds.
"""
import numpy as np
import scipy.sparse as sp
import torch
import torch.nn as nn

from . import step_port, variants_port


def operator_f64(A):
    """scipy matrix -> torch sparse fp64 with fp32-rounded values."""
    return variants_port.to_torch_sparse(sp.csr_matrix(A).astype(np.float32).astype(np.float64))


class AdaptiveTrainer:
    def __init__(self, x, edge_index, U_base, K_list, M_list, lam_target, weights, biases, mode_scales,
                 lr=1e-3, weight_decay=1e-5, corr_scale=10.0, w_res=1000.0, w_orth=10.0, w_trace=0.0, w_order=0.0,
                 w_eigen=0.0, w_smooth=0.0, w_smooth_corr=0.0, grad_clip=10.0, ramp_epochs=5000.0):
        self.x = torch.as_tensor(x).double()
        self.ei = torch.as_tensor(edge_index).long()
        self.U_base = torch.as_tensor(U_base).double()
        self.K = [operator_f64(K) for K in K_list]
        self.M = [operator_f64(M) for M in M_list]
        self.n = [K.shape[0] for K in K_list]
        self.offsets = [0] + list(np.cumsum(self.n[:-1]))
        self.lam_target = None if lam_target is None else torch.as_tensor(lam_target).double()
        k = len(mode_scales)
        self.k = k
        hidden = [w.shape[0] for w in weights[:-1]]
        self.model = variants_port.AdaptiveCorrector(self.x.shape[1], k, hidden).double()
        with torch.no_grad():
            linears = [m for m in self.model.net if isinstance(m, nn.Linear)]
            for lin, W, b in zip(linears, weights, biases):
                lin.weight.copy_(torch.as_tensor(W))
                lin.bias.copy_(torch.as_tensor(b))
            self.model.mode_scales.copy_(torch.as_tensor(mode_scales))
        self.linears = linears
        self.params = list(self.model.parameters())
        self.opt = torch.optim.Adam(self.params, lr=lr, weight_decay=weight_decay)
        self.corr_scale, self.ramp, self.grad_clip = corr_scale, ramp_epochs, grad_clip
        self.w = dict(res=w_res, orth=w_orth, trace=w_trace, order=w_order, eigen=w_eigen, smooth=w_smooth,
                      smooth_corr=w_smooth_corr)

    def scale_for(self, epoch):
        return self.corr_scale * min(1.0, epoch / self.ramp)

    def losses(self, epoch):
        """(total, w_res sum L_res, w_orth sum L_orth, smoothness (both parts, weighted), U_pred)."""
        corr = self.model(self.x, self.ei)
        U_pred = self.U_base + self.scale_for(epoch) * corr
        w, k = self.w, self.k
        eye = torch.eye(k, dtype=torch.float64)
        res = orth = smooth = torch.zeros((), dtype=torch.float64)
        lams = []
        for K, M, off, n in zip(self.K, self.M, self.offsets, self.n):
            U = U_pred[off:off + n]
            KU, MU = torch.sparse.mm(K, U), torch.sparse.mm(M, U)
            lam = (U * KU).sum(0) / ((U * MU).sum(0) + 1e-12)
            lams.append(lam)
            res = res + ((KU - MU * lam[None, :]) ** 2).mean()
            orth = orth + ((U.t() @ MU - eye) ** 2).sum() / k
            l_corr, l_total = variants_port.smoothness_loss(corr[off:off + n], U, K)
            smooth = smooth + w["smooth"] * l_total + w["smooth_corr"] * l_corr
        extra = step_port.eigenvalue_losses(lams[0], self.lam_target, 0.0, w["trace"], w["order"], w["eigen"])
        total = w["res"] * res + w["orth"] * orth + smooth + sum(e.double() for e in extra)
        return total, w["res"] * res, w["orth"] * orth, smooth, U_pred

    def step(self, epoch):
        self.opt.zero_grad()
        total, l_res, l_orth, smooth, _ = self.losses(epoch)
        total.backward()
        torch.nn.utils.clip_grad_norm_(self.params, self.grad_clip)
        self.opt.step()
        return [float(total), float(l_res), float(l_orth), float(smooth)]
