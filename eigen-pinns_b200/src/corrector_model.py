"""Corrector networks: one aggregation step, then a ReLU MLP on [x | agg].

Drop-in for reference src/corrector_model.py: same constructors, same `.net` (an
nn.Sequential of nn.Linear / nn.ReLU / nn.Dropout, so `state_dict` keys are `net.<i>.weight|bias`
and `model.net[-1].weight` works), same forward signatures.  The arithmetic runs in the
hand-written CUDA kernels:
  * SimpleCorrector   mean over incoming edges   -> ep_neighbor_mean_concat_f32  (:23-30)
  * SpectralCorrector agg = A_norm @ x           -> ep_spmm_concat_f32           (:76-79)
  * every Linear(+ReLU) pair                      -> ep_linear_fwd_f32 / ep_linear_bwd_f32
The graph structure and (for inputs that do not require grad) the concatenated input are cached
between calls, because the training loop feeds the same features every epoch.
"""
from typing import List

import torch
import torch.nn as nn

import _backend

_ops = _backend.module("ops")
_sparse = _backend.module("sparse")


def _build_net(in_dim, out_dim, hidden_layers, dropout):
    layers, prev = [], 2 * in_dim
    for width in hidden_layers:
        layers += [nn.Linear(prev, width), nn.ReLU(inplace=True)]
        if dropout > 0.0:
            layers.append(nn.Dropout(dropout))
        prev = width
    layers.append(nn.Linear(prev, out_dim))
    return nn.Sequential(*layers)


def _run_net(net, h, training):
    """Walk the Sequential, fusing each Linear with a directly following ReLU into one kernel."""
    mods = list(net)
    i = 0
    while i < len(mods):
        m = mods[i]
        if isinstance(m, nn.Linear):
            fuse = i + 1 < len(mods) and isinstance(mods[i + 1], nn.ReLU)
            h = _ops.linear(h, m.weight, m.bias, relu=fuse)
            i += 2 if fuse else 1
        elif isinstance(m, nn.ReLU):
            h = torch.relu(h)
            i += 1
        elif isinstance(m, nn.Dropout):
            h = torch.nn.functional.dropout(h, m.p, training)
            i += 1
        else:
            raise TypeError("unsupported layer in corrector net: %r" % (m,))
    return h


class _GraphCache:
    """Remembers the CSR graph and the concatenated input [x | agg] of the last call.  An entry is reused only
    for the SAME tensor object at the same in-place version; the cache keeps a strong reference to the keyed
    tensors, so neither their storage nor their id() can be recycled for a different tensor while the entry
    lives (the reference recomputes the aggregation on every call)."""

    def __init__(self):
        self.graph_obj, self.graph_ver, self.n, self.csr = None, None, None, None
        self.x_obj, self.x_ver, self.h = None, None, None

    @staticmethod
    def _ver(t):
        return t._version if torch.is_tensor(t) else 0

    def graph_hit(self, obj, n):
        return self.graph_obj is obj and self.graph_ver == self._ver(obj) and self.n == n

    def set_graph(self, obj, n, csr):
        self.graph_obj, self.graph_ver, self.n, self.csr = obj, self._ver(obj), n, csr
        self.x_obj, self.x_ver, self.h = None, None, None

    def input_hit(self, x):
        return self.x_obj is x and self.x_ver == x._version

    def set_input(self, x, h):
        self.x_obj, self.x_ver, self.h = x, x._version, h


class SimpleCorrector(nn.Module):
    """aggregation='mean' is the reference (src/corrector_model.py:23-30).  aggregation='sum' is the notebook variant
    without the degree division (SURVEY 8a-bis, `SimpleGNN` of transfer_learning_downsampling.ipynb cell 0): the same
    gather kernel with unit edge weights (ep_spmm_concat_f32 on the multi-adjacency, duplicates kept)."""

    def __init__(self, in_dim, out_dim, hidden_layers, dropout, aggregation="mean"):
        super().__init__()
        if aggregation not in ("mean", "sum"):
            raise ValueError(f"aggregation must be 'mean' or 'sum', got '{aggregation}'")
        self.aggregation = aggregation
        self.net = _build_net(in_dim, out_dim, hidden_layers, dropout)
        self._cache = _GraphCache()

    def corrector_input(self, x, edge_index):
        c = self._cache
        if not c.graph_hit(edge_index, x.shape[0]):
            csr = _sparse.CsrMatrix.from_edge_index(edge_index, x.shape[0], x.device)
            if self.aggregation == "sum":
                csr.val = torch.ones(csr.nnz, dtype=torch.float32, device=x.device)
            c.set_graph(edge_index, x.shape[0], csr)
        if x.requires_grad:
            raise NotImplementedError("gradients w.r.t. the node features are not part of the hot path")
        if not c.input_hit(x):
            c.set_input(x, _ops.neighbor_mean_concat(x, c.csr) if self.aggregation == "mean"
                        else _ops.spmm_concat(x, c.csr))
        return c.h

    def forward(self, x, edge_index):
        return _run_net(self.net, self.corrector_input(x, edge_index), self.training)


class AdaptiveCorrector(SimpleCorrector):
    """Notebook variant with learnable per-mode scales (SURVEY 8a-bis, `AdaptiveCorrector` of
    delta_pinns_validation/multigrid_gnn_refine_fixed.ipynb cell 4): correction = net([x, mean_nbr x]) * mode_scales.
    Runs on the same kernels through autograd (aggregation, fused Linear+ReLU GEMMs); the scales are a torch parameter.
    MultigridGNN (model_type 'adaptive') trains it in the fused TrainStepEngine: the scales are the last k entries of
    the flat parameter buffer (clip + Adam like every weight), U_pred = U_base + scale * (net o mode_scales) and the
    scale gradient come from ep_mode_scale_fwd_f32 / ep_mode_scale_bwd_f32, in fp32 and bf16 MLP mode, eager or
    graph-replayed.  The vertex-sharded engine refuses it."""

    def __init__(self, in_dim, out_dim, hidden_layers=(128, 64, 32), dropout=0.0, init_scale=0.01):
        super().__init__(in_dim, out_dim, list(hidden_layers), dropout)
        self.mode_scales = nn.Parameter(torch.ones(out_dim) * init_scale)

    def forward(self, x, edge_index):
        return super().forward(x, edge_index) * self.mode_scales.unsqueeze(0)


class SpectralCorrector(nn.Module):
    def __init__(self, in_dim: int, out_dim: int, hidden_layers: List[int], dropout: float):
        super().__init__()
        self.net = _build_net(in_dim, out_dim, hidden_layers, dropout)
        self._cache = _GraphCache()

    def corrector_input(self, x, A_norm_sparse):
        c = self._cache
        if not c.graph_hit(A_norm_sparse, x.shape[0]):
            csr = A_norm_sparse if isinstance(A_norm_sparse, _sparse.CsrMatrix) else \
                _sparse.CsrMatrix.from_torch_sparse(A_norm_sparse, x.device)
            c.set_graph(A_norm_sparse, x.shape[0], csr)
        if not c.input_hit(x):
            if x.requires_grad:
                raise NotImplementedError("gradients w.r.t. the node features are not part of the hot path")
            c.set_input(x, _ops.spmm_concat(x.detach(), c.csr))
        return c.h

    def forward(self, x: torch.Tensor, A_norm_sparse) -> torch.Tensor:
        return _run_net(self.net, self.corrector_input(x, A_norm_sparse), self.training)
