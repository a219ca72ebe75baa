"""Autograd-free training step of the single-mode eigenfunction network
(delta_pinns_validation/iterative_eigenvalues_on_cloud.ipynb cell 1, SURVEY 8a-bis): variants.EigenfunctionNN on
variants.single_mode_loss, trained with Adam, one eigenfunction at a time with deflation against the earlier modes.

One step() is, on fixed buffers and with no autograd:
    fold lambda = |w| into the biases (ep_single_mode_fold_fwd_*)  ->  four sin layers (ep_linear_act_fwd_*)
    -> L u, M u (ep_spmm2_csr_* at k = 1) -> loss terms and backward coefficients (ep_single_mode_fwd_*)
    -> gL, gM, D (ep_single_mode_bwd_*) -> dL/du = L gL + M gM + D (ep_spmm2_sum_csr_*, L and M symmetric)
    -> four layer backwards (ep_linear_act_bwd_*) -> dW, db, dw (ep_single_mode_fold_bwd_*) -> Adam (one launch).
fp32 or fp64 by the dtype of the network and the operators.  enable_graph() replays the whole step as one CUDA graph;
replay and eager steps are bit-identical.  The loss terms are fp64 [total, eig, norm, ortho] in the first four entries
of a device buffer that engine.LossReader reads back.
"""
import numpy as np
import torch

from . import ops
from ._cabi import EpError, query
from .engine import LossReader
from .variants import EigenfunctionNN


class SingleModeTrainer:
    """Trains `net` (variants.EigenfunctionNN, on the device) on mean((L u - lambda M u)^2) + (u^T M u - 1)^2 +
    ortho_weight * sum_p (u^T M u_p)^2 with torch.optim.Adam's update (no weight decay, no clipping).

    X: n x d vertex coordinates; pair: sparse.OperatorPair (L, M) of the same dtype, symmetric; previous: earlier
    eigenfunctions (n or n x 1 each), detached, M u_p computed once here.  The module's parameters become views of one
    flat buffer (its state_dict keys and fc* attributes are unchanged), so after training the module holds the
    trained values."""

    def __init__(self, net: EigenfunctionNN, X, pair, previous=(), ortho_weight=1.0, lr=1e-3, betas=(0.999, 0.9999),
                 eps=1e-8):
        fcs = [net.fc1, net.fc2, net.fc3, net.fc4]
        dtype = fcs[0].weight.dtype
        if dtype not in (torch.float32, torch.float64):
            raise TypeError("the network must be float32 or float64, not %s" % dtype)
        if pair.dtype != dtype or X.dtype != dtype:
            raise TypeError("network %s, operators %s and X %s must share one dtype" % (dtype, pair.dtype, X.dtype))
        if not (X.is_cuda and fcs[0].weight.is_cuda):
            raise EpError("SingleModeTrainer needs the network and X on the GPU (no CPU fallback exists)")
        if not pair.symmetric:
            raise ValueError("the single-mode step needs symmetric operators (L^T = L, M^T = M)")
        n = pair.n
        if X.dim() != 2 or X.shape[0] != n:
            raise ValueError("X must be n x d with n = %d rows" % n)
        P = len(previous)
        if P > ops.single_mode_max_prev():
            raise EpError("%d earlier modes: the single-mode kernels take at most %d" % (P, ops.single_mode_max_prev()))
        dev = X.device
        self.net, self.pair, self.n, self.dtype, self.dev = net, pair, n, dtype, dev
        self.X = ops._check(X.contiguous(), dtype)
        self.ortho_weight, self.lr, self.betas, self.eps = float(ortho_weight), float(lr), tuple(betas), float(eps)
        self.dims = [fcs[0].in_features - 1] + [fc.out_features for fc in fcs]
        like = dict(dtype=dtype, device=dev)

        # flat parameters [W_l | b_l ... | w] (include/eigenpinns_b200.h), adopted by the module
        total = sum(fc.weight.numel() + fc.bias.numel() for fc in fcs) + 1
        self.flat = torch.empty(total, **like)
        off = 0
        for fc in fcs:
            for p in (fc.weight, fc.bias):
                view = self.flat[off:off + p.numel()].view(p.shape)
                view.copy_(p.detach())
                p.data = view
                off += p.numel()
        wl = net.eigenvalue_layer.weight
        self.flat[off:].copy_(wl.detach().reshape(1))
        wl.data = self.flat[off:].view(wl.shape)
        self.w = self.flat[off:]
        self.grad, self.m, self.v = (torch.zeros_like(self.flat) for _ in range(3))

        # folded layers [W_eff,l | b_eff,l] and their gradients
        self.eff = torch.empty(sum(o * (d + 1) for d, o in zip(self.dims[:-1], self.dims[1:])), **like)
        self.grad_eff = torch.zeros_like(self.eff)
        self.W_eff, self.b_eff, self.dW_eff, self.db_eff = [], [], [], []
        off = 0
        for d, o in zip(self.dims[:-1], self.dims[1:]):
            for buf, gbuf, shape, store, gstore in ((self.eff, self.grad_eff, (o, d), self.W_eff, self.dW_eff),
                                                    (self.eff, self.grad_eff, (o,), self.b_eff, self.db_eff)):
                size = int(np.prod(shape))
                store.append(buf[off:off + size].view(shape))
                gstore.append(gbuf[off:off + size].view(shape))
                off += size

        h = self.dims[1:-1]
        self.Y = [torch.empty((n, w_), **like) for w_ in h]          # sin(Z) of the hidden layers
        self.Z = [torch.empty((n, w_), **like) for w_ in h]
        self.dX = [torch.empty((n, max(h)), **like) for _ in range(2)]
        self.u, self.Lu, self.Mu, self.gL, self.gM, self.D, self.du = (torch.empty((n, 1), **like) for _ in range(7))
        self.Q = None
        if P:
            U_prev = torch.stack([p.detach().reshape(-1).to(**like) for p in previous], dim=1).contiguous()
            self.Q = ops.spmm(pair.M, U_prev)
        self.loss = torch.zeros(ops.N_LOSS_TERMS, dtype=torch.float64, device=dev)
        self.coef = torch.zeros(3 + P, dtype=torch.float64, device=dev)
        self.dloss_dlam = self.coef[2:3]
        self.ws = ops.single_mode_workspace(P, dev)
        wq = "ep_linear_bwd_workspace_bytes" + ("_f64" if dtype == torch.float64 else "")
        self.bwd_ws = torch.empty(max(query(wq, n, d, o) for d, o in zip(self.dims[:-1], self.dims[1:])),
                                  dtype=torch.uint8, device=dev)
        self.step_count = 0
        self.use_graph, self._graph, self.hyper = False, None, None

    # ---- pieces
    def forward(self):
        """u (n x 1, the trainer's buffer) of the current parameters; lambda = |w| is self.w.abs()."""
        ops.single_mode_fold_fwd(self.dims, self.flat, self.eff)
        x, last = self.X, len(self.W_eff) - 1
        for l in range(last + 1):
            hidden = l < last
            x = ops.linear_act_fwd(x, self.W_eff[l], self.b_eff[l], "sin" if hidden else "none",
                                   Y=self.Y[l] if hidden else self.u, Z=self.Z[l] if hidden else None)
        return self.u

    def loss_forward(self):
        ops.spmm2(self.pair, self.u, out_K=self.Lu, out_M=self.Mu)
        ops.single_mode_fwd(self.u, self.Lu, self.Mu, self.Q, self.w, self.ortho_weight, self.loss, self.coef,
                            self.ws)
        return self.loss

    def backward(self):
        """grad = dL/d(flat parameters) from the coefficients of loss_forward."""
        ops.single_mode_bwd(self.Lu, self.Mu, self.Q, self.w, self.coef, self.gL, self.gM, self.D)
        ops.spmm2_sum(self.pair.KT, self.pair.MT, self.gL, self.gM, D=self.D, out=self.du)
        g = self.du
        for l in reversed(range(len(self.W_eff))):
            if l > 0:
                dx = self.dX[l & 1][:, :self.dims[l]]
                ops.linear_act_bwd(self.Y[l - 1], self.Z[l - 1], "sin", self.W_eff[l], g, True, dW=self.dW_eff[l],
                                   db=self.db_eff[l], dX=dx, workspace=self.bwd_ws)
                g = dx
            else:
                ops.linear_act_bwd(self.X, None, "none", self.W_eff[0], g, False, dW=self.dW_eff[0],
                                   db=self.db_eff[0], workspace=self.bwd_ws)
        ops.single_mode_fold_bwd(self.dims, self.flat, self.grad_eff, self.dloss_dlam, self.grad)
        return self.grad

    def optimizer_step(self, lr, hyper_dev=None):
        if hyper_dev is None:
            self.step_count += 1
        b1, b2 = self.betas
        ops.adam_clip_step(self.flat, self.grad, self.m, self.v, lr, b1, b2, self.eps, 0.0, max(self.step_count, 1),
                           0.0, None, hyper_dev)

    def _body(self, lr, hyper_dev=None):
        self.forward()
        self.loss_forward()
        self.backward()
        self.optimizer_step(lr, hyper_dev)

    # ---- steps
    def step(self, lr=None):
        """One Adam step; returns the device buffer of the loss terms before the update ([total, eig, norm, ortho] in
        its first four entries, fp64).  Reading it on the host is the caller's sync (engine.LossReader pipelines it)."""
        lr = self.lr if lr is None else float(lr)
        if self.use_graph:
            return self._step_graph(lr)
        self._body(lr)
        return self.loss

    def enable_graph(self, on=True):
        """Replay the step as one CUDA graph (call after an eager warm-up step); lr and the step count live in device
        memory, so replay follows them and stays bit-identical to eager steps."""
        self.use_graph, self._graph = bool(on), None

    def _write_hyper(self, lr):
        """{lr, step} -> device: {float, int32} for an fp32 network (ep_adam_clip_step_f32), {double, double} for
        fp64."""
        slot = self._slot = (self._slot + 1) % len(self._host)
        self._evt[slot].synchronize()                # the upload that last used this pinned slot has finished
        host = self._host[slot]
        host[0] = lr
        if self.dtype == torch.float64:
            host[1] = float(self.step_count + 1)
        else:
            host.view(torch.int32)[1] = self.step_count + 1
        self.hyper.copy_(host, non_blocking=True)
        self._evt[slot].record()

    def _step_graph(self, lr):
        if self.hyper is None:
            self.hyper = torch.zeros(2, dtype=self.dtype, device=self.dev)
            self._host = [torch.zeros(2, dtype=self.dtype).pin_memory() for _ in range(8)]
            self._evt = [torch.cuda.Event() for _ in range(8)]
            self._slot = -1
        self._write_hyper(lr)
        if self._graph is None:
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._body(0.0, hyper_dev=self.hyper)
            self._graph = g
        self._graph.replay()
        self.step_count += 1
        return self.loss

    def run(self, epochs, graph=True, history=None):
        """`epochs` steps, the first eager, the rest replayed when graph; history (list) receives the loss terms
        [total, eig, norm, ortho] of every step, read back through an engine.LossReader with a delay of a few steps."""
        reader = LossReader() if history is not None else None
        tickets = []
        for e in range(epochs):
            if graph and e == 1:
                self.enable_graph()
            acc = self.step()
            if reader is not None:
                tickets.append(reader.push(acc))
                if len(tickets) == len(reader.buf):
                    history.append(reader.get(tickets.pop(0))[:4])
        for t in tickets:
            history.append(reader.get(t)[:4])
        self.enable_graph(False)


def train_modes(X, pair, n_modes, epochs, *, initial_eigenvalues, hidden_dim=64, ortho_weight=1.0, lr=1e-3,
                betas=(0.999, 0.9999), eps=1e-8, graph=True, losses=None):
    """The notebook's outer loop: train mode 0, append its u to the earlier modes, train mode 1 against it, and so on;
    each mode gets a fresh EigenfunctionNN(hidden_dim, X.shape[1], initial_eigenvalues[i]) (torch's current RNG draws
    its initial weights) and its own trainer / CUDA graph.  The dtype follows pair.  Returns (eigenvalues (n_modes,),
    U (n x n_modes)) with lambda = |w| and u of the trained networks.  losses (list, optional) receives one
    epochs x 4 array [total, eig, norm, ortho] per mode."""
    if len(initial_eigenvalues) < n_modes:
        raise ValueError("need one initial eigenvalue per mode")
    X = X.to(device=pair.K.device, dtype=pair.dtype).contiguous()
    prev, eigs = [], []
    for i in range(n_modes):
        net = EigenfunctionNN(hidden_dim, X.shape[1], initial_eigenvalue=float(initial_eigenvalues[i]))
        net = net.to(device=X.device, dtype=pair.dtype)
        trainer = SingleModeTrainer(net, X, pair, previous=prev, ortho_weight=ortho_weight, lr=lr, betas=betas,
                                    eps=eps)
        history = [] if losses is not None else None
        trainer.run(epochs, graph=graph, history=history)
        if losses is not None:
            losses.append(np.array(history).reshape(-1, 4))
        prev.append(trainer.forward().clone())
        eigs.append(trainer.w.abs().clone())
    return torch.cat(eigs), torch.cat(prev, dim=1)
