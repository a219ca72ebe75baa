"""Explicit (autograd-free) training step of the corrector network on the eigen-loss.

One `step()` is one epoch body of the reference loop (src/multigrid_model.py:237-261):
    corrector forward -> U_pred = U_base + scale * corr -> per level K U, M U -> Rayleigh
    quotient / residual / Gram terms -> analytic backward -> MLP backward -> clip + Adam.
All buffers are allocated once; every arithmetic kernel is one of ours (include/eigenpinns_b200.h).

Two MLP back ends share this driver:
  "fp32"  layer-by-layer SIMT GEMMs, fp32 end to end       (parity mode, <= 1e-5 vs. the reference)
  "bf16"  fused tcgen05 forward / backward over vertex tiles (perf mode, tolerance stated in DESIGN.md)
"""
import ctypes

import numpy as np
import torch

from . import ops
from ._cabi import call, query, EpError


class FlatParams:
    """Weights and biases of the corrector MLP in ONE contiguous fp32 buffer (plus gradient and
    Adam moments of the same shape).  nn.Module parameters are re-pointed at views of it so the
    module's state_dict keeps working while the optimiser kernel updates everything in one launch."""

    def __init__(self, weights, biases, device, mode_scales=None):
        self.shapes = [(tuple(w.shape), tuple(b.shape)) for w, b in zip(weights, biases)]
        n_scales = 0 if mode_scales is None else mode_scales.numel()
        total = sum(w.numel() + b.numel() for w, b in zip(weights, biases)) + n_scales
        self.flat = torch.empty(total, dtype=torch.float32, device=device)
        self.grad = torch.zeros_like(self.flat)
        self.m = torch.zeros_like(self.flat)
        self.v = torch.zeros_like(self.flat)
        self.W, self.b, self.dW, self.db = [], [], [], []
        self.layer_range = []                       # (first, last) element of layer l's [W | b] block in the flat buffers
        off = 0
        for w, b in zip(weights, biases):
            self.layer_range.append((off, off + w.numel() + b.numel()))
            for src, store, gstore in ((w, self.W, self.dW), (b, self.b, self.db)):
                n = src.numel()
                view = self.flat[off:off + n].view(src.shape)
                view.copy_(src.detach().to(device=device, dtype=torch.float32))
                store.append(view)
                gstore.append(self.grad[off:off + n].view(src.shape))
                off += n
        # learnable per-mode scales of the AdaptiveCorrector: k values after the last bias (None without them)
        self.mode_scales = self.d_mode_scales = None
        if mode_scales is not None:
            self.mode_scales = self.flat[off:off + n_scales]
            self.mode_scales.copy_(mode_scales.detach().reshape(-1).to(device=device, dtype=torch.float32))
            self.d_mode_scales = self.grad[off:off + n_scales]
        self.step_count = 0
        self.sq_norm = torch.zeros(1, dtype=torch.float64, device=device)

    @classmethod
    def adopt(cls, linears, mode_scales=None):
        """Build from nn.Linear modules (and the per-mode scale parameter, if any) and make their parameters views of
        the flat buffer."""
        dev = linears[0].weight.device
        fp = cls([l.weight for l in linears], [l.bias for l in linears], dev, mode_scales=mode_scales)
        for lin, W, b in zip(linears, fp.W, fp.b):
            lin.weight.data = W
            lin.bias.data = b
        if mode_scales is not None:
            mode_scales.data = fp.mode_scales
        return fp

    @property
    def dims(self):
        return [self.W[0].shape[1]] + [w.shape[0] for w in self.W]


class Fp32Mlp:
    """Layer-wise fp32 forward / backward with saved activations.  dropout (ops.Dropout or None): dropout after every
    hidden ReLU, hidden layer l drawing the masks of layer index l at the step passed to forward()."""

    def __init__(self, n, params: FlatParams, device, dropout=None):
        self.p = params
        self.dropout = dropout
        dims = params.dims
        self.acts = [torch.empty((n, d), dtype=torch.float32, device=device) for d in dims[1:]]
        wmax = max(dims[1:-1]) if len(dims) > 2 else dims[0]
        self.dx = [torch.empty((n, wmax), dtype=torch.float32, device=device) for _ in range(2)]

    def forward(self, h, U_base=None, scale=0.0, U_pred=None, scale_dev=None, step=0, step_dev=None):
        x = h
        L = len(self.p.W)
        for l in range(L):
            if self.dropout is not None and l < L - 1:
                ops.linear_fwd_dropout(x, self.p.W[l], self.p.b[l], self.dropout, step, l, step_dev=step_dev,
                                       out=self.acts[l])
            else:
                ops.linear_fwd(x, self.p.W[l], self.p.b[l], relu=(l < L - 1), out=self.acts[l])
            x = self.acts[l]
        if U_pred is not None:
            ops.axpy_out(U_base, x, scale, out=U_pred, alpha_dev=scale_dev)
        return x                                    # corr_raw (n x k)

    def backward(self, h, d_out, on_layer_grads=None):
        """on_layer_grads(l): called as soon as dW / db of layer l are enqueued (the sharded engine starts that
        layer's gradient all-reduce there, overlapping it with the remaining layers)."""
        L = len(self.p.W)
        dy = d_out
        for l in range(L - 1, -1, -1):
            x = self.acts[l - 1] if l > 0 else h
            need_dx = l > 0
            dx = self.dx[l & 1][:, :x.shape[1]] if need_dx else None
            if need_dx and self.dropout is not None:
                ops.linear_bwd_dropout(x, self.p.W[l], dy, self.dropout, dW=self.p.dW[l], db=self.p.db[l], dX=dx)
            else:
                ops.linear_bwd(x, self.p.W[l], dy, need_dx, relu_mask=need_dx, dW=self.p.dW[l], db=self.p.db[l],
                               dX=dx)
            if on_layer_grads is not None:
                on_layer_grads(l)
            dy = dx


class StepConfig:
    def __init__(self, lr=1e-3, weight_decay=1e-5, corr_scale=10.0, w_res=1000.0, w_orth=10.0, w_trace=0.0,
                 w_order=0.0, w_eigen=0.0, grad_clip=10.0, beta1=0.9, beta2=0.999, eps=1e-8, ramp_epochs=5000.0,
                 w_mean=0.0, w_smooth=0.0, w_smooth_corr=0.0, dropout=0.0, dropout_seed=None):
        # dropout: probability of the nn.Dropout after every hidden ReLU (parameters.yml `dropout`), in [0, 1);
        # dropout_seed: 64-bit key of the keep masks (None: one draw from torch's generator when the engine is built)
        self.dropout = ops.check_dropout_p(dropout)
        self.dropout_seed = dropout_seed
        # w_mean / w_smooth: per-level zero-mean and smoothness terms of the notebook variants (SURVEY 8a-bis);
        # w_smooth_corr: the smoothness of the correction, w sum corr o (K corr) / (n k) per level
        self.w_mean, self.w_smooth, self.w_smooth_corr = w_mean, w_smooth, w_smooth_corr
        self.lr, self.weight_decay, self.corr_scale = lr, weight_decay, corr_scale
        self.w_res, self.w_orth, self.w_trace, self.w_order, self.w_eigen = w_res, w_orth, w_trace, w_order, w_eigen
        self.grad_clip, self.beta1, self.beta2, self.eps = grad_clip, beta1, beta2, eps
        self.ramp_epochs = ramp_epochs


class TrainStepEngine:
    """Single-GPU step.  h: (sum N) x 2d corrector input, U_base: (sum N) x k, pairs: OperatorPair per
    level, offsets: first row of each level in the stacked arrays."""

    def __init__(self, h, U_base, pairs, offsets, params: FlatParams, cfg: StepConfig, lam_target=None,
                 mlp_mode="fp32"):
        self.h, self.U_base, self.pairs, self.cfg, self.params = h, U_base.contiguous(), pairs, cfg, params
        self.offsets = [int(o) for o in offsets]
        self.dev = h.device
        self.n_total, self.k = U_base.shape
        k = self.k
        f32 = dict(dtype=torch.float32, device=self.dev)
        self.U_pred = torch.empty((self.n_total, k), **f32)
        # K U and M U of a vertex sit side by side in one row of width 2k: the backward gather reads both with one
        # 8k-byte access per neighbour, and the vertex-sharded engine exchanges their halo rows as ONE message
        self.KUMU = torch.empty((self.n_total, 2 * k), **f32)
        self.KU, self.MU = self.KUMU[:, :k], self.KUMU[:, k:]
        self._bwd_scratch = None       # KU_bar, MU_bar, D: only the unfused (non-symmetric) backward needs them
        self.dCorr = torch.empty((self.n_total, k), **f32)
        ws = ops.EigenWorkspace.get(k, self.dev)
        self.partials = [torch.empty(ws.plen, dtype=torch.float64, device=self.dev) for _ in pairs]
        self.coefs = [torch.empty(ws.clen, **f32) for _ in pairs]
        self.lams = [torch.empty(k, **f32) for _ in pairs]
        self.loss_acc = torch.zeros(ops.N_LOSS_TERMS, dtype=torch.float64, device=self.dev)
        self.projections = {}          # level index -> ops.ProjectionTerm (optional notebook-variant term)
        self.lam_target = lam_target.to(**f32).contiguous() if lam_target is not None else None
        self.mlp_mode = mlp_mode
        self.n_mlp = self._mlp_rows()                  # rows the corrector is evaluated on (all, unless sharded)
        self.dropout = None
        if cfg.dropout > 0.0:
            seed = cfg.dropout_seed
            if seed is None:
                seed = int(torch.randint(0, 2 ** 63 - 1, (1,)).item())
            self.dropout = ops.Dropout(cfg.dropout, seed)
        if mlp_mode == "fp32":
            self.mlp = Fp32Mlp(self.n_mlp, params, self.dev, dropout=self.dropout)
        elif mlp_mode == "bf16":
            from .mlp_tc import TcMlp
            self.mlp = TcMlp(self.n_mlp, params, self.dev, h[:self.n_mlp], dropout=self.dropout)
            self.mlp.want_corr = False
        else:
            raise ValueError("mlp_mode must be 'fp32' or 'bf16'")
        # Per-mode scales and / or the smoothness of the correction: the MLP writes the raw output c, then
        # ep_mode_scale_fwd_f32 forms U_pred and ep_mode_scale_bwd_f32 runs after the eigen-loss backward.  Decided once
        # here; without either the step keeps the plain path (the chain writes U_pred itself).
        self.adaptive = params.mode_scales is not None or float(cfg.w_smooth_corr) != 0.0
        self.Kc = None
        if self.adaptive:
            if mlp_mode == "bf16":
                self.mlp.want_corr = True
            if float(cfg.w_smooth_corr) != 0.0:
                for li, pair in enumerate(pairs):
                    if not pair.symmetric:
                        raise ValueError("w_smooth_corr needs a symmetric K (level %d is not): the gradient uses "
                                         "K^T = K" % li)
                self.Kc = torch.empty((self.n_mlp, k), **f32)
        self.launches_per_step = None
        self.use_graph, self._graph, self.hyper = False, None, None

    # ---- pieces (also used one by one by the tests)
    def add_projection_term(self, level, P, U_coarse, w_proj):
        """Enable w_proj * sum (P^T U_level - U_coarse)^2 / (n_c k) on `level` (P: scipy n_level x n_c prolongation)."""
        from .sparse import CsrMatrix
        import scipy.sparse as sp
        P = sp.csr_matrix(P)
        self.projections[level] = ops.ProjectionTerm(CsrMatrix.from_scipy(P, self.dev), CsrMatrix.from_scipy(P.T.tocsr(), self.dev),
                                                     U_coarse.to(device=self.dev, dtype=torch.float32), w_proj)
        self._graph = None

    def scale_for(self, epoch):
        return self.cfg.corr_scale * min(1.0, epoch / self.cfg.ramp_epochs)

    def forward(self, scale, scale_dev=None, step_dev=None):
        """step_dev (device int32, graph replay) or else params.step_count + 1: the Adam step this forward feeds, which
        selects the dropout masks."""
        m = self.n_mlp
        step = self.params.step_count + 1
        if not self.adaptive:
            return self.mlp.forward(self.h[:m], U_base=self.U_base[:m], scale=scale, U_pred=self.U_pred[:m],
                                    scale_dev=scale_dev, step=step, step_dev=step_dev)
        self.mlp.forward(self.h[:m], step=step, step_dev=step_dev)
        self.mode_scale_forward(scale, scale_dev)
        return self.corr_raw

    @property
    def corr_raw(self):
        """Raw MLP output c (n_mlp x k, fp32): the last activation (fp32 mode) or the chain's corr output (bf16)."""
        return self.mlp.acts[-1] if self.mlp_mode == "fp32" else self.mlp.corr

    def mode_scale_forward(self, scale, scale_dev=None):
        """U_pred = U_base + scale * (c o mode_scales) and, with w_smooth_corr, K c per level."""
        m, c = self.n_mlp, self.corr_raw
        ops.mode_scale_fwd(c, self.U_base[:m], self.params.mode_scales, scale, out=self.U_pred[:m], sigma_dev=scale_dev)
        if self.Kc is not None:
            for li, pair in enumerate(self.pairs):
                s = self._level_slices(li)
                ops.spmm(pair.K, c[s], out=self.Kc[s])

    def mode_scale_backward(self):
        """Per level: dCorr -> dL/dc in place, dL/dmode_scales into the flat gradient, smoothness of the correction
        into loss_acc[8] / [5]."""
        c, p = self.corr_raw, self.params
        for li in range(len(self.pairs)):
            s = self._level_slices(li)
            ops.mode_scale_bwd(c[s], self.Kc[s] if self.Kc is not None else None, p.mode_scales, self.cfg.w_smooth_corr,
                               self.dCorr[s], n_global=self._n_global(li), grad_s=p.d_mode_scales, accumulate=li > 0,
                               loss_acc=self.loss_acc)

    def mlp_backward(self):
        m = self.n_mlp
        self.mlp.backward(self.h[:m], self.dCorr[:m], on_layer_grads=self._layer_grads_ready)

    def _level_slices(self, li):
        off, n = self.offsets[li], self.pairs[li].n
        return slice(off, off + n)

    def loss_forward(self):
        c = self.cfg
        for li, pair in enumerate(self.pairs):
            s = self._level_slices(li)
            ops.spmm2(pair, self.U_pred[s], out_K=self.KU[s], out_M=self.MU[s])
            ops.eigen_partials(self.U_pred[s], self.KU[s], self.MU[s], out=self.partials[li])
            self._reduce_partials(li)
            ops.eigen_finalize(self.k, self._n_global(li), self.partials[li], c.w_res, c.w_orth, self.loss_acc,
                               coef=self.coefs[li], lam_out=self.lams[li], level0=(li == 0),
                               lam_target=self.lam_target, w_trace=c.w_trace, w_order=c.w_order, w_eigen=c.w_eigen,
                               overwrite=(li == 0), w_mean=c.w_mean, w_smooth=c.w_smooth)
        for li, term in self.projections.items():
            term.forward(self.U_pred[self._level_slices(li)], self.loss_acc)

    def _bwd_scratch_rows(self, s):
        """KU_bar, MU_bar, D rows of level slice s for the general backward, allocated on first use."""
        if self._bwd_scratch is None:                 # same row stride as KU / MU (halves of the interleaved rows)
            two = torch.empty_like(self.KUMU)
            self._bwd_scratch = [two[:, :self.k], two[:, self.k:], torch.empty_like(self.KUMU)[:, :self.k]]
        return [t[s] for t in self._bwd_scratch]

    def loss_backward(self, scale, scale_dev=None):
        for li, pair in enumerate(self.pairs):
            s = self._level_slices(li)
            ops.eigen_loss_bwd(pair, self.U_pred[s], self.KU[s], self.MU[s], self.coefs[li], scale, self.dCorr[s],
                               scale_dev, scratch=lambda: self._bwd_scratch_rows(s))
            if li in self.projections:
                self.projections[li].backward(self.dCorr[s], scale, scale_dev)
        if self.adaptive:
            self.mode_scale_backward()

    def optimizer_step(self, lr, hyper_dev=None):
        p, c = self.params, self.cfg
        self._reduce_grads()
        ops.grad_sqnorm(p.grad, p.sq_norm)
        if hyper_dev is None:
            p.step_count += 1
        ops.adam_clip_step(p.flat, p.grad, p.m, p.v, lr, c.beta1, c.beta2, c.eps, c.weight_decay,
                           max(p.step_count, 1), c.grad_clip, p.sq_norm, hyper_dev)

    # hooks for the vertex-sharded engine
    def _mlp_rows(self):
        return self.n_total

    def _n_global(self, li):
        return self.pairs[li].n

    def _reduce_partials(self, li):
        pass

    def _reduce_grads(self):
        pass

    _layer_grads_ready = None          # sharded engine: per-layer gradient all-reduce, started inside the backward

    def step(self, epoch, lr=None, marks=None):
        """One epoch body.  Returns the device tensor loss_acc = [res, orth, trace, order, eigen, total]
        (weighted, fp64); reading it on the host is the caller's one sync per step.
        marks: optional list that receives (phase, cuda event) pairs recorded on the current stream."""
        if self.use_graph and marks is None:
            return self._step_graph(epoch, self.cfg.lr if lr is None else lr)

        def mark(name):
            if marks is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                marks.append((name, ev))
        scale = self.scale_for(epoch)
        mark("start")
        self.forward(scale)
        mark("mlp_fwd")
        self.loss_forward()
        mark("loss_fwd")
        self.loss_backward(scale)
        mark("loss_bwd")
        self.mlp_backward()
        mark("mlp_bwd")
        self.optimizer_step(self.cfg.lr if lr is None else lr)
        mark("optim")
        return self.loss_acc

    # ---- CUDA-graph replay: the whole step is captured once; per-step scalars live in device memory
    def _write_hyper(self, epoch, lr):
        """{float scale, float lr, int32 step} -> device.  The Adam bias corrections are derived from the integer
        step inside the kernel (in double), exactly as in the eager launch, so replay == eager bit for bit."""
        t = self.params.step_count + 1
        slot = self._hyper_slot = (self._hyper_slot + 1) % len(self._hyper_host)
        self._hyper_evt[slot].synchronize()          # the upload that last used this pinned slot has finished
        host = self._hyper_host[slot]
        host[0] = self.scale_for(epoch)
        host[1] = lr
        host.view(torch.int32)[2] = t
        self.hyper.copy_(host, non_blocking=True)
        self._hyper_evt[slot].record()

    def _step_body_dev(self):
        sd = self.hyper[0:1]
        self.forward(0.0, scale_dev=sd, step_dev=self.hyper.view(torch.int32)[2:3])
        self.loss_forward()
        self.loss_backward(0.0, scale_dev=sd)
        self.mlp_backward()
        self.optimizer_step(0.0, hyper_dev=self.hyper[1:3])

    def _step_graph(self, epoch, lr):
        if self.hyper is None:
            self.hyper = torch.zeros(4, dtype=torch.float32, device=self.dev)
            self._hyper_host = [torch.zeros(4, dtype=torch.float32).pin_memory() for _ in range(16)]
            self._hyper_evt = [torch.cuda.Event() for _ in range(16)]
            self._hyper_slot = -1
        self._write_hyper(epoch, lr)
        if self._graph is None:
            from . import _cabi
            torch.cuda.synchronize()
            before, by0 = _cabi.launch_counter, dict(_cabi.launch_by_entry)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._step_body_dev()
            self.launches_per_step = _cabi.launch_counter - before
            self.launches_by_entry = {k_: v - by0.get(k_, 0) for k_, v in _cabi.launch_by_entry.items()
                                      if v - by0.get(k_, 0) > 0}
            self._graph = g
            self._captured_ptrs = self._io_ptrs()
        elif self._io_ptrs() != self._captured_ptrs:
            raise EpError("the captured step reads h / U_base at fixed addresses: copy new data INTO engine.h / "
                          "engine.U_base (or call enable_graph() again) instead of rebinding them")
        self._graph.replay()
        self.params.step_count += 1
        return self.loss_acc

    def _io_ptrs(self):
        return (self.h.data_ptr(), self.U_base.data_ptr())

    def enable_graph(self, on=True):
        """Replay the step as one CUDA graph (call after a few eager warm-up steps).  Changing the shape of the
        problem or the input tensor objects requires enable_graph() again to re-capture."""
        self.use_graph, self._graph = bool(on), None

    def step_from_host(self, h_host, U_base_host, epoch, lr=None):
        """Simplest end-to-end variant: this step's corrector input and base subspace arrive in (pinned) host
        memory, the loss goes back to the host (one synchronising D2H copy)."""
        self.h.copy_(h_host, non_blocking=True)
        self.U_base.copy_(U_base_host, non_blocking=True)
        if hasattr(self.mlp, "input_changed"):
            self.mlp.input_changed(self.h[:self.n_mlp])
        return self.step(epoch, lr).cpu().numpy()


class LossReader:
    """Pipelined read-back of the six loss terms: `push(acc)` enqueues a 48-byte D2H copy into a pinned ring and returns
    a ticket, `get(ticket)` waits for that copy only.  Reading with a delay of one step keeps the host one step ahead
    of the GPU, so the reference's `total_loss.item()` every epoch (src/multigrid_model.py:261) costs no bubble."""

    def __init__(self, depth=4):
        self.buf = [torch.empty(ops.N_LOSS_TERMS, dtype=torch.float64).pin_memory() for _ in range(depth)]
        self.evt = [torch.cuda.Event() for _ in range(depth)]
        self.n = 0

    def push(self, acc):
        slot = self.n % len(self.buf)
        self.buf[slot].copy_(acc, non_blocking=True)
        self.evt[slot].record()
        self.n += 1
        return self.n - 1

    def get(self, ticket):
        assert self.n - ticket <= len(self.buf), "ticket expired (ring depth)"
        slot = ticket % len(self.buf)
        self.evt[slot].synchronize()
        return self.buf[slot].numpy().copy()


class HostFedPipeline:
    """End-to-end driver with HOST inputs every step: node features x (n x d) and the base subspace U_base
    (n x k) live in pinned host memory.  Uploads go through a copy stream into one of two staging sets, so the
    upload of step i+1 overlaps the kernels of step i; the aggregation [x | mean_nbr x] and (bf16 mode) the
    packing run on the device; the six loss terms return through a pinned 48-byte buffer.

        handle = pipe.submit(x_host, U_host, epoch, lr)      # asynchronous
        losses = pipe.result(handle)                         # waits for that step only
    """

    def __init__(self, engine, aggregate):
        """aggregate(x_dev, out) fills out = corrector input h from the uploaded features."""
        self.e, self.aggregate = engine, aggregate
        dev = engine.dev
        n, d2 = engine.h.shape
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.x_dev = [torch.empty((n, d2 // 2), dtype=torch.float32, device=dev) for _ in range(2)]
        self.u_dev = [torch.empty_like(engine.U_base) for _ in range(2)]
        self.uploaded = [torch.cuda.Event() for _ in range(2)]
        self.consumed = [torch.cuda.Event() for _ in range(2)]
        self.loss_host = [torch.empty(ops.N_LOSS_TERMS, dtype=torch.float64).pin_memory() for _ in range(2)]
        self.done = [torch.cuda.Event() for _ in range(2)]
        self.count = 0
        self.h2d_bytes = self.x_dev[0].numel() * 4 + self.u_dev[0].numel() * 4
        self.d2h_bytes = 8 * ops.N_LOSS_TERMS

    def submit(self, x_host, U_host, epoch, lr=None):
        s = self.count & 1
        main = torch.cuda.current_stream()
        with torch.cuda.stream(self.copy_stream):
            if self.count >= 2:
                self.copy_stream.wait_event(self.consumed[s])
            self.x_dev[s].copy_(x_host, non_blocking=True)
            self.u_dev[s].copy_(U_host, non_blocking=True)
            self.uploaded[s].record(self.copy_stream)
        main.wait_event(self.uploaded[s])
        self.aggregate(self.x_dev[s], self.e.h)
        if hasattr(self.e.mlp, "input_changed"):
            self.e.mlp.input_changed(self.e.h[:self.e.n_mlp])
        # the engine (and a captured CUDA graph of its step) reads U_base at a FIXED address: copy, never rebind
        self.e.U_base.copy_(self.u_dev[s], non_blocking=True)
        acc = self.e.step(epoch, lr)
        self.consumed[s].record(main)
        self.loss_host[s].copy_(acc, non_blocking=True)
        self.done[s].record(main)
        self.count += 1
        return s

    def result(self, handle):
        self.done[handle].synchronize()
        return self.loss_host[handle].numpy().copy()
