"""MultigridGNN: trains a graph corrector so that U_base + scale * corr solves K u = lambda M u
on every level of a mesh hierarchy.

Drop-in for reference src/multigrid_model.py (class, constructor, public and underscore methods
keep their names, argument order and return types).  What changed underneath:
  * the epoch body (:237-261) is one call of the explicit TrainStepEngine (no autograd graph, no
    per-epoch scipy->torch conversions, fused eigen-loss forward/backward, one Adam launch);
  * `_compute_residual_ortho_loss`, `_forward_pass`, `_normalize_eigenvectors`,
    `refine_eigenvectors` run on the CUDA kernels and stay usable on their own (autograd works
    through them), so reference-style call sites and tests keep functioning;
  * there is no CPU device fallback: constructing the trainer without a GPU raises.
"""
import numpy as np
import torch
import torch.nn as nn
import torch.optim as optim
from scipy.linalg import eigh

import _backend
import utils
from corrector_model import AdaptiveCorrector, SimpleCorrector, SpectralCorrector

_ops = _backend.module("ops")
_engine = _backend.module("engine")
_sparse = _backend.module("sparse")


class MultigridGNN:
    """Multigrid graph-corrector trainer for generalised eigenvectors."""

    def __init__(self, config):
        if not torch.cuda.is_available():
            raise RuntimeError("MultigridGNN (B200 build) needs a CUDA device; there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device())
        self.model = None
        self.model_type = config.model_type.lower()
        if self.model_type not in ['simple', 'spectral', 'adaptive']:
            raise ValueError(f"model_type must be 'simple', 'spectral' or 'adaptive', got '{self.model_type}'")
        for src, dst in (("epochs", "epochs"), ("learning_rate", "lr"), ("corrector_scale", "corr_scale"),
                         ("weight_residual", "w_res"), ("weight_orthogonal", "w_orth"),
                         ("weight_projection", "w_proj"), ("weight_trace", "w_trace"), ("w_order", "w_order"),
                         ("w_eigen", "w_eigen"), ("gradient_clipping", "grad_clip"), ("weight_decay", "weight_decay"),
                         ("log_every", "log_every"), ("hidden_layers", "hidden_layers"), ("dropout", "dropout"),
                         ("n_modes", "n_modes")):
            setattr(self, dst, getattr(config, src))
        self.mlp_mode = getattr(config, "mlp_mode", "fp32")
        self.cgc_mode = getattr(config, "cgc_mode", "reference")
        self.cgc_shift = float(getattr(config, "cgc_shift", 1e-3))
        self.offset_edges = bool(getattr(config, "offset_edges", False))
        self.aggregation = getattr(config, "aggregation", "mean")
        self.loss_read_delay = int(getattr(config, "loss_read_delay", 1))
        self.graph_after_epochs = 3 if getattr(config, "cuda_graph", True) else -1
        self.seed = getattr(config, "seed", None)
        # notebook variant (multigrid_gnn_refine_fixed.ipynb cell 4): 'adaptive' = SimpleCorrector times learnable
        # per-mode scales; smoothness of U_pred and of the correction, w sum u o (K u) / (n k) per level
        self.mode_scale_init = float(getattr(config, "mode_scale_init", 0.01))
        self.w_smooth = float(getattr(config, "weight_smooth", 0.0))
        self.w_smooth_corr = float(getattr(config, "weight_smooth_corr", 0.0))
        self.loss_history = []

    # ------------------------------------------------------------------ top level
    def train_multiresolution(self, sampler):
        offsets = self._compute_node_offsets(sampler.X_list)
        U_cgc, lambda_list = self._initialize_cgc_hierarchy(sampler.U_list, sampler.K_list, sampler.M_list,
                                                            sampler.P_list)
        U_norm = self._normalize_eigenvectors(U_cgc, sampler.M_list)
        U_all = torch.cat(U_norm, dim=0)
        x_feats, edge_index, A_norm = self._build_features(sampler.X_list, U_norm, lambda_list,
                                                           sampler.edge_index_list, sampler.K_list, sampler.M_list)
        self._initialize_model(x_feats.shape[1], self.n_modes, self.hidden_layers, self.dropout)
        optimizer, scheduler = self._create_optimizer(self.lr, self.weight_decay)
        self._training_loop(x_feats, edge_index, A_norm, U_all, sampler.K_list, sampler.M_list, lambda_list,
                            offsets, optimizer, scheduler)
        U_pred = self._generate_final_predictions(x_feats, edge_index, A_norm, U_all, U_norm, sampler.M_list)
        return self._refine_final_predictions(sampler, U_pred)

    def _compute_node_offsets(self, X_list):
        sizes = [X.shape[0] for X in X_list[:-1]]
        return [0] + list(np.cumsum(sizes))

    # ------------------------------------------------------------------ set-up
    def _dev_f32(self, a):
        if torch.is_tensor(a):
            return a.to(device=self.device, dtype=torch.float32).contiguous()
        return torch.from_numpy(np.ascontiguousarray(a)).to(device=self.device, dtype=torch.float32)

    def _pair(self, K, M):
        return utils.device_pair(K, M, self.device)

    def _initialize_cgc_hierarchy(self, U_init_list, K_list, M_list, P_list):
        print("\nApplying Coarse Grid Correction (CGC) to all fine levels...")
        U_out = [self._dev_f32(U_init_list[0])]
        lambdas = []
        for i in range(1, len(K_list)):
            U_fine = self._dev_f32(U_init_list[i])
            if self.cgc_mode == "skip":
                vals, _ = self.refine_eigenvectors(U_fine, K_list[i], M_list[i])
                U_c, lam = U_fine, self._dev_f32(vals)
            else:
                U_c, lam = self.apply_coarse_grid_correction(U_fine, K_list[i], M_list[i], K_list[i - 1],
                                                             P_list[i - 1], M_coarse=M_list[i - 1])
            U_out.append(U_c)
            lambdas.append(lam)
        vals0, _ = self.refine_eigenvectors(U_init_list[0], K_list[0], M_list[0])
        lambdas.insert(0, self._dev_f32(vals0))
        return U_out, lambdas

    def _normalize_eigenvectors(self, U_CGC_list, M_list):
        out = []
        for U, M in zip(U_CGC_list, M_list):
            Mt = utils.device_operator(M, self.device)
            out.append(_ops.m_normalize_columns(self._dev_f32(U), Mt))
        return out

    def _build_features(self, X_list, U_normalized_list, lambda_list, edge_index_list, K_list, M_list):
        print("Building physics-informed features from normalized U_CGC...")
        feats, edges = [], []
        n_levels = len(K_list)
        for i, (X, U, lam, ei) in enumerate(zip(X_list, U_normalized_list, lambda_list, edge_index_list)):
            f = self._compute_level_features(X, U, lam, ei, K_list[i], M_list[i], i, n_levels)
            print(f"--- features have shape: {f.shape} ---")
            feats.append(f)
            edges.append(ei)
        x_all = torch.cat(feats, dim=0).contiguous()
        # NB: like the reference, per-level edge lists are concatenated without node offsets (SURVEY Q3);
        # `offset_edges: true` applies the offsets like the notebooks do (edge_index + node_offset)
        if self.offset_edges:
            edge_all = utils.offset_edge_lists(edges, [f.shape[0] for f in feats])
        else:
            edge_all = torch.cat(edges, dim=1)
        A_norm = utils.build_A_norm(edge_all, x_all.shape[0], self.device) if self.model_type == 'spectral' else None
        return x_all, edge_all, A_norm

    def _compute_level_features(self, X, U_norm, lambdas, edge_index, K_np, M_np, level_idx, n_levels):
        n = X.shape[0]
        dev = self.device
        U = self._dev_f32(U_norm)
        lam = self._dev_f32(lambdas)
        coords = self._dev_f32(X)
        level = torch.full((n, 1), float(n_levels - 1 - level_idx), dtype=torch.float32, device=dev)
        deg = torch.bincount(edge_index[0].to(dev), minlength=n).to(torch.float32).unsqueeze(1)
        deg = deg / (deg.max() + 1e-12)
        Kd = self._dev_f32(K_np.diagonal()).unsqueeze(1)
        Md = self._dev_f32(M_np.diagonal()).unsqueeze(1)
        KU, MU = _ops.spmm2(self._pair(K_np, M_np), U)
        rmag = torch.norm(KU - MU * lam.unsqueeze(0), dim=1, keepdim=True)
        rmag = rmag / (rmag.max() + 1e-12)
        ray = (U * KU).sum(1, keepdim=True) / ((U * MU).sum(1, keepdim=True) + 1e-12)
        ray = ray / (lam.max() + 1e-12)
        return torch.cat([coords, level, deg, Kd, Md, rmag, ray, U], dim=1)

    def _initialize_model(self, input_dim, n_modes, hidden_layers, dropout):
        if self.model is not None:
            return
        if self.seed is not None:
            torch.manual_seed(self.seed)
        if self.model_type == 'simple':
            self.model = SimpleCorrector(input_dim, n_modes, hidden_layers, dropout, aggregation=self.aggregation)
        elif self.model_type == 'adaptive':
            self.model = AdaptiveCorrector(input_dim, n_modes, hidden_layers, dropout, init_scale=self.mode_scale_init)
        else:
            self.model = SpectralCorrector(input_dim, n_modes, hidden_layers, dropout)
        self.model = self.model.to(self.device)
        nn.init.normal_(self.model.net[-1].weight, mean=0.0, std=0.01)      # escape the "do nothing" minimum
        nn.init.zeros_(self.model.net[-1].bias)
        print(f"Model initialized ({self.model_type}): input_dim={input_dim}, output_dim={n_modes}")
        print("Applied small random initialization to output layer.")

    def _create_optimizer(self, lr, weight_decay):
        """torch objects are returned for API compatibility; they carry the hyper-parameters and the
        plateau schedule, while the update itself is the fused clip+Adam kernel of the engine."""
        optimizer = optim.Adam(self.model.parameters(), lr=lr, weight_decay=weight_decay)
        scheduler = optim.lr_scheduler.ReduceLROnPlateau(optimizer, mode='min', factor=0.5, patience=2000,
                                                         min_lr=1e-6)
        return optimizer, scheduler

    # ------------------------------------------------------------------ hot loop
    def _make_engine(self, x_feats, edge_index, A_norm, U_base, K_list, M_list, lambda_target, node_offsets,
                     optimizer):
        x_feats = self._dev_f32(x_feats)
        if self.model_type in ('simple', 'adaptive'):
            h = self.model.corrector_input(x_feats, edge_index.to(self.device))
        else:
            h = self.model.corrector_input(x_feats, A_norm)
        linears = [m for m in self.model.net if isinstance(m, nn.Linear)]
        params = _engine.FlatParams.adopt(linears, mode_scales=getattr(self.model, "mode_scales", None))
        group = optimizer.param_groups[0]
        cfg = _engine.StepConfig(lr=group['lr'], weight_decay=group['weight_decay'], corr_scale=self.corr_scale,
                                 w_res=self.w_res, w_orth=self.w_orth, w_trace=self.w_trace, w_order=self.w_order,
                                 w_eigen=self.w_eigen, grad_clip=self.grad_clip, beta1=group['betas'][0],
                                 beta2=group['betas'][1], eps=group['eps'], w_smooth=self.w_smooth,
                                 w_smooth_corr=self.w_smooth_corr, dropout=float(self.dropout or 0.0),
                                 dropout_seed=self.seed)
        pairs = [self._pair(K, M) for K, M in zip(K_list, M_list)]
        return _engine.TrainStepEngine(h, self._dev_f32(U_base), pairs, node_offsets, params, cfg,
                                       lam_target=lambda_target, mlp_mode=self.mlp_mode)

    def _training_loop(self, x_feats, edge_index, A_norm, U_base, K_list, M_list, lambda_list, node_offsets,
                       optimizer, scheduler):
        print("\nStarting training loop...")
        engine = self._make_engine(x_feats, edge_index, A_norm, U_base, K_list, M_list, lambda_list[0],
                                   node_offsets, optimizer)
        self.engine = engine
        best, stale, max_stale = float('inf'), 0, 5000
        self.model.train()
        # The step is replayed as one CUDA graph after a few eager epochs, and the loss is read back with a delay of
        # one epoch (pinned ring), so the host never stalls the GPU.  Consequence, documented deviation from the
        # reference's synchronous `.item()` (:261): ReduceLROnPlateau and the early-stopping counter see the loss of
        # epoch e while epoch e+1 is already in flight, i.e. a learning-rate change or a stop takes effect one epoch
        # later.  `loss_read_delay = 0` restores the fully synchronous behaviour.
        delay = int(getattr(self, "loss_read_delay", 1))
        reader = _engine.LossReader(depth=4)
        graph_after = int(getattr(self, "graph_after_epochs", 3))
        pending = []                                                   # (epoch, ticket, scale)
        stop = False

        def consume(epoch, ticket, scale):
            nonlocal best, stale, stop
            acc = reader.get(ticket)
            total = float(acc[5])
            self.loss_history.append(total)
            scheduler.step(total)
            if total < best:
                best, stale = total, 0
            else:
                stale += 1
            if stale > max_stale:
                print(f"\nEarly stopping at epoch {epoch} (no improvement for {max_stale} epochs)")
                stop = True
            if epoch % self.log_every == 0 or epoch == self.epochs - 1:
                t = [torch.tensor(float(v)) for v in (acc[5], acc[0], acc[1], 0.0, acc[2], acc[3], acc[4])]
                self._log_training_progress(epoch, *t, scale)

        for epoch in range(self.epochs):
            if epoch == graph_after and graph_after >= 0:
                engine.enable_graph()
            lr = optimizer.param_groups[0]['lr']
            acc = engine.step(epoch, lr=lr)
            pending.append((epoch, reader.push(acc), engine.scale_for(epoch)))
            while len(pending) > delay:
                consume(*pending.pop(0))
            if stop:
                break
        while pending and not stop:
            consume(*pending.pop(0))

    def _forward_pass(self, x_feats, edge_index, A_norm):
        x_feats = x_feats.to(self.device)
        if self.model_type in ('simple', 'adaptive'):
            return self.model(x_feats, edge_index.to(self.device))
        return self.model(x_feats, A_norm)

    def _compute_residual_ortho_loss(self, U_pred, K_list, M_list, node_offsets, w_res, w_orth, n_modes):
        """(w_res * sum_l mean((K U - M U lam)^2), w_orth * sum_l ||U^T M U - I||^2 / k, [lam_l]) - fused
        forward with an analytic backward (autograd flows into U_pred and out of the returned lambdas)."""
        assert U_pred.shape[1] == n_modes
        pairs = [self._pair(K, M) for K, M in zip(K_list, M_list)]
        return _ops.eigen_loss(U_pred, pairs, [int(o) for o in node_offsets], w_res, w_orth)

    def _compute_eigenvalue_losses(self, M_list, lambda_target, lambda_pred_list, w_proj, w_trace, w_order, w_eigen):
        lam = lambda_pred_list[0]                                   # coarsest level only, like the reference
        zero = torch.zeros((), device=lam.device)
        trace = lam.mean()
        order = torch.relu(lam[:-1] - lam[1:]).sum()
        eigen = ((lam - lambda_target.to(lam.device)) ** 2).mean() if lambda_target is not None else zero
        return w_proj * zero, w_trace * trace, w_order * order, w_eigen * eigen

    def _log_training_progress(self, epoch, total_loss, loss_res, loss_orth, loss_proj, loss_trace, loss_order,
                               loss_eigen, scale):
        vals = [float(v) for v in (total_loss, loss_res, loss_orth, loss_proj, loss_trace, loss_order, loss_eigen)]
        print("Epoch %4d: Loss=%.6f | Res=%.6f | Orth=%.6f | Mean=%.6f | Trace=%.6f | Order=%.6f | Eigen=%.6f | "
              "Scale=%.4f" % ((epoch,) + tuple(vals) + (scale,)))

    # ------------------------------------------------------------------ after the loop
    def _generate_final_predictions(self, x_feats, edge_index, A_norm, U_base, U_normalized_list, M_list):
        with torch.no_grad():
            self.model.eval()
            corr = self._forward_pass(x_feats, edge_index, A_norm)
            U_pred = _ops.axpy_out(self._dev_f32(U_base), corr.contiguous(), self.corr_scale)
            out, off = [], 0
            for U_lvl, M in zip(U_normalized_list, M_list):
                n = U_lvl.shape[0]
                out.append(_ops.m_normalize_columns(U_pred[off:off + n], utils.device_operator(M, self.device)))
                off += n
            return torch.cat(out, dim=0).cpu().numpy()

    def refine_eigenvectors(self, U_pred, K, M):
        """Rayleigh-Ritz: eigh(U^T K U, U^T M U) on the host (k x k), U @ C."""
        U = self._dev_f32(U_pred)
        A, B = _ops.gram_pair(U, self._pair(K, M))
        vals, C = eigh(A.to(torch.float32).cpu().numpy(), B.to(torch.float32).cpu().numpy())
        return vals, U.cpu().numpy() @ C

    def apply_coarse_grid_correction(self, U_fine, K_fine, M_fine, K_coarse, P_np, M_coarse=None):
        """U - P A_c^{-1} P^T (K U - M U diag(lambda)) with lambda from Rayleigh-Ritz (reference :410-450).
        cgc_mode 'reference': A_c = K_c, dense fp32 LU like the reference - fails the same way on a singular K_c
        (SURVEY Q12: FEM stiffness matrices of closed or multi-component meshes are singular).
        cgc_mode 'regularized': A_c = K_c + cgc_shift * M_c (or + cgc_shift * I without M_c), never densified: Jacobi-
        preconditioned block CG whose operator application is the CSR SpMM kernel, all k right-hand sides at once."""
        lam_np, _ = self.refine_eigenvectors(U_fine, K_fine, M_fine)
        lam = self._dev_f32(lam_np)
        U = self._dev_f32(U_fine)
        KU, MU = _ops.spmm2(self._pair(K_fine, M_fine), U)
        R_f = KU - MU * lam.unsqueeze(0)
        P = utils.device_operator(P_np, self.device)
        R_c = _ops.spmm(P.transpose(), R_f)
        if self.cgc_mode == "regularized":
            delta_c = self._coarse_solve_cg(K_coarse, M_coarse, R_c)
        else:
            K_c = torch.from_numpy(np.asarray(K_coarse.todense(), dtype=np.float32)).to(self.device)
            delta_c = torch.linalg.solve(K_c, R_c)
        U_cgc = U - _ops.spmm(P, delta_c.contiguous())
        return U_cgc.detach(), lam.detach()

    def _coarse_solve_cg(self, K_coarse, M_coarse, B, tol=1e-6, max_iter=5000):
        """Solve (K_c + shift M_c) X = B for all columns of B (fp32, device).  Per iteration: one SpMM
        (ep_spmm_csr_f32) and a handful of column reductions."""
        import scipy.sparse as sp
        Kc = sp.csr_matrix(K_coarse).astype(np.float64)
        reg = sp.csr_matrix(M_coarse).astype(np.float64) if M_coarse is not None else sp.identity(Kc.shape[0], format="csr")
        A_host = (Kc + self.cgc_shift * reg).tocsr()
        A = utils.device_operator(A_host, self.device)
        d_inv = self._dev_f32(1.0 / A_host.diagonal()).unsqueeze(1)
        B = B.contiguous()
        X = torch.zeros_like(B)
        R = B.clone()
        Z = d_inv * R
        Pd = Z.clone()
        rz = (R * Z).sum(0)
        b_norm = B.norm(dim=0).clamp_min(1e-30)
        self.cgc_iterations = 0
        for it in range(max_iter):
            AP = _ops.spmm(A, Pd)
            alpha = rz / (Pd * AP).sum(0).clamp_min(1e-30)
            X += Pd * alpha.unsqueeze(0)
            R -= AP * alpha.unsqueeze(0)
            self.cgc_iterations = it + 1
            if it % 8 == 7 and float((R.norm(dim=0) / b_norm).max()) < tol:       # one host sync per 8 iterations
                break
            Z = d_inv * R
            rz_new = (R * Z).sum(0)
            Pd = Z + Pd * (rz_new / rz.clamp_min(1e-30)).unsqueeze(0)
            rz = rz_new
        return X

    def _refine_final_predictions(self, sampler, U_pred_all):
        hierarchy = sampler.actual_hierarchy
        start = sum(hierarchy[:-1])
        print("\n--- Extracting finest level ---")
        print(f"Node offset: {start}")
        print(f"Total nodes in U_pred_all: {U_pred_all.shape[0]}")
        print(f"Expected finest level nodes: {hierarchy[-1]}")
        U_finest = U_pred_all[start:start + hierarchy[-1]]
        print(f"Extracted U_finest shape: {U_finest.shape}")
        assert U_finest.shape[0] == hierarchy[-1], f"Mismatch! Got {U_finest.shape[0]}, expected {hierarchy[-1]}"
        print("\n--- Rayleigh-Ritz refinement on finest level ---")
        vals, U_refined = self.refine_eigenvectors(U_finest, sampler.K_list[-1], sampler.M_list[-1])
        print(f"Refined eigenvalues (first 10): {np.round(vals[:10], 6)}")
        return U_refined
