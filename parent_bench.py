#!/usr/bin/env python
"""Benchmark of the eigen-pinns hot path on B200: training steps per second of the corrector on the
eigen-loss (BASELINE.json metric "train steps/s at 1M/16M verts, k=32 eigs").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME]

One "step" = one epoch body of the reference loop (src/multigrid_model.py:237-261) on the whole mesh:
corrector forward, U_pred, K U / M U, Rayleigh / residual / Gram terms, analytic backward, MLP
backward, clip + Adam.  Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for the roofline
arithmetic used below.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
SRC = os.path.join(ROOT, "eigen-pinns_b200", "src")

WORKLOADS = {
    # name: (kind, size parameter, k)
    "icosphere1m": ("icosphere", 316, 32),      # 998,562 vertices, BASELINE config 4
    "icosphere100k": ("icosphere", 100, 32),    # bounded CPU sample of the same workload
    "icosphere10k": ("icosphere", 32, 32),
    "torus16m": ("torus", 4096, 64),            # 16,777,216 vertices, BASELINE config 5
    "torus1m": ("torus", 1024, 64),
    "torus4m": ("torus", 2048, 64),
}
HIDDEN = [256] * 6                               # reference default (src/parameters.yml)
# dram__bytes_read.sum + dram__bytes_write.sum per launch / vertices from the committed ncu --set full captures
# (profiles/r02_ncu_chain2_summary.csv: tc_chain2_kernel<FWD> 0.3249 GB + 3.3334 GB at 998,562 vertices, k = 32;
#  profiles/r01_final_ncu_full_summary.csv: spmm_kernel<4,1> 0.4330 GB)
NCU_TRAFFIC_CHAIN_FWD_PER_VERTEX = (0.324922e9 + 3.333443e9) / 998562
NCU_TRAFFIC_SPMM2_PER_VERTEX = 0.4330e9 / 998562
MIN_TIMED_MS = 1000.0                            # every timed region lasts at least this long (clock sampling, sustained rates)


def pkg(name=None):
    return importlib.import_module("eigen-pinns_b200" + ("." + name if name else ""))


def mlp_flops_per_vertex(d_in, hidden, k):
    """fwd 2S + bwd (4S - 2*d_in*h0): no input-gradient GEMM for the first layer (SURVEY 8d)."""
    dims = [d_in] + list(hidden) + [k]
    S = sum(dims[i] * dims[i + 1] for i in range(len(dims) - 1))
    return 6 * S - 2 * dims[0] * dims[1]


def build_host_workload(name, band_order=False):
    """Synthetic mesh, FEM operators, initial subspace and node features on the host (float64 / numpy).
    band_order: relabel the icosphere's vertices in latitude bands (used when the mesh is sharded over GPUs)."""
    kind, size, k = WORKLOADS[name]
    fem, syn = pkg("fem"), pkg("synthetic")
    rng = np.random.default_rng(0)
    if kind == "icosphere":
        verts, tris = syn.icosphere(size)
        if band_order:
            # latitude-band vertex order: contiguous vertex ranges (one per GPU) then touch two neighbours each and the
            # halos are balanced (the generator's face-by-face order puts every icosahedron edge vertex on rank 0).
            # Not used on one GPU: the face-by-face order has the better gather locality (0.29 vs 0.45 ms loss backward)
            part = pkg("partition")
            verts, tris = part.permute_mesh(verts, tris, part.z_order(verts))
        unit = verts.copy()
        verts = fem.normalize_verts(verts)
        modes, degs = syn.real_spherical_harmonics(unit, k)
        radius2 = float((verts ** 2).sum(1).mean())
        lam_analytic = degs * (degs + 1) / (2.0 * radius2)     # reference mass matrix is 2x the lumped area
    else:
        verts, tris = syn.torus(size, size)
        verts = fem.normalize_verts(verts)
        modes, lam_analytic = syn.torus_trial_modes(size, size, k), None
    K, M = fem.assemble_stiffness_mass(verts, tris)
    edges = fem.connectivity_edges(tris)
    U0 = (modes + 0.05 * rng.standard_normal(modes.shape)).astype(np.float32)
    return dict(name=name, k=k, verts=verts, tris=tris, K=K, M=M, edges=edges, U0=U0, modes=modes,
                lam_analytic=lam_analytic)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, col in (("hw_slowdown", 3), ("hw_thermal_slowdown", 4), ("sw_thermal_slowdown", 5),
                              ("sw_power_cap", 6)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], bf16_burst=p["bf16_tflops"], bf16_sustained=p.get("bf16_tflops_sustained",
                    p["bf16_tflops"]), source="measured")
    return dict(hbm=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback")


# ------------------------------------------------------------------------------------------ CPU oracle / reference arm
def oracle_trainer(w):
    """CPU oracle (torch-CPU port of the reference step, oracle/step_port.py) on a host workload."""
    import torch
    from oracle import step_port
    k = w["k"]
    U_base = step_port.m_normalize(torch.from_numpy(w["U0"]), w["M"])
    ei = torch.from_numpy(w["edges"])
    lam = torch.zeros(k)
    x = step_port.level_features(w["verts"], U_base, torch.linspace(0, 1, k), ei, w["K"], w["M"], 0, 1)
    tr = step_port.CorrectorTrainer(x, ei, U_base, [w["K"]], [w["M"]], lam, HIDDEN, k)
    tr.epoch = 2500
    return tr


def time_oracle(w, steps, warmup, threads, budget_s=None):
    """Wall-clock steps/s of the oracle on all host cores.  With a time budget the number of timed steps is cut
    (never below 2) and the number actually executed is reported - nothing is extrapolated."""
    import torch
    if threads:
        torch.set_num_threads(threads)
    tr = oracle_trainer(w)
    t0 = time.perf_counter()
    for _ in range(max(1, warmup)):
        tr.step()
    t_warm = (time.perf_counter() - t0) / max(1, warmup)
    n = steps
    if budget_s is not None:
        n = max(2, min(steps, int(budget_s / max(t_warm, 1e-6))))
    t0 = time.perf_counter()
    for _ in range(n):
        tr.step()
    dt = (time.perf_counter() - t0) / n
    return dict(ms_per_step=dt * 1e3, steps_per_s=1.0 / dt, steps_run=n, threads=torch.get_num_threads(),
                vertices=int(w["verts"].shape[0]))


def reference_workload_name(args):
    """The reference arm runs the NAMED configuration when it fits the host (1 M vertices: ~3-4 s per step on 16 cores);
    the 16 M-vertex torus needs > 120 GB of autograd state on the CPU (SURVEY 8d), so there the 1 M torus is timed and
    the line says so in config.workload / cpu_baseline.sample."""
    kind, size, k = WORKLOADS[args.workload]
    if kind == "torus" and size > 1024:
        return "torus1m"
    return args.workload


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    name = reference_workload_name(args)
    kind, size, k = WORKLOADS[name]
    w = build_host_workload(name)
    # torchrun pins OMP_NUM_THREADS=1; the reference arm is entitled to every host core
    r = time_oracle(w, args.steps, min(args.warmup, 1), threads=os.cpu_count(), budget_s=150.0)
    sample_txt = ("oracle/step_port.py (torch-CPU port of the reference epoch body, src/multigrid_model.py:237-261) on the "
                  "full %s workload (%d vertices, k = %d), %d timed steps of %.0f ms, wall clock, %d threads"
                  % (name, r["vertices"], k, r["steps_run"], r["ms_per_step"], r["threads"]))
    line = {"impl": "reference", "metric": "train_steps_per_s", "value": r["steps_per_s"], "unit": "steps/s",
            "n_gpus": args.gpus, "steps": r["steps_run"], "steps_requested": args.steps, "warmup": min(args.warmup, 1),
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": name, "vertices": r["vertices"], "k": k, "hidden": HIDDEN},
            "cpu_baseline": {"value": r["steps_per_s"], "unit": "steps/s", "cores": r["threads"], "kind": "port",
                             "sample": sample_txt},
            "e2e": {"value": r["steps_per_s"], "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ our arm
def build_engine(args, dev, rank, world, workload=None):
    """Set-up (untimed): workload -> training-step engine.  Triangle meshes built on the host go through the
    reference-shaped API (MultigridGNN._normalize_eigenvectors / _build_features / _initialize_model / _make_engine);
    the torus grids are generated, assembled and sharded on the device (eigen-pinns_b200/workloads.py)."""
    import torch
    workload = workload or args.workload
    kind, size, k = WORKLOADS[workload]
    if kind == "torus":
        eng, x_feats, adj, U_norm, n, nnz = pkg("workloads").build_torus_engine(size, k, dev, args.mlp_mode, HIDDEN,
                                                                               rank, world)
        return dict(engine=eng, n=n, k=k, nnz=nnz, lam_err=None, x_feats=x_feats, U_norm=U_norm, edge_index=None,
                    adjacency=adj, host=None)
    if SRC not in sys.path:
        sys.path.insert(0, SRC)
    import config as cfg_mod
    import multigrid_model
    w = build_host_workload(workload, band_order=world > 1)
    n = w["verts"].shape[0]
    cfg = cfg_mod.PINNConfig.from_yaml(os.path.join(SRC, "parameters.yml"))
    cfg.n_modes, cfg.mlp_mode, cfg.seed, cfg.hidden_layers = k, args.mlp_mode, 0, HIDDEN
    stdout, sys.stdout = sys.stdout, open(os.devnull, "w")      # the drop-in modules print like the reference
    try:
        gnn = multigrid_model.MultigridGNN(cfg)
        edges = torch.from_numpy(w["edges"])
        U_norm = gnn._normalize_eigenvectors([w["U0"]], [w["M"]])
        vals_rr, _ = gnn.refine_eigenvectors(w["modes"].astype(np.float32), w["K"], w["M"])
        lam0 = torch.from_numpy(vals_rr.astype(np.float32))
        x_feats, edge_all, A_norm = gnn._build_features([w["verts"]], U_norm, [lam0], [edges], [w["K"]], [w["M"]])
        gnn._initialize_model(x_feats.shape[1], k, HIDDEN, 0.0)
        opt, _ = gnn._create_optimizer(gnn.lr, gnn.weight_decay)
        if world > 1:
            eng = pkg("dist_engine").make_sharded_engine(gnn, x_feats, edge_all, U_norm[0], w["K"], w["M"], lam0, opt,
                                                         rank, world)
        else:
            eng = gnn._make_engine(x_feats, edge_all, A_norm, U_norm[0], [w["K"]], [w["M"]], lam0, [0], opt)
    finally:
        sys.stdout = stdout
    lam_err = None
    if w["lam_analytic"] is not None:             # Rayleigh-Ritz of the analytic harmonics vs l(l+1)/(2 rho^2)
        ref = w["lam_analytic"]
        nz = ref > 0
        lam_err = float(np.max(np.abs(np.sort(vals_rr)[nz] - ref[nz]) / ref[nz]))
    return dict(engine=eng, n=n, k=k, nnz=int(w["K"].nnz), lam_err=lam_err, x_feats=x_feats, U_norm=U_norm[0],
                edge_index=edge_all, adjacency=None, host=w)


def timed_steps(eng, args, dev, rank, world, epoch0, clock_sampler=None):
    """Warm-up (eager, then phase timing, then CUDA-graph capture), then the timed region: K steps x R repeats with
    R chosen so that the region lasts >= MIN_TIMED_MS.  The loss of every step is read back on the host with a delay
    of one step (pinned ring), as the drop-in training loop does.  Returns a dict of measurements (ms = max over ranks)."""
    import torch
    import torch.distributed as dist
    cabi, engine_mod = pkg("_cabi"), pkg("engine")

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        eng.step(epoch0 + i)
    marks_all, n_phase = [], 5
    for i in range(n_phase):
        marks = []
        eng.step(epoch0 + args.warmup + i, marks=marks)
        marks_all.append(marks)
    torch.cuda.synchronize()
    phase = {}
    for marks in marks_all:
        for (a, ea), (b, eb) in zip(marks[:-1], marks[1:]):
            phase[b] = phase.get(b, 0.0) + ea.elapsed_time(eb)
    phase = {p: v / n_phase for p, v in phase.items()}
    if not args.no_graph:
        eng.enable_graph()
        try:
            for i in range(2):
                eng.step(epoch0 + args.warmup + n_phase + i)
        except Exception as exc:                      # same kernels either way; only the launch mechanism differs
            sys.stderr.write("CUDA-graph capture failed (%r); timing eager launches instead\n" % (exc,))
            eng.enable_graph(False)
    # estimate -> number of repeats
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(3):
        eng.step(epoch0 + i)
    e1.record()
    torch.cuda.synchronize()
    est = torch.tensor([e0.elapsed_time(e1) / 3.0], device=dev)
    if world > 1:
        dist.all_reduce(est, op=dist.ReduceOp.MAX)
    repeats = max(1, int(np.ceil(MIN_TIMED_MS / (float(est.item()) * args.steps))))
    n_timed = args.steps * repeats
    reader = engine_mod.LossReader(depth=4)
    if clock_sampler is not None:
        clock_sampler.start()
    launches0 = cabi.launch_counter
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_start.record()
    prev, loss_now = None, None
    for i in range(n_timed):
        ticket = reader.push(eng.step(epoch0 + 3 + i))
        if prev is not None:
            loss_now = reader.get(prev)               # loss of the previous step: the host stays one step ahead
        prev = ticket
    t_end.record()
    barrier()
    loss_now = reader.get(prev)
    clk = clock_sampler.stop() if clock_sampler is not None else None
    launches = cabi.launch_counter - launches0
    if eng.use_graph and eng.launches_per_step:
        launches = eng.launches_per_step * n_timed
    ms_total = t_start.elapsed_time(t_end)
    if world > 1:
        t = torch.tensor([ms_total], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    return dict(ms_step=ms_total / n_timed, n_timed=n_timed, repeats=repeats, phase=phase, clocks=clk,
                launches=int(launches), loss=float(loss_now[5]), timed_ms=ms_total,
                launches_by_entry=getattr(eng, "launches_by_entry", None))


def trained_accuracy(mlp_mode, epochs=10000):
    """BASELINE "lambda rel err" of a TRAINED run, through the drop-in surface: coarse FEM level (1057 vertices) + bunny
    (2503 vertices) from tests/golden/bunny_fem.npz, k = 16, MLP 50 -> 256 x 6 -> 16, MultigridGNN.train_multiresolution
    for `epochs` epochs (CUDA-graph replayed, loss read back every epoch), Rayleigh-Ritz on the finest level, eigenvalues
    against scipy's eigsh on the same FEM operators.  profiles/r02_trained_accuracy_*.json holds the same problem trained
    by the CPU oracle for comparison (the reference's own accuracy level; 10 000 epochs is the reference's default, the
    correction scale ramps up over the first 5 000, src/multigrid_model.py:243)."""
    import types
    import torch
    import scipy.sparse as sp
    from scipy.sparse.linalg import eigsh
    if SRC not in sys.path:
        sys.path.insert(0, SRC)
    import config as cfg_mod
    import multigrid_model
    import utils
    fem = pkg("fem")
    g = np.load(os.path.join(ROOT, "tests", "golden", "bunny_fem.npz"))
    n, k = g["verts"].shape[0], 16
    K = sp.csr_matrix((g["K_data"], g["K_indices"], g["K_indptr"]), shape=(n, n))
    M = sp.csr_matrix((g["M_data"], g["M_indices"], g["M_indptr"]), shape=(n, n))
    Kc, Mc = fem.assemble_stiffness_mass(g["coarse_verts"], g["coarse_tris"])
    s = types.SimpleNamespace()
    s.X_list = [g["coarse_verts"], g["verts"]]
    s.K_list, s.M_list = [Kc.tocoo(), K.tocoo()], [Mc.tocoo(), M.tocoo()]
    s.edge_index_list = [utils.build_knn_graph(X, k=8) for X in s.X_list]
    vals_c, U0 = eigsh(Kc.tocsc(), k=k, M=Mc.tocsc(), sigma=-1e-6, which="LM")
    U0 = U0[:, np.argsort(vals_c)]
    P = utils.build_prolongation(s.X_list[0], s.X_list[1], k=8)
    s.P_list, s.U_list = [P], [U0, utils.jacobi_smooth(M, K, P @ U0, alpha=0.1, n_iters=10)]
    s.actual_hierarchy = [X.shape[0] for X in s.X_list]
    exact = np.sort(eigsh(K.tocsc(), k=k, M=M.tocsc(), sigma=-1e-6, which="LM")[0])
    cfg = cfg_mod.PINNConfig.from_yaml(os.path.join(SRC, "parameters.yml"))
    cfg.n_modes, cfg.hidden_layers, cfg.epochs, cfg.log_every = k, HIDDEN, epochs, 10 ** 9
    cfg.mlp_mode, cfg.cgc_mode, cfg.seed = mlp_mode, "skip", 0
    stdout, sys.stdout = sys.stdout, open(os.devnull, "w")
    try:
        gnn = multigrid_model.MultigridGNN(cfg)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        U = gnn.train_multiresolution(s)
        torch.cuda.synchronize()
        secs = time.perf_counter() - t0
        vals, _ = gnn.refine_eigenvectors(U, s.K_list[-1], s.M_list[-1])
    finally:
        sys.stdout = stdout
    rel = np.abs(np.sort(vals)[1:] - exact[1:]) / np.abs(exact[1:])
    return {"problem": "coarse(1057) + bunny(2503), k=16, MLP 50->256x6->16, %d epochs, %s" % (epochs, mlp_mode),
            "lambda_rel_err_trained_first10_max": float(rel[:9].max()), "lambda_rel_err_trained_mean": float(rel.mean()),
            "final_loss": float(gnn.loss_history[-1]), "first_loss": float(gnn.loss_history[0]),
            "train_seconds_incl_setup": secs, "epochs_per_s": epochs / secs,
            "oracle_cpu_same_problem": {"epochs": 10000, "lambda_rel_err_trained_first10_max": 0.195, "final_loss": 0.145,
                                        "epochs_per_s": 5.8, "source": "profiles/r02_trained_accuracy_oracle_10k.json "
                                        "(CPU oracle, fp32, 1726 s; after 3000 epochs: 0.559, r02_trained_accuracy_oracle.json)"}}


def time_call(fn, reps_min=20):
    """CUDA-event time of one call of fn (ms), repeated so that the timed region lasts >= 100 ms."""
    import torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(3):
        fn()
    e1.record()
    torch.cuda.synchronize()
    reps = max(reps_min, int(100.0 / max(e0.elapsed_time(e1) / 3.0, 1e-3)))
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def run_ours(args):
    import ctypes
    import torch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback exists for the product path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    pkg().require_library()
    cabi, ops = pkg("_cabi"), pkg("ops")
    wl = build_engine(args, dev, rank, world)
    eng, n, k, nnz, lam_err = wl["engine"], wl["n"], wl["k"], wl["nnz"], wl["lam_err"]
    x_feats, U_norm, edge_all, adj_dev = wl["x_feats"], [wl["U_norm"]], wl["edge_index"], wl["adjacency"]
    device_built = adj_dev is not None
    d_in = eng.h.shape[1]
    flops_v = mlp_flops_per_vertex(d_in, HIDDEN, k)
    epoch0 = 2500                                            # mid-ramp: correction scale 5.0, non-zero gradients
    peaks = measured_peaks()

    m = timed_steps(eng, args, dev, rank, world, epoch0, ClockSampler(local_rank) if rank == 0 else None)
    ms_step, phase = m["ms_step"], m["phase"]

    # ---- kernels timed alone (burst peaks apply): dual SpMM, forward chain of the MLP
    pair = eng.pairs[-1]
    s = eng._level_slices(len(eng.pairs) - 1)
    spmm_ms = time_call(lambda: ops.spmm2(pair, eng.U_pred[s], out_K=eng.KU[s], out_M=eng.MU[s]))
    n_loc = pair.n
    spmm_bytes = 12 * pair.K.nnz + 4 * (n_loc + 1) + 12 * n_loc * k
    chain_ms, chain_bytes, chain_flops = None, 0, 0
    if args.mlp_mode == "bf16" and getattr(eng.mlp, "chain_fwd", False):
        mm = eng.mlp
        chain_ms = time_call(lambda: mm.forward(eng.h, U_base=eng.U_base, scale=5.0, U_pred=eng.U_pred))
        pw_ms = time_call(mm._pack_weights)                 # forward() re-packs the weights first: subtract that launch group
        chain_ms -= pw_ms
        n_rows = mm.n
        # algorithmic bytes: packed input read, every hidden activation + ReLU mask written once, U_base read, U_pred written
        chain_bytes = n_rows * (2 * mm.pd[0] + sum(2 * w + w // 8 for w in mm.pd[1:-1]) + 8 * k)
        chain_flops = 2.0 * n_rows * sum(mm.dims[i] * mm.dims[i + 1] for i in range(mm.L))

    # ---- samplers at BASELINE config 3 size (1 M-point cloud): FPS iterations and one voxel hierarchy
    samplers_info = None
    if world == 1 and not args.no_samplers:
        sampling = pkg("sampling")
        cloud = torch.from_numpy(np.random.default_rng(1234).standard_normal((1_000_000, 3))).to(dev)
        sampling.fps_order(cloud, 64, 7)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sampling.fps_order(cloud, 1024, 7)
        torch.cuda.synchronize()
        fps_ms = (time.perf_counter() - t0) * 1e3
        sampling.voxel_levels(cloud, [256, 512, 1024])          # warm-up (kernel loading, workspace), like the FPS call above
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sampling.voxel_levels(cloud, [256, 512, 1024])
        vox_ms = (time.perf_counter() - t0) * 1e3
        samplers_info = {"points": 1000000, "fps_1024_samples_ms": fps_ms, "fps_us_per_iteration": fps_ms * 1e3 / 1023,
                         "voxel_hierarchy_256_512_1024_ms": vox_ms,
                         "reference_cpu": "43.4 ms per FPS iteration, 1.25 s per voxel level (SURVEY 6, 8 cores)"}
        del cloud

    # ---- host issue time (how long Python + ctypes take to enqueue one step)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(5):
        eng.step(epoch0 + i)
    host_issue_ms = (time.perf_counter() - t0) / 5 * 1e3
    torch.cuda.synchronize()

    # ---- end to end through the public host-fed API: every step uploads its inputs (node features x and the base
    # subspace U_base) from pinned host memory and returns the loss to the host
    e2e = None
    if world == 1 and not args.no_e2e:
        engine_mod = pkg("engine")
        sparse = pkg("sparse")
        adj = adj_dev if device_built else sparse.CsrMatrix.from_edge_index(edge_all, n, dev)
        pipe = engine_mod.HostFedPipeline(eng, lambda x, out: ops.neighbor_mean_concat(x, adj, out=out))
        x_host = x_feats.detach().cpu().pin_memory()
        ub_host = U_norm[0].detach().cpu().pin_memory()
        prev = pipe.submit(x_host, ub_host, epoch0)
        for i in range(1, 3):
            cur = pipe.submit(x_host, ub_host, epoch0 + i)
            pipe.result(prev)
            prev = cur
        pipe.result(prev)
        torch.cuda.synchronize()
        n_e2e = max(args.steps, int(np.ceil(MIN_TIMED_MS / max(ms_step * 1.5, 1e-3))))
        t0 = time.perf_counter()
        prev = pipe.submit(x_host, ub_host, epoch0)
        e2e_loss = None
        for i in range(1, n_e2e + 1):
            cur = pipe.submit(x_host, ub_host, epoch0 + i) if i < n_e2e else None
            e2e_loss = pipe.result(prev)
            prev = cur
        dt = (time.perf_counter() - t0) / n_e2e
        e2e = {"value": 1.0 / dt, "unit": "steps/s", "h2d_bytes_per_step": int(pipe.h2d_bytes),
               "d2h_bytes_per_step": int(pipe.d2h_bytes), "ms_per_step": dt * 1e3, "steps_timed": n_e2e,
               "api": "engine.HostFedPipeline.submit/result (x_feats + U_base uploaded from pinned host memory every "
                      "step, aggregation + packing on the device, six loss terms read back)",
               "loss": float(e2e_loss[5])}
        del pipe, x_host, ub_host

    # ---- CPU baseline beside it: the oracle on the SAME workload (bounded: 1 warm-up + 3 timed steps), rank 0, N = 1
    cpu = None
    if not args.no_cpu_baseline and world == 1 and rank == 0:
        host = wl["host"] if wl["host"] is not None else build_host_workload(reference_workload_name(args))
        r = time_oracle(host, 3, 1, threads=os.cpu_count())
        cpu = {"value": r["steps_per_s"], "unit": "steps/s", "cores": r["threads"], "kind": "port",
               "sample": "oracle/step_port.py on the %s workload (%d vertices), 3 timed steps of %.0f ms after 1 warm-up, "
                         "wall clock" % (args.workload if wl["host"] is not None else reference_workload_name(args),
                                         r["vertices"], r["ms_per_step"])}

    # ---- accuracy of a trained run (BASELINE "lambda rel err"), small enough to train inside the benchmark
    trained = None
    if world == 1 and rank == 0 and not args.no_trained:
        try:
            trained = trained_accuracy(args.mlp_mode)
        except Exception as exc:
            trained = {"error": repr(exc)[:300]}

    # ---- BASELINE config 5 (north star): 16 M-vertex torus, k = 64, same engine, same number of GPUs
    torus = None
    if not args.no_torus and args.workload != "torus16m":
        del eng, wl, x_feats, U_norm, m["phase"]
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        try:
            twl = build_engine(args, dev, rank, world, workload="torus16m")
            targs = argparse.Namespace(**vars(args))
            targs.steps, targs.warmup = max(3, min(args.steps, 10)), 3
            tm = timed_steps(twl["engine"], targs, dev, rank, world, epoch0)
            torus = {"workload": "torus16m", "vertices": twl["n"], "k": twl["k"], "ms_per_step": tm["ms_step"],
                     "steps_per_s": 1000.0 / tm["ms_step"], "timed_steps": tm["n_timed"], "phase_ms": tm["phase"],
                     "loss": tm["loss"], "n_gpus": world, "scaling": "strong",
                     "mlp_tflops": mlp_flops_per_vertex(twl["engine"].h.shape[1], HIDDEN, twl["k"]) * twl["n"] / world /
                                   ((tm["phase"].get("mlp_fwd", 0) + tm["phase"].get("mlp_bwd", 0)) * 1e-3) / 1e12}
            del twl
        except Exception as exc:                                   # e.g. not enough memory: say so, keep the headline
            torus = {"workload": "torus16m", "error": repr(exc)[:300]}
    ms_phase = phase

    def finish():
        """Multi-rank exit: tearing the NCCL communicator down while captured graphs still reference it can block
        for minutes, so the ranks synchronise and leave without the orderly shutdown."""
        sys.stdout.flush()
        sys.stderr.flush()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
            os._exit(0)

    if rank != 0:
        finish()
        return
    mlp_ms = ms_phase.get("mlp_fwd", 0.0) + ms_phase.get("mlp_bwd", 0.0)
    n_global = n
    tflops = flops_v * n_global / world / (mlp_ms * 1e-3) / 1e12 if mlp_ms > 0 else 0.0
    eager_ms = sum(ms_phase.values())
    shares = {p: v / eager_ms for p, v in ms_phase.items()} if eager_ms > 0 else {}
    mlp_roof = {"bound": "tensor", "kernel": "corrector MLP forward + backward, all layers (%s)" % args.mlp_mode,
                "achieved": tflops, "peak": peaks["bf16_sustained"], "unit": "TFLOP/s",
                "frac": tflops / peaks["bf16_sustained"], "frac_of_burst_peak": tflops / peaks["bf16_burst"],
                "peak_source": peaks["source"] + " bf16 sustained (kernels timed inside the >= 1 s step loop)",
                "ms_per_step": mlp_ms, "flop_per_vertex": flops_v, "share_of_step": shares.get("mlp_fwd", 0) + shares.get("mlp_bwd", 0)}
    if chain_ms is not None:
        gbs = chain_bytes / (chain_ms * 1e-3) / 1e9
        roofline = {"bound": "hbm",
                    "kernel": "tc_chain2_kernel<FWD> (tcgen05 cta_group::2: all %d layers of the corrector, persistent CTA pairs, two "
                              "128-vertex tiles per CTA in ping-pong; activations + ReLU masks streamed to HBM once, never read "
                              "back)" % eng_layers(d_in, k),
                    "achieved": gbs, "peak": peaks["hbm"], "unit": "GB/s", "frac": gbs / peaks["hbm"],
                    "traffic": NCU_TRAFFIC_CHAIN_FWD_PER_VERTEX * n_loc,
                    "peak_source": peaks["source"] + " hbm copy (kernel timed alone)", "ms": chain_ms,
                    "bytes_per_launch": chain_bytes, "launches_per_step": 1, "share_of_step": chain_ms / ms_step,
                    "arithmetic_intensity_flop_per_byte": chain_flops / chain_bytes,
                    "tflops_this_kernel": chain_flops / (chain_ms * 1e-3) / 1e12,
                    "frac_of_tensor_burst_peak": chain_flops / (chain_ms * 1e-3) / 1e12 / peaks["bf16_burst"],
                    "why_hbm": "AI = %.0f flop/B is below the ridge %.0f flop/B of the measured peaks"
                               % (chain_flops / chain_bytes, peaks["bf16_burst"] * 1e3 / peaks["hbm"])}
    else:
        roofline = dict(mlp_roof, traffic=None)
    spmm_gbs = spmm_bytes / (spmm_ms * 1e-3) / 1e9
    spmm_roof = {"bound": "hbm", "kernel": "ep_spmm2_csr_f32 (K U and M U, shared pattern)", "achieved": spmm_gbs,
                 "peak": peaks["hbm"], "unit": "GB/s", "frac": spmm_gbs / peaks["hbm"], "ms": spmm_ms,
                 "bytes_per_launch": spmm_bytes, "traffic": NCU_TRAFFIC_SPMM2_PER_VERTEX * n_loc,
                 "share_of_step": spmm_ms / ms_step}
    line = {"metric": "train_steps_per_s", "value": 1000.0 / ms_step, "unit": "steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32" if args.mlp_mode == "fp32" else "bf16",
            "data": "synthetic",
            "config": {"workload": args.workload, "vertices": n_global, "k": k, "hidden": HIDDEN, "mlp_in": d_in,
                       "nnz_per_operator": int(nnz), "mlp_mode": args.mlp_mode, "levels": 1,
                       "parallelism": "vertex-shard x%d" % world, "cuda_graph": bool(args.no_graph is False),
                       "l2": "inputs larger than L2 (U, KU, MU, activations >> 126 MB)",
                       "timed_region": "%d steps x %d repeats = %d steps, %.0f ms; loss read back every step with a "
                                       "delay of one step" % (args.steps, m["repeats"], m["n_timed"], m["timed_ms"])},
            "timed_steps": m["n_timed"], "clocks": m["clocks"], "gpu_launches": m["launches"],
            "launches_per_step_by_entry": m["launches_by_entry"], "e2e": e2e, "roofline": roofline,
            "mlp_roofline": mlp_roof, "spmm_roofline": spmm_roof, "cpu_baseline": cpu, "samplers": samplers_info,
            "phase_ms": ms_phase, "phase_share_of_eager_step": shares, "host_issue_ms": host_issue_ms,
            "loss": m["loss"], "lambda_rel_err_rayleigh_ritz": lam_err, "lambda_rel_err_trained": trained,
            "north_star_torus16m": torus}
    print(json.dumps(line))
    finish()


def eng_layers(d_in, k):
    return len(HIDDEN) + 1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="icosphere1m", choices=sorted(WORKLOADS))
    ap.add_argument("--mlp-mode", default=os.environ.get("EP_MLP_MODE", "bf16"), choices=["fp32", "bf16"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-samplers", action="store_true")
    ap.add_argument("--no-torus", action="store_true", help="skip the 16 M-vertex torus block (BASELINE config 5)")
    ap.add_argument("--no-trained", action="store_true", help="skip the small trained-accuracy run")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of replaying a CUDA graph")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
