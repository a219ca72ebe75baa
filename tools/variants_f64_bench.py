"""fp64 against fp32 kernels of the notebook variants on the 998,562-vertex icosphere (synthetic.icosphere(316) plus the
FEM operators); prints one JSON line (and writes it to --out).

    python tools/variants_f64_bench.py [--out FILE] [--min-seconds 1.0] [--rounds 2]

Items, each timed with CUDA events over a region of at least --min-seconds, fp64 and fp32 alternating in one process:
  spmm2            K U, M U at k = 32; achieved bytes/s from the algorithmic bytes
                   fp64 20 nnz + 4 (n+1) + 24 n k,  fp32 12 nnz + 4 (n+1) + 12 n k
  eigen_partials   k = 50; algorithmic bytes 24 n k (fp64), 12 n k (fp32)
  layers           linear_fwd + linear_bwd of the notebook network 3 -> 256 -> 256 -> 128 -> 50 over all vertices,
                   also torch fp64 on the same GPU (torch.nn.functional.linear and matmuls; reported, not a target)
  train_step       one step of CoordinateMLP + whitened_subspace_loss (k = 50) + Adam, in fp64 kernels, fp32 kernels
                   and torch fp64 (torch.sparse.mm + dense); steps/s
The card name, power limit and SM clocks are read with nvidia-smi in the same run."""
import argparse
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def pkg(name):
    return importlib.import_module("eigen-pinns_b200." + name)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [s.strip() for s in out.split(",")]))
    except (OSError, subprocess.SubprocessError):
        return {"nvidia-smi": "unavailable"}


def timed(fn, min_seconds):
    """Seconds per call: warm-up, then a CUDA-event-timed region of >= min_seconds."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    reps = 1
    while True:
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for _ in range(reps):
            fn()
        stop.record()
        stop.synchronize()
        sec = start.elapsed_time(stop) / 1e3
        if sec >= min_seconds:
            return sec / reps
        reps = max(reps * 2, int(reps * 1.2 * min_seconds / max(sec, 1e-6)) + 1)


def alternate(variants, min_seconds, rounds):
    """{name: best seconds per call} over `rounds` alternating passes through the variants."""
    best = {}
    for _ in range(rounds):
        for name, fn in variants.items():
            t = timed(fn, min_seconds)
            best[name] = min(best.get(name, t), t)
    return best


def torch_whitened_loss(U, Kt, Mt):
    """whitened_subspace_loss with torch.sparse.mm for the two products (default weights)."""
    k = U.shape[1]
    A, B = U.t() @ torch.sparse.mm(Kt, U), U.t() @ torch.sparse.mm(Mt, U)
    eye = torch.eye(k, dtype=B.dtype, device=B.device)
    V, S, _ = torch.linalg.svd(B)
    W = V @ torch.diag_embed(1.0 / torch.sqrt(torch.clamp(S, min=1e-7))) @ V.t()
    R = W @ A @ W
    e, _ = torch.sort(torch.diagonal(R))
    eig_loss = (100.0 * e[0] ** 2 + 5.0 * e[1:].sum() / (k - 1) + 2.0 * torch.relu(1e-4 - (e[1:] - e[:-1])).sum() / (k - 1)
                + ((R * (1 - eye)) ** 2).sum() / (k * (k - 1)))
    orth = torch.linalg.norm(W @ B @ W - eye) ** 2
    ordering = torch.relu(e[:-1] - e[1:]).sum() / k
    stability = torch.relu(S.max() / (S.min() + 1e-10) - 1e3) / 1e3
    return eig_loss + orth + 0.05 * ordering + 0.1 * stability


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--freq", type=int, default=316)
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "variants_f64_bench measures on a GPU"
    dev = torch.device("cuda", 0)
    info_before = gpu_info()
    ep = importlib.import_module("eigen-pinns_b200")
    ep.require_library()
    ops, sparse, variants, fem, syn = pkg("ops"), pkg("sparse"), pkg("variants"), pkg("fem"), pkg("synthetic")
    from oracle import variants_port as vp

    verts, tris = syn.icosphere(args.freq)
    verts = fem.normalize_verts(verts)
    K, M = fem.assemble_stiffness_mass(verts, tris)
    n, nnz = K.shape[0], K.nnz
    pairs = {dt: sparse.OperatorPair(K, M, dev, dtype=dt) for dt in (torch.float64, torch.float32)}
    rng = np.random.default_rng(0)
    res = {"workload": "icosphere(%d)" % args.freq, "n": n, "nnz": int(nnz), "min_seconds": args.min_seconds,
           "rounds": args.rounds}

    # ---- spmm2, k = 32
    k = 32
    X = {dt: torch.from_numpy(rng.standard_normal((n, k))).to(dev, dt) for dt in pairs}
    outs = {dt: (torch.empty_like(X[dt]), torch.empty_like(X[dt])) for dt in pairs}
    t = alternate({"f64": lambda: ops.spmm2(pairs[torch.float64], X[torch.float64], *outs[torch.float64]),
                   "f32": lambda: ops.spmm2(pairs[torch.float32], X[torch.float32], *outs[torch.float32])},
                  args.min_seconds, args.rounds)
    b64, b32 = 20 * nnz + 4 * (n + 1) + 24 * n * k, 12 * nnz + 4 * (n + 1) + 12 * n * k
    res["spmm2_k32"] = {"f64_ms": t["f64"] * 1e3, "f32_ms": t["f32"] * 1e3, "f64_GBps": b64 / t["f64"] / 1e9,
                        "f32_GBps": b32 / t["f32"] / 1e9, "f64_over_f32_bandwidth": (b64 / t["f64"]) / (b32 / t["f32"])}
    del X, outs

    # ---- eigen_partials, k = 50
    k = 50
    T3 = {dt: [torch.from_numpy(rng.standard_normal((n, k))).to(dev, dt) for _ in range(3)] for dt in pairs}
    P = {dt: torch.empty(k * k + 5 * k, dtype=torch.float64, device=dev) for dt in pairs}
    t = alternate({"f64": lambda: ops.eigen_partials(*T3[torch.float64], out=P[torch.float64]),
                   "f32": lambda: ops.eigen_partials(*T3[torch.float32], out=P[torch.float32])},
                  args.min_seconds, args.rounds)
    res["eigen_partials_k50"] = {"f64_ms": t["f64"] * 1e3, "f32_ms": t["f32"] * 1e3,
                                 "f64_GBps": 24 * n * k / t["f64"] / 1e9, "f32_GBps": 12 * n * k / t["f32"] / 1e9,
                                 "f64_over_f32_time": t["f64"] / t["f32"]}
    del T3, P

    # ---- dense layers 3 -> 256 -> 256 -> 128 -> 50, forward + backward over all vertices
    widths = [3, 256, 256, 128, 50]
    layers = {}
    for dt in pairs:
        g = torch.Generator().manual_seed(1)
        Ws = [(torch.randn(o, i, generator=g) / np.sqrt(i)).to(dev, dt) for i, o in zip(widths[:-1], widths[1:])]
        bs = [torch.zeros(o, device=dev, dtype=dt) for o in widths[1:]]
        acts = [torch.from_numpy(verts).to(dev, dt)] + [torch.empty(n, w, device=dev, dtype=dt) for w in widths[1:]]
        grads = [torch.empty(n, w, device=dev, dtype=dt) for w in widths]
        grads[-1].normal_()
        layers[dt] = (Ws, bs, acts, grads)

    def kernels(dt):
        Ws, bs, acts, grads = layers[dt]

        def run():
            for li in range(4):
                ops.linear_fwd(acts[li], Ws[li], bs[li], False, out=acts[li + 1])
            for li in reversed(range(4)):
                ops.linear_bwd(acts[li], Ws[li], grads[li + 1], li > 0, relu_mask=False,
                               dX=grads[li] if li > 0 else None)
        return run

    def torch_layers():
        Ws, bs, acts, grads = layers[torch.float64]
        F = torch.nn.functional
        for li in range(4):
            acts[li + 1] = F.linear(acts[li], Ws[li], bs[li])
        for li in reversed(range(4)):
            if li > 0:
                grads[li] = grads[li + 1] @ Ws[li]
            _ = grads[li + 1].t() @ acts[li], grads[li + 1].sum(0)

    t = alternate({"f64": kernels(torch.float64), "f32": kernels(torch.float32), "torch_f64": torch_layers},
                  args.min_seconds, args.rounds)
    flops = sum(2 * n * i * o * (3 if li > 0 else 2) for li, (i, o) in enumerate(zip(widths[:-1], widths[1:])))
    res["layers_3_256_256_128_50"] = {"f64_ms": t["f64"] * 1e3, "f32_ms": t["f32"] * 1e3,
                                      "torch_f64_ms": t["torch_f64"] * 1e3, "f64_over_f32_time": t["f64"] / t["f32"],
                                      "f64_TFLOPs": flops / t["f64"] / 1e12, "f32_TFLOPs": flops / t["f32"] / 1e12,
                                      "torch_f64_TFLOPs": flops / t["torch_f64"] / 1e12}
    del layers

    # ---- one training step: CoordinateMLP + whitened_subspace_loss (k = 50) + Adam
    Kn, Mn, _, _ = variants.frobenius_normalised(K, M)
    wpairs = {dt: sparse.OperatorPair(Kn, Mn, dev, dtype=dt) for dt in pairs}
    Xv = {dt: torch.from_numpy(verts).to(dev, dt) for dt in pairs}
    torch.manual_seed(0)
    ref_net = vp.CoordinateMLP(3, 50, (256, 256, 128), "silu").double()
    steps = {}
    for dt, name in ((torch.float64, "f64"), (torch.float32, "f32")):
        net = variants.CoordinateMLP(3, 50, (256, 256, 128), "silu").to(dev, dt)
        net.load_state_dict(ref_net.state_dict())
        opt = torch.optim.Adam(net.parameters(), lr=1e-4)

        def step(net=net, opt=opt, dt=dt):
            opt.zero_grad()
            loss, _, _ = variants.whitened_subspace_loss(net(Xv[dt]), wpairs[dt])
            loss.backward()
            opt.step()
        steps[name] = step
    tnet = vp.CoordinateMLP(3, 50, (256, 256, 128), "silu").double().to(dev)
    tnet.load_state_dict(ref_net.state_dict())
    topt = torch.optim.Adam(tnet.parameters(), lr=1e-4)
    Kt, Mt = vp.to_torch_sparse(Kn).to(dev), vp.to_torch_sparse(Mn).to(dev)

    def torch_step():
        topt.zero_grad()
        torch_whitened_loss(tnet(Xv[torch.float64]), Kt, Mt).backward()
        topt.step()
    steps["torch_f64"] = torch_step
    t = alternate(steps, args.min_seconds, args.rounds)
    res["train_step_k50"] = {name + "_steps_per_s": 1.0 / sec for name, sec in t.items()}
    res["train_step_k50"].update({name + "_ms": sec * 1e3 for name, sec in t.items()})

    res["gpu_before"], res["gpu_after"] = info_before, gpu_info()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
