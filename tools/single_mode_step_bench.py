"""Training steps per second of the single-mode eigenfunction network (delta_pinns_validation/
iterative_eigenvalues_on_cloud.ipynb cell 1) on three paths, alternating in one process; prints one JSON line (and
writes it to --out).

    python tools/single_mode_step_bench.py [--out FILE] [--min-seconds 1.0] [--rounds 2] [--freq 316]

Paths, each step = network forward, loss, backward, Adam(betas=(0.999, 0.9999)):
  autograd   variants.EigenfunctionNN + variants.single_mode_loss + loss.backward() + torch.optim.Adam (what the library
             offered before single_mode.SingleModeTrainer; the layers and SpMMs already run on its kernels)
  eager      SingleModeTrainer.step(), eager launches
  graph      SingleModeTrainer.step() replayed as one CUDA graph
Workloads: the bunny of tests/golden/bunny_fem.npz (N = 2503, the operators K_*, M_* and verts), hidden 64 and 128,
P = 0 and 9 earlier modes, fp32 and fp64; the 998,562-vertex icosphere(316) (FEM K, M of the normalised sphere) at
hidden 128, P = 9, where the layer GEMMs dominate.  Times are CUDA-event times over a region of at least --min-seconds
per path (host-bound paths included: the events bracket everything the host enqueued); it/s = 1 / time per step.
The earlier modes are fixed random vectors: the step's cost does not depend on their values.
The reference publishes 360-490 it/s for this network on the bunny (hidden 128, fp32) on a GPU it does not name; that
range is written beside the results as a number of unknown hardware.
The card name, power limit and SM clocks are read with nvidia-smi in the same run."""
import argparse
import importlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))


def pkg(name):
    return importlib.import_module("eigen-pinns_b200." + name)


def autograd_step(net, X, pair, prev, opt):
    v = pkg("variants")

    def step():
        opt.zero_grad(set_to_none=True)
        u, lam = net(X)
        v.single_mode_loss(u, lam, pair, prev)[0].backward()
        opt.step()
    return step


def measure(name, verts, K, M, hidden, P, dtype, dev, args, alternate):
    sparse, v, sm, cabi = pkg("sparse"), pkg("variants"), pkg("single_mode"), pkg("_cabi")
    pair = sparse.OperatorPair(K, M, dev, dtype=dtype)
    n = pair.n
    X = torch.from_numpy(np.ascontiguousarray(verts)).to(device=dev, dtype=dtype)
    gen = torch.Generator().manual_seed(1)
    prev = [(torch.randn(n, 1, generator=gen, dtype=torch.float64) / n ** 0.5).to(device=dev, dtype=dtype)
            for _ in range(P)]
    torch.manual_seed(0)
    base = v.EigenfunctionNN(hidden, 3, initial_eigenvalue=1.0).to(device=dev, dtype=dtype)
    net_a = v.EigenfunctionNN(hidden, 3).to(device=dev, dtype=dtype)
    net_a.load_state_dict(base.state_dict())
    opt = torch.optim.Adam(net_a.parameters(), lr=args.lr, betas=(0.999, 0.9999), eps=1e-8)
    tr_e = sm.SingleModeTrainer(base, X, pair, previous=prev, lr=args.lr)
    net_g = v.EigenfunctionNN(hidden, 3).to(device=dev, dtype=dtype)
    net_g.load_state_dict(base.state_dict())
    tr_g = sm.SingleModeTrainer(net_g, X, pair, previous=prev, lr=args.lr)
    before = cabi.launch_counter
    tr_g.step()
    launches = cabi.launch_counter - before
    tr_g.enable_graph()
    tr_g.step()
    t = alternate({"autograd": autograd_step(net_a, X, pair, prev, opt), "eager": tr_e.step, "graph": tr_g.step},
                  args.min_seconds, args.rounds)
    res = {"workload": name, "n": n, "dtype": str(dtype).replace("torch.", ""), "hidden": hidden, "P": P,
           "launches_per_step": launches}
    for k_, sec in t.items():
        res[k_ + "_ms"] = sec * 1e3
        res[k_ + "_it_per_s"] = 1.0 / sec
    res["graph_vs_autograd"] = t["autograd"] / t["graph"]
    res["eager_vs_autograd"] = t["autograd"] / t["eager"]
    print(json.dumps(res), file=sys.stderr)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--freq", type=int, default=316)
    ap.add_argument("--lr", type=float, default=1e-4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "single_mode_step_bench measures on a GPU"
    from variants_f64_bench import gpu_info, alternate
    from conftest import load_golden, csr_from_golden
    fem, syn = pkg("fem"), pkg("synthetic")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    info_before = gpu_info()
    g = load_golden("bunny_fem.npz")
    n = g["verts"].shape[0]
    K, M = csr_from_golden(g, "K", n), csr_from_golden(g, "M", n)
    results = []
    for dtype in (torch.float32, torch.float64):
        for hidden in (64, 128):
            for P in (0, 9):
                results.append(measure("bunny", g["verts"], K, M, hidden, P, dtype, dev, args, alternate))
    verts, tris = syn.icosphere(args.freq)
    verts = fem.normalize_verts(verts)
    Ki, Mi = fem.assemble_stiffness_mass(verts, tris)
    for dtype in (torch.float32, torch.float64):
        results.append(measure("icosphere(%d)" % args.freq, verts, Ki, Mi, 128, 9, dtype, dev, args, alternate))
        torch.cuda.empty_cache()
    out = {"min_seconds": args.min_seconds, "rounds": args.rounds, "lr": args.lr,
           "reference": {"it_per_s": [360, 490], "workload": "bunny, N = 2503, hidden 128, fp32",
                         "hardware": "unknown (the reference does not name its GPU)"},
           "results": results, "gpu_before": info_before, "gpu_after": gpu_info()}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
