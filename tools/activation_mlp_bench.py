"""Activation epilogues in the layer kernels (ops.mlp_act) against the composition they replace, on the 998,562 vertices
of synthetic.icosphere(316); prints one JSON line (and writes it to --out).

    python tools/activation_mlp_bench.py [--out FILE] [--min-seconds 1.0] [--rounds 3]

Items, each timed with CUDA events over a region of at least --min-seconds after a warm-up, fused and composed
alternating in one process, fp32 and fp64:
  coordinate_mlp   CoordinateMLP(3, 50, (256, 256, 128), "silu") on the vertex coordinates: forward alone (autograd
                   recording, as in training) and forward + backward of sum(out * R)
                   fused:    CoordinateMLP.forward = ops.mlp_act, SiLU in the GEMM epilogues
                   composed: the same modules applied one by one, net.net(x): KernelLinear (ops.linear) and torch
                             nn.SiLU through autograd
  eigenfunction_nn EigenfunctionNN(64): forward + backward of sum(u * R) + lambda
                   fused:    EigenfunctionNN.forward (lambda folded into the biases, ops.mlp_act with sin)
                   composed: torch.cat([h, lambda]) before each KernelLinear, torch.sin between them
The working set (activations of 998,562 rows) is far larger than the 126 MB L2.  Outputs of the two versions are
compared on the same weights (max relative difference, reported).  The card name, power limit and SM clocks are read
with nvidia-smi in the same run."""
import argparse
import importlib
import json
import os
import subprocess
import sys

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
    """{name: [seconds per call of each round]} over `rounds` alternating passes through the variants."""
    times = {name: [] for name in variants}
    for _ in range(rounds):
        for name, fn in variants.items():
            times[name].append(timed(fn, min_seconds))
    return times


def summary(times):
    """ms per call: best and spread (max - min) over the rounds, and fused / composed of the best."""
    out = {}
    for name, t in times.items():
        out[name + "_ms"] = min(t) * 1e3
        out[name + "_spread_ms"] = (max(t) - min(t)) * 1e3
    out["fused_over_composed"] = min(times["fused"]) / min(times["composed"])
    return out


def rel(a, b):
    return ((a - b).abs().max() / b.abs().max()).item()


def composed_eigenfunction(net, x):
    """EigenfunctionNN.forward as it was built before the activation epilogues: n x (d + 1) concatenations, KernelLinear
    layers and torch.sin."""
    eigenvalue = torch.abs(net.eigenvalue_layer.weight).reshape(1, 1)
    lam = eigenvalue.expand(x.shape[0], 1)
    h = torch.sin(net.fc1(torch.cat([x, lam], dim=1)))
    h = torch.sin(net.fc2(torch.cat([h, lam], dim=1)))
    h = torch.sin(net.fc3(torch.cat([h, lam], dim=1)))
    return net.fc4(torch.cat([h, lam], dim=1)), eigenvalue


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--freq", type=int, default=316)
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "activation_mlp_bench measures on a GPU"
    dev = torch.device("cuda", 0)
    info_before = gpu_info()
    ep = importlib.import_module("eigen-pinns_b200")
    ep.require_library()
    variants, fem, syn = pkg("variants"), pkg("fem"), pkg("synthetic")
    verts, _ = syn.icosphere(args.freq)
    verts = fem.normalize_verts(verts)
    n = verts.shape[0]
    res = {"workload": "icosphere(%d) vertex coordinates" % args.freq, "n": n, "min_seconds": args.min_seconds,
           "rounds": args.rounds}

    for dt, name in ((torch.float32, "f32"), (torch.float64, "f64")):
        x = torch.from_numpy(verts).to(dev, dt)
        torch.manual_seed(0)
        net = variants.CoordinateMLP(3, 50, (256, 256, 128), "silu").to(dev, dt)
        R = torch.randn(n, 50, device=dev, dtype=dt)
        params = list(net.parameters())

        def fwd(f):
            def run():
                f(x)
            return run

        def fwd_bwd(f):
            def run():
                for p in params:
                    p.grad = None
                (f(x) * R).sum().backward()
            return run
        with torch.no_grad():
            diff = rel(net(x), net.net(x))
        t_f = alternate({"fused": fwd(net), "composed": fwd(net.net)}, args.min_seconds, args.rounds)
        t_fb = alternate({"fused": fwd_bwd(net), "composed": fwd_bwd(net.net)}, args.min_seconds, args.rounds)
        res["coordinate_mlp_silu_" + name] = {"forward": summary(t_f), "forward_backward": summary(t_fb),
                                              "fused_vs_composed_output_rel_diff": diff}
        del net, R, x

        x = torch.from_numpy(verts).to(dev, dt)
        torch.manual_seed(1)
        enet = variants.EigenfunctionNN(64, 3, initial_eigenvalue=0.7).to(dev, dt)
        Ru = torch.randn(n, 1, device=dev, dtype=dt)
        eparams = list(enet.parameters())

        def estep(f):
            def run():
                for p in eparams:
                    p.grad = None
                u, lam = f(enet, x)
                ((u * Ru).sum() + lam.sum()).backward()
            return run
        with torch.no_grad():
            diff = rel(enet(x)[0], composed_eigenfunction(enet, x)[0])
        t = alternate({"fused": estep(lambda m, xx: m(xx)), "composed": estep(composed_eigenfunction)},
                      args.min_seconds, args.rounds)
        res["eigenfunction_nn_64_" + name] = {"forward_backward": summary(t), "fused_vs_composed_output_rel_diff": diff}
        del enet, Ru, x
        torch.cuda.empty_cache()

    res["gpu_before"], res["gpu_after"] = info_before, gpu_info()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
