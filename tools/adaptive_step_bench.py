"""Cost of the AdaptiveCorrector options in the fused training step on the 998,562-vertex icosphere (k = 32, corrector
82 -> 256 x 6 -> 32), bf16 and fp32 MLP modes; prints one JSON line (and writes it to --out).

    python tools/adaptive_step_bench.py [--out FILE] [--min-seconds 1.0] [--rounds 2]

Items, each timed with CUDA events over a region of at least --min-seconds, the variants alternating in one process:
  step      per-step phases (mlp_fwd, loss_fwd, loss_bwd, mlp_bwd, optim; eager launches with events between the phases)
            and the whole step as a replayed CUDA graph, for
              plain        no per-mode scales, w_smooth_corr = 0 (the path bench.py times)
              scales       per-mode scales (ep_mode_scale_fwd_f32 / ep_mode_scale_bwd_f32 on top of the plain step)
              scales_sc    per-mode scales and w_smooth_corr != 0 (plus K c per level: one ep_spmm_csr_f32)
            The three engines share the input, the operators and the initial weights.
  kernels   ep_mode_scale_fwd_f32 and ep_mode_scale_bwd_f32 (with K c, with scales) alone; achieved bytes/s from the
            bytes the algorithm moves: forward reads c and U_base, writes U_pred (12 n k); backward reads c, g and K c,
            writes dc (16 n k); and that rate over the 7.7 TB/s HBM3e data-sheet bandwidth of one B200.
The card name, power limit and SM clocks are read with nvidia-smi in the same run."""
import argparse
import importlib
import json
import os
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

HBM_BYTES_PER_S = 7.7e12
PHASES = ("mlp_fwd", "loss_fwd", "loss_bwd", "mlp_bwd", "optim")


def pkg(name):
    return importlib.import_module("eigen-pinns_b200." + name)


def variant_engine(base, mode_scales, w_smooth_corr):
    """A TrainStepEngine on the inputs of `base` with fresh copies of its initial weights."""
    engine = pkg("engine")
    p = base.params
    params = engine.FlatParams([w.detach().clone() for w in p.W], [b.detach().clone() for b in p.b], base.dev,
                               mode_scales=mode_scales)
    cfg = engine.StepConfig(**dict(vars(base.cfg), w_smooth_corr=w_smooth_corr))
    return engine.TrainStepEngine(base.h, base.U_base, base.pairs, base.offsets, params, cfg,
                                  lam_target=base.lam_target, mlp_mode=base.mlp_mode)


def phase_times(eng, epoch, min_seconds):
    """Mean ms per phase over eager steps with events between the phases (>= min_seconds of steps)."""
    eng.use_graph = False
    for _ in range(3):
        eng.step(epoch)
    torch.cuda.synchronize()
    sums, steps, total = dict.fromkeys(PHASES, 0.0), 0, 0.0
    while total < min_seconds * 1e3:
        marks = []
        eng.step(epoch, marks=marks)
        marks[-1][1].synchronize()
        for (_, a), (name, b) in zip(marks[:-1], marks[1:]):
            ms = a.elapsed_time(b)
            sums[name] += ms
            total += ms
        steps += 1
    return {k: v / steps for k, v in sums.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--workload", default="icosphere1m")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "adaptive_step_bench measures on a GPU"
    from variants_f64_bench import gpu_info, alternate
    import bench
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    info_before = gpu_info()
    ops = pkg("ops")
    res = {"workload": args.workload, "min_seconds": args.min_seconds, "rounds": args.rounds}
    epoch = 2500
    for mlp_mode in ("bf16", "fp32"):
        built = bench.build_engine(types.SimpleNamespace(workload=args.workload, mlp_mode=mlp_mode), dev, 0, 1)
        plain = built["engine"]
        n, k = built["n"], built["k"]
        res.update(n=n, k=k, hidden=bench.HIDDEN, mlp_in=plain.params.dims[0])
        scales = torch.linspace(0.5, 1.5, k)
        engines = {"plain": variant_engine(plain, None, 0.0), "scales": variant_engine(plain, scales, 0.0),
                   "scales_sc": variant_engine(plain, scales, 1.0)}
        del plain, built
        out = {}
        phases = {}
        for _ in range(args.rounds):
            for name, eng in engines.items():
                t = phase_times(eng, epoch, args.min_seconds)
                phases[name] = t if name not in phases else {p: min(phases[name][p], t[p]) for p in PHASES}
        for eng in engines.values():
            eng.enable_graph()
            eng.step(epoch)
        graph = alternate({name: (lambda e=eng: e.step(epoch)) for name, eng in engines.items()},
                          args.min_seconds, args.rounds)
        for name in engines:
            out[name] = {"graph_step_ms": graph[name] * 1e3, "phases_ms": phases[name],
                         "launches_per_step": engines[name].launches_per_step}
        for name in ("scales", "scales_sc"):
            out[name]["overhead_ms"] = out[name]["graph_step_ms"] - out["plain"]["graph_step_ms"]
            out[name]["overhead_rel"] = out[name]["overhead_ms"] / out["plain"]["graph_step_ms"]
        res["step_" + mlp_mode] = out
        if mlp_mode == "fp32":
            eng = engines["scales_sc"]
            c, s = eng.corr_raw, eng.params.mode_scales
            U_pred = torch.empty_like(eng.U_pred)
            g = torch.randn_like(c)
            Kc = eng.Kc
            grad_s = torch.empty(k, device=dev)
            acc = torch.zeros(9, dtype=torch.float64, device=dev)
            t = alternate({"fwd": lambda: ops.mode_scale_fwd(c, eng.U_base, s, 5.0, out=U_pred),
                           "bwd": lambda: ops.mode_scale_bwd(c, Kc, s, 1.0, g, grad_s=grad_s, loss_acc=acc)},
                          args.min_seconds, args.rounds)
            fwd_bytes, bwd_bytes = 12 * n * k, 16 * n * k
            res["kernels"] = {
                "mode_scale_fwd": {"ms": t["fwd"] * 1e3, "bytes": fwd_bytes, "TBps": fwd_bytes / t["fwd"] / 1e12,
                                   "of_hbm_peak": fwd_bytes / t["fwd"] / HBM_BYTES_PER_S},
                "mode_scale_bwd": {"ms": t["bwd"] * 1e3, "bytes": bwd_bytes, "TBps": bwd_bytes / t["bwd"] / 1e12,
                                   "of_hbm_peak": bwd_bytes / t["bwd"] / HBM_BYTES_PER_S}}
        del engines
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
