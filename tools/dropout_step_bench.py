"""Cost of dropout in the fused training step on the 998,562-vertex icosphere (k = 32, corrector 82 -> 256 x 6 -> 32,
bf16 MLP mode); prints one JSON line and writes it to --out (default profiles/r05_dropout_step.json).

    python tools/dropout_step_bench.py [--out FILE] [--min-seconds 1.0] [--rounds 2]

Two engines share the input, the operators and the initial weights: p = 0 (the path bench.py times) and p = 0.1
(the dropout kernel instances: tc_chain2_dropout_kernel forward, tc_linear_dropout_kernel<MODE_DX> backward).  Timed
with CUDA events, the variants alternating in one process:
  phases_ms      mlp_fwd, loss_fwd, loss_bwd, mlp_bwd, optim of eager steps with events between the phases
  graph_step_ms  the whole step as a replayed CUDA graph
The card name, power limit and SM clocks are read with nvidia-smi in the same run."""
import argparse
import json
import os
import sys
import types

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from adaptive_step_bench import pkg, phase_times, PHASES      # noqa: E402


def variant_engine(base, p):
    engine = pkg("engine")
    bp = base.params
    params = engine.FlatParams([w.detach().clone() for w in bp.W], [b.detach().clone() for b in bp.b], base.dev)
    cfg = engine.StepConfig(**dict(vars(base.cfg), dropout=p, dropout_seed=1234))
    return engine.TrainStepEngine(base.h, base.U_base, base.pairs, base.offsets, params, cfg,
                                  lam_target=base.lam_target, mlp_mode=base.mlp_mode)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--min-seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--workload", default="icosphere1m")
    ap.add_argument("--p", type=float, default=0.1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_dropout_step.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "dropout_step_bench measures on a GPU"
    from variants_f64_bench import gpu_info, alternate
    import bench
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    info_before = gpu_info()
    res = {"workload": args.workload, "mlp_mode": "bf16", "min_seconds": args.min_seconds, "rounds": args.rounds}
    epoch = 2500
    built = bench.build_engine(types.SimpleNamespace(workload=args.workload, mlp_mode="bf16"), dev, 0, 1)
    base = built["engine"]
    res.update(n=built["n"], k=built["k"], hidden=bench.HIDDEN, mlp_in=base.params.dims[0])
    engines = {"p0": variant_engine(base, 0.0), "p%g" % args.p: variant_engine(base, args.p)}
    del base, built
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
    out = {name: {"graph_step_ms": graph[name] * 1e3, "phases_ms": phases[name],
                  "launches_by_entry": engines[name].launches_by_entry} for name in engines}
    drop = "p%g" % args.p
    out[drop]["overhead_ms"] = out[drop]["graph_step_ms"] - out["p0"]["graph_step_ms"]
    out[drop]["overhead_rel"] = out[drop]["overhead_ms"] / out["p0"]["graph_step_ms"]
    for ph in ("mlp_fwd", "mlp_bwd"):
        out[drop][ph + "_overhead_ms"] = out[drop]["phases_ms"][ph] - out["p0"]["phases_ms"][ph]
    res["step"] = out
    res["gpu_before"], res["gpu_after"] = info_before, gpu_info()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
