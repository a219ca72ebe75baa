"""Micro-benchmarks of single kernels with CUDA events (development aid; not part of the bench contract)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def timeit(fn, reps=20):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ops, sparse, cabi, engine = bench.pkg("ops"), bench.pkg("sparse"), bench.pkg("_cabi"), bench.pkg("engine")
    name = sys.argv[1] if len(sys.argv) > 1 else "icosphere1m"
    w = bench.build_host_workload(name)
    dev = torch.device("cuda")
    pair = sparse.OperatorPair(w["K"], w["M"], dev, assume_symmetric=True)
    n, k = w["verts"].shape[0], w["k"]
    U = 0.3 * torch.randn(n, k, device=dev)
    KU, MU, dU = torch.empty_like(U), torch.empty_like(U), torch.empty_like(U)
    nbytes = 12 * pair.K.nnz + 4 * (n + 1) + 12 * n * k
    for waves in (1, 2, 4, 16):
        cabi.call("ep_tune_set", 1, waves)
        ms = timeit(lambda: ops.spmm2(pair, U, out_K=KU, out_M=MU))
        print("spmm2 waves %2d: %.4f ms, %.0f GB/s" % (waves, ms, nbytes / ms / 1e6))
    cabi.call("ep_tune_set", 1, 1)
    P = ops.eigen_partials(U, KU, MU)
    ms = timeit(lambda: ops.eigen_partials(U, KU, MU, out=P))
    print("partials (+reduce): %.4f ms, %.0f GB/s" % (ms, 12 * n * k / ms / 1e6))
    acc = torch.zeros(6, dtype=torch.float64, device=dev)
    lam, coef = ops.eigen_finalize(k, n, P, 1000.0, 10.0, acc)
    ms = timeit(lambda: ops.eigen_loss_bwd(pair, U, KU, MU, coef, 1.0, dU))
    print("fused bwd: %.4f ms, %.0f GB/s" % (ms, nbytes / ms / 1e6))


if __name__ == "__main__":
    main()
