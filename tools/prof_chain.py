"""Times (CUDA events) the tensor-core MLP at the benchmark size: forward chain against layer-by-layer forward (same
backward), the forward chain without its activation / mask copies, and the in-kernel clock64 trace of the chain.
    python tools/prof_chain.py [n] [k] [reps]"""
import ctypes
import importlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
engine = importlib.import_module("eigen-pinns_b200.engine")
tcm = importlib.import_module("eigen-pinns_b200.mlp_tc")
cabi = importlib.import_module("eigen-pinns_b200._cabi")


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 998562
    k = int(sys.argv[2]) if len(sys.argv) > 2 else 32
    reps = int(sys.argv[3]) if len(sys.argv) > 3 else 10
    dev = torch.device("cuda", 0)
    dims = [2 * (9 + k)] + [256] * 6 + [k]
    g = torch.Generator().manual_seed(0)
    Ws = [torch.randn(dims[i + 1], dims[i], generator=g) / np.sqrt(dims[i]) for i in range(len(dims) - 1)]
    bs = [0.1 * torch.randn(dims[i + 1], generator=g) for i in range(len(dims) - 1)]
    h = torch.randn(n, dims[0], device=dev)
    U = torch.randn(n, k, device=dev)
    d_out = torch.randn(n, k, device=dev) / n
    up = torch.empty_like(U)
    out = {}
    for chain in (True, False):
        p = engine.FlatParams(Ws, bs, dev)
        m = tcm.TcMlp(n, p, dev, h, chain_fwd=chain)
        m.want_corr = False
        ev = lambda: torch.cuda.Event(enable_timing=True)
        for _ in range(2):
            m.forward(h, U, 0.5, up)
            m.backward(h, d_out)
        torch.cuda.synchronize()
        e0, e1, e2 = ev(), ev(), ev()
        tf = tb = 0.0
        for _ in range(reps):
            e0.record()
            m.forward(h, U, 0.5, up)
            e1.record()
            m.backward(h, d_out)
            e2.record()
            torch.cuda.synchronize()
            tf += e0.elapsed_time(e1)
            tb += e1.elapsed_time(e2)
        out["chain" if chain else "layerwise"] = (tf / reps, tb / reps)
        if chain:
            P = lambda t: ctypes.c_void_p(t.data_ptr())
            st = lambda: ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            # in-kernel timeline of CTA 0 (clock64 stamps per (layer, slot) step): ep_tune_set keys 3 / 4 carry a device
            # pointer
            trace = torch.zeros(64 * 8, dtype=torch.int64, device=dev)
            ptr = trace.data_ptr()
            cabi.call("ep_tune_set", 3, ctypes.c_int(ptr & 0xFFFFFFFF if (ptr & 0xFFFFFFFF) < 2**31 else (ptr & 0xFFFFFFFF) - 2**32))
            cabi.call("ep_tune_set", 4, ctypes.c_int(ptr >> 32))
            m.forward(h, U, 0.5, up)
            torch.cuda.synchronize()
            cabi.call("ep_tune_set", 3, 0)
            cabi.call("ep_tune_set", 4, 0)
            tr = trace.view(64, 8).cpu().numpy()
            t0 = tr[0, 0]
            print("step (layer, slot): ready issued acc_full drained arrived  (clk since first)")
            for gi in range(30):
                r = tr[gi] - t0
                print("%2d (l%d u%d): %7d %7d %7d %7d %7d   issue %5d tail %5d epi %5d arrive %4d" % (
                    gi, (gi // 2) % m.L, gi % 2, r[0], r[1], r[2], r[3], r[4], r[1] - r[0], r[2] - r[1], r[3] - r[2],
                    r[4] - r[3]))
            # experiment: the forward chain without the HBM copies of activations / masks (not a product path)
            for label, acts_t, masks_t in (("fwd_no_act_no_mask", None, None), ("fwd_no_mask", m._t_acts, None),
                                           ("fwd_no_act", None, m._t_masks)):
                e0.record()
                for _ in range(reps):
                    cabi.call("ep_tc_chain_fwd_bf16", m.n, m.L, m._t_pd, m._t_out, P(m.x0), m._t_Wp, m._t_b, acts_t, masks_t,
                              None, k, P(U), 0.5, None, P(up), k, st())
                e1.record()
                torch.cuda.synchronize()
                out[label] = e0.elapsed_time(e1) / reps
        del m, p
        torch.cuda.empty_cache()
    flops = 2 * n * sum(dims[i] * dims[i + 1] for i in range(len(dims) - 1))
    print("n=%d k=%d" % (n, k))
    for name, v in out.items():
        print(name, v)
    tf, tb = out["chain"]
    print("chain fwd %.3f ms = %.0f TFLOP/s; fwd+bwd %.3f ms = %.0f TFLOP/s (3x fwd flops - first-layer dX)"
          % (tf, flops / tf / 1e9, tf + tb, (3 * flops - 2 * n * dims[0] * dims[1]) / (tf + tb) / 1e9))


if __name__ == "__main__":
    main()
