"""bench.py on small workloads: --steps is the number of optimizer steps the timed region executes, and --dump-outputs
writes what the last of them computed, from the same inputs on every run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from gpu_util import pkg

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps, workload, mlp_mode):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "3",
           "--workload", workload, "--mlp-mode", mlp_mode, "--no-e2e", "--no-samplers", "--no-torus", "--no-trained",
           "--no-cpu-baseline", "--dump-outputs", str(out_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=str(out_dir.parent))
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    return json.loads(lines[-1])


# icosphere10k: all 10,242 rows of U_pred are written; icosphere100k: the seeded sample of DUMP_ROWS rows, bf16 path
@pytest.mark.parametrize("workload,mlp_mode", [("icosphere10k", "fp32"), ("icosphere100k", "bf16")])
def test_steps_and_dump_outputs(workload, mlp_mode, tmp_path):
    import bench
    line = _bench(tmp_path / "a", 7, workload, mlp_mode)
    # timed_steps is the change of the optimizer's step counter over the timed region
    assert line["timed_steps"] == 7 and line["steps"] == 7
    got = {name: np.load(str(tmp_path / "a" / (name + ".npy")))
           for name in ("loss_terms", "eigenvalues", "params", "U_pred_sample")}
    assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in got.values())
    k, n = line["config"]["k"], line["config"]["vertices"]
    assert got["loss_terms"].shape == (pkg("ops").N_LOSS_TERMS,) and got["eigenvalues"].shape == (1, k)
    assert got["U_pred_sample"].shape == (min(n, bench.DUMP_ROWS), k)
    assert got["loss_terms"][5] == pytest.approx(line["loss"], rel=1e-12)
    assert sum(a.nbytes for a in got.values()) <= 64 << 20
    # seeded inputs and fixed-order reductions (no floating-point atomics): a second run is bit-identical
    _bench(tmp_path / "b", 7, workload, mlp_mode)
    for name, a in got.items():
        assert np.array_equal(np.load(str(tmp_path / "b" / (name + ".npy"))), a), name
