"""eigen-pinns, B200-native hot path.

Package layout
  csrc/            hand-written sm_100a CUDA kernels + the C ABI (include/eigenpinns_b200.h)
  _cabi.py         ctypes binding of that ABI (no fallback: a missing library raises)
  sparse.py        device-resident CSR operators (K, M pairs with a shared pattern)
  ops.py           tensor-level wrappers and autograd Functions
  engine.py        explicit training step (forward, eigen-loss, analytic backward, clip + Adam)
  sampling.py      host side of the FPS / voxel down-samplers
  partition.py     vertex sharding + halo plans for the multi-GPU step
  fem.py           sparse linear-FEM assembly (host, fp64);  synthetic.py: benchmark meshes
  src/             reference-shaped drop-in surface (main.py, config.py, multigrid_model.py, ...)
"""
from . import _cabi

__version__ = "0.3.0"


def library_version():
    return _cabi.query("ep_version")


def require_library():
    """Load the CUDA library now (raises with build instructions if it is missing)."""
    return _cabi.load()
