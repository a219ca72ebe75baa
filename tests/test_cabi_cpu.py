"""CPU-side checks of the boundary: the shared library loads and exports every symbol the public
header declares, the ctypes table mirrors the header, and the product refuses CPU tensors."""
import ctypes
import importlib
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "eigenpinns_b200.h")


def _declared():
    text = open(HEADER).read()
    return sorted(set(re.findall(r"EP_API\s+[\w\s\*]+?\b(ep_\w+)\s*\(", text)))


def test_header_declares_entry_points():
    names = _declared()
    assert len(names) >= 35
    for must in ("ep_spmm2_csr_f32", "ep_eigen_partials_f32", "ep_fps_f64", "ep_voxel_select_f64",
                 "ep_linear_fwd_f32", "ep_adam_clip_step_f32", "ep_tc_linear_fwd_bf16"):
        assert must in names


def test_library_exports_every_declared_symbol():
    cabi = importlib.import_module("eigen-pinns_b200._cabi")
    lib = cabi.load()
    for name in _declared():
        assert hasattr(lib, name), "library does not export " + name
    assert lib.ep_version() >= 100


def test_ctypes_table_matches_header():
    cabi = importlib.import_module("eigen-pinns_b200._cabi")
    assert sorted(cabi.SIGNATURES) == _declared()
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    for name, (_, args) in cabi.SIGNATURES.items():
        m = re.search(r"\b%s\s*\(([^;]*?)\)\s*;" % name, text, flags=re.S)
        assert m, name
        params = m.group(1).strip()
        n = 0 if params in ("void", "") else params.count(",") + 1
        assert n == len(args), "%s: header has %d parameters, ctypes table %d" % (name, n, len(args))


def test_sizes_without_gpu():
    cabi = importlib.import_module("eigen-pinns_b200._cabi")
    assert cabi.query("ep_eigen_partials_len", 32) == 32 * 32 + 5 * 32       # G | num | sKK | sKM | sMM | colsum(MU)
    assert cabi.query("ep_eigen_coef_len", 64) == 1 + 4 * 64 + 64 * 64         # c_res | lam | num_bar | den_bar | G_bar | g_mean


@pytest.mark.parametrize("k", [k for k in range(4, 129, 4) if k != 64])
def test_gram_term_tf32x3_accepts_k_64_only(k):
    """The tensor-core k x k term of the loss backward is built for k = 64 alone: any other k returns EP_ERR_UNSUPPORTED
    before anything is launched (so no GPU is needed; the pointers are never dereferenced)."""
    cabi = importlib.import_module("eigen-pinns_b200._cabi")
    fake = ctypes.c_void_p(256)
    with pytest.raises(cabi.EpError, match=r"status -3\).*k must be 64"):
        cabi.call("ep_eigen_bwd_gram_term_tf32x3", 0, 1000, k, fake, 2 * k, fake, 1.0, None, fake, k, None)


def test_ops_reject_cpu_tensors():
    import torch
    ops = importlib.import_module("eigen-pinns_b200.ops")
    cabi = importlib.import_module("eigen-pinns_b200._cabi")
    with pytest.raises((cabi.EpError, AssertionError, RuntimeError)):
        ops.linear_fwd(torch.zeros(4, 4), torch.zeros(4, 4), torch.zeros(4), relu=False)


def test_trainer_refuses_to_run_without_gpu():
    import sys
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    src = os.path.join(ROOT, "eigen-pinns_b200", "src")
    sys.path.insert(0, src)
    try:
        for m in ("config", "multigrid_model", "corrector_model", "utils", "Mesh", "mesh_helpers", "samplers"):
            sys.modules.pop(m, None)
        import config
        import multigrid_model
        cfg = config.PINNConfig.from_yaml(os.path.join(src, "parameters.yml"))
        with pytest.raises(RuntimeError):
            multigrid_model.MultigridGNN(cfg)
    finally:
        sys.path.remove(src)


def test_multi_gpu_entry_points_resolve_nccl_at_run_time():
    """The library has no link-time NCCL dependency; the halo / all-reduce entry points find libnccl.so.2 when called and
    reject bad arguments before touching it."""
    import ctypes
    import subprocess
    cabi = importlib.import_module("eigen-pinns_b200._cabi")
    needed = subprocess.run(["objdump", "-p", cabi.LIB_PATH], capture_output=True, text=True).stdout
    assert "libnccl" not in needed
    assert cabi.query("ep_dist_nccl_version") >= 0                     # 0 when no NCCL can be found: not an error here
    with pytest.raises(cabi.EpError):
        cabi.call("ep_halo_exchange_f32", None, 1, None, None, None, None, 4, None, 4, None, None, None)
    cabi.call("ep_halo_exchange_f32", None, 0, None, None, None, None, 4, None, 4, None, None, None)   # no peers: no-op
    cabi.call("ep_allreduce_sum_f64", ctypes.c_void_p(1), 0, None, None)                                 # empty: no-op


def test_header_is_plain_c_and_links_from_c(tmp_path):
    """The boundary is a C ABI: the header compiles as C99 (-pedantic) and as C++, and a C program links against the
    shared library and calls it (no GPU needed for ep_version / the size queries)."""
    import shutil
    import subprocess
    cabi = importlib.import_module("eigen-pinns_b200._cabi")
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    src = tmp_path / "use_abi.c"
    src.write_text('#include <stdio.h>\n#include "eigenpinns_b200.h"\n'
                   'int main(void) {\n'
                   '  if (ep_version() <= 0) return 1;\n'
                   '  if (ep_eigen_partials_len(32) != 32 * 32 + 5 * 32) return 2;\n'
                   '  if (ep_tc_pad_features(82, 0) != 96) return 3;\n'
                   '  /* bad arguments are reported, not crashed on */\n'
                   '  if (ep_spmm_csr_f32(-1, 4, 0, 0, 0, 0, 4, 0, 4, 0) == EP_OK) return 4;\n'
                   '  if (ep_last_error_string() == 0) return 5;\n'
                   '  printf("ok\\n");\n  return 0;\n}\n')
    inc = os.path.join(ROOT, "include")
    lib_dir = os.path.dirname(cabi.LIB_PATH)
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", inc, "-c", str(src), "-o",
                    str(tmp_path / "a.o")], check=True)
    subprocess.run(["g++", "-std=c++11", "-Wall", "-Werror", "-I", inc, "-x", "c++", "-c", str(src), "-o",
                    str(tmp_path / "b.o")], check=True)
    exe = tmp_path / "use_abi"
    subprocess.run(["gcc", str(tmp_path / "a.o"), "-o", str(exe), "-L", lib_dir, "-leigenpinns_b200",
                    "-Wl,-rpath," + lib_dir], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.strip() == "ok", (out.returncode, out.stdout, out.stderr)
