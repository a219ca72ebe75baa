"""ctypes binding of include/eigenpinns_b200.h (the C ABI of the sm_100a kernels).

There is deliberately NO fallback: if the shared library has not been built
(`python -c "import __graft_entry__ as g; g.build()"` or `make -C eigen-pinns_b200/csrc`)
loading raises, and every wrapper raises `EpError` on a non-zero status.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libeigenpinns_b200.so")

c_int, c_i64, c_sz, c_u64 = ctypes.c_int, ctypes.c_int64, ctypes.c_size_t, ctypes.c_uint64
c_f, c_d, c_p = ctypes.c_float, ctypes.c_double, ctypes.c_void_p

# name -> (restype, argtypes); mirrors the header one to one
SIGNATURES = {
    "ep_version": (c_int, []),
    "ep_last_error_string": (ctypes.c_char_p, []),
    "ep_device_info": (c_int, [c_p, c_p, c_p]),
    "ep_tune_set": (c_int, [c_int, c_int]),
    "ep_spmm_csr_f32": (c_int, [c_int, c_int, c_p, c_p, c_p, c_p, c_int, c_p, c_int, c_p]),
    "ep_spmm2_csr_f32": (c_int, [c_int, c_int, c_p, c_p, c_p, c_p, c_p, c_int, c_p, c_p, c_int, c_p]),
    "ep_spmm2_sum_csr_f32": (c_int, [c_int, c_int, c_p, c_p, c_p, c_p, c_p, c_p, c_int, c_p, c_int, c_f, c_p,
                                     c_p, c_int, c_p]),
    "ep_spmm_csr_f64": (c_int, [c_int, c_int, c_p, c_p, c_p, c_p, c_int, c_p, c_int, c_p]),
    "ep_spmm2_csr_f64": (c_int, [c_int, c_int, c_p, c_p, c_p, c_p, c_p, c_int, c_p, c_p, c_int, c_p]),
    "ep_spmm2_sum_csr_f64": (c_int, [c_int, c_int, c_p, c_p, c_p, c_p, c_p, c_p, c_int, c_p, c_int, c_d, c_p,
                                     c_p, c_int, c_p]),
    "ep_neighbor_mean_concat_f32": (c_int, [c_int, c_int, c_p, c_p, c_p, c_int, c_p, c_int, c_p]),
    "ep_spmm_concat_f32": (c_int, [c_int, c_int, c_p, c_p, c_p, c_p, c_int, c_p, c_int, c_p]),
    "ep_eigen_partials_len": (c_sz, [c_int]),
    "ep_eigen_partials_workspace_bytes": (c_sz, [c_int]),
    "ep_eigen_partials_f32": (c_int, [c_int, c_int, c_p, c_int, c_p, c_p, c_int, c_p, c_p, c_sz, c_p]),
    "ep_eigen_partials_f64": (c_int, [c_int, c_int, c_p, c_int, c_p, c_p, c_int, c_p, c_p, c_sz, c_p]),
    "ep_eigen_coef_len": (c_sz, [c_int]),
    "ep_eigen_finalize_f32": (c_int, [c_int, c_d, c_p, c_f, c_f, c_int, c_p, c_f, c_f, c_f, c_f, c_f, c_p, c_p, c_p, c_p,
                                      c_p]),
    "ep_loss_add_sum_f64": (c_int, [c_int, c_p, c_d, c_int, c_p, c_p]),
    "ep_eigen_bwd_prepare_f32": (c_int, [c_int, c_int, c_p, c_int, c_p, c_p, c_int, c_p, c_p, c_p, c_p, c_p]),
    "ep_eigen_bwd_fused_sym_rows_f32": (c_int, [c_int, c_int, c_int, c_p, c_p, c_p, c_p, c_p, c_p, c_int, c_p, c_f, c_p, c_p,
                                                c_int, c_p]),
    "ep_eigen_bwd_gram_term_tf32x3": (c_int, [c_int, c_int, c_int, c_p, c_int, c_p, c_f, c_p, c_p, c_int, c_p]),
    "ep_eigen_bwd_gather_sym_rows_f32": (c_int, [c_int, c_int, c_int, c_p, c_p, c_p, c_p, c_p, c_p, c_int, c_p, c_f, c_p, c_p,
                                                 c_int, c_int, c_p]),
    "ep_scale_columns_rsqrt_f32": (c_int, [c_int, c_int, c_p, c_int, c_p, c_int, c_d, c_p, c_int, c_p]),
    "ep_axpy_out_f32": (c_int, [c_sz, c_f, c_p, c_p, c_p, c_p, c_p]),
    "ep_mode_scale_fwd_f32": (c_int, [c_int, c_int, c_p, c_int, c_p, c_int, c_p, c_f, c_p, c_p, c_int, c_p]),
    "ep_mode_scale_bwd_workspace_bytes": (c_sz, [c_int]),
    "ep_mode_scale_bwd_f32": (c_int, [c_int, c_int, c_d, c_p, c_int, c_p, c_int, c_p, c_f, c_p, c_int, c_p, c_int,
                                      c_p, c_p, c_sz, c_p]),
    "ep_linear_fwd_f32": (c_int, [c_int, c_int, c_int, c_p, c_int, c_p, c_p, c_p, c_int, c_int, c_p]),
    "ep_linear_bwd_workspace_bytes": (c_sz, [c_int, c_int, c_int]),
    "ep_linear_bwd_f32": (c_int, [c_int, c_int, c_int, c_p, c_int, c_p, c_p, c_int, c_p, c_int, c_int,
                                  c_p, c_p, c_p, c_sz, c_p]),
    "ep_linear_fwd_f64": (c_int, [c_int, c_int, c_int, c_p, c_int, c_p, c_p, c_p, c_int, c_int, c_p]),
    "ep_linear_bwd_workspace_bytes_f64": (c_sz, [c_int, c_int, c_int]),
    "ep_linear_bwd_f64": (c_int, [c_int, c_int, c_int, c_p, c_int, c_p, c_p, c_int, c_p, c_int, c_int,
                                  c_p, c_p, c_p, c_sz, c_p]),
    "ep_linear_act_fwd_f32": (c_int, [c_int, c_int, c_int, c_p, c_int, c_p, c_p, c_p, c_int, c_p, c_int, c_int, c_p]),
    "ep_linear_act_fwd_f64": (c_int, [c_int, c_int, c_int, c_p, c_int, c_p, c_p, c_p, c_int, c_p, c_int, c_int, c_p]),
    "ep_linear_act_bwd_f32": (c_int, [c_int, c_int, c_int, c_p, c_int, c_p, c_int, c_int, c_p, c_p, c_int, c_p, c_int,
                                      c_p, c_p, c_p, c_sz, c_p]),
    "ep_linear_act_bwd_f64": (c_int, [c_int, c_int, c_int, c_p, c_int, c_p, c_int, c_int, c_p, c_p, c_int, c_p, c_int,
                                      c_p, c_p, c_p, c_sz, c_p]),
    "ep_tc_pad_features": (c_int, [c_int, c_int]),
    "ep_tc_packed_rows_bytes": (c_sz, [c_int, c_int]),
    "ep_tc_packed_weight_bytes": (c_sz, [c_int, c_int]),
    "ep_tc_pack_rows_bf16": (c_int, [c_int, c_int, c_int, c_p, c_int, c_p, c_p]),
    "ep_tc_pack_weight_bf16": (c_int, [c_int, c_int, c_int, c_int, c_p, c_p, c_p, c_p]),
    "ep_tc_relu_mask_bytes": (c_sz, [c_int, c_int]),
    "ep_tc_linear_fwd_bf16": (c_int, [c_int, c_int, c_int, c_int, c_p, c_p, c_p, c_int, c_p, c_p, c_p]),
    "ep_tc_linear_final_bf16": (c_int, [c_int, c_int, c_int, c_int, c_p, c_p, c_p, c_p, c_int, c_p, c_f, c_p,
                                        c_p, c_int, c_p]),
    "ep_tc_linear_dx_bf16": (c_int, [c_int, c_int, c_int, c_p, c_p, c_p, c_p, c_int, c_p]),
    "ep_tc_chain_fwd_bf16": (c_int, [c_int, c_int, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_int, c_p, c_f, c_p, c_p,
                                     c_int, c_p]),
    "ep_dropout_keep_mask_u8": (c_int, [c_i64, c_int, c_f, c_u64, c_int, c_p, c_int, c_i64, c_p, c_p]),
    "ep_linear_fwd_dropout_f32": (c_int, [c_int, c_int, c_int, c_p, c_int, c_p, c_p, c_p, c_int, c_f, c_u64, c_int, c_p,
                                          c_int, c_i64, c_p]),
    "ep_linear_bwd_dropout_f32": (c_int, [c_int, c_int, c_int, c_p, c_int, c_p, c_p, c_int, c_p, c_int, c_f, c_p, c_p,
                                          c_p, c_sz, c_p]),
    "ep_tc_linear_fwd_dropout_bf16": (c_int, [c_int, c_int, c_int, c_int, c_p, c_p, c_p, c_p, c_p, c_f, c_u64, c_int,
                                              c_p, c_int, c_i64, c_p]),
    "ep_tc_linear_dx_dropout_bf16": (c_int, [c_int, c_int, c_int, c_p, c_p, c_p, c_p, c_f, c_int, c_p]),
    "ep_tc_chain_fwd_dropout_bf16": (c_int, [c_int, c_int, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_int, c_p, c_f, c_p,
                                             c_p, c_int, c_p, c_f, c_u64, c_int, c_p, c_i64, c_p]),
    "ep_tc_dw_workspace_bytes": (c_sz, []),
    "ep_tc_linear_dw_bf16": (c_int, [c_int, c_int, c_int, c_int, c_int, c_p, c_p, c_p, c_p, c_p, c_sz, c_int, c_p]),
    "ep_grad_sqnorm_f32": (c_int, [c_sz, c_p, c_p, c_p]),
    "ep_adam_clip_step_f32": (c_int, [c_sz, c_p, c_p, c_p, c_p, c_f, c_p, c_f, c_f, c_f, c_f, c_int, c_f,
                                      c_p, c_p]),
    "ep_grad_sqnorm_f64": (c_int, [c_sz, c_p, c_p, c_p]),
    "ep_adam_clip_step_f64": (c_int, [c_sz, c_p, c_p, c_p, c_p, c_d, c_p, c_d, c_d, c_d, c_d, c_int, c_d,
                                      c_p, c_p]),
    "ep_single_mode_max_prev": (c_int, []),
    "ep_single_mode_workspace_bytes": (c_sz, [c_int]),
    "ep_single_mode_fwd_f32": (c_int, [c_int, c_int, c_p, c_p, c_p, c_p, c_int, c_p, c_d, c_p, c_p, c_p, c_sz, c_p]),
    "ep_single_mode_fwd_f64": (c_int, [c_int, c_int, c_p, c_p, c_p, c_p, c_int, c_p, c_d, c_p, c_p, c_p, c_sz, c_p]),
    "ep_single_mode_bwd_f32": (c_int, [c_int, c_int, c_p, c_p, c_p, c_int, c_p, c_p, c_p, c_p, c_p, c_p]),
    "ep_single_mode_bwd_f64": (c_int, [c_int, c_int, c_p, c_p, c_p, c_int, c_p, c_p, c_p, c_p, c_p, c_p]),
    "ep_single_mode_fold_fwd_f32": (c_int, [c_int, c_p, c_p, c_p, c_p]),
    "ep_single_mode_fold_fwd_f64": (c_int, [c_int, c_p, c_p, c_p, c_p]),
    "ep_single_mode_fold_bwd_f32": (c_int, [c_int, c_p, c_p, c_p, c_p, c_p, c_p]),
    "ep_single_mode_fold_bwd_f64": (c_int, [c_int, c_p, c_p, c_p, c_p, c_p, c_p]),
    "ep_fps_workspace_bytes": (c_sz, [c_i64]),
    "ep_fps_f64": (c_int, [c_i64, c_p, c_int, c_i64, c_p, c_p, c_sz, c_p]),
    "ep_fps_f64_host": (c_int, [c_i64, c_p, c_int, c_i64, c_p]),
    "ep_bounds_f64": (c_int, [c_i64, c_p, c_p, c_p]),
    "ep_voxel_workspace_bytes": (c_sz, [c_i64, c_i64]),
    "ep_voxel_select_f64": (c_int, [c_i64, c_p, c_p, c_d, c_p, c_p, c_i64, c_p, c_p, c_sz, c_p]),
    "ep_voxel_select_f64_host": (c_int, [c_i64, c_p, c_p, c_d, c_p, c_p, c_i64, c_p]),
    "ep_fem_elements_f64": (c_int, [c_i64, c_p, c_p, c_i64, c_p, c_p, c_p, c_p]),
    "ep_fem_segment_sum_f64": (c_int, [c_i64, c_p, c_p, c_p, c_p, c_p, c_p, c_i64, c_p, c_p, c_p, c_p, c_p, c_p]),
    "ep_knn_grid_f64": (c_int, [c_i64, c_p, c_i64, c_p, c_p, c_p, c_p, c_d, c_p, c_int, c_p, c_p, c_p]),
    "ep_gather_rows_f32": (c_int, [c_int, c_int, c_p, c_p, c_int, c_p, c_int, c_p]),
    "ep_scatter_add_rows_f32": (c_int, [c_int, c_int, c_p, c_p, c_int, c_p, c_int, c_p]),
    "ep_dist_nccl_version": (c_int, []),
    "ep_halo_exchange_f32": (c_int, [c_p, c_int, c_p, c_p, c_p, c_p, c_int, c_p, c_int, c_p, c_p, c_p]),
    "ep_allreduce_sum_f64": (c_int, [c_p, c_sz, c_p, c_p]),
    "ep_allreduce_sum_f32": (c_int, [c_p, c_sz, c_p, c_p]),
}


class EpError(RuntimeError):
    pass


_lib = None

# kernels launched by one call of each entry point (for bench.py's "gpu_launches" claim)
KERNELS_PER_CALL = {
    "ep_spmm_csr_f32": 1, "ep_spmm2_csr_f32": 1, "ep_spmm2_sum_csr_f32": 1, "ep_neighbor_mean_concat_f32": 1,
    "ep_spmm_concat_f32": 2, "ep_eigen_partials_f32": 2, "ep_eigen_finalize_f32": 1, "ep_loss_add_sum_f64": 1, "ep_eigen_bwd_prepare_f32": 1, "ep_eigen_bwd_fused_sym_rows_f32": 1, "ep_eigen_bwd_gram_term_tf32x3": 1, "ep_eigen_bwd_gather_sym_rows_f32": 1,
    "ep_scale_columns_rsqrt_f32": 1, "ep_axpy_out_f32": 1, "ep_linear_fwd_f32": 1, "ep_linear_bwd_f32": 5,
    "ep_grad_sqnorm_f32": 2, "ep_adam_clip_step_f32": 1, "ep_fps_f64": 1, "ep_bounds_f64": 2,
    "ep_voxel_select_f64": 6, "ep_gather_rows_f32": 1, "ep_knn_grid_f64": 1, "ep_fem_elements_f64": 1, "ep_fem_segment_sum_f64": 1, "ep_scatter_add_rows_f32": 1,
    "ep_tc_pack_rows_bf16": 1, "ep_tc_pack_weight_bf16": 1, "ep_tc_linear_fwd_bf16": 1, "ep_tc_linear_final_bf16": 1,
    "ep_tc_linear_dx_bf16": 1, "ep_tc_linear_dw_bf16": 2, "ep_tc_chain_fwd_bf16": 1,
    "ep_halo_exchange_f32": 1,
    "ep_spmm_csr_f64": 1, "ep_spmm2_csr_f64": 1, "ep_spmm2_sum_csr_f64": 1, "ep_eigen_partials_f64": 2,
    "ep_linear_fwd_f64": 1, "ep_linear_bwd_f64": 5,
    "ep_linear_act_fwd_f32": 1, "ep_linear_act_fwd_f64": 1, "ep_linear_act_bwd_f32": 5, "ep_linear_act_bwd_f64": 5,
    "ep_mode_scale_fwd_f32": 1, "ep_mode_scale_bwd_f32": 2,
    "ep_dropout_keep_mask_u8": 1, "ep_linear_fwd_dropout_f32": 1, "ep_linear_bwd_dropout_f32": 5,
    "ep_tc_linear_fwd_dropout_bf16": 1, "ep_tc_linear_dx_dropout_bf16": 1, "ep_tc_chain_fwd_dropout_bf16": 1,
    "ep_grad_sqnorm_f64": 2, "ep_adam_clip_step_f64": 1,
    "ep_single_mode_fwd_f32": 2, "ep_single_mode_fwd_f64": 2, "ep_single_mode_bwd_f32": 1, "ep_single_mode_bwd_f64": 1,
    "ep_single_mode_fold_fwd_f32": 1, "ep_single_mode_fold_fwd_f64": 1, "ep_single_mode_fold_bwd_f32": 1,
    "ep_single_mode_fold_bwd_f64": 1,
}
launch_counter = 0
launch_by_entry = {}          # entry point -> kernels launched through it (bench.py reports the per-step table)


def load():
    """Load the shared library (once) and attach the signatures.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise EpError(
            "eigenpinns_b200: %s is missing - build it first (make -C eigen-pinns_b200/csrc, or "
            "__graft_entry__.build()).  There is no CPU / PyTorch fallback for the hot path." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)            # AttributeError here = header / library out of sync
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def call(name, *args):
    """Call a status-returning entry point; raise EpError with the library's message on failure."""
    global launch_counter
    lib = load()
    rc = getattr(lib, name)(*args)
    nk = KERNELS_PER_CALL.get(name, 0)
    launch_counter += nk
    if nk:
        launch_by_entry[name] = launch_by_entry.get(name, 0) + nk
    if rc != 0:
        msg = lib.ep_last_error_string()
        raise EpError("%s failed (status %d): %s" % (name, rc, msg.decode() if msg else "?"))


def query(name, *args):
    """Call a size / version query (returns the value)."""
    return getattr(load(), name)(*args)
