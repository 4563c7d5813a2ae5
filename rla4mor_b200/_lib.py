"""ctypes binding of librla_b200.so (the C ABI declared in include/rla_b200.h).

There is no fallback: if the shared library is missing or a call fails, an
exception is raised.  Nothing in this package imports `oracle/`.
"""
import ctypes
import os
from ctypes import c_int, c_int64, c_size_t, c_void_p, c_double, c_float, c_uint64, c_char_p, POINTER

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "librla_b200.so")


class RlaError(RuntimeError):
    pass


_lib = None

_vp = c_void_p
_SIGS = {
    "rla_version": (c_int, []),
    "rla_last_error": (c_char_p, []),
    "rla_launch_count": (ctypes.c_ulonglong, []),
    "rla_launch_count_add": (None, [ctypes.c_longlong]),
    "rla_copy2d_async": (c_int, [_vp, c_size_t, _vp, c_size_t, c_size_t, c_size_t, c_int, _vp]),
    "rla_srht_plan_create": (c_int, [POINTER(c_void_p), _vp, c_int64, _vp, c_int64, c_int]),
    "rla_srht_plan_destroy": (None, [_vp]),
    "rla_srht_plan_device_bytes": (c_size_t, [_vp]),
    "rla_srht_plan_upload": (c_int, [_vp, _vp, _vp]),
    "rla_srht_plan_passes": (c_int, [_vp]),
    "rla_srht_workspace_bytes": (c_size_t, [_vp, c_int64]),
    "rla_srht_apply_f64": (c_int, [_vp, _vp, c_int64, c_int64, c_double, _vp, c_int64, _vp, c_size_t, _vp]),
    "rla_srht_apply_f32": (c_int, [_vp, _vp, c_int64, c_int64, c_float, _vp, c_int64, _vp, c_size_t, _vp]),
    "rla_srht_rows_f64": (c_int, [_vp, c_int64, _vp, _vp, c_int64, c_double, _vp, c_int64, _vp]),
    "rla_fwht_f64": (c_int, [_vp, c_int64, c_int64, c_int64, _vp, c_int64, c_double, _vp]),
    "rla_fwht_f32": (c_int, [_vp, c_int64, c_int64, c_int64, _vp, c_int64, c_float, _vp]),
    "rla_srht_adjoint_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "rla_srht_adjoint_f64": (c_int, [_vp, c_int64, _vp, _vp, c_int64, _vp, c_int64, c_int64, c_double, _vp, c_int64,
                                     _vp, c_size_t, _vp]),
    "rla_gemm_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "rla_gemm_rng_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "rla_philox4x32_10_host": (c_int, [_vp, c_int64, _vp]),
    "rla_philox4x32_10_device": (c_int, [_vp, c_int64, _vp, _vp]),
    "rla_dmma_peak_tflops": (c_int, [POINTER(c_double), _vp, _vp]),
    "rla_gauss_apply_explicit_f64": (c_int, [_vp, c_int64, c_int64, c_int64, _vp, c_int64, c_int64, _vp, c_int64,
                                             _vp, c_size_t, _vp]),
    "rla_embed_apply_rng_f64": (c_int, [c_uint64, c_int, c_double, c_int64, c_int64, c_int64, c_int64, _vp, c_int64,
                                        c_int64, _vp, c_int64, c_int, _vp, c_size_t, _vp]),
    "rla_gemm32_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "rla_embed_apply_rng_f32": (c_int, [c_uint64, c_int, c_double, c_int64, c_int64, c_int64, c_int64, _vp, c_int64,
                                        c_int64, _vp, c_int64, c_int, _vp, c_size_t, _vp]),
    "rla_theta_materialize_f64": (c_int, [c_uint64, c_int, c_double, c_int64, c_int64, c_int64, c_int64, _vp, c_int64, _vp]),
    "rla_embed_adjoint_rng_f64": (c_int, [c_int, c_double, _vp, _vp, c_int64, c_int64, _vp, c_int64, c_int64, _vp,
                                          c_int64, _vp]),
    "rla_mt19937_segment_words": (c_int64, []),
    "rla_mt19937_plan_create": (c_int, [POINTER(c_void_p), _vp, _vp, c_int64]),
    "rla_mt19937_plan_destroy": (None, [_vp]),
    "rla_mt19937_plan_workspace_bytes": (c_size_t, [_vp]),
    "rla_mt19937_plan_build": (c_int, [_vp, _vp, c_size_t, _vp]),
    "rla_mt19937_plan_pairs": (c_int64, [_vp, c_int64]),
    "rla_mt19937_execute_workspace_bytes": (c_size_t, [_vp, c_int64]),
    "rla_mt19937_normal_f64": (c_int, [_vp, _vp, _vp, _vp, c_double, c_double, _vp, c_int64, _vp, c_size_t, c_int64,
                                       _vp, POINTER(c_int64), _vp]),
    "rla_mt19937_jump_host": (c_int, [_vp, c_uint64, _vp]),
    "rla_mt19937_attempts_host": (c_int, [_vp, c_int64, _vp, _vp, _vp, _vp]),
    "rla_mt19937_ext_log_host": (c_int, [_vp, c_int64, c_double, _vp, _vp, _vp]),
    "rla_libm_log_host": (c_int, [_vp, c_int64, _vp]),
    "rla_gemm_nn_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "rla_gemm_nn_f64": (c_int, [_vp, c_int64, c_int64, c_int64, _vp, c_int64, c_int64, _vp, c_int64, _vp, c_size_t, _vp]),
    "rla_spmm_csr_f64": (c_int, [_vp, _vp, _vp, c_int64, c_int64, _vp, c_int64, c_int64, _vp, c_int64, _vp]),
    "rla_gram_schmidt_f64": (c_int, [_vp, c_int64, c_int64, c_int64, c_int64, _vp, _vp, c_double, c_double, c_double, _vp]),
    "rla_svd_jacobi_f64": (c_int, [_vp, c_int64, c_int64, c_int64, _vp, _vp, _vp, _vp, c_int, c_double,
                                   POINTER(c_int), _vp]),
    "rla_residual_norm_f64": (c_int, [_vp, c_int64, c_int64, c_int64, _vp, _vp, _vp, c_int64, _vp, _vp, _vp]),
    "rla_rom_solve_batch_max_r": (c_int, []),
    "rla_rom_solve_batch_f64": (c_int, [_vp, c_int64, c_int64, _vp, c_int64, _vp, c_int64, _vp, c_int64, c_int64,
                                        _vp, c_int64, _vp, _vp]),
    "rla_rom_lstsq_batch_max_r": (c_int, []),
    "rla_rom_lstsq_batch_f64": (c_int, [_vp, c_int64, c_int64, c_int64, c_int64, c_int64, _vp, c_int64, _vp, c_int64,
                                        c_int64, _vp, c_int64, _vp, _vp]),
    "rla_residual_norm_batch_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "rla_residual_norm_batch_f64": (c_int, [_vp, c_int64, c_int64, c_int64, c_int64, c_int64, _vp, c_int64, _vp,
                                            c_int64, _vp, c_int64, c_int64, _vp, _vp, c_size_t, _vp]),
    "rla_affine_cg_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "rla_affine_spmm_f64": (c_int, [_vp, _vp, _vp, c_int64, c_int64, c_int64, _vp, c_int64, _vp, c_int64, c_int64, _vp,
                                    c_int64, _vp, _vp, c_size_t, _vp]),
    "rla_row_dot_partials_f64": (c_int, [_vp, c_int64, _vp, c_int64, c_int64, c_int64, _vp, _vp, c_size_t, _vp]),
    "rla_row_dot_sum_f64": (c_int, [_vp, c_size_t, c_int64, c_int64, _vp, _vp]),
    "rla_affine_cg_start_f64": (c_int, [_vp, _vp, c_size_t, c_int64, c_int64, c_double, c_int64, _vp, _vp, _vp]),
    "rla_affine_cg_alpha_f64": (c_int, [_vp, c_size_t, c_int64, c_int64, _vp, _vp, _vp]),
    "rla_affine_cg_update_r_f64": (c_int, [_vp, c_int64, _vp, c_int64, c_int64, c_int64, _vp, _vp, _vp]),
    "rla_affine_cg_beta_f64": (c_int, [_vp, c_size_t, c_int64, c_int64, c_double, c_int64, _vp, _vp, _vp]),
    "rla_affine_cg_update_xp_f64": (c_int, [_vp, c_int64, _vp, c_int64, _vp, c_int64, c_int64, c_int64, _vp, _vp, _vp]),
    "rla_affine_gmres_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "rla_affine_gmres_hess_bytes": (c_size_t, [c_int64, c_int64]),
    "rla_affine_gmres_dots_f64": (c_int, [_vp, _vp, _vp, c_int64, c_int64, c_int64, _vp, _vp, _vp, c_size_t, _vp]),
    "rla_affine_gmres_orth_f64": (c_int, [_vp, _vp, _vp, _vp, _vp, c_int64, c_int64, c_int64, _vp, _vp, _vp, c_size_t,
                                          _vp]),
    "rla_affine_gmres_dgks_f64": (c_int, [_vp, _vp, c_int64, c_int64, _vp, _vp, _vp, _vp]),
    "rla_affine_gmres_step_f64": (c_int, [_vp, _vp, c_int64, c_int64, c_double, c_int64, _vp, _vp, _vp, _vp]),
    "rla_affine_gmres_residual_f64": (c_int, [_vp, _vp, c_int64, c_int64, _vp, _vp]),
    "rla_affine_gmres_normalize_f64": (c_int, [_vp, _vp, _vp, _vp, _vp, c_int64, c_int64, c_int64, _vp, _vp, _vp]),
    "rla_affine_gmres_update_f64": (c_int, [_vp, _vp, _vp, c_int64, c_int64, c_int64, _vp, _vp, _vp]),
    "rla_gram_schmidt_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "rla_gram_schmidt_status_offset": (c_int64, [c_int64, c_int64]),
    "rla_gram_schmidt_ws_f64": (c_int, [_vp, c_int64, c_int64, c_int64, c_int64, _vp, _vp, c_double, c_double, c_double,
                                        _vp, c_size_t, _vp]),
    "rla_svd_jacobi_block_rows": (c_int, [c_int64, c_int64, c_int]),
    "rla_svd_jacobi_block_scratch_ints": (c_size_t, [c_int64, c_int, c_int]),
    "rla_svd_jacobi_block_f64": (c_int, [_vp, c_int64, c_int64, c_int64, _vp, _vp, _vp, c_int, _vp, c_int, c_double, _vp]),
    "rla_svd_jacobi_cluster_size": (c_int, [c_int64, c_int64, c_int]),
    "rla_svd_jacobi_cluster_f64": (c_int, [_vp, c_int64, c_int64, c_int64, _vp, _vp, _vp, c_int, c_double, _vp]),
    "rla_trinv_upper_f64": (c_int, [_vp, c_int64, c_int64, _vp, c_int64, _vp]),
    "rla_sptrsv_plan_host": (c_int, [c_int64, _vp, _vp, _vp, c_int, c_int, c_int, c_int, _vp, _vp, _vp, _vp, _vp, _vp,
                                     _vp, _vp, _vp, _vp, POINTER(c_int64), _vp, _vp, _vp, _vp, POINTER(c_int64),
                                     POINTER(ctypes.c_int32)]),
    "rla_sptrsv_transpose_in_f64": (c_int, [_vp, c_int64, c_int64, c_int64, _vp, _vp, c_int64, _vp]),
    "rla_sptrsv_transpose_out_f64": (c_int, [_vp, c_int64, c_int64, c_int64, _vp, _vp, c_int64, _vp]),
    "rla_sptrsv_group_inverses_host": (c_int, [c_int64, _vp, _vp, _vp, _vp, _vp, c_int64, _vp, _vp, _vp, _vp, _vp]),
    "rla_sptrsv_permute_rows_f64": (c_int, [_vp, _vp, _vp, c_int64, c_int64, _vp]),
    "rla_sptrsv_solve_f64": (c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, c_int64, _vp, c_int64,
                                     c_int64, _vp]),
    "rla_peer_buffer_create": (c_int, [c_size_t, POINTER(c_void_p), _vp]),
    "rla_peer_buffer_open": (c_int, [_vp, POINTER(c_void_p)]),
    "rla_peer_buffer_close": (c_int, [_vp]),
    "rla_peer_buffer_destroy": (c_int, [_vp]),
    "rla_peer_allreduce_f64": (c_int, [_vp, _vp, c_int, c_int, c_uint64, c_int64, c_int64, c_int64, _vp, _vp, c_int64,
                                       _vp, c_double, _vp]),
}

EXPORTED_SYMBOLS = tuple(_SIGS)


def lib():
    """Load librla_b200.so once; raise if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            # a fresh checkout has no binary: compile the CUDA sources once (needs nvcc);
            # there is no CPU fallback, so without the library every call fails
            try:
                from . import _build
                _build.build_library()
            except Exception as exc:
                raise RlaError(
                    f"{LIB_PATH} is missing and could not be built ({exc}); build it with "
                    "`python -m rla4mor_b200._build` (there is no CPU fallback for the sketching kernels)") from exc
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(status, what=""):
    if status != 0:
        msg = lib().rla_last_error()
        raise RlaError(f"{what} failed with status {status}: {msg.decode() if msg else ''}")


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise RlaError("rla4mor_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch


def stream_ptr():
    import torch
    return c_void_p(torch.cuda.current_stream().cuda_stream)
